/* bnbp.h — C ABI of libbnbp: batched loopy belief propagation (Pearl pi/lambda) on B200.
 *
 * This is the only boundary between host code (the drop-in C++ headers under
 * include/bayesian/, the Python host in bayesiannetwork_b200/, or any FFI) and the
 * CUDA backend.  POD structs, plain pointers and sizes only; no STL, no torch types.
 *
 * Each entry point names the reference interface it replaces.  File:line citations are
 * relative to the reference tree (godai0519/BayesianNetwork):
 *
 *   bnbp_create        <- belief_propagation::belief_propagation(graph_t const&)
 *                         bayesian/inference/belief_propagation.hpp:16-19 (+ the topology
 *                         queries graph.hpp:362-433 and CPT lookups graph.hpp:117-147 that
 *                         the reference repeats on every sweep; here they run once)
 *   bnbp_run_batch     <- belief_propagation::operator()(precondition, epsilon)
 *                         belief_propagation.hpp:31-159, for n_cases evidence sets at once
 *   bnbp_run_batch_device  same, evidence / marginals already resident in device memory
 *   bnbp_create_multi / bnbp_comm_* / bnbp_get_summary  (new: SURVEY 8e, cases sharded over the GPUs of a box;
 *                         the reference runs one evidence set on one core)
 *   bnbp_host_alloc/free  (new: page-locked result buffers for bnbp_run_batch)
 *   bnbp_check_errors  (evidence validation of the asynchronous device-path call; no reference counterpart)
 *   bnbp_run_batch_log_evidence / bnbp_run_batch_device_log_evidence  (new: per-case Bethe log-evidence)
 *   bnbp_run_batch_expected_counts / bnbp_run_batch_device_expected_counts  (new: the E-step of EM)
 *   bnbp_destroy       <- belief_propagation::~belief_propagation()   :21
 *   bnbp_last_error    <- (the reference has no error channel; UB / NaN / endless loop)
 *   bnbp_refresh_cpt   <- the reference reads vertex_t::cpt at call time (graph.hpp:157-161), so
 *                         CPT edits between calls are visible; here they need this call
 *   bnbp_precompile / bnbp_spec_source  (new: the network compiler, see BNBP_SPEC_* below)
 *   bnbp_lw_run_batch  <- likelihood_weighting::operator()  bayesian/inference/likelihood_weighting.hpp:28-59
 *   bnbp_estimate_cpt  <- sampler::make_cpt                  bayesian/sampler.hpp:81-163
 *   bnbp_netfile_*     <- serializer::bif::parse (serializer/bif.hpp:41-132) and serializer::dsc::parse
 *                         (serializer/dsc.hpp:33-232): network files -> bnbp_flat_network
 *
 * Semantics reproduced exactly (belief_propagation.hpp:75-148): synchronous (Jacobi)
 * schedule, no damping unless asked, evidence vector written into both pi and lambda of the
 * node and never updated, delta = max(DBL_MIN, max |new-old| over all message entries) with
 * NaN ignored, stop when delta < epsilon (strict), belief = normalize(pi .* lambda).
 */
#ifndef BNBP_H
#define BNBP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNBP_VERSION 2

/* status codes */
enum {
    BNBP_OK = 0,
    BNBP_ERR_INVALID = 1,   /* bad argument / malformed network or evidence */
    BNBP_ERR_CUDA = 2,      /* CUDA runtime error (message in bnbp_last_error) */
    BNBP_ERR_NO_DEVICE = 3, /* no usable sm_100 device: there is NO CPU fallback */
    BNBP_ERR_NOMEM = 4
};

enum { BNBP_FP64 = 0, BNBP_FP32 = 1 };

/* Sweep-kernel family.  The reference walks hash maps on every sweep; libbnbp has two GPU kernels:
 * a generic one that interprets the flat network (any network), and one COMPILED FOR THE NETWORK
 * at run time (NVRTC, sm_100a; cubins cached on disk) in which cardinalities, slot offsets and the
 * CPT arena are compile-time constants.  AUTO specialises eligible networks (small enough to
 * unroll, CPT arena <= 60 KB of constant bank) once a batch has >= 4096 cases.  Both are GPU
 * paths with identical semantics; neither is a CPU fallback.
 *
 * Independently of the family, nodes with LARGE CPTs (>= bnbp_options.dense_min_cpt entries, e.g. the
 * 32^4-entry tables of a card-32 node with 3 parents) take the dense contraction path: their CPT
 * is multiplied with the whole batch as two matrix products per sweep (csrc/bnbp_dense.cuh) and the
 * sweep kernel finishes from the per-case result tables.  Networks with such nodes are not
 * specialised. */
enum { BNBP_SPEC_AUTO = 0, BNBP_SPEC_ALWAYS = 1, BNBP_SPEC_NEVER = 2 };

/* Flat (CSR) description of a discrete Bayesian network.
 *   node i      = i-th entry of graph_t::vertex_list()                (graph.hpp:214)
 *   card[i]     = vertex_t::selectable_num                            (graph.hpp:159)
 *   parents of i = graph_t::in_vertexes(vertex i), ascending index    (graph.hpp:389-413)
 *   cpt         = row-major per node: cpt[cpt_off[i] + q*card[i] + x] = P(X_i = x | config q)
 *                 q enumerates parent configurations in mixed radix with the FIRST parent
 *                 slowest, the order of all_combination_pattern (belief_propagation.hpp:269-295)
 * Children lists (graph_t::out_vertexes, graph.hpp:378-386) are derived by the library. */
typedef struct bnbp_flat_network {
    int32_t        n_nodes;
    const int32_t* card;        /* [n_nodes]                        */
    const int32_t* parent_off;  /* [n_nodes+1]                      */
    const int32_t* parents;     /* [parent_off[n_nodes]]            */
    const int64_t* cpt_off;     /* [n_nodes+1]                      */
    const double*  cpt;         /* [cpt_off[n_nodes]]               */
} bnbp_flat_network;

typedef struct bnbp_options {
    int32_t precision;          /* BNBP_FP64 (default, the reference's arithmetic) or BNBP_FP32 */
    int32_t device;             /* CUDA device ordinal; -1 = current device                     */
    int64_t max_resident_cases; /* cases kept in HBM at once (0 = pick from free memory)         */
    int32_t specialize;         /* BNBP_SPEC_AUTO (default) / ALWAYS (error if impossible) / NEVER */
    int32_t dense_min_cpt;      /* nodes whose CPT has >= this many entries meet the batch as matrix
                                   products (dense contraction path); 0 = default 256, < 0 = never  */
    int32_t dense_tensor;       /* fp32 handles: large dense products run on the tensor cores (tcgen05, fp32
                                   accumulators in TMEM, every operand split hi + lo into two tf32 values:
                                   csrc/bnbp_dense_tc.cuh).  0 = default (products with K >= 32, N >= 128),
                                   1 = every dense product, -1 = never (CUDA-core FMA products)             */
    int32_t onchip;             /* the ON-CHIP kernel (csrc/bnbp_onchip.cuh): a specialised network whose per-case state fits
                                   shared memory runs init, every sweep, the stopping rule and the beliefs of a case in ONE
                                   launch, 32 cases per CTA, the node walk split over 4 warps; HBM sees evidence in and
                                   marginals out only.  0 = default (eligible networks, specialize == AUTO, hard evidence,
                                   fixed sweep count without damping, batches >= 4096 cases), 1 = always (error if
                                   impossible; also epsilon mode and damping), -1 = never (streaming kernels)            */
    int32_t reserved[4];
} bnbp_options;

/* Evidence for a batch, CSR over cases.  Entry e of case c (ev_off[c] <= e < ev_off[c+1])
 * observes node ev_node[e]:
 *   hard evidence (ev_values == NULL): one-hot row with state ev_state[e]
 *                 (the condition_t form, graph.hpp:18 / example main.cpp:50-55);
 *   soft evidence (ev_values != NULL): the row ev_values[ev_val_off[e] .. +card[node])
 *                 (the unordered_map<vertex_type, matrix_type> form, belief_propagation.hpp:31,69-73).
 * A node listed twice in one case: the last entry wins. */
typedef struct bnbp_evidence {
    int64_t        n_cases;
    const int64_t* ev_off;      /* [n_cases+1]            */
    const int32_t* ev_node;     /* [ev_off[n_cases]]      */
    const int32_t* ev_state;    /* [nnz] or NULL          */
    const int64_t* ev_val_off;  /* [nnz+1] or NULL        */
    const double*  ev_values;   /* [ev_val_off[nnz]] or NULL */
} bnbp_evidence;

enum { BNBP_OUT_DEFAULT = 0, BNBP_OUT_FP64 = 1, BNBP_OUT_FP32 = 2 };
enum { BNBP_SUM_PRODUCT = 0, BNBP_MAX_PRODUCT = 1 };

typedef struct bnbp_run_params {
    double  epsilon;        /* stop a case when its delta < epsilon (reference default 0.001).
                               epsilon <= 0 disables the test (fixed sweep count, no old-message reads) */
    int32_t max_sweeps;     /* cap per case; <= 0 means 1<<30 (the reference has no cap)                */
    double  damping;        /* 0 = reference behaviour; msg = (1-d)*new + d*old otherwise (extension)   */
    int32_t check_interval; /* test convergence every n-th sweep; 1 = reference semantics                */
    /* ---- what leaves the device (all 0 / NULL = the reference's "every node, in double") ------------------
     * The marginals are 8 * sum r_X bytes per case; on a host link of ~50 GB/s that copy, not the kernels,
     * bounds bnbp_run_batch (alarm37: 840 B per case, 881 MB per 1M cases). */
    int32_t out_precision;  /* bnbp_run_batch: BNBP_OUT_DEFAULT / BNBP_OUT_FP64 = out_marginals is double*;
                               BNBP_OUT_FP32 (fp32 handles only) = out_marginals is float*: half the copy.
                               bnbp_run_batch_device always writes the handle's precision.               */
    int32_t gather;         /* bnbp_run_batch_device on a handle with a communicator (bnbp_comm_init): out_marginals
                               is the gathered buffer [world][n_cases][row]; the rank's kernels write straight into
                               its slot and the slots travel over NCCL chunk by chunk behind the kernels of the next
                               chunk.  Every rank must pass the same n_cases.                           */
    int32_t n_query;        /* > 0: only the marginals of query_nodes[0..n_query) are written, in that order: a row
                               is sum card[query_nodes[i]] values instead of sum r_X (0 = every node)   */
    const int32_t* query_nodes;   /* host array, read during the call                                   */
    int32_t semiring;       /* BNBP_SUM_PRODUCT (default: the reference, belief_propagation.hpp:174-266) or
                               BNBP_MAX_PRODUCT (extension, SURVEY 8 f4): every sum over parent configurations and
                               child states becomes a maximum, beliefs are max-marginals (exact on polytrees); same
                               schedule, normalisation and stopping rule.  Runs on the generic sweep kernel.        */
    int32_t reserved[3];
} bnbp_run_params;

/* Convergence summary of a sharded run (SURVEY 8e: the only collective besides the gather). */
typedef struct bnbp_summary {
    int64_t n_cases;        /* over all ranks / devices */
    int64_t case_sweeps;    /* sum of sweeps executed   */
    int64_t not_converged;  /* cases whose last tested delta was not < epsilon (all of them when epsilon <= 0) */
    int64_t max_sweeps;     /* most sweeps any case ran */
} bnbp_summary;

typedef struct bnbp_stats {
    int64_t state_values_per_case;   /* S = 2*sum r_X + 2*sum_{U->X} r_U                        */
    int64_t msg_values_per_case;     /* 2*sum_{U->X} r_U                                        */
    int64_t belief_values_per_case;  /* sum r_X                                                  */
    int64_t cpt_values;              /* reference-layout CPT entries                             */
    int64_t bytes_per_value;         /* 8 or 4                                                   */
    int64_t last_case_sweeps;        /* sum over cases of sweeps executed by the last run       */
    int64_t last_sweep_launches;     /* sweeps enqueued by the last run (a fixed-count run of a specialised
                                        network puts its middle sweeps into ONE looping launch)  */
    int64_t last_kernel_launches;    /* all kernel launches of the last run                     */
    double  last_sweep_ms;           /* device time of the sweep launches (CUDA events)         */
    double  last_total_ms;           /* device time init..beliefs of the last run               */
    int64_t resident_cases;          /* cases per HBM-resident chunk                            */
    int64_t last_specialised;        /* 1 if the last run used the network-specialised sweep kernel */
    int64_t cases_per_tile;          /* 128 x cases per thread of the kernel family of the last run */
    double  spec_compile_ms;         /* NVRTC time spent by this handle (0 when served by the cache) */
    int64_t dense_nodes;             /* nodes on the dense contraction path                       */
    int64_t dense_values_per_case;   /* per-case slots of their result tables T1/T2 (HBM scratch) */
    double  dense_flops_per_case_sweep; /* 4 * sum |CPT| over the dense nodes                    */
    int64_t last_dense_launches;     /* dense-contraction launches of the last run               */
    double  last_dense_ms;           /* device time of (up to the first 512 sweeps') dense launches */
    int64_t dense_tensor_jobs;       /* dense products (two per node) that run on the tensor cores */
    double  dense_tensor_flops_per_case_sweep; /* their algorithmic flops, 2*K*N each (x3 issued: hi/lo split) */
    int64_t last_dense_tensor_launches;
    int64_t last_fused;              /* 1 if the last run formed the time-0 state inside the first sweep and the
                                        marginals inside the last one (no separate init / belief kernels) */
    int64_t last_compactions;        /* eps mode: how often the still-active cases were gathered into dense tiles */
    double  last_host_ms;            /* wall clock of the last bnbp_run_batch call, entry to return (-1: none yet)  */
    double  last_host_wait_ms;       /* of which: the final waits for the streams                                   */
    int64_t last_onchip;             /* 1 if the last run used the on-chip kernel (state in shared memory for all sweeps) */
    int64_t onchip_roles;            /* warps that share the node walk of a 32-case group (0: network not eligible)   */
    int64_t onchip_smem_bytes;       /* shared memory of one group: (PL + 2M) * 32 values + reduction scratch          */
    int64_t onchip_blocks_per_sm;    /* resident groups per SM of the loaded on-chip kernel (0: none loaded yet)        */
    double  onchip_role_imbalance;   /* busiest role / mean role cost of the node partition (1 = perfectly balanced)    */
    int64_t spec_class_count;        /* node shape classes of a CLASS-LOOPED specialised walk (networks too large to unroll
                                        node by node: one unrolled body per class, looped over its nodes); 0 otherwise   */
} bnbp_stats;

typedef struct bnbp_handle bnbp_handle;

int  bnbp_device_count(void);
const char* bnbp_last_error(void);           /* thread-local, never NULL */

/* Lays the network out on the device (replaces belief_propagation::belief_propagation(graph_t const&),
 * belief_propagation.hpp:16-19).  Validates what the reference leaves undefined (parent ids, ascending parent lists, cycles,
 * CPT sizes: BNBP_ERR_INVALID with the reason in bnbp_last_error()).  Limits the reference does not have: at most 128 states
 * per node and 8 parents per node.  The first run on a network compiles its kernels (NVRTC, cached on disk; see
 * bnbp_precompile for doing that ahead of time, without a GPU). */
int  bnbp_create(const bnbp_flat_network* net, const bnbp_options* opt, bnbp_handle** out);
void bnbp_destroy(bnbp_handle* h);

/* Host buffers in, host buffers out (copies are part of the call).
 *   out_marginals [n_cases][belief_values_per_case] doubles, node i at offset sum_{j<i} card[j]
 *   out_sweeps    [n_cases] sweeps executed per case (may be NULL)
 *   out_converged [n_cases] 1 if the case's last tested delta < epsilon (may be NULL)   */
int  bnbp_run_batch(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm,
                    void* out_marginals, int32_t* out_sweeps, uint8_t* out_converged);

/* Page-locked host memory for the buffers of bnbp_run_batch: a pageable destination makes every device-to-host
 * copy go through a driver bounce buffer (~7 GB/s instead of the link rate) and blocks the calling thread.
 * The drop-in headers allocate their flat results here.  The memory is not zero-filled. */
void* bnbp_host_alloc(size_t bytes);
void  bnbp_host_free(void* p);

/* ---- several GPUs of one box (SURVEY 8e) -----------------------------------------------------------------
 * Evidence cases are independent (belief_propagation.hpp keeps all state per call, :162-172), so a batch shards
 * by contiguous case ranges with the network replicated; NCCL carries the two exchanges the path has: the
 * convergence summary (all-reduce) and, on request, the gather of the marginals.  libbnbp owns the communicators.
 *
 * One process, several devices: bnbp_create_multi returns a GROUP handle (one member handle, host thread and
 * stream set per device, an NCCL communicator over them).  bnbp_run_batch on it cuts the caller's CSR evidence
 * into contiguous ranges (range g = [g*n/G, (g+1)*n/G) up to one case), every device copies its marginals
 * straight into its rows of the caller's buffers, and the summary is all-reduced in the library
 * (bnbp_get_summary).  devices == NULL: ordinals 0..n_devices-1; n_devices <= 0: every visible device.
 * Results are bit-identical to a one-device handle: a case's arithmetic does not depend on where it runs.
 *
 * One process per device (torchrun, MPI): every rank creates an ordinary handle, rank 0 draws an id with
 * bnbp_comm_unique_id and ships it to the others by whatever means the launcher has, all call bnbp_comm_init;
 * bnbp_run_batch_device with bnbp_run_params.gather then leaves ALL marginals on every rank, and
 * bnbp_comm_summary all-reduces the per-case counts of the last run.
 * Allocation and collectives: an NCCL collective is a kernel that spins until every rank has joined, and with peer
 * access on, a cudaMalloc on one rank waits for its peers' devices.  A handle allocates on the FIRST call of a given
 * shape (state arena, staging); make that call without `gather` (or give every rank the same first call and no other
 * allocating work around it), and synchronise the ranks on the host, not with an NCCL barrier, around phases that
 * allocate (new handles, pinned buffers).  bench.py does both. */
int  bnbp_create_multi(const bnbp_flat_network* net, const bnbp_options* opt, const int32_t* devices, int32_t n_devices,
                       bnbp_handle** out);
int  bnbp_get_summary(const bnbp_handle* h, bnbp_summary* out);      /* of the last bnbp_run_batch of a group handle */
#define BNBP_COMM_ID_BYTES 128
int  bnbp_comm_unique_id(void* id_out);                              /* BNBP_COMM_ID_BYTES bytes */
int  bnbp_comm_init(bnbp_handle* h, int32_t world, int32_t rank, const void* id);
/* d_sweeps / d_converged: the DEVICE arrays the last bnbp_run_batch_device of this rank filled (n_cases entries).
 * Synchronises `stream`; *out (host) holds the totals over all ranks. */
int  bnbp_comm_summary(bnbp_handle* h, const int32_t* d_sweeps, const uint8_t* d_converged, int64_t n_cases,
                       bnbp_summary* out, void* stream);

/* Same, but every pointer inside *ev and every out_* pointer is a DEVICE pointer on the
 * handle's device; out_marginals has the handle's precision (double or float).  The work is
 * enqueued on `stream` (a cudaStream_t passed as void*; NULL = the handle's own stream) and the
 * call returns without synchronising unless epsilon > 0 forces host-side termination polls. */
int  bnbp_run_batch_device(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm,
                           void* out_marginals, int32_t* out_sweeps, uint8_t* out_converged,
                           void* stream);

/* The device-path call above does not wait for the device, so malformed evidence it meets there (node id or
 * state out of range, soft row of the wrong length: such entries are skipped) cannot fail the call itself
 * unless epsilon > 0 made it synchronise.  After synchronising `stream`, this returns BNBP_ERR_INVALID with
 * the reason if the last device-path run skipped evidence, BNBP_OK otherwise.  Every run clears the flag
 * when it starts, so an unchecked error never fails a later call.  (The reference has no error channel:
 * evidence on a vertex outside the graph is silently ignored, belief_propagation.hpp:69-73.) */
int  bnbp_check_errors(bnbp_handle* h, void* stream);

/* Log-evidence (no reference counterpart): bnbp_run_batch / bnbp_run_batch_device that also return, per case,
 * the Bethe estimate log Z_B of ln P(e) from the state the run ends with -- exactly ln P(e) on a polytree run to
 * convergence, BP's standard approximation of it on a loopy network.  With the rows lambda_X of the final state and
 * the pi-messages pm_j the case's last sweep read (the committed messages of the sweep before, damped if damping is
 * on), per node X with parents U_j, m_X children and CPT P(x|u):
 *   Z_X = sum_{x,u} P(x|u) lambda_X(x) prod_j pm_j(u_j),  b_X = that product / Z_X,
 *   log Z_B = sum_X [ ln Z_X - sum_x b_X(x) ln lambda_X(x) - sum_j sum_u b_X(u_j=u) ln pm_j(u) + m_X sum_x b_X(x) ln b_X(x) ]
 * A term of weight 0 contributes 0; a NaN Z_X makes the case NaN, else a zero Z_X makes it -inf (evidence impossible
 * given the messages).  fp64 sums in both precisions.  out_log_evidence [n_cases] doubles (host / device memory as
 * the call's other outputs).  out_marginals may be NULL: then no marginals are written or copied.  Group handles
 * slice it like out_sweeps.  The run takes the streaming kernels (not the on-chip kernel, the fused first / last
 * sweeps or the split convergence test: AUTO steps around them, onchip = ALWAYS is refused).  BNBP_ERR_INVALID with
 * the reason for soft evidence, BNBP_MAX_PRODUCT, handles with dense-path nodes (create with dense_min_cpt = -1)
 * and gather; the handle stays usable. */
int  bnbp_run_batch_log_evidence(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm,
                                 void* out_marginals, int32_t* out_sweeps, uint8_t* out_converged,
                                 double* out_log_evidence);
int  bnbp_run_batch_device_log_evidence(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm,
                                        void* out_marginals, int32_t* out_sweeps, uint8_t* out_converged,
                                        double* out_log_evidence, void* stream);

/* Expected family counts (no reference counterpart): the E-step of EM parameter learning from incomplete evidence.
 * The run of bnbp_run_batch_log_evidence, whose scoring launches also add, for every case c of weight w_c (1 when
 * case_weights is NULL) with a finite log-evidence, the family posterior b_X of the log-evidence above into counts:
 *   counts[cpt_off[X] + q r_X + x] += w_c P(x|u_q) lambda_X(x) prod_j pm_j(u_qj) / Z_X      for every X, q, x
 * with lambda_X and pm_j of the case's last executed sweep as above.  counts has the layout of the CPT arena
 * (cpt_off[n_nodes] doubles), so sampler::make_cpt's normalisation of each row is the M-step.  A case whose
 * log-evidence is NaN or -inf (some Z_X is NaN or 0: the evidence is impossible under the CPT) adds nothing; it still
 * gets its log-evidence, sweeps and flag.  Summed over x and u the counts of a node are sum_c w_c b_X(x), the node
 * marginal, at any sweep count; on a polytree run to its fixed point they are sum_c w_c P(x, u | e_c).
 * The call ADDS INTO counts: zero it once and stream a data set larger than one call through several calls before
 * an M-step.  Sums are fp64 in both precisions, but atomics leave their order open: counts agree between runs to
 * rounding, not bit for bit.  case_weights [n_cases] must be finite and >= 0 (the host call checks this and refuses
 * otherwise; the device call reads them as given).  case_weights, out_marginals and out_log_evidence may be NULL.
 * Host call: host buffers, the handle's own zeroed device count arena is added into counts when the call returns;
 * group handles add the members' counts in member order.  Device call: device pointers, counts is added into on
 * the device, in stream order.  Kernels and refusals are log-evidence's, plus BNBP_ERR_INVALID for a NULL counts;
 * the handle stays usable after a refusal. */
int  bnbp_run_batch_expected_counts(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm,
                                    const double* case_weights, double* counts,
                                    void* out_marginals, int32_t* out_sweeps, uint8_t* out_converged,
                                    double* out_log_evidence);
int  bnbp_run_batch_device_expected_counts(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm,
                                           const double* case_weights, double* counts,
                                           void* out_marginals, int32_t* out_sweeps, uint8_t* out_converged,
                                           double* out_log_evidence, void* stream);

/* Likelihood weighting for a batch of HARD-evidence cases (SURVEY 8 f2): the independent statistical
 * check of BP marginals on loopy networks.  Replaces likelihood_weighting::operator()(evidence_list,
 * sample_num) (bayesian/inference/likelihood_weighting.hpp:28-59, weighted_sample :122-173) for
 * n_cases evidence sets at once.  The reference seeds a mt19937 from std::random_device; here the
 * uniform variate of (case, sample, node) is a pure function of `seed` (splitmix64), so a run is
 * reproducible and independent of how cases are spread over launches or GPUs.
 *   out_marginals  [n_cases][belief_values_per_case], same layout as bnbp_run_batch
 *   out_weight_sum [n_cases] total sample weight (estimate of n_samples * P(evidence)); may be NULL */
int  bnbp_lw_run_batch(bnbp_handle* h, const bnbp_evidence* ev, int64_t n_samples, uint64_t seed,
                       double* out_marginals, double* out_weight_sum);

/* CPT estimation from a table of samples on the device (SURVEY 8 f3).  Replaces sampler::make_cpt
 * (bayesian/sampler.hpp:81-163): samples[row][node] is the state of every node in one distinct sample,
 * multiplicity[row] how often it occurred (NULL = once; the first column of the reference's sample
 * file, sampler.hpp:53-76).  out_cpt gets the CPT arena in the layout of bnbp_flat_network.cpt
 * (net->cpt itself is not read): count / row total, uniform 1/card for configurations never seen. */
int  bnbp_estimate_cpt(const bnbp_flat_network* net, const int32_t* samples, const int64_t* multiplicity,
                       int64_t n_rows, int32_t device, double* out_cpt);

int  bnbp_get_stats(const bnbp_handle* h, bnbp_stats* out);

/* Re-upload CPT values after the host network changed them (topology must be unchanged). */
int  bnbp_refresh_cpt(bnbp_handle* h, const double* cpt, int64_t n_values);

/* Network compiler without a GPU (build machines, tests): generate the specialised sweep kernel of
 * `net` for opt->precision and compile it into the cubin cache ($BNBP_CACHE_DIR, default
 * <dir of libbnbp.so>/jitcache), so that bnbp_create/run on the GPU box finds it there.
 * variant_mask: bit 0 plain (fixed sweeps), bit 1 freeze, bit 2 freeze+check (epsilon mode, damping),
 *               bit 3 plain-first (time-0 messages are all 1: not loaded), bit 4 plain-last (messages
 *               of the last sweep are never read: not stored), bits 5-7 the fused first / last sweeps;
 *               bits 8-11 the on-chip kernel: 8 fixed sweeps, 9 the same with double marginals from a
 *               float kernel, 10 / 11 the epsilon / damping flavour of the two.
 * Returns BNBP_ERR_INVALID with the reason if the network is not eligible. */
int  bnbp_precompile(const bnbp_flat_network* net, const bnbp_options* opt, int32_t variant_mask);

/* The generated CUDA source of one variant (0..7 streaming, 8 / 9 on-chip plain / check), for inspection and tests.  Writes at most
 * cap bytes including the terminating NUL and returns the full length via *needed. */
int  bnbp_spec_source(const bnbp_flat_network* net, const bnbp_options* opt, int32_t variant,
                      char* buf, int64_t cap, int64_t* needed);

/* ---- network files (host only, no GPU needed) --------------------------------------------------------
 * BIF / DSC text -> the flat network above.  Replaces the reference loaders
 * bn::serializer::bif::parse (bayesian/serializer/bif.hpp:41-132, grammar :138-263, Boost.Spirit) and
 * bn::serializer::dsc::parse (bayesian/serializer/dsc.hpp:33-232); the parsers are the drop-in headers
 * include/bayesian/serializer/{bif,dsc}.hpp, this is their FFI face.  Node i of the flat network is
 * the i-th `variable` / `node` section of the file (the reference's vertex_list() order); parents are
 * listed in ascending node index and CPT rows in the layout of bnbp_flat_network whatever order the
 * file used. */
enum { BNBP_FORMAT_AUTO = 0, BNBP_FORMAT_BIF = 1, BNBP_FORMAT_DSC = 2 };

typedef struct bnbp_network_file bnbp_network_file;

int  bnbp_netfile_parse(const char* text, int64_t len, int32_t format, bnbp_network_file** out);
int  bnbp_netfile_load(const char* path, int32_t format, bnbp_network_file** out);  /* AUTO: by extension, then content */
/* the arrays stay owned by the file object and live until bnbp_netfile_free */
const bnbp_flat_network* bnbp_netfile_network(const bnbp_network_file* nf);
const char* bnbp_netfile_name(const bnbp_network_file* nf);
const char* bnbp_netfile_node_name(const bnbp_network_file* nf, int32_t node);                  /* NULL if out of range */
const char* bnbp_netfile_state_name(const bnbp_network_file* nf, int32_t node, int32_t state);  /* NULL if out of range */
void bnbp_netfile_free(bnbp_network_file* nf);

#ifdef __cplusplus
}
#endif
#endif /* BNBP_H */
