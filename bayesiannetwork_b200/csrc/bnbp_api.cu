// bnbp_api.cu — C ABI of libbnbp (include/bnbp.h): network flattening into the device arena,
// batch orchestration, error channel.  The reference keeps the network as hash maps of hash maps
// and re-queries topology on every sweep (graph.hpp:362-481, :117-147); here all of that happens
// ONCE in bnbp_create and the sweeps touch only flat device arrays.
#include "../../include/bnbp.h"
#include "bnbp_kernels.cuh"
#include "bnbp_lw.cuh"
#include "bnbp_variants.h"
#include "bnbp_jit.h"
#include "bnbp_dense.h"
#include "bnbp_dense_tc.cuh"

#include <nccl.h>
#include <nvtx3/nvToolsExt.h>      // header-only; ranges cost nothing unless a profiler is attached

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <thread>
#include <vector>

using namespace bnbp;

#include <dlfcn.h>
#include <mutex>

// NCCL is bound at FIRST USE of a communicator, not at link time.  libbnbp is loaded into processes that bring their
// own NCCL (PyTorch bundles a newer libnccl.so.2 than the system's): a link-time dependency makes the loader map the
// SYSTEM library first, and a later `import torch` then fails on the symbols only the newer one has (r02b: undefined
// symbol ncclDevCommCreate).  dlopen("libnccl.so.2") returns the copy the process already holds when there is one.
namespace bnbp_nccl {
struct Api {
    void* so = nullptr;
    std::string load_error;
    decltype(&::ncclAllReduce) AllReduce = nullptr;
    decltype(&::ncclBroadcast) Broadcast = nullptr;
    decltype(&::ncclCommDestroy) CommDestroy = nullptr;
    decltype(&::ncclCommAbort) CommAbort = nullptr;
    decltype(&::ncclCommInitAll) CommInitAll = nullptr;
    decltype(&::ncclCommInitRank) CommInitRank = nullptr;
    decltype(&::ncclGetErrorString) GetErrorString = nullptr;
    decltype(&::ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&::ncclGroupStart) GroupStart = nullptr;
    decltype(&::ncclGroupEnd) GroupEnd = nullptr;
};
static Api& api()
{
    static Api a;
    static std::once_flag once;
    std::call_once(once, [] {
        for (const char* nm : {"libnccl.so.2", "libnccl.so"}) {
            a.so = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
            if (a.so) break;
        }
        if (!a.so) { a.load_error = std::string("libnccl.so.2 not found: ") + dlerror(); return; }
#define BNBP_NCCL_SYM(field, name)                                                  \
    a.field = reinterpret_cast<decltype(a.field)>(dlsym(a.so, name));               \
    if (!a.field) { a.load_error = std::string("libnccl lacks ") + name; return; }
        BNBP_NCCL_SYM(AllReduce, "ncclAllReduce")
        BNBP_NCCL_SYM(Broadcast, "ncclBroadcast")
        BNBP_NCCL_SYM(CommDestroy, "ncclCommDestroy")
        BNBP_NCCL_SYM(CommAbort, "ncclCommAbort")
        BNBP_NCCL_SYM(CommInitAll, "ncclCommInitAll")
        BNBP_NCCL_SYM(CommInitRank, "ncclCommInitRank")
        BNBP_NCCL_SYM(GetErrorString, "ncclGetErrorString")
        BNBP_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
        BNBP_NCCL_SYM(GroupStart, "ncclGroupStart")
        BNBP_NCCL_SYM(GroupEnd, "ncclGroupEnd")
#undef BNBP_NCCL_SYM
    });
    return a;
}
} // namespace bnbp_nccl

namespace {

thread_local std::string g_err = "";

int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}

}  // namespace

// the error channel for the other translation units of the library (bnbp_netfile.cpp)
namespace bnbp {
int set_error(int code, const std::string& msg) { return fail(code, msg); }
}

namespace {

#define CU_TRY(expr)                                                                      \
    do {                                                                                  \
        cudaError_t e__ = (expr);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            return fail(e__ == cudaErrorMemoryAllocation ? BNBP_ERR_NOMEM : BNBP_ERR_CUDA, \
                        std::string(#expr) + ": " + cudaGetErrorString(e__));             \
        }                                                                                 \
    } while (0)

// Wait for a stream; BNBP_SPIN_SYNC=1 polls instead of sleeping on the driver's interrupt.  (Tried as the
// default against the 30-120 ms host-side stalls that hit bursts of bnbp_run_batch calls on the boxes of this
// pool at a constant 27.0 ms of device time -- r01y/r01z: neither polling nor switching Python's garbage
// collector off removes them, so the default stays the sleeping wait, which leaves the core to others.)
cudaError_t wait_stream(cudaStream_t s)
{
    static const bool blocking = getenv("BNBP_SPIN_SYNC") == nullptr;
    if (!blocking) {
        const auto t0 = std::chrono::steady_clock::now();
        for (unsigned spin = 0;; ++spin) {
            const cudaError_t e = cudaStreamQuery(s);
            if (e != cudaErrorNotReady) return e;
            if ((spin & 1023u) == 1023u &&
                std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 2.0) break;
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
        }
    }
    return cudaStreamSynchronize(s);
}

// NVTX range over a scope: the phases of a call show up by name on an nsys / ncu timeline (SURVEY section 5)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};

constexpr int BLOCK_THREADS = 128;   // sweep-kernel block; a tile holds BLOCK_THREADS * vec cases

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need)
    {
        if (need <= bytes) return BNBP_OK;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        CU_TRY(cudaMalloc(&p, need));
        bytes = need;
        return BNBP_OK;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};

} // namespace

struct bnbp_handle {
    int device = 0;
    int precision = BNBP_FP64;
    size_t tsize = 8;
    int N = 0, E = 0;
    int PL = 0, M = 0, W = 0, V = 0;
    int rmax = 2;              // template bound actually used (2,4,8,16,32,64)
    int knet = 2;              // in-degree bound actually used (2,4,8)
    int vec = 1;
    int tb = 128;              // cases per tile = BLOCK_THREADS * vec
    int scratch_vals = 0;      // per-thread scratch values (x VEC)
    int64_t cpt_values = 0;
    int64_t max_resident = 0;
    std::vector<NodeMeta> nodes;
    std::vector<double> cost_prefix;   // [N+1]
    std::vector<int32_t> card;
    std::vector<int32_t> e_card, e_lam_out, c_pi_out;   // per in-edge / out-edge tables (host copies)
    std::vector<double> cpt_host;      // reference-layout CPT values (for the specialised kernels' constant bank)
    // network-specialised sweep kernels (bnbp_jit.h); index = variant 0 plain, 1 freeze, 2 freeze+check
    int specialize = 0;                // BNBP_SPEC_AUTO / ALWAYS / NEVER
    bool spec_eligible_ = false;
    std::string spec_why;              // why the network is not specialised
    int spec_vec = 1, spec_minb = 1, spec_ahead = 1;
    bool spec_classloop = false;       // the specialised walk loops over node SHAPE classes (networks too large to unroll)
    int spec_classes_n = 0;
    bool spec_auto_ok = true;          // may AUTO compile the specialised kernels at first use? (false: NVRTC would need minutes
    bool oc_auto_ok = true;            //  for an unrolled walk of this size and no cubin is cached -- ALWAYS still compiles them)
    static constexpr int NSPEC = 8;    // variants of bnbp_spec.cuh
    SpecKernel spec[NSPEC];            // + 3 plain-first (no message loads), 4 plain-last (no message stores),
                                       //   5 first + K0, 6/7 last + K4 (marginals in T / in double)
    int spec_state[NSPEC] = {0, 0, 0, 0, 0, 0, 0, 0};   // 0 untried, 1 loaded, -1 failed
    bool fuse = false;                 // this run: K0 inside the first sweep, K4 inside the last (variants 5, 6/7)
    int last_fused = 0;
    double last_host_ms = -1.0, last_host_wait_ms = -1.0;   // wall clock of the last bnbp_run_batch call / of its final waits
    bool fuse_ok = true;               // cleared when a fused variant failed to build: the unfused launch sequence runs
    // eps mode: compaction of the still-active cases into a second arena (compact_* kernels, bnbp_kernels.cuh)
    DevBuf d_pl2, d_msg2[2], d_evbits2, d_orig[2], d_src_pos, d_tile_count;
    bool split = false;                // this run: plain sweeps + delta_retire_kernel instead of the freeze/check variants
    bool compact_ok = true;            // cleared when the second arena does not fit
    int64_t last_compactions = 0;
    DevBuf d_evst;                     // [tiles][N][tb] evidence-state bytes of the resident chunk
    bool run_spec = false;             // kernel family of the current run
    int last_specialised = 0;
    // on-chip multi-sweep kernel (bnbp_onchip.cuh): index = (check ? 2 : 0) + (marginals in double from a float kernel ? 1 : 0)
    int onchip = 0;                    // bnbp_options.onchip: 0 auto, 1 always, -1 never
    bool oc_eligible = false;
    std::string oc_why;
    int oc_roles = 4, oc_minb = 1, oc_ahead = 1;
    size_t oc_smem = 0;
    SpecKernel oc[4];
    int oc_state[4] = {0, 0, 0, 0};    // 0 untried, 1 loaded, -1 failed
    bool run_onchip = false;           // this run: the whole case (init, every sweep, beliefs) in one on-chip kernel
    int reserve_sms = 0;               // this run: SMs the on-chip grid leaves to the concurrent NCCL exchange (gather)
    int last_onchip = 0;
    double oc_imbalance = 1.0;         // busiest role / mean role cost of the node partition
    double spec_compile_ms = 0.0;
    // dense contraction path (bnbp_dense.h): nodes whose CPT has >= dense_min entries
    int64_t dense_min = 256;           // < 0: never
    bool dense_mma = true;             // fp64: DMMA (tensor pipe) instead of DFMA for the products
    int TS = 0;                        // per-case slots of the contraction scratch (T1 / T2 tables)
    int dense_nodes = 0;
    double dense_flops_per_case = 0.0; // 4 * sum |CPT| over the dense nodes, per sweep
    std::vector<DenseJob> djobs;       // sorted by factor count
    struct DenseGroup { int nf, tnt, n_y, ytab0, max_rows; };
    std::vector<DenseGroup> dgroups;   // one launch each
    std::vector<int32_t> dytab;
    std::vector<unsigned long long> ddig;
    std::vector<int64_t> dense_pt_off; // per node: offset of the transposed CPT copy in arena 1 (-1: not dense)
    int64_t cpt_t_values = 0;
    DevBuf d_djobs, d_dytab, d_ddig, d_cpt_t, d_tscr;
    // tensor-core variant of the products (bnbp_dense_tc.cuh), fp32 handles
    int dense_tc = 0;                  // bnbp_options.dense_tensor: 0 default thresholds, 1 every product, -1 never
    struct TcGroup { int n_y, ytab0, max_rows, stages; };
    std::vector<TcGroup> tcgroups;     // one launch each
    struct TcPack { int64_t src_off, sk, sn, out_off; int K, N; };
    std::vector<TcPack> tcpack;        // how each tensor-core job's B operand is cut out of the CPT arena
    int64_t tc_values = 0;             // floats of the pre-tiled hi/lo arena
    int dense_tc_jobs = 0;
    double dense_tc_flops_per_case = 0.0;
    int64_t last_dense_tc_launches = 0;
    DevBuf d_cpt_tc;
    std::vector<cudaEvent_t> ev_dense; // pairs around the dense launches of a sweep
    int ev_dense_used = 0;
    int64_t last_dense_launches = 0;
    // device network
    DevBuf d_nodes, d_e_card, d_e_lam_out, d_c_pi_out, d_cpt, d_pl_init;
    // device state for the resident chunk
    int64_t cap = 0;
    DevBuf d_pl, d_msg[2], d_evbits, d_delta, d_status, d_sweeps, d_misc;
    // staging for the host API (outputs double-buffered: D2H of chunk i overlaps the sweeps of chunk i+1)
    DevBuf s_ev_off, s_ev_node, s_ev_state, s_ev_val_off, s_ev_values, s_out[2], s_out_sweeps, s_out_conv;   // sweeps/conv: whole batch
    // likelihood weighting (bnbp_lw.cuh): parent ids, a topological order and the fp64 CPT arena, uploaded on first use
    std::vector<int32_t> par_host;
    DevBuf d_lw_order, d_lw_par, d_lw_cpt, d_lw_out, d_lw_wsum;
    bool lw_ready = false;
    void* pin_counts = nullptr;         // pinned host staging of the per-case sweep counts / converged flags
    size_t pin_counts_bytes = 0;
    DevBuf s_out_all;                   // whole-batch output staging (used when HBM has the room)
    cudaStream_t copy_stream = nullptr, h2d_stream = nullptr;
    std::vector<cudaEvent_t> ev_chunk;  // per chunk of the host-buffer call: uploaded, computed, copied
    // column groups of the tiled belief kernel, per (tile width, output element size)
    struct BeliefPlan { DevBuf groups; int n_groups = 0; int stride = 0; size_t smem = 0; bool ok = false; };
    std::map<int, BeliefPlan> belief_plans;
    int32_t* pinned_poll = nullptr;    // [4]
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_total[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> ev_sweep;  // pairs per chunk
    int ev_sweep_used = 0;
    cudaEvent_t ev_poll[2] = {nullptr, nullptr};
    // stats of the last run
    int64_t last_case_sweeps = -1, last_sweep_launches = 0, last_kernel_launches = 0;
    bool total_recorded = false;
    // what leaves the device (bnbp_run_params.n_query / query_nodes)
    std::vector<int32_t> q_nodes;      // the query the device tables describe (empty: every node)
    bool q_valid = false;
    int Vout = 0;                      // values per output row of the current run
    DevBuf d_belcol;                   // [N] column of node x's marginal in an output row, -1: not written
    DevBuf d_colmap;                   // [Vout] source column (full-width row) of output column j
    DevBuf s_full;                     // full-width rows of a chunk (streaming kernels under a query), gathered into the output
    // host link / memory rates for the chunk planner (measured once per handle, not assumed)
    double link_gbs = 0.0, hbm_gbs = 0.0;
    // multi-GPU (SURVEY 8e): the communicator this handle owns, and -- for a group handle -- its members
    ncclComm_t comm = nullptr;
    int comm_rank = 0, comm_world = 1;
    cudaStream_t comm_stream = nullptr;
    std::vector<cudaEvent_t> ev_comm;  // per gather chunk: computed, gathered
    DevBuf d_summary;                  // 4 x int64: case sweeps, not converged, max sweeps, cases
    int64_t* pin_summary = nullptr;    // pinned [4]
    std::vector<bnbp_handle*> members; // group handle: one member per device (the group itself holds no device state)
    bnbp_summary last_summary = {0, 0, 0, 0};
};

namespace {

int pick_rmax(int maxcard)
{
    for (int r : {2, 4, 8, 16, 32, 64, 128})
        if (maxcard <= r) return r;
    return -1;
}

// ---- launch dispatch ----------------------------------------------------------------------------
template <typename T>
cudaError_t launch_sweep(const bnbp_handle* h, const SweepArgs<T>& a, dim3 grid, size_t smem, bool freeze,
                         bool check, cudaStream_t st, bool maxp = false)
{
#define BNBP_X(TT, V, R, K) \
    if (h->vec == V && h->rmax == R && h->knet == K) return launch_sweep_vr<TT, V, R, K>(a, grid, smem, freeze, check, st, maxp);
    BNBP_SWEEP_VARIANTS(BNBP_X, T)
#undef BNBP_X
    return cudaErrorInvalidConfiguration;
}

template <typename T>
cudaError_t set_smem(const bnbp_handle* h, int bytes)
{
#define BNBP_X(TT, V, R, K) \
    if (h->vec == V && h->rmax == R && h->knet == K) return set_sweep_smem<TT, V, R, K>(bytes);
    BNBP_SWEEP_VARIANTS(BNBP_X, T)
#undef BNBP_X
    return cudaErrorInvalidConfiguration;
}

// node ranges of roughly equal cost for grid.y
void make_chunks(const bnbp_handle* h, int n_chunks, int32_t* off)
{
    const double total = h->cost_prefix[h->N];
    off[0] = 0;
    int x = 0;
    for (int c = 1; c < n_chunks; ++c) {
        const double target = total * c / n_chunks;
        while (x < h->N && h->cost_prefix[x + 1] <= target) ++x;
        off[c] = std::max(x, off[c - 1]);
    }
    off[n_chunks] = h->N;
}

int ensure_state(bnbp_handle* h, int64_t n_cases)
{
    const int64_t TBMAX = 512;          // every kernel family's tile width divides this
    int64_t want = (n_cases + TBMAX - 1) / TBMAX * TBMAX;
    const size_t per_case = (size_t)(h->PL + 2 * (size_t)h->M + (size_t)h->TS) * h->tsize + (size_t)h->W * 4 + 3 * h->tsize + 8;
    // fast path first: cudaMemGetInfo below is an ioctl into the kernel driver, and on a shared host it
    // waits behind whatever else queries the GPU (monitoring daemons): 20-90 ms on 1 call in ~5 (r01chk4:
    // the slow host-buffer calls spent their extra time before the first kernel was enqueued)
    if (want <= h->cap) return h->fuse ? h->d_evst.ensure((size_t)h->cap * h->N) : BNBP_OK;
    int64_t limit = h->max_resident;
    if (limit <= 0) {
        size_t free_b = 0, total_b = 0;
        CU_TRY(cudaMemGetInfo(&free_b, &total_b));
        size_t held = h->d_pl.bytes + h->d_msg[0].bytes + h->d_msg[1].bytes + h->d_evbits.bytes + h->d_tscr.bytes;
        // leave room for output staging (V doubles per case) and the caller's own buffers
        double usable = 0.80 * (double)(free_b + held);
        limit = (int64_t)(usable / (double)(per_case + (size_t)h->V * 8));
    }
    limit = std::max<int64_t>(TBMAX, limit / TBMAX * TBMAX);
    want = std::min(want, limit);
    if (want <= h->cap) return h->fuse ? h->d_evst.ensure((size_t)h->cap * h->N) : BNBP_OK;
    // grow: release first so the new allocation can reuse the space
    h->d_pl.release(); h->d_msg[0].release(); h->d_msg[1].release(); h->d_evbits.release(); h->d_tscr.release();
    h->d_delta.release(); h->d_status.release(); h->d_sweeps.release();
    h->cap = 0;
    int rc;
    if ((rc = h->d_pl.ensure((size_t)want * h->PL * h->tsize))) return rc;
    if ((rc = h->d_msg[0].ensure(std::max<size_t>(16, (size_t)want * h->M * h->tsize)))) return rc;
    if ((rc = h->d_msg[1].ensure(std::max<size_t>(16, (size_t)want * h->M * h->tsize)))) return rc;
    if ((rc = h->d_evbits.ensure((size_t)want * h->W * 4))) return rc;
    if (h->TS > 0 && (rc = h->d_tscr.ensure((size_t)want * h->TS * h->tsize))) return rc;
    if ((rc = h->d_delta.ensure((size_t)want * 3 * h->tsize))) return rc;
    if ((rc = h->d_status.ensure((size_t)want))) return rc;
    if ((rc = h->d_sweeps.ensure((size_t)want * 4))) return rc;
    h->cap = want;
    h->d_evst.release();
    return h->fuse ? h->d_evst.ensure((size_t)h->cap * h->N) : BNBP_OK;
}

SpecLayout spec_layout(const bnbp_handle* h)
{
    SpecLayout L;
    L.N = h->N; L.PL = h->PL; L.M = h->M; L.W = h->W; L.V = h->V;
    L.cpt_values = h->cpt_values;
    L.nodes = h->nodes.data();
    L.e_card = h->e_card.data();
    L.e_lam_out = h->e_lam_out.data();
    L.c_pi_out = h->c_pi_out.data();
    return L;
}

// __launch_bounds__ min blocks per SM of variant v.  The freeze+check variant (2) also holds the old value
// of every message it emits (the delta of :105-131): under the register cap of 3 (fp64) / 4 (fp32) blocks
// per SM it spills (alarm37 fp64: 364 B of spill stores per thread, 2.4 ms per sweep instead of 1.1,
// r01q); one block per SM less lets it keep everything in registers.
int spec_minb_for(const bnbp_handle* h, int v)
{
    int mb = h->spec_minb;
    if (v == 2 && !getenv("BNBP_SPEC_MINB")) {
        mb = std::max(1, mb - 1);
        if (const char* e = getenv("BNBP_SPEC_MINB_CHECK")) mb = std::min(16, std::max(1, atoi(e)));
    }
    return mb;
}

// Make variant v of the specialised kernel available (compile or fetch from the cache, load, upload
// the CPT arena into its constant bank).
int ensure_spec(bnbp_handle* h, int v)
{
    if (h->spec_state[v] == 1) return BNBP_OK;
    if (h->spec_state[v] < 0) return fail(BNBP_ERR_INVALID, "specialised kernel unavailable: " + h->spec_why);
    h->spec_state[v] = -1;
    SpecConfig cfg;
    cfg.fp32 = h->precision == BNBP_FP32;
    cfg.vec = h->spec_vec; cfg.minb = spec_minb_for(h, v); cfg.variant = v; cfg.ahead = h->spec_ahead;
    cfg.classloop = h->spec_classloop;
    if (cfg.classloop && v > 4) return fail(BNBP_ERR_INVALID, "class-looped walks exist for variants 0-4");
    const std::string src = spec_source(spec_layout(h), cfg);
    std::vector<char> cubin;
    std::string err;
    bool cached = false;
    double ms = 0;
    if (!spec_compile(src, &cubin, &cached, &ms, &err)) { h->spec_why = err; return fail(BNBP_ERR_CUDA, err); }
    h->spec_compile_ms += ms;
    if (!spec_load(cubin, &h->spec[v], &err)) {
        // a cached cubin that does not load (another driver / a damaged file) is replaced once
        if (!cached || !spec_compile(src, &cubin, &cached, &ms, &err, true) || !spec_load(cubin, &h->spec[v], &err)) {
            h->spec_why = err;
            return fail(BNBP_ERR_CUDA, err);
        }
        h->spec_compile_ms += ms;
    }
    h->spec[v].from_cache = cached;
    h->spec[v].compile_ms = ms;
    bool ok;
    if (cfg.fp32) {
        std::vector<float> tmp(h->cpt_host.begin(), h->cpt_host.end());
        ok = spec_upload_cpt(h->spec[v], tmp.data(), tmp.size() * 4, &err);
    } else {
        ok = spec_upload_cpt(h->spec[v], h->cpt_host.data(), h->cpt_host.size() * 8, &err);
    }
    if (!ok) { spec_unload(&h->spec[v]); h->spec_why = err; return fail(BNBP_ERR_CUDA, err); }
    h->spec_state[v] = 1;
    return BNBP_OK;
}

// Same for the on-chip kernel (variants 8 / 9 of the generated source, entry bnbp_onchip_run).
int ensure_onchip(bnbp_handle* h, int idx)
{
    if (h->oc_state[idx] == 1) return BNBP_OK;
    if (h->oc_state[idx] < 0) return fail(BNBP_ERR_INVALID, "on-chip kernel unavailable: " + h->oc_why);
    h->oc_state[idx] = -1;
    SpecConfig cfg;
    cfg.fp32 = h->precision == BNBP_FP32;
    cfg.vec = 1; cfg.minb = h->oc_minb; cfg.variant = 8 + (idx >> 1); cfg.ahead = h->oc_ahead;
    cfg.roles = h->oc_roles; cfg.out_double = (idx & 1) != 0;
    const std::string src = spec_source(spec_layout(h), cfg);
    std::vector<char> cubin;
    std::string err;
    bool cached = false;
    double ms = 0;
    if (!spec_compile(src, &cubin, &cached, &ms, &err)) { h->oc_why = err; return fail(BNBP_ERR_CUDA, err); }
    h->spec_compile_ms += ms;
    const int threads = 32 * h->oc_roles;
    if (!spec_load(cubin, &h->oc[idx], &err, "bnbp_onchip_run", threads, h->oc_smem)) {
        if (!cached || !spec_compile(src, &cubin, &cached, &ms, &err, true) ||
            !spec_load(cubin, &h->oc[idx], &err, "bnbp_onchip_run", threads, h->oc_smem)) {
            h->oc_why = err;
            return fail(BNBP_ERR_CUDA, err);
        }
        h->spec_compile_ms += ms;
    }
    h->oc[idx].from_cache = cached;
    h->oc[idx].compile_ms = ms;
    bool ok;
    if (cfg.fp32) {
        std::vector<float> tmp(h->cpt_host.begin(), h->cpt_host.end());
        ok = spec_upload_cpt(h->oc[idx], tmp.data(), tmp.size() * 4, &err);
    } else {
        ok = spec_upload_cpt(h->oc[idx], h->cpt_host.data(), h->cpt_host.size() * 8, &err);
    }
    if (!ok) { spec_unload(&h->oc[idx]); h->oc_why = err; return fail(BNBP_ERR_CUDA, err); }
    if (h->oc[idx].blocks_per_sm < 1) {
        spec_unload(&h->oc[idx]);
        h->oc_why = "the on-chip kernel does not fit an SM (registers / shared memory)";
        return fail(BNBP_ERR_CUDA, h->oc_why);
    }
    h->oc_state[idx] = 1;
    return BNBP_OK;
}

// Kernel family of one run.  Decided before the state is initialised because the tile width
// (cases per thread) belongs to the family.  ALWAYS: failure is an error; AUTO: the generic GPU
// kernel takes over (still CUDA: there is no CPU path).
int choose_kernels(bnbp_handle* h, int64_t n_cases, const bnbp_run_params& prm, bool soft_evidence, bool out_double)
{
    h->run_spec = false;
    h->fuse = false;
    h->split = false;
    h->run_onchip = false;
    h->last_onchip = 0;
    if (prm.semiring == BNBP_MAX_PRODUCT) {
        // opt-in extension: the generic kernel's max flavour (one kernel per network shape class); matrix products
        // cannot take a maximum, so handles whose large CPTs sit on the dense contraction path refuse it
        if (h->TS > 0) return fail(BNBP_ERR_INVALID, "max-product: create the handle with dense_min_cpt = -1 (the dense contraction path sums)");
        h->tb = BLOCK_THREADS * h->vec;
        h->last_specialised = 0;
        return BNBP_OK;
    }
    {
        // the on-chip kernel: the whole case in one launch, state in shared memory (hard evidence; soft rows
        // take the streaming kernels).  AUTO: eligible networks, batches worth a persistent grid.
        int mode = h->onchip;
        if (const char* e = getenv("BNBP_ONCHIP")) mode = atoi(e) > 0 ? 1 : (atoi(e) < 0 || !strcmp(e, "0") ? -1 : 0);
        // AUTO takes it for fixed sweep counts only: in epsilon mode its check flavour (10 k instructions of straight-line
        // code per sweep, a retire / refill path every few sweeps) runs at 302 M executed case-sweeps/s on alarm37 against
        // 357-381 M for the streaming kernels with the split convergence test (r02b vs r01fin)
        const bool plain_run = !(prm.epsilon > 0.0) && prm.damping == 0.0;
        const bool want_oc = mode > 0 || (mode == 0 && h->specialize == BNBP_SPEC_AUTO && h->oc_eligible && h->oc_auto_ok &&
                                          !soft_evidence && n_cases >= 4096 && plain_run);
        if (want_oc) {
            if (!h->oc_eligible) return fail(BNBP_ERR_INVALID, "onchip=ALWAYS but the network is not eligible: " + h->oc_why);
            if (soft_evidence) return fail(BNBP_ERR_INVALID, "onchip=ALWAYS: soft evidence rows take the streaming kernels");
            const int idx = ((prm.epsilon > 0.0 || prm.damping != 0.0) ? 2 : 0) + ((h->precision == BNBP_FP32 && out_double) ? 1 : 0);
            const int rc = ensure_onchip(h, idx);
            if (rc == BNBP_OK) {
                h->run_onchip = true;
                h->last_onchip = 1;
                h->last_specialised = 1;
                h->tb = 32;
                return BNBP_OK;
            }
            if (mode > 0) return rc;
        }
    }
    bool want = h->specialize == BNBP_SPEC_ALWAYS ||
                (h->specialize == BNBP_SPEC_AUTO && h->spec_eligible_ && h->spec_auto_ok && n_cases >= 4096);
    if (want && h->spec_classloop && h->specialize == BNBP_SPEC_AUTO) {
        // A class-looped walk covers a batch that does not fill the SMs with node slices in grid.y -- in its PLAIN variants.
        // The freeze / check variants (epsilon mode below the split threshold, damping) keep per-case state one block must
        // own, so a small batch would leave most SMs idle; the generic kernel splits its node walk in every flavour.
        const bool plain_variants = (!(prm.epsilon > 0.0) && prm.damping == 0.0) ||
                                    (prm.epsilon > 0.0 && prm.damping == 0.0 && n_cases >= 16384 && !getenv("BNBP_NO_SPLIT"));
        if (!plain_variants && n_cases < 32768) want = false;
    }
    if (want) {
        if (!h->spec_eligible_)
            return fail(BNBP_ERR_INVALID, "specialize=ALWAYS but the network is not eligible: " + h->spec_why);
        const bool eps_mode = prm.epsilon > 0.0;
        const int interval = prm.check_interval > 0 ? prm.check_interval : 1;
        const bool plain = !eps_mode && prm.damping == 0.0;
        // fixed sweep count: the first sweep knows every message is 1 (:44-55) and the last sweep's
        // messages are never read, so neither is moved through HBM (variants 3 and 4)
        // eps mode without damping on a batch worth it: the convergence test is a kernel of its own
        // (delta_retire_kernel) and the sweeps run as the plain variant
        const bool split = eps_mode && prm.damping == 0.0 && n_cases >= 16384 && h->TS == 0 && !getenv("BNBP_NO_SPLIT");
        bool need[5] = {(plain && prm.max_sweeps != 2) || split, eps_mode && interval > 1 && prm.damping == 0.0 && !split,
                        (eps_mode && !split) || prm.damping != 0.0, plain && prm.max_sweeps >= 2, plain && prm.max_sweeps >= 2};
        bool ok = true;
        for (int v = 0; v < 5 && ok; ++v)
            if (need[v] && ensure_spec(h, v) != BNBP_OK) ok = false;
        if (!ok && h->specialize == BNBP_SPEC_ALWAYS) return BNBP_ERR_CUDA;   // message already set
        h->run_spec = ok;
        h->split = ok && split;
        // fixed sweep count, hard evidence, one case per thread: K0 runs inside the first sweep and K4
        // inside the last (variants 5 and 6/7), so neither the time-0 pi/lambda nor the final ones
        // cross HBM.  Soft evidence rows do not fit a state byte: the unfused sequence handles them.
        if (ok && need[3] && !soft_evidence && h->spec_vec == 1 && h->fuse_ok && !getenv("BNBP_NO_FUSE")) {
            const int vlast = (h->precision == BNBP_FP32 && out_double) ? 7 : 6;
            if (ensure_spec(h, 5) == BNBP_OK && ensure_spec(h, vlast) == BNBP_OK) h->fuse = true;
            else h->fuse_ok = false;
        }
    }
    if (!h->run_spec)        // the generic family splits the convergence test off the same way (plain sweep + delta_retire_kernel)
        h->split = prm.epsilon > 0.0 && prm.damping == 0.0 && n_cases >= 16384 && h->TS == 0 && !getenv("BNBP_NO_SPLIT");
    h->tb = BLOCK_THREADS * (h->run_spec ? h->spec_vec : h->vec);
    h->last_specialised = h->run_spec ? 1 : 0;
    return BNBP_OK;
}

// Column groups for belief_tiled_kernel: consecutive nodes whose marginals fit one per-warp
// shared-memory tile of [32 cases][width] output elements (32 columns: 8.4 KB per warp in fp64).
int belief_plan(bnbp_handle* h, int tb, int out_size, bnbp_handle::BeliefPlan** out)
{
    const int key = tb * 16 + out_size;
    bnbp_handle::BeliefPlan& p = h->belief_plans[key];
    *out = &p;
    if (p.n_groups) return BNBP_OK;
    int width = 32;                                      // every node fits a group: width >= max cardinality
    for (int x = 0; x < h->N; ++x) width = std::max(width, (int)h->nodes[x].card);
    std::vector<BeliefGroup> groups;
    for (int x = 0; x < h->N;) {
        BeliefGroup g;
        g.n0 = x; g.j0 = h->nodes[x].bel_off;
        int w = 0;
        while (x < h->N && w + h->nodes[x].card <= width) { w += h->nodes[x].card; ++x; }
        g.n1 = x; g.j1 = g.j0 + w;
        groups.push_back(g);
    }
    p.ok = true;
    p.n_groups = (int)groups.size();
    p.stride = width | 1;                                // odd row stride: conflict-free phase 1
    p.smem = (size_t)tb * p.stride * out_size;           // tb/32 warps x [32][stride]
    int rc = p.groups.ensure(groups.size() * sizeof(BeliefGroup));
    if (rc) return rc;
    CU_TRY(cudaMemcpy(p.groups.p, groups.data(), groups.size() * sizeof(BeliefGroup), cudaMemcpyHostToDevice));
    return BNBP_OK;
}

struct DevEvidence {       // device pointers, offsets absolute with the given bases
    const int64_t* ev_off; int64_t ev_base;
    const int32_t* ev_node; const int32_t* ev_state;
    const int64_t* ev_val_off; const double* ev_values; int64_t ev_val_base;
};

// Runs init -> sweeps -> beliefs for n (<= cap) cases whose evidence is on the device.
template <typename T, typename OUT>
int run_chunk(bnbp_handle* h, int64_t n, const DevEvidence& de, const bnbp_run_params& prm, OUT* d_out,
              int32_t* d_out_sweeps, uint8_t* d_out_conv, cudaStream_t st, int64_t* planned_sweeps)
{
    NvtxRange nvtx_chunk("bnbp: chunk (init, sweeps, beliefs) streaming kernels");
    const int tiles = (int)((n + h->tb - 1) / h->tb);
    int32_t* d_last_active = reinterpret_cast<int32_t*>(h->d_misc.p);
    int32_t* d_error = d_last_active + 1;
    const bool eps_mode = prm.epsilon > 0.0;
    const int max_sweeps = prm.max_sweeps > 0 ? prm.max_sweeps : (1 << 30);
    const int interval = prm.check_interval > 0 ? prm.check_interval : 1;
    if (!eps_mode && prm.max_sweeps <= 0)
        return fail(BNBP_ERR_INVALID, "epsilon <= 0 needs a positive max_sweeps (the loop would never end)");

    CU_TRY(cudaMemsetAsync(d_last_active, 0xFF, 4, st));   // -1
    const bool fuse = h->fuse && h->run_spec && !eps_mode && prm.damping == 0.0 && max_sweeps >= 2 && !de.ev_values;
    h->last_fused = fuse ? 1 : 0;
    if (fuse) {
        // K0 is part of the first sweep (variant 5): only the observed states are scattered here
        CU_TRY(cudaMemsetAsync(h->d_evst.p, 0, (size_t)tiles * h->tb * h->N, st));
        CU_TRY(cudaMemsetAsync(h->d_evbits.p, 0, (size_t)tiles * h->tb * h->W * 4, st));
        EvidenceArgs ea;
        ea.nodes = (const NodeMeta*)h->d_nodes.p;
        ea.evst = (uint8_t*)h->d_evst.p; ea.evbits = (uint32_t*)h->d_evbits.p;
        ea.W = h->W; ea.TB = h->tb; ea.n_nodes = h->N; ea.n_valid = n;
        ea.ev_off = de.ev_off; ea.ev_base = de.ev_base; ea.ev_node = de.ev_node; ea.ev_state = de.ev_state;
        ea.error_flag = d_error;
        evidence_kernel<<<tiles, h->tb, 0, st>>>(ea);
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
    } else {
        InitArgs<T> ia;
        ia.nodes = (const NodeMeta*)h->d_nodes.p;
        ia.pl_init = (const T*)h->d_pl_init.p;
        ia.pl = (T*)h->d_pl.p; ia.msg0 = (T*)h->d_msg[0].p; ia.evbits = (uint32_t*)h->d_evbits.p;
        ia.PL = h->PL; ia.M = h->M; ia.W = h->W; ia.TB = h->tb; ia.n_nodes = h->N;
        ia.n_valid = n;
        ia.ev_off = de.ev_off; ia.ev_base = de.ev_base; ia.ev_node = de.ev_node; ia.ev_state = de.ev_state;
        ia.ev_val_off = de.ev_val_off; ia.ev_values = de.ev_values; ia.ev_val_base = de.ev_val_base;
        ia.delta = (T*)h->d_delta.p; ia.cap = h->cap;
        ia.status = (uint8_t*)h->d_status.p; ia.sweeps = (int32_t*)h->d_sweeps.p;
        ia.error_flag = d_error;
        // the specialised first sweep (variant 3) does not read the time-0 messages
        ia.write_msgs = (h->run_spec && !eps_mode && prm.damping == 0.0 && max_sweeps >= 2) ? 0 : 1;
        init_kernel<T><<<tiles, h->tb, 0, st>>>(ia);
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
    }

    // the arena the sweeps work on: the handle's own, or (eps mode, after a compaction) the second one
    T* pl_p = (T*)h->d_pl.p;
    T* msg_p[2] = {(T*)h->d_msg[0].p, (T*)h->d_msg[1].p};
    uint32_t* evb_p = (uint32_t*)h->d_evbits.p;
    int arena_set = 0;
    int64_t n_cur = n;                       // cases (positions) of the current arena
    int tiles_cur = tiles;
    const int32_t* orig = nullptr;           // position -> case of the chunk (nullptr: identity)
    int orig_set = 0;
    // Compaction pays when the sweep counts spread (alarm37, eps 1e-6: mean 13, max 40 sweeps).  Not with
    // dense nodes (their per-case tables live in a third arena) and not for small batches.
    const bool trace_compact = getenv("BNBP_TRACE") != nullptr;
    const auto t_chunk = std::chrono::steady_clock::now();
    const bool compact = eps_mode && h->compact_ok && h->TS == 0 && n >= 16384 && !getenv("BNBP_NO_COMPACT");
    const bool split = h->split && eps_mode && prm.damping == 0.0;
    bool have_total = false;                 // split: a delta_retire_kernel has counted the active cases

    SweepArgs<T> sa;
    memset(&sa, 0, sizeof sa);
    sa.nodes = (const NodeMeta*)h->d_nodes.p;
    sa.e_card = (const int32_t*)h->d_e_card.p;
    sa.e_lam_out = (const int32_t*)h->d_e_lam_out.p;
    sa.c_pi_out = (const int32_t*)h->d_c_pi_out.p;
    sa.cpt = (const T*)h->d_cpt.p;
    sa.pl = pl_p;
    sa.evbits = evb_p;
    sa.PL = h->PL; sa.M = h->M; sa.W = h->W; sa.TS = h->TS;
    sa.tscr = (const T*)h->d_tscr.p;
    // enough threads to fill 148 SMs a few times over: split the node walk when the batch is small
    const int64_t threads_per_row = (int64_t)tiles * BLOCK_THREADS;
    int n_chunks = (int)std::min<int64_t>(std::min(MAX_CHUNKS, std::max(1, h->N / 8)),
                                          std::max<int64_t>(1, (148 * 2048 * 2 + threads_per_row - 1) / threads_per_row));
    sa.n_chunks = n_chunks;
    make_chunks(h, n_chunks, sa.chunk_off);
    sa.status = (uint8_t*)h->d_status.p;
    sa.sweeps = (int32_t*)h->d_sweeps.p;
    sa.last_active = d_last_active;
    sa.eps = (T)prm.epsilon;
    sa.damping = (T)prm.damping;
    {
        // next-node L2 prefetch: pays where a node is a handful of rows and the walk is pure latency (grid100, cardinality 2:
        // +9 %, r02d), costs where a node has dozens of rows and the kernel already issues at 22 % (dag2000, cardinality <= 8: -10 %)
        static const int knob = getenv("BNBP_PREFETCH") ? atoi(getenv("BNBP_PREFETCH")) : -1;      // tuning knob (A/B runs)
        sa.prefetch = knob >= 0 ? knob : (h->rmax <= 4 ? 1 : 0);
    }
    T* delta = (T*)h->d_delta.p;
    const size_t smem = (size_t)BLOCK_THREADS * (size_t)h->scratch_vals * h->vec * sizeof(T);
    dim3 grid(tiles, n_chunks);
    auto regrid = [&]() {                    // after a compaction: fewer tiles, maybe more node chunks
        const int64_t tpr = (int64_t)tiles_cur * BLOCK_THREADS;
        n_chunks = (int)std::min<int64_t>(std::min(MAX_CHUNKS, std::max(1, h->N / 8)),
                                          std::max<int64_t>(1, (148 * 2048 * 2 + tpr - 1) / tpr));
        sa.n_chunks = n_chunks;
        make_chunks(h, n_chunks, sa.chunk_off);
        grid = dim3(tiles_cur, n_chunks);
    };

    // event pair around the sweeps of this chunk
    if ((int)h->ev_sweep.size() < 2 * (h->ev_sweep_used + 1)) {
        cudaEvent_t a, b;
        CU_TRY(cudaEventCreate(&a));
        CU_TRY(cudaEventCreate(&b));
        h->ev_sweep.push_back(a);
        h->ev_sweep.push_back(b);
    }
    CU_TRY(cudaEventRecord(h->ev_sweep[2 * h->ev_sweep_used], st));

    int t = 0;
    bool prev_tested = false;
    const int POLL = (compact || split) ? 4 : 8;
    int polls_issued = 0;
    bool stop = false;
    while (t < max_sweeps && !stop) {
        const int t_end = (int)std::min<int64_t>((int64_t)t + POLL, max_sweeps);
        for (; t < t_end; ++t) {
            const bool tested = eps_mode && (((t + 1) % interval) == 0 || t + 1 >= max_sweeps);
            const bool check = tested || prm.damping != 0.0;
            sa.msg_cur = msg_p[t & 1];
            sa.msg_nxt = msg_p[(t + 1) & 1];
            sa.delta_prev = delta + (size_t)((t + 2) % 3) * h->cap;
            sa.delta_cur = delta + (size_t)(t % 3) * h->cap;
            sa.delta_next = delta + (size_t)((t + 1) % 3) * h->cap;
            sa.sweep_index = t;
            sa.prev_tested = prev_tested ? 1 : 0;
            int n_inner = 1;
            if (h->TS > 0) {
                // dense nodes: this sweep's CPT x batch products (time-t messages and lambda_X), before
                // the sweep kernel overwrites lambda_X in place
                const bool timed = h->ev_dense_used < 512;
                if (timed) {
                    if ((int)h->ev_dense.size() < 2 * (h->ev_dense_used + 1)) {
                        cudaEvent_t e0, e1;
                        CU_TRY(cudaEventCreate(&e0));
                        CU_TRY(cudaEventCreate(&e1));
                        h->ev_dense.push_back(e0);
                        h->ev_dense.push_back(e1);
                    }
                    CU_TRY(cudaEventRecord(h->ev_dense[2 * h->ev_dense_used], st));
                }
                DenseArgs<T> da;
                da.jobs = (const DenseJob*)h->d_djobs.p;
                da.dig = (const unsigned long long*)h->d_ddig.p;
                da.arena0 = (const T*)h->d_cpt.p;
                da.arena1 = (const T*)h->d_cpt_t.p;
                da.pl = (const T*)h->d_pl.p;
                da.msg_cur = sa.msg_cur;
                da.tscr = (T*)h->d_tscr.p;
                da.PL = h->PL; da.M = h->M; da.TS = h->TS; da.TBC = h->tb;
                da.status = eps_mode ? (const uint8_t*)h->d_status.p : nullptr;
                for (const bnbp_handle::DenseGroup& g : h->dgroups) {
                    da.ytab = (const int32_t*)h->d_dytab.p + g.ytab0;
                    cudaError_t e = launch_dense<T>(da, g.nf, g.tnt, h->dense_mma, dim3((unsigned)((int64_t)tiles * h->tb / DT_M), (unsigned)g.n_y),
                                                    dense_smem_bytes(g.max_rows, g.tnt, sizeof(T)), st);
                    if (e != cudaSuccess) return fail(BNBP_ERR_CUDA, std::string("dense launch: ") + cudaGetErrorString(e));
                    h->last_dense_launches++;
                    h->last_kernel_launches++;
                }
                if constexpr (sizeof(T) == 4) {
                    // tensor-core products (tcgen05, 3xTF32): 256 cases x 256 columns per CTA
                    DenseTcArgs ta;
                    ta.jobs = da.jobs; ta.dig = da.dig;
                    ta.arena_tc = (const float*)h->d_cpt_tc.p;
                    ta.pl = (const float*)da.pl; ta.msg_cur = (const float*)da.msg_cur; ta.tscr = (float*)da.tscr;
                    ta.PL = da.PL; ta.M = da.M; ta.TS = da.TS; ta.TBC = da.TBC;
                    ta.n_cases = (int64_t)tiles * h->tb;
                    ta.status = da.status;
                    for (const bnbp_handle::TcGroup& g : h->tcgroups) {
                        ta.ytab = (const int32_t*)h->d_dytab.p + g.ytab0;
                        ta.stages = g.stages;
                        cudaError_t e = launch_dense_tc(ta, dim3((unsigned)((ta.n_cases + TC_M - 1) / TC_M), (unsigned)g.n_y),
                                                        tc_smem_bytes(g.max_rows, g.stages), st);
                        if (e != cudaSuccess) return fail(BNBP_ERR_CUDA, std::string("tensor-core dense launch: ") + cudaGetErrorString(e));
                        h->last_dense_launches++;
                        h->last_dense_tc_launches++;
                        h->last_kernel_launches++;
                    }
                }
                if (timed) {
                    CU_TRY(cudaEventRecord(h->ev_dense[2 * h->ev_dense_used + 1], st));
                    h->ev_dense_used++;
                }
            }
            if (h->run_spec) {
                // network-specialised kernel: variant 0 plain, 1 freeze, 2 freeze + check
                int variant = check ? 2 : (eps_mode ? 1 : 0);
                if (split) variant = 0;
                else if (variant == 0 && max_sweeps >= 2) variant = t == 0 ? 3 : (t == max_sweeps - 1 ? 4 : 0);
                if (fuse && variant == 3) variant = 5;
                if (fuse && variant == 4) variant = (sizeof(T) == 4 && sizeof(OUT) == 8) ? 7 : 6;
                SpecAux<T> ax;
                ax.delta_prev = sa.delta_prev; ax.delta_cur = sa.delta_cur; ax.delta_next = sa.delta_next;
                ax.status = sa.status; ax.sweeps = sa.sweeps; ax.last_active = sa.last_active;
                ax.sweep_index = sa.sweep_index; ax.prev_tested = sa.prev_tested; ax.eps = sa.eps; ax.damping = sa.damping;
                ax.evst = (const unsigned char*)h->d_evst.p; ax.out = d_out; ax.n_valid = n;
                // fixed-count runs: the plain sweeps between the first and the last can go out as ONE launch
                // (cases are independent, no barrier between their sweeps is needed).  A looped launch ends with
                // ONE tail of up to a whole block lifetime (n_inner sweeps), separate launches with n_inner short
                // ones: looping wins for grids of whole waves and for short grids (the chunks of the host-buffer
                // pipeline, +3 % e2e), separate launches for one long ragged grid (18.45 waves: -3 %, r01o).
                ax.n_inner = 1;
                // class-looped walk on a batch that does not fill the SMs (cfg 3 sharded 8 ways: 64 tiles for 148 SMs): the
                // plain variants take node SLICES in grid.y -- block (tile, y) walks the y-th slice of every node class -- until
                // one wave of blocks is resident.  Such a launch is one sweep (slices of sweep t+1 read what every slice of
                // sweep t wrote), so it does not loop.
                unsigned node_slices = 1;
                if (h->spec_classloop && (variant == 0 || variant == 3 || variant == 4) && !getenv("BNBP_NO_NODE_SLICES")) {
                    int sms = 148;
                    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
                    const int64_t wave_blocks = (int64_t)sms * std::max(1, h->spec[variant].blocks_per_sm);
                    // as many slices as keep the grid within ONE wave (a second, sparse wave costs a whole block lifetime:
                    // 512 tiles on 444 slots ran at 0.72 of HBM against 0.95 on 592 slots, r02r)
                    if (tiles_cur < wave_blocks) node_slices = (unsigned)std::min<int64_t>(32, std::max<int64_t>(1, wave_blocks / tiles_cur));
                    if (const char* e = getenv("BNBP_NODE_SLICES")) node_slices = (unsigned)std::min(64, std::max(1, atoi(e)));      // tuning / test knob
                }
                if (node_slices == 1 && variant == 0 && !eps_mode && prm.damping == 0.0 && !getenv("BNBP_NO_LOOP")) {
                    int sms = 148;
                    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
                    const int64_t wave_blocks = (int64_t)sms * std::max(1, h->spec[0].blocks_per_sm);
                    if (tiles_cur % wave_blocks == 0 || tiles_cur < 12 * wave_blocks || getenv("BNBP_LOOP_ALWAYS"))
                        ax.n_inner = (max_sweeps >= 2 ? max_sweeps - 1 : max_sweeps) - t;
                }
                n_inner = ax.n_inner;
                std::string err;
                if (!spec_launch(h->spec[variant], (unsigned)tiles_cur, st, sa.pl, sa.msg_cur, sa.msg_nxt, sa.evbits, &ax, &err, node_slices))
                    return fail(BNBP_ERR_CUDA, err);
            } else {
                cudaError_t e = launch_sweep<T>(h, sa, grid, smem, eps_mode && !split, check && !split, st, prm.semiring == BNBP_MAX_PRODUCT);
                if (e != cudaSuccess) return fail(BNBP_ERR_CUDA, std::string("sweep launch: ") + cudaGetErrorString(e));
            }
            if (split && tested) {
                // the convergence test of this sweep (:105-131,:147), retirement of the cases it stops, census
                int rc;
                if ((rc = h->d_tile_count.ensure((size_t)tiles * 8))) return rc;
                int32_t* const d_total = d_last_active + 2;
                CU_TRY(cudaMemsetAsync(d_total, 0, 4, st));
                delta_retire_kernel<T, OUT><<<tiles_cur, h->tb, 0, st>>>(
                    (const NodeMeta*)h->d_nodes.p, h->N, h->PL, h->M, h->V, pl_p, sa.msg_cur, sa.msg_nxt, (uint8_t*)h->d_status.p,
                    (T)prm.epsilon, t + 1, n_cur, orig, d_out, d_out_sweeps, d_out_conv, (int32_t*)h->d_tile_count.p, d_total);
                CU_TRY(cudaGetLastError());
                h->last_kernel_launches++;
                have_total = true;
            }
            prev_tested = tested;
            h->last_sweep_launches += n_inner;      // counted in sweeps: a looped launch stands for n_inner of them
            h->last_kernel_launches++;
            t += n_inner - 1;
        }
        if ((split && have_total && t < max_sweeps) || (compact && !split && t < max_sweeps && t >= 8)) {
            // census: the freeze rule of the next launch, active cases per tile and in total (one host
            // round trip per POLL sweeps; the grid that follows is sized by its answer).  In split mode
            // the last delta_retire_kernel has already counted.
            int rc;
            if ((rc = h->d_tile_count.ensure((size_t)tiles * 8))) return rc;
            int32_t* const d_total = d_last_active + 2;
            int32_t* const d_tile_cnt = (int32_t*)h->d_tile_count.p;
            int32_t* const d_tile_off = d_tile_cnt + tiles;
            if (!split) {
                CU_TRY(cudaMemsetAsync(d_total, 0, 4, st));
                compact_census_kernel<T><<<tiles_cur, h->tb, 0, st>>>((uint8_t*)h->d_status.p, (int32_t*)h->d_sweeps.p,
                                                                      delta + (size_t)((t + 2) % 3) * h->cap, prev_tested ? 1 : 0,
                                                                      (T)prm.epsilon, t, d_tile_cnt, d_total);
                CU_TRY(cudaGetLastError());
                h->last_kernel_launches++;
            }
            CU_TRY(cudaMemcpyAsync(&h->pinned_poll[2], d_total, 4, cudaMemcpyDeviceToHost, st));
            CU_TRY(wait_stream(st));
            const int64_t n_active = h->pinned_poll[2];
            if (trace_compact)
                fprintf(stderr, "[bnbp] census after sweep %d: %lld of %lld positions active, %.3f ms since the chunk started\n", t,
                        (long long)n_active, (long long)n_cur,
                        std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_chunk).count());
            if (n_active == 0) {
                stop = true;
            } else if (compact && n_active * 10 <= n_cur * 7 && n_cur >= 8192) {
                const int64_t tiles_new = (n_active + h->tb - 1) / h->tb;
                const size_t want = (size_t)tiles_new * h->tb;
                DevBuf* pl_b[2] = {&h->d_pl, &h->d_pl2};
                DevBuf* m0_b[2] = {&h->d_msg[0], &h->d_msg2[0]};
                DevBuf* m1_b[2] = {&h->d_msg[1], &h->d_msg2[1]};
                DevBuf* ev_b[2] = {&h->d_evbits, &h->d_evbits2};
                const int dst = arena_set ^ 1;
                bool fits = true;
                if (dst == 1) {                                  // set 0 is the handle's full-size arena
                    cudaGetLastError();
                    fits = h->d_pl2.ensure(want * h->PL * sizeof(T)) == BNBP_OK &&
                           h->d_msg2[0].ensure(std::max<size_t>(16, want * h->M * sizeof(T))) == BNBP_OK &&
                           h->d_msg2[1].ensure(std::max<size_t>(16, want * h->M * sizeof(T))) == BNBP_OK &&
                           h->d_evbits2.ensure(want * h->W * 4) == BNBP_OK;
                    if (!fits) {                                 // HBM is full: carry on in place, never try again
                        cudaGetLastError();
                        h->d_pl2.release(); h->d_msg2[0].release(); h->d_msg2[1].release(); h->d_evbits2.release();
                        h->compact_ok = false;
                    }
                }
                if (fits && (h->d_orig[0].ensure((size_t)h->cap * 4) || h->d_orig[1].ensure((size_t)h->cap * 4) ||
                             h->d_src_pos.ensure((size_t)h->cap * 4)))
                    fits = false;
                if (fits && split) have_total = false;           // the counts describe the old arena
                if (fits && !split) {
                    // 1. retire the converged cases: their state is final (:135-147), write their beliefs now
                    bnbp_handle::BeliefPlan* plan = nullptr;
                    if ((rc = belief_plan(h, h->tb, (int)sizeof(OUT), &plan))) return rc;
                    if (plan->smem > 48 * 1024)
                        CU_TRY(cudaFuncSetAttribute(belief_tiled_kernel<T, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan->smem));
                    belief_tiled_kernel<T, OUT><<<tiles_cur, h->tb, plan->smem, st>>>(
                        (const NodeMeta*)h->d_nodes.p, (const BeliefGroup*)plan->groups.p, plan->n_groups, pl_p, h->PL,
                        h->tb, h->V, plan->stride, n_cur, d_out, (const uint8_t*)h->d_status.p, (const int32_t*)h->d_sweeps.p,
                        d_out_sweeps, d_out_conv, orig, 1);
                    CU_TRY(cudaGetLastError());
                    h->last_kernel_launches++;
                }
                if (fits) {
                    // 2. new position -> old position (stable), 3. gather into the other arena
                    compact_scan_kernel<<<1, 1024, 0, st>>>(d_tile_cnt, d_tile_off, tiles_cur);
                    int32_t* const orig_new = (int32_t*)h->d_orig[orig_set ^ 1].p;
                    compact_index_kernel<<<tiles_cur, h->tb, 0, st>>>((const uint8_t*)h->d_status.p, d_tile_off, orig,
                                                                      (int32_t*)h->d_src_pos.p, orig_new);
                    CU_TRY(cudaGetLastError());
                    T* const pl_d = (T*)pl_b[dst]->p;
                    T* const md[2] = {(T*)m0_b[dst]->p, (T*)m1_b[dst]->p};
                    uint32_t* const ev_d = (uint32_t*)ev_b[dst]->p;
                    compact_gather_kernel<T><<<(unsigned)tiles_new, h->tb, 0, st>>>(
                        (const int32_t*)h->d_src_pos.p, (int32_t)n_active, h->tb, h->PL, h->M, h->W, pl_p, msg_p[t & 1], evb_p,
                        pl_d, md[t & 1], ev_d, (uint8_t*)h->d_status.p, delta, h->cap);
                    CU_TRY(cudaGetLastError());
                    h->last_kernel_launches += 3;
                    h->last_compactions++;
                    pl_p = pl_d; msg_p[0] = md[0]; msg_p[1] = md[1]; evb_p = ev_d;
                    arena_set = dst;
                    orig = orig_new; orig_set ^= 1;
                    n_cur = n_active; tiles_cur = (int)tiles_new;
                    sa.pl = pl_p; sa.evbits = evb_p;
                    regrid();
                    prev_tested = false;                         // the census already froze what the last test found
                }
            }
        } else if (eps_mode && !compact && !split && t < max_sweeps) {
            // asynchronous termination poll: keep one batch of launches in flight while the flag
            // of the batch before travels back (speculative launches exit on the device at once)
            const int slot = polls_issued & 1;
            if (polls_issued >= 2) {
                CU_TRY(cudaEventSynchronize(h->ev_poll[slot]));
                // value copied after the sweeps [.., t_prev) of two batches ago
                const int t_prev = t - 2 * POLL;
                if (h->pinned_poll[slot] < t_prev - 1) stop = true;
            }
            if (!stop) {
                CU_TRY(cudaMemcpyAsync(&h->pinned_poll[slot], d_last_active, 4, cudaMemcpyDeviceToHost, st));
                CU_TRY(cudaEventRecord(h->ev_poll[slot], st));
                polls_issued++;
            }
        }
    }
    const int total_sweeps = t;
    CU_TRY(cudaEventRecord(h->ev_sweep[2 * h->ev_sweep_used + 1], st));
    h->ev_sweep_used++;
    if (eps_mode) {
        const int last = total_sweeps - 1;
        finalize_kernel<T><<<(unsigned)(((int64_t)tiles_cur * h->tb + 255) / 256), 256, 0, st>>>(
            (uint8_t*)h->d_status.p, (int32_t*)h->d_sweeps.p, delta + (size_t)(last % 3) * h->cap,
            (prev_tested && !split) ? 1 : 0, (T)prm.epsilon, total_sweeps, (int64_t)tiles_cur * h->tb);
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
    } else {
        CU_TRY(cudaMemsetAsync(h->d_status.p, 0, (size_t)tiles * h->tb, st));
        // sweeps[] = total for every case
        finalize_kernel<T><<<(unsigned)((h->cap + 255) / 256), 256, 0, st>>>(
            (uint8_t*)h->d_status.p, (int32_t*)h->d_sweeps.p, delta, 0, (T)0, total_sweeps, (int64_t)tiles * h->tb);
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
    }

    if (fuse) {
        // K4 ran inside the last sweep (variants 6/7); only the per-case counts are left
        if (d_out_sweeps || d_out_conv) {
            counts_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const uint8_t*)h->d_status.p, (const int32_t*)h->d_sweeps.p,
                                                                        d_out_sweeps, d_out_conv, n);
            CU_TRY(cudaGetLastError());
            h->last_kernel_launches++;
        }
    } else {
        bnbp_handle::BeliefPlan* plan = nullptr;
        int rc = belief_plan(h, h->tb, (int)sizeof(OUT), &plan);
        if (rc) return rc;
        if (plan->ok) {
            if (plan->smem > 48 * 1024)
                CU_TRY(cudaFuncSetAttribute(belief_tiled_kernel<T, OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan->smem));
            belief_tiled_kernel<T, OUT><<<tiles_cur, h->tb, plan->smem, st>>>(
                (const NodeMeta*)h->d_nodes.p, (const BeliefGroup*)plan->groups.p, plan->n_groups, pl_p, h->PL,
                h->tb, h->V, plan->stride, n_cur, d_out, (const uint8_t*)h->d_status.p, (const int32_t*)h->d_sweeps.p,
                d_out_sweeps, d_out_conv, orig, split ? 2 : 0);
        } else {
            belief_kernel<T, OUT><<<tiles, h->tb, 0, st>>>((const NodeMeta*)h->d_nodes.p, h->N, (const T*)h->d_pl.p, h->PL, h->tb,
                                                        h->V, n, d_out, (const uint8_t*)h->d_status.p,
                                                        (const int32_t*)h->d_sweeps.p, d_out_sweeps, d_out_conv);
        }
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
    }
    if (planned_sweeps) *planned_sweeps = eps_mode ? -1 : (int64_t)total_sweeps * n;
    return BNBP_OK;
}

// The whole path for n cases in ONE launch of the on-chip kernel (bnbp_onchip.cuh): init, every sweep, the
// stopping rule and the beliefs; nothing but evidence in and marginals out touches HBM.
template <typename T, typename OUT>
int run_onchip(bnbp_handle* h, int64_t n, const DevEvidence& de, const bnbp_run_params& prm, OUT* d_out,
               int32_t* d_out_sweeps, uint8_t* d_out_conv, cudaStream_t st, int64_t* planned_sweeps)
{
    NvtxRange nvtx_chunk("bnbp: chunk, on-chip kernel (init, every sweep, beliefs in one launch)");
    const bool eps_mode = prm.epsilon > 0.0;
    if (!eps_mode && prm.max_sweeps <= 0)
        return fail(BNBP_ERR_INVALID, "epsilon <= 0 needs a positive max_sweeps (the loop would never end)");
    if (de.ev_values) return fail(BNBP_ERR_INVALID, "the on-chip kernel takes hard evidence");
    const int idx = ((eps_mode || prm.damping != 0.0) ? 2 : 0) + (sizeof(OUT) != sizeof(T) ? 1 : 0);
    const SpecKernel& k = h->oc[idx];
    if (h->oc_state[idx] != 1) return fail(BNBP_ERR_INVALID, "on-chip kernel not loaded");
    int32_t* const misc = reinterpret_cast<int32_t*>(h->d_misc.p);
    unsigned long long* const ticket = reinterpret_cast<unsigned long long*>(misc + 8);
    CU_TRY(cudaMemsetAsync(ticket, 0, 8, st));
    OnchipArgs<T> a;
    a.ev_off = reinterpret_cast<const long long*>(de.ev_off); a.ev_base = de.ev_base;
    a.ev_node = de.ev_node; a.ev_state = de.ev_state;
    a.n_cases = n;
    a.out = d_out; a.out_sweeps = d_out_sweeps; a.out_conv = d_out_conv;
    a.bel_col = (const int*)h->d_belcol.p; a.out_stride = h->Vout;
    a.ticket = ticket; a.error_flag = misc + 1;
    a.eps = (T)prm.epsilon; a.damping = (T)prm.damping;
    a.max_sweeps = prm.max_sweeps > 0 ? prm.max_sweeps : (1 << 30);
    a.interval = prm.check_interval > 0 ? prm.check_interval : 1;
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    a.first_reserved_sm = sms - std::min(std::max(0, h->reserve_sms), sms / 2);
    const int64_t groups = (n + 31) / 32;
    const unsigned blocks = (unsigned)std::min<int64_t>(groups, (int64_t)sms * std::max(1, k.blocks_per_sm));
    if ((int)h->ev_sweep.size() < 2 * (h->ev_sweep_used + 1)) {
        cudaEvent_t e0, e1;
        CU_TRY(cudaEventCreate(&e0));
        CU_TRY(cudaEventCreate(&e1));
        h->ev_sweep.push_back(e0);
        h->ev_sweep.push_back(e1);
    }
    CU_TRY(cudaEventRecord(h->ev_sweep[2 * h->ev_sweep_used], st));
    std::string err;
    if (!onchip_launch(k, blocks, (unsigned)(32 * h->oc_roles), h->oc_smem, st, &a, &err)) return fail(BNBP_ERR_CUDA, err);
    CU_TRY(cudaEventRecord(h->ev_sweep[2 * h->ev_sweep_used + 1], st));
    h->ev_sweep_used++;
    h->last_kernel_launches++;
    h->last_sweep_launches += eps_mode ? 1 : a.max_sweeps;      // counted in sweeps: the launch runs them all
    h->last_fused = 1;
    if (planned_sweeps) *planned_sweeps = eps_mode ? -1 : (int64_t)a.max_sweeps * n;
    return BNBP_OK;
}

// ---- what leaves the device ---------------------------------------------------------------------------
// Row layout of the marginals of this run: every node (the reference's result map, :151-158) or the queried
// nodes only.  The device tables are rebuilt only when the query changes.
int query_columns(const bnbp_handle* h, const bnbp_run_params& prm, std::vector<int32_t>* q, std::vector<int32_t>* belcol,
                  std::vector<int32_t>* colmap)
{
    if (prm.n_query < 0) return fail(BNBP_ERR_INVALID, "n_query < 0");
    if (prm.n_query > 0 && !prm.query_nodes) return fail(BNBP_ERR_INVALID, "query_nodes is NULL");
    q->assign(prm.query_nodes, prm.query_nodes + prm.n_query);
    belcol->assign((size_t)h->N, -1);
    colmap->clear();
    if (q->empty()) {
        for (int x = 0; x < h->N; ++x) {
            (*belcol)[(size_t)x] = h->nodes[x].bel_off;
            for (int i = 0; i < h->nodes[x].card; ++i) colmap->push_back(h->nodes[x].bel_off + i);
        }
        return BNBP_OK;
    }
    for (int32_t x : *q) {
        if (x < 0 || x >= h->N) return fail(BNBP_ERR_INVALID, "query node id out of range");
        if ((*belcol)[(size_t)x] >= 0) return fail(BNBP_ERR_INVALID, "query node listed twice");
        (*belcol)[(size_t)x] = (int32_t)colmap->size();
        for (int i = 0; i < h->nodes[x].card; ++i) colmap->push_back(h->nodes[x].bel_off + i);
    }
    return BNBP_OK;
}

int set_query(bnbp_handle* h, const bnbp_run_params& prm)
{
    std::vector<int32_t> q, belcol, colmap;
    int rc = query_columns(h, prm, &q, &belcol, &colmap);
    if (rc) return rc;
    if (h->q_valid && q == h->q_nodes) return BNBP_OK;
    CU_TRY(cudaDeviceSynchronize());          // an earlier asynchronous run may still read the old tables
    if ((rc = h->d_belcol.ensure(belcol.size() * 4)) || (rc = h->d_colmap.ensure(std::max<size_t>(16, colmap.size() * 4)))) return rc;
    CU_TRY(cudaMemcpy(h->d_belcol.p, belcol.data(), belcol.size() * 4, cudaMemcpyHostToDevice));
    if (!colmap.empty()) CU_TRY(cudaMemcpy(h->d_colmap.p, colmap.data(), colmap.size() * 4, cudaMemcpyHostToDevice));
    h->q_nodes.swap(q);
    h->Vout = (int)colmap.size();
    h->q_valid = true;
    return BNBP_OK;
}

template <typename OUT>
__global__ void gather_columns_kernel(const OUT* __restrict__ src, OUT* __restrict__ dst, int64_t n, int V, int Vout,
                                      const int32_t* __restrict__ colmap)
{
    const int64_t total = n * Vout;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t c = i / Vout;
        dst[i] = src[c * V + colmap[i - c * Vout]];
    }
}

// One chunk through whichever kernel family the run chose; under a query the streaming kernels write full-width
// rows into a staging buffer and the asked-for columns are gathered into the output (the on-chip kernel writes
// only those in the first place).
template <typename T, typename OUT>
int run_any(bnbp_handle* h, int64_t n, const DevEvidence& de, const bnbp_run_params& prm, OUT* d_out, int32_t* d_out_sweeps,
            uint8_t* d_out_conv, cudaStream_t st, int64_t* planned_sweeps)
{
    if (h->run_onchip) return run_onchip<T, OUT>(h, n, de, prm, d_out, d_out_sweeps, d_out_conv, st, planned_sweeps);
    if (h->q_nodes.empty()) return run_chunk<T, OUT>(h, n, de, prm, d_out, d_out_sweeps, d_out_conv, st, planned_sweeps);
    int rc = h->s_full.ensure((size_t)n * h->V * sizeof(OUT));
    if (rc) return rc;
    if ((rc = run_chunk<T, OUT>(h, n, de, prm, (OUT*)h->s_full.p, d_out_sweeps, d_out_conv, st, planned_sweeps))) return rc;
    const int64_t total = n * h->Vout;
    if (total > 0) {
        gather_columns_kernel<OUT><<<(unsigned)std::min<int64_t>((total + 255) / 256, 148 * 16), 256, 0, st>>>(
            (const OUT*)h->s_full.p, d_out, n, h->V, h->Vout, (const int32_t*)h->d_colmap.p);
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
    }
    return BNBP_OK;
}

// ---- rates the chunk planner needs: measured on this handle's device, once --------------------------------
int measure_rates(bnbp_handle* h)
{
    if (h->link_gbs > 0.0) return BNBP_OK;
    // device-to-host over the link this GPU sits on: 32 MB from device memory into pinned memory, second of two copies
    const size_t bytes = 32u << 20;
    void* dev = nullptr;
    void* host = nullptr;
    CU_TRY(cudaMalloc(&dev, bytes));
    if (cudaMallocHost(&host, bytes) != cudaSuccess) { cudaFree(dev); cudaGetLastError(); h->link_gbs = 25.0; }
    else {
        cudaEvent_t e0, e1;
        cudaEventCreate(&e0);
        cudaEventCreate(&e1);
        cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, h->copy_stream);
        cudaEventRecord(e0, h->copy_stream);
        cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, h->copy_stream);
        cudaEventRecord(e1, h->copy_stream);
        float ms = 0.f;
        if (cudaEventSynchronize(e1) == cudaSuccess && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess && ms > 0.f)
            h->link_gbs = (double)bytes / (ms * 1e-3) / 1e9;
        else
            h->link_gbs = 25.0;
        cudaEventDestroy(e0);
        cudaEventDestroy(e1);
        cudaFreeHost(host);
        cudaFree(dev);
        cudaGetLastError();
    }
    // HBM: 0.8 of the interface rate the device reports (memory clock x bus width, double data rate)
    int khz = 0, bits = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrMemoryClockRate, h->device);
    cudaDeviceGetAttribute(&bits, cudaDevAttrGlobalMemoryBusWidth, h->device);
    h->hbm_gbs = khz > 0 && bits > 0 ? 0.8 * 2.0 * (double)khz * 1e3 * (double)bits / 8.0 / 1e9 : 4000.0;
    cudaGetLastError();
    return BNBP_OK;
}

// ---- multi-GPU: summary of a shard on the device, all-reduced over the handle's communicator ----------------
__global__ void summary_kernel(const int32_t* __restrict__ sweeps, const uint8_t* __restrict__ conv, int64_t n,
                               unsigned long long* __restrict__ out)
{
    unsigned long long s = 0, nc = 0, mx = 0, cnt = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long v = (unsigned long long)sweeps[i];
        s += v;
        nc += conv[i] ? 0u : 1u;
        mx = v > mx ? v : mx;
        ++cnt;
    }
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        nc += __shfl_xor_sync(0xffffffffu, nc, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        const unsigned long long m2 = __shfl_xor_sync(0xffffffffu, mx, o);
        mx = m2 > mx ? m2 : mx;
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&out[0], s);
        atomicAdd(&out[1], nc);
        atomicAdd(&out[2], cnt);
        atomicMax(&out[4], mx);
    }
}

int comm_resources(bnbp_handle* h)
{
    if (h->comm_stream) return BNBP_OK;
    CU_TRY(cudaSetDevice(h->device));
    CU_TRY(cudaStreamCreateWithFlags(&h->comm_stream, cudaStreamNonBlocking));
    int rc = h->d_summary.ensure(8 * 8);
    if (rc) return rc;
    CU_TRY(cudaMallocHost((void**)&h->pin_summary, 8 * 8));
    return BNBP_OK;
}

#define NCCL_TRY(expr)                                                                              \
    do {                                                                                            \
        if (!bnbp_nccl::api().load_error.empty()) return fail(BNBP_ERR_CUDA, bnbp_nccl::api().load_error); \
        ncclResult_t r__ = (expr);                                                                  \
        if (r__ != ncclSuccess) return fail(BNBP_ERR_CUDA, std::string(#expr) + ": " + bnbp_nccl::api().GetErrorString(r__)); \
    } while (0)
#define NCCL(fn) bnbp_nccl::api().fn

// enqueue: local reduction of (sweeps, converged) of n cases, then the two all-reduces (sum / max); the totals land
// in h->pin_summary once `st` has drained
int enqueue_summary(bnbp_handle* h, const int32_t* d_sweeps, const uint8_t* d_conv, int64_t n, cudaStream_t st)
{
    unsigned long long* d = (unsigned long long*)h->d_summary.p;
    CU_TRY(cudaMemsetAsync(d, 0, 8 * 8, st));
    if (n > 0) {
        summary_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8), 256, 0, st>>>(d_sweeps, d_conv, n, d);
        CU_TRY(cudaGetLastError());
    }
    if (h->comm && h->comm_world > 1) {
        NCCL_TRY(NCCL(AllReduce)(d, d, 4, ncclUint64, ncclSum, h->comm, st));
        NCCL_TRY(NCCL(AllReduce)(d + 4, d + 4, 1, ncclUint64, ncclMax, h->comm, st));
    }
    return BNBP_OK;
}

// the totals into pinned host memory (its own step: inside an ncclGroupStart / ncclGroupEnd bracket the all-reduces are
// only ENQUEUED at ncclGroupEnd, so a copy issued with them would overtake them -- r02c: a group of two devices
// reported one device's share)
int fetch_summary(bnbp_handle* h, cudaStream_t st)
{
    CU_TRY(cudaMemcpyAsync(h->pin_summary, h->d_summary.p, 8 * 8, cudaMemcpyDeviceToHost, st));
    return BNBP_OK;
}

void read_summary(const bnbp_handle* h, bnbp_summary* out)
{
    out->case_sweeps = h->pin_summary[0];
    out->not_converged = h->pin_summary[1];
    out->n_cases = h->pin_summary[2];
    out->max_sweeps = h->pin_summary[4];
}

void shard_range(int64_t n, int g, int G, int64_t* lo, int64_t* hi)
{
    const int64_t base = n / G, rem = n % G;
    *lo = g * base + std::min<int64_t>(g, rem);
    *hi = *lo + base + (g < rem ? 1 : 0);
}

// Cases one full wave of the sweep grid holds (blocks resident on the 148 SMs x cases per tile).
// The specialised kernels report their occupancy; the generic family is taken at 4 blocks per SM.
int64_t wave_cases(const bnbp_handle* h, const bnbp_run_params& prm)
{
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    int blocks = 4;
    if (h->run_onchip) {
        // persistent grid: one "wave" = 4 rounds of 32 cases on every resident CTA
        int nb = 1;
        for (int i = 0; i < 4; ++i) if (h->oc_state[i] == 1) nb = std::max(nb, h->oc[i].blocks_per_sm);
        return (int64_t)sms * nb * 32 * 4;
    }
    if (h->run_spec) {
        const bool plain = !(prm.epsilon > 0.0) && prm.damping == 0.0;
        const SpecKernel& k = h->spec[plain ? (prm.max_sweeps != 2 ? 0 : 3) : (h->split ? 0 : 2)];
        if (k.blocks_per_sm > 0) blocks = k.blocks_per_sm;
    }
    if (const char* e = getenv("BNBP_WAVE_BLOCKS")) blocks = std::max(1, atoi(e));
    return (int64_t)sms * blocks * h->tb;
}

// Chunk sizes (cases) of the host-buffer call, whole waves each; the last chunk takes the remainder.
// rho = estimated copy time / compute time of a chunk (an upper bound: the compute estimate is the HBM
// floor of the sweeps).  Every chunk boundary costs ~20 dependent-launch drains (0.3 ms on alarm37,
// r01l trace), so the plan is as short as the overlap allows:
//   compute-bound (rho < 0.9): 5 chunks shrinking by ~rho, so each copy hides behind the next chunk's
//                 kernels and the exposed tail copy is the smallest chunk;
//   copy-bound:   a 1-wave and a 2-wave chunk start the copy engine early, the rest goes in 4 chunks.
std::vector<int64_t> plan_chunks(int64_t n, int64_t wave, double rho)
{
    std::vector<int64_t> plan;
    const int64_t W = wave > 0 ? n / wave : 0;
    if (W < 3 || getenv("BNBP_ONE_CHUNK")) { plan.push_back(n); return plan; }
    std::vector<int64_t> w;
    int64_t rest = W;
    double ratio = std::min(0.8, std::max(0.5, rho));
    int k = 5;                                         // r01end sweep, alarm37 fp64: 4 chunks 27.6 ms, 5: 26.9, 6: 27.2, 8: 27.4
    if (rho >= 0.9) {
        if (W >= 10) { w = {1, 2}; rest -= 3; }
        else if (W >= 5) { w = {1}; rest -= 1; }
        ratio = 1.0;
        k = 4;                                         // fp32: 3 chunks after the ramp 20.9 ms, 4: 19.4, 5: 19.5
    }
    if (const char* e = getenv("BNBP_CHUNKS")) k = std::max(1, atoi(e));
    k = (int)std::min<int64_t>(k, rest);
    std::vector<double> ideal((size_t)k);
    double sum = 0.0, term = 1.0;
    for (int i = 0; i < k; ++i, term *= ratio) { ideal[(size_t)i] = term; sum += term; }
    std::vector<int64_t> g((size_t)k);
    int64_t used = 0;
    for (int i = 0; i < k; ++i) {
        ideal[(size_t)i] *= (double)rest / sum;
        g[(size_t)i] = std::max<int64_t>(1, (int64_t)ideal[(size_t)i]);
        used += g[(size_t)i];
    }
    while (used < rest) {                              // largest remainder first
        int best = 0;
        for (int i = 1; i < k; ++i)
            if (ideal[(size_t)i] - (double)g[(size_t)i] > ideal[(size_t)best] - (double)g[(size_t)best]) best = i;
        g[(size_t)best]++; used++;
    }
    while (used > rest) {                              // the floor of 1 wave overshot: take from the largest
        int best = 0;
        for (int i = 1; i < k; ++i) if (g[(size_t)i] > g[(size_t)best]) best = i;
        g[(size_t)best]--; used--;
    }
    w.insert(w.end(), g.begin(), g.end());
    int64_t placed = 0;
    for (int64_t x : w) if (x > 0) { plan.push_back(x * wave); placed += x * wave; }
    plan.back() += n - placed;                         // the fraction of a wave that is left
    return plan;
}

// Chunk sizes for the on-chip kernel, where the kernels of a batch and the copy of its marginals take about the same
// time (alarm37 fp64: 15.2 ms vs 15.4 ms per 1M cases).  With equal rates the copy of chunk i runs beside the kernels of
// chunk i+1 and the call costs T/k + T: EQUAL chunks, as many as the launch overhead allows (14 of two waves each for 1M
// cases).  Measured: the copy-bound plan of the streaming kernels (7 % + 14 % + 4 x 20 %) 19.8 ms per call, a grow-and-shrink
// plan (1 2 3 4 5 4 3 2 1) 20.9 ms -- the copy engine waits while the chunks grow and falls behind when they shrink (r02d, r02i).
std::vector<int64_t> plan_chunks_balanced(int64_t n, int64_t wave)
{
    std::vector<int64_t> plan;
    const int64_t W = wave > 0 ? n / wave : 0;
    if (W < 3 || getenv("BNBP_ONE_CHUNK")) { plan.push_back(n); return plan; }
    int64_t k = std::min<int64_t>(16, (W + 1) / 2);            // two waves per chunk, at most 16 chunks
    if (const char* e = getenv("BNBP_CHUNKS")) k = std::max(1, atoi(e));
    k = std::max<int64_t>(1, std::min(k, W));
    // W whole waves over k chunks, as evenly as they divide (the first W % k chunks get one more); the last chunk also
    // takes the cases beyond the last whole wave (< 1 wave).  (r02j: the remainder of W / k went to the last chunk, which
    // then held half the batch -- 25 ms per call instead of 17.)
    const int64_t base = W / k, extra = W % k;
    for (int64_t i = 0; i < k; ++i) plan.push_back((base + (i < extra ? 1 : 0)) * wave);
    plan.back() += n - W * wave;
    return plan;
}

int check_error_flag(bnbp_handle* h, cudaStream_t st)
{
    // into pinned memory: a device-to-PAGEABLE copy makes the driver itself sleep until the stream has drained
    int32_t* d_error = reinterpret_cast<int32_t*>(h->d_misc.p) + 1;
    h->pinned_poll[3] = 0;
    CU_TRY(cudaMemcpyAsync(&h->pinned_poll[3], d_error, 4, cudaMemcpyDeviceToHost, st));
    CU_TRY(wait_stream(st));
    const int32_t flag = h->pinned_poll[3];
    if (flag) {
        cudaMemsetAsync(d_error, 0, 4, st);
        const char* what = flag == 1 ? "evidence node id out of range"
                         : flag == 2 ? "soft evidence row length != cardinality of the node"
                                     : "hard evidence state out of range";
        return fail(BNBP_ERR_INVALID, what);
    }
    return BNBP_OK;
}

int validate_params(const bnbp_run_params* prm)
{
    if (!prm) return fail(BNBP_ERR_INVALID, "run params are NULL");
    if (std::isnan(prm->epsilon)) return fail(BNBP_ERR_INVALID, "epsilon is NaN");
    if (!(prm->damping >= 0.0 && prm->damping < 1.0)) return fail(BNBP_ERR_INVALID, "damping must be in [0,1)");
    if (prm->semiring != BNBP_SUM_PRODUCT && prm->semiring != BNBP_MAX_PRODUCT) return fail(BNBP_ERR_INVALID, "semiring out of range");
    return BNBP_OK;
}

template <typename T>
int upload_cpt(bnbp_handle* h, const double* cpt, int64_t n)
{
    std::vector<T> tmp((size_t)std::max<int64_t>(n, 1));
    for (int64_t i = 0; i < n; ++i) tmp[(size_t)i] = (T)cpt[i];
    int rc = h->d_cpt.ensure(tmp.size() * sizeof(T));
    if (rc) return rc;
    CU_TRY(cudaMemcpy(h->d_cpt.p, tmp.data(), tmp.size() * sizeof(T), cudaMemcpyHostToDevice));
    // pi of a root starts as the RAW prior row (belief_propagation.hpp:58-64)
    std::vector<T> init((size_t)h->PL, T(1));
    for (int x = 0; x < h->N; ++x)
        if (h->nodes[x].k == 0)
            for (int i = 0; i < h->nodes[x].card; ++i)
                init[(size_t)h->nodes[x].pl_off + i] = (T)cpt[h->nodes[x].cpt_off + i];
    rc = h->d_pl_init.ensure(init.size() * sizeof(T));
    if (rc) return rc;
    CU_TRY(cudaMemcpy(h->d_pl_init.p, init.data(), init.size() * sizeof(T), cudaMemcpyHostToDevice));
    if (h->cpt_t_values > 0) {
        // arena 1: P^T [(uB,x)][uA] of every dense node, the B operand of GEMM 2 (bnbp_dense.h)
        std::vector<T> pt((size_t)h->cpt_t_values);
        for (int x = 0; x < h->N; ++x) {
            if (h->dense_pt_off[x] < 0) continue;
            const NodeMeta& nd = h->nodes[x];
            int64_t QA = 1;
            for (int j = 0; j < nd.dense_s; ++j) QA *= h->e_card[nd.e0 + j];
            const int64_t cptn = (x + 1 < h->N ? h->nodes[x + 1].cpt_off : n) - nd.cpt_off;
            const int64_t QBr = cptn / QA;
            const double* P = cpt + nd.cpt_off;
            T* out = pt.data() + h->dense_pt_off[x];
            for (int64_t ua = 0; ua < QA; ++ua)
                for (int64_t c = 0; c < QBr; ++c) out[c * QA + ua] = (T)P[ua * QBr + c];
        }
        rc = h->d_cpt_t.ensure(pt.size() * sizeof(T));
        if (rc) return rc;
        CU_TRY(cudaMemcpy(h->d_cpt_t.p, pt.data(), pt.size() * sizeof(T), cudaMemcpyHostToDevice));
    }
    if (h->tc_values > 0) {
        // tensor-core jobs: B operands split hi/lo and pre-tiled into the MMA's shared-memory image
        std::vector<float> tc((size_t)h->tc_values);
        for (const bnbp_handle::TcPack& pk : h->tcpack)
            tc_pack_job(tc.data() + pk.out_off, cpt + pk.src_off, pk.K, pk.N, pk.sk, pk.sn);
        rc = h->d_cpt_tc.ensure(tc.size() * sizeof(float));
        if (rc) return rc;
        CU_TRY(cudaMemcpy(h->d_cpt_tc.p, tc.data(), tc.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    return BNBP_OK;
}

// Dense contraction plan (bnbp_dense.h): which nodes meet the batch as matrix products, where their
// parents are split, the GEMM job list (sorted by factor count = one launch per count), the digit
// table that maps an operand row to its factor rows, and the slots of the per-case result tables.
int plan_dense(bnbp_handle* h, const bnbp_flat_network* net, const std::vector<int32_t>& e_pin)
{
    h->djobs.clear(); h->dgroups.clear(); h->dytab.clear(); h->ddig.clear();
    h->tcgroups.clear(); h->tcpack.clear();
    h->tc_values = 0; h->dense_tc_jobs = 0; h->dense_tc_flops_per_case = 0.0;
    h->dense_pt_off.assign(h->N, -1);
    h->TS = 0; h->dense_nodes = 0; h->dense_flops_per_case = 0.0; h->cpt_t_values = 0;
    if (h->dense_min < 0) return BNBP_OK;
    // which products run on the tensor cores (fp32 handles): worth a 256 x 256 CTA tile, factor rows
    // fit next to >= 2 operand stages, pre-tiled arena within 16 GB
    constexpr size_t TC_SMEM_LIMIT = 227 * 1024;                 // opt-in shared memory per CTA, sm_100
    int tc_min_k = 32, tc_min_n = 128;
    if (const char* ev = getenv("BNBP_TC_MIN_K")) tc_min_k = atoi(ev);
    if (const char* ev = getenv("BNBP_TC_MIN_N")) tc_min_n = atoi(ev);
    auto tc_ok = [&](const DenseJob& j) {
        if (h->dense_tc < 0 || h->precision != BNBP_FP32) return false;
        if (tc_stages_for(j.n_rows, TC_SMEM_LIMIT) < 2) return false;
        if (h->tc_values + tc_job_floats(j.K, j.N) > ((int64_t)1 << 32)) return false;
        return h->dense_tc > 0 || (j.K >= tc_min_k && j.N >= tc_min_n);
    };
    std::vector<int> tc_of;                                       // per job: index into tcpack or -1
    int64_t ts = 0;
    std::vector<DenseJob> jobs;
    std::vector<std::vector<unsigned long long>> digs;
    auto make_digits = [&](const DenseJob& jb) {
        const int kpad = (jb.K + DT_K - 1) / DT_K * DT_K + DT_K;       // the kernel prefetches one stage past the end
        std::vector<unsigned long long> d((size_t)kpad);
        std::vector<int> stride(jb.nf), base(jb.nf);
        int st = 1, rows = 0;
        for (int f = jb.nf - 1; f >= 0; --f) { stride[f] = st; st *= jb.f_card[f]; }
        for (int f = 0; f < jb.nf; ++f) { base[f] = rows; rows += jb.f_card[f]; }
        for (int kk = 0; kk < kpad; ++kk) {
            unsigned long long v = 0;
            for (int f = 0; f < jb.nf; ++f) {
                const int row = kk < jb.K ? base[f] + (kk / stride[f]) % jb.f_card[f] : rows;   // rows = the zero row
                v |= (unsigned long long)row << (8 * f);
            }
            d[(size_t)kk] = v;
        }
        return d;
    };
    for (int x = 0; x < h->N; ++x) {
        NodeMeta& nd = h->nodes[x];
        const int k = nd.k, r = nd.card;
        const int64_t cptn = net->cpt_off[x + 1] - net->cpt_off[x];
        if (k == 0 || cptn < h->dense_min || cptn > (int64_t)1 << 30) continue;
        int best_s = -1;
        int64_t best_cost = 0;
        int64_t QA = 1;
        int rowsA = 0, rows_all = r;
        for (int j = 0; j < k; ++j) rows_all += h->e_card[nd.e0 + j];
        for (int s = 1; s <= k; ++s) {
            QA *= h->e_card[nd.e0 + s - 1];
            rowsA += h->e_card[nd.e0 + s - 1];
            const int rowsB = rows_all - rowsA;
            if (s > DENSE_MAXF || k - s + 1 > DENSE_MAXF || rowsA > DENSE_MAXROWS || rowsB > DENSE_MAXROWS) continue;
            const int64_t cost = QA + cptn / QA;              // per-case result slots: QA + QB*r
            if (best_s < 0 || cost < best_cost) { best_s = s; best_cost = cost; }
        }
        if (best_s < 0 || ts + best_cost > (int64_t)1 << 30) continue;
        const int s = best_s;
        QA = 1;
        for (int j = 0; j < s; ++j) QA *= h->e_card[nd.e0 + j];
        const int64_t QBr = cptn / QA;
        nd.dense_s = s;
        nd.t1_off = (int32_t)ts; ts += QBr;
        nd.t2_off = (int32_t)ts; ts += QA;
        DenseJob g1;                                          // T1 = WA x P
        memset(&g1, 0, sizeof g1);
        g1.arena = 0; g1.b_off = nd.cpt_off; g1.K = (int32_t)QA; g1.N = (int32_t)QBr; g1.t_off = nd.t1_off; g1.nf = s;
        for (int j = 0; j < s; ++j) { g1.f_slot[j] = e_pin[nd.e0 + j]; g1.f_card[j] = h->e_card[nd.e0 + j]; g1.n_rows += g1.f_card[j]; }
        DenseJob g2;                                          // T2 = WB x P^T
        memset(&g2, 0, sizeof g2);
        g2.arena = 1; g2.b_off = 0; g2.K = (int32_t)QBr; g2.N = (int32_t)QA; g2.t_off = nd.t2_off; g2.nf = k - s + 1;
        for (int j = s; j < k; ++j) { g2.f_slot[j - s] = e_pin[nd.e0 + j]; g2.f_card[j - s] = h->e_card[nd.e0 + j]; g2.n_rows += g2.f_card[j - s]; }
        g2.f_slot[k - s] = -(nd.pl_off + r + 1);              // lambda_X, fastest digit (x)
        g2.f_card[k - s] = r;
        g2.n_rows += r;
        for (int which = 0; which < 2; ++which) {
            DenseJob& g = which == 0 ? g1 : g2;
            if (tc_ok(g)) {
                // B[k][n]: GEMM 1 reads the reference layout P[uA][(uB,x)] as is, GEMM 2 reads it transposed
                bnbp_handle::TcPack pk;
                pk.src_off = nd.cpt_off; pk.K = g.K; pk.N = g.N; pk.out_off = h->tc_values;
                pk.sk = which == 0 ? g.N : 1; pk.sn = which == 0 ? 1 : g.K;
                g.arena = 2; g.b_off = h->tc_values;
                h->tc_values += tc_job_floats(g.K, g.N);
                tc_of.push_back((int)h->tcpack.size());
                h->tcpack.push_back(pk);
                h->dense_tc_jobs++;
                h->dense_tc_flops_per_case += 2.0 * (double)g.K * (double)g.N;
            } else {
                tc_of.push_back(-1);
                if (which == 1) {                             // CUDA-core GEMM 2 reads a transposed copy (arena 1)
                    h->dense_pt_off[x] = h->cpt_t_values;
                    g.b_off = h->cpt_t_values;
                    h->cpt_t_values += cptn;
                }
            }
            jobs.push_back(g); digs.push_back(make_digits(g));
        }
        h->dense_flops_per_case += 4.0 * (double)cptn;
        h->dense_nodes++;
    }
    h->TS = (int)ts;
    if (jobs.empty()) return BNBP_OK;
    // one launch per factor count (and per 65535 grid rows)
    std::vector<int> order(jobs.size());
    for (size_t i = 0; i < order.size(); ++i) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
        return std::make_pair(jobs[a].nf, -dense_tnt(jobs[a].N)) < std::make_pair(jobs[b].nf, -dense_tnt(jobs[b].N));
    });
    for (int idx : order) {                                   // tensor-core jobs: one launch (nf is a run-time loop there)
        if (tc_of[(size_t)idx] < 0) continue;
        DenseJob jb = jobs[(size_t)idx];
        const int ny = (jb.N + TC_N - 1) / TC_N;
        if (h->tcgroups.empty() || h->tcgroups.back().n_y + ny > 65535)
            h->tcgroups.push_back({0, (int)h->dytab.size(), 0, 0});
        bnbp_handle::TcGroup& g = h->tcgroups.back();
        jb.y0 = g.n_y;
        jb.dig_off = (int64_t)h->ddig.size();
        h->ddig.insert(h->ddig.end(), digs[(size_t)idx].begin(), digs[(size_t)idx].end());
        for (int y = 0; y < ny; ++y) h->dytab.push_back((int32_t)h->djobs.size());
        g.n_y += ny;
        g.max_rows = std::max(g.max_rows, (int)jb.n_rows);
        g.stages = tc_stages_for(g.max_rows, TC_SMEM_LIMIT);
        h->djobs.push_back(jb);
    }
    for (int idx : order) {
        if (tc_of[(size_t)idx] >= 0) continue;
        DenseJob jb = jobs[(size_t)idx];
        const int tnt = dense_tnt(jb.N);
        const int ny = (jb.N + 16 * tnt - 1) / (16 * tnt);
        if (h->dgroups.empty() || h->dgroups.back().nf != jb.nf || h->dgroups.back().tnt != tnt ||
            h->dgroups.back().n_y + ny > 65535)
            h->dgroups.push_back({jb.nf, tnt, 0, (int)h->dytab.size(), 0});
        bnbp_handle::DenseGroup& g = h->dgroups.back();
        jb.y0 = g.n_y;
        jb.dig_off = (int64_t)h->ddig.size();
        h->ddig.insert(h->ddig.end(), digs[(size_t)idx].begin(), digs[(size_t)idx].end());
        for (int y = 0; y < ny; ++y) h->dytab.push_back((int32_t)h->djobs.size());
        g.n_y += ny;
        g.max_rows = std::max(g.max_rows, (int)jb.n_rows);
        h->djobs.push_back(jb);
    }
    return BNBP_OK;
}

// Host-only part of bnbp_create: validation, slot layout, kernel-family choice.  No CUDA calls, so
// bnbp_precompile / bnbp_spec_source can run it on a machine without a GPU.
size_t generic_smem(const bnbp_handle* h)
{
    return (size_t)BLOCK_THREADS * (size_t)h->scratch_vals * h->vec * h->tsize;
}

int build_layout(const bnbp_flat_network* net, const bnbp_options* opt, bnbp_handle* h)
{
    if (!net) return fail(BNBP_ERR_INVALID, "network is NULL");
    const int N = net->n_nodes;
    if (N <= 0 || !net->card || !net->parent_off || !net->cpt_off || !net->cpt)
        return fail(BNBP_ERR_INVALID, "bnbp_create: empty or incomplete network");
    const int E = net->parent_off[N];
    if (net->parent_off[0] != 0 || net->cpt_off[0] != 0 || E < 0 || (E > 0 && !net->parents))
        return fail(BNBP_ERR_INVALID, "bnbp_create: malformed offset arrays");
    h->precision = (opt && opt->precision == BNBP_FP32) ? BNBP_FP32 : BNBP_FP64;
    h->tsize = h->precision == BNBP_FP32 ? 4 : 8;
    h->max_resident = opt ? opt->max_resident_cases : 0;
    h->specialize = opt ? opt->specialize : BNBP_SPEC_AUTO;
    if (const char* ev = getenv("BNBP_SPECIALIZE")) {      // tuning / test knob, overrides the option
        if (!strcmp(ev, "always")) h->specialize = BNBP_SPEC_ALWAYS;
        else if (!strcmp(ev, "never")) h->specialize = BNBP_SPEC_NEVER;
        else if (!strcmp(ev, "auto")) h->specialize = BNBP_SPEC_AUTO;
    }
    h->dense_min = (opt && opt->dense_min_cpt != 0) ? opt->dense_min_cpt : 256;
    h->dense_tc = opt ? opt->dense_tensor : 0;
    h->onchip = opt ? opt->onchip : 0;
    if (h->onchip < -1 || h->onchip > 1) return fail(BNBP_ERR_INVALID, "bnbp_options.onchip out of range");
    if (const char* ev = getenv("BNBP_DENSE_TC")) h->dense_tc = atoi(ev);      // tuning / test knob: -1 never, 1 every product
    if (const char* ev = getenv("BNBP_DENSE_MMA")) h->dense_mma = atoi(ev) != 0;   // tuning knob: 0 = DFMA products
    if (const char* ev = getenv("BNBP_DENSE_MIN")) h->dense_min = atoll(ev);   // tuning / test knob (< 0: never)
    if (h->specialize < BNBP_SPEC_AUTO || h->specialize > BNBP_SPEC_NEVER)
        return fail(BNBP_ERR_INVALID, "bnbp_options.specialize out of range");
    h->N = N;
    h->E = E;
    h->card.assign(net->card, net->card + N);
    h->par_host.assign(net->parents, net->parents + E);

    // ---- validate + derive topology (the checks the reference leaves as UB, graph.hpp:117-124) ----
    int maxcard = 1;
    for (int x = 0; x < N; ++x) {
        if (net->card[x] < 1) return fail(BNBP_ERR_INVALID, "node " + std::to_string(x) + ": cardinality < 1");
        maxcard = std::max(maxcard, (int)net->card[x]);
    }
    h->rmax = pick_rmax(maxcard);
    if (h->rmax < 0) return fail(BNBP_ERR_INVALID, "cardinality > 128 is not supported");
    std::vector<int> nchild(N, 0);
    for (int x = 0; x < N; ++x) {
        const int k = net->parent_off[x + 1] - net->parent_off[x];
        if (k < 0) return fail(BNBP_ERR_INVALID, "parent_off not monotone");
        if (k > KMAX) return fail(BNBP_ERR_INVALID, "node " + std::to_string(x) + ": in-degree > " + std::to_string(KMAX) + " is not supported");
        int64_t Q = 1;
        for (int e = net->parent_off[x]; e < net->parent_off[x + 1]; ++e) {
            const int u = net->parents[e];
            if (u < 0 || u >= N || u == x) return fail(BNBP_ERR_INVALID, "node " + std::to_string(x) + ": bad parent id");
            if (e > net->parent_off[x] && net->parents[e - 1] >= u)
                return fail(BNBP_ERR_INVALID, "node " + std::to_string(x) + ": parents must be strictly ascending");
            Q *= net->card[u];
            nchild[u]++;
        }
        if (net->cpt_off[x + 1] - net->cpt_off[x] != Q * net->card[x])
            return fail(BNBP_ERR_INVALID, "node " + std::to_string(x) + ": CPT size does not match parent configurations (missing rows)");
    }
    {   // DAG check (graph_t::add_edge refuses cycles, graph.hpp:268-275)
        std::vector<int> indeg(N), stack;
        std::vector<std::vector<int>> ch(N);
        for (int x = 0; x < N; ++x) {
            indeg[x] = net->parent_off[x + 1] - net->parent_off[x];
            for (int e = net->parent_off[x]; e < net->parent_off[x + 1]; ++e) ch[net->parents[e]].push_back(x);
            if (!indeg[x]) stack.push_back(x);
        }
        int seen = 0;
        while (!stack.empty()) {
            int u = stack.back(); stack.pop_back(); ++seen;
            for (int c : ch[u]) if (--indeg[c] == 0) stack.push_back(c);
        }
        if (seen != N) return fail(BNBP_ERR_INVALID, "network has a directed cycle");
    }

    // ---- slot layout -------------------------------------------------------------------------------
    // pi/lambda region: [pi_X | lambda_X] per node.  Message buffer: pi-messages in in-edge order
    // (grouped by child), then lambda-messages in out-edge order (grouped by parent), so that
    // everything node X READS is contiguous; what it writes is scattered to its neighbours' blocks.
    h->nodes.resize(N);
    std::vector<int32_t>& e_card = h->e_card;
    std::vector<int32_t>& e_lam_out = h->e_lam_out;
    std::vector<int32_t>& c_pi_out = h->c_pi_out;
    e_card.assign(std::max(E, 1), 0); e_lam_out.assign(std::max(E, 1), 0); c_pi_out.assign(std::max(E, 1), 0);
    std::vector<int32_t> e_pin(std::max(E, 1));      // slot of pi-msg of in-edge e
    int pl = 0, bel = 0, pin = 0;
    for (int x = 0; x < N; ++x) {
        NodeMeta& nd = h->nodes[x];
        nd.card = net->card[x];
        nd.k = net->parent_off[x + 1] - net->parent_off[x];
        nd.m = nchild[x];
        nd.pl_off = pl; pl += 2 * nd.card;
        nd.bel_off = bel; bel += nd.card;
        nd.e0 = net->parent_off[x];
        nd.cpt_off = net->cpt_off[x];
        nd.pin_off = pin;
        nd.scr_half = 0;
        for (int e = nd.e0; e < nd.e0 + nd.k; ++e) {
            e_card[e] = net->card[net->parents[e]];
            e_pin[e] = pin;
            pin += e_card[e];
        }
    }
    h->PL = pl;
    h->V = bel;
    int lin = pin, c0 = 0;
    for (int x = 0; x < N; ++x) {
        h->nodes[x].lin_off = lin; lin += nchild[x] * net->card[x];
        h->nodes[x].c0 = c0; c0 += nchild[x];
    }
    h->M = lin;
    h->W = (N + 31) / 32;
    {   // children in ascending child index (graph_t::out_vertexes scans the adjacency row, graph.hpp:362-386)
        std::vector<int> fill(N, 0);
        for (int x = 0; x < N; ++x)
            for (int e = h->nodes[x].e0; e < h->nodes[x].e0 + h->nodes[x].k; ++e) {
                const int u = net->parents[e];
                const int ci = fill[u]++;
                e_lam_out[e] = h->nodes[u].lin_off + ci * net->card[u];   // X writes lambda-msg here, U reads it
                c_pi_out[h->nodes[u].c0 + ci] = e_pin[e];                 // U writes pi-msg here, X reads it
            }
    }
    for (int x = 0; x < N; ++x) { h->nodes[x].dense_s = 0; h->nodes[x].t1_off = h->nodes[x].t2_off = 0; h->nodes[x].pad_ = 0; }
    {
        // Small networks keep the network-specialised kernel (CPT in the constant bank, everything
        // unrolled): the dense path only takes over by default where specialisation is impossible.
        // An explicit threshold (option or BNBP_DENSE_MIN) is honoured as given.
        h->cpt_values = net->cpt_off[N];
        const bool explicit_dense = (opt && opt->dense_min_cpt != 0) || getenv("BNBP_DENSE_MIN") != nullptr;
        std::string why;
        if (!explicit_dense && h->specialize != BNBP_SPEC_NEVER &&
            spec_eligible(spec_layout(h), h->precision == BNBP_FP32, &why))
            h->dense_min = -1;
        int rc = plan_dense(h, net, e_pin);
        if (rc) return rc;
    }
    // scratch: outer parents' messages + accumulators
    int so_max = 0;
    h->cost_prefix.assign(N + 1, 0.0);
    for (int x = 0; x < N; ++x) {
        const NodeMeta& nd = h->nodes[x];
        int so = 0, sin = 0;
        for (int j = 0; j < nd.k; ++j) { sin += e_card[nd.e0 + j]; if (j < nd.k - 1) so += e_card[nd.e0 + j]; }
        so_max = std::max(so_max, so);
        const double cptn = (double)(net->cpt_off[x + 1] - net->cpt_off[x]);
        // a dense node reads its per-case tables (QA + QB*r coalesced loads) instead of walking the CPT
        double table = 0.5 * cptn;
        if (nd.dense_s) {
            double QA = 1.0;
            for (int j = 0; j < nd.dense_s; ++j) QA *= e_card[nd.e0 + j];
            table = 2.0 * (QA + cptn / QA);
        }
        h->cost_prefix[x + 1] = h->cost_prefix[x] + 2.0 * (2 * nd.card + sin + nd.m * nd.card) + table +
                                (double)nd.m * nd.m * nd.card;
    }
    h->scratch_vals = 2 * so_max;
    for (int x = 0; x < N; ++x) h->nodes[x].scr_half = so_max;
    int kmax = 0;
    for (int x = 0; x < N; ++x) kmax = std::max(kmax, (int)h->nodes[x].k);
    h->knet = kmax <= 2 ? 2 : (kmax <= 4 ? 4 : 8);
    if (h->rmax == 8 && h->knet < 4) h->knet = 4;
    if (h->rmax > 8) h->knet = 8;
    h->vec = (h->rmax <= 4) ? 2 : 1;
    if (const char* ev = getenv("BNBP_VEC")) {           // tuning knob: cases per thread
        const int v = atoi(ev);
        if ((v == 1 || v == 2) && h->rmax <= 8) h->vec = v;
    }
    h->tb = BLOCK_THREADS * h->vec;
    h->cpt_values = net->cpt_off[N];
    if (generic_smem(h) > 200 * 1024) return fail(BNBP_ERR_INVALID, "parent sets too wide for the shared-memory scratch");


    h->cpt_host.assign(net->cpt, net->cpt + net->cpt_off[N]);
    // ---- network-specialised kernel: eligibility and tuning ---------------------------------------
    {
        SpecLayout L = spec_layout(h);
        h->spec_eligible_ = spec_eligible(L, h->precision == BNBP_FP32, &h->spec_why);
        if (h->spec_eligible_ && h->TS > 0) {
            h->spec_eligible_ = false;
            h->spec_why = "the dense contraction path is active for this network";
        }
        // measured on B200 (profiles/r01c): one case per thread beats 2/4 in both precisions -- the
        // kernel is HBM-latency bound, so resident warps (registers per thread) matter more than
        // wider accesses; fp64 1.147 ms/sweep at (1,3,1), fp32 0.620 ms at (1,4,1) for 1M alarm37 cases
        h->spec_vec = 1;
        h->spec_minb = h->precision == BNBP_FP32 ? 4 : 3;
        h->spec_ahead = 1;
        auto env_knobs = [&]() {                       // tuning knobs win over every rule below
            if (const char* ev = getenv("BNBP_SPEC_VEC")) {
                const int v = atoi(ev);
                if (v == 1 || v == 2 || (v == 4 && h->tsize == 4)) h->spec_vec = v;
            }
            if (const char* ev = getenv("BNBP_SPEC_MINB")) h->spec_minb = std::min(16, std::max(1, atoi(ev)));
            if (const char* ev = getenv("BNBP_SPEC_AHEAD")) h->spec_ahead = std::min(4, std::max(0, atoi(ev)));
        };
        env_knobs();
        // What the FIRST use of an unrolled walk costs: NVRTC time grows like N^2.4 with the node count (one variant, measured on
        // the build box: 37 nodes 13 s, 49: 21 s, 64: 44 s, 100: 144 s, 144: 451 s) and a run needs two to four variants.  Above
        // 64 nodes the unrolled kernels are therefore taken only when their cubin is already in the cache (bnbp_precompile, or an
        // earlier ALWAYS run); otherwise the class-looped walk is preferred where the network allows it -- its compile time grows
        // with the CLASS count (10 000-node grid, 6 classes: 3 s; 100-node DAG, 63 classes: 31 s) -- and else the generic kernel.
        constexpr int UNROLL_FAST_NODES = 64;
        const bool static_ok = h->spec_eligible_;
        bool static_slow = false;
        if (static_ok && h->N > UNROLL_FAST_NODES) {
            SpecConfig cfg;
            cfg.fp32 = h->precision == BNBP_FP32;
            cfg.vec = h->spec_vec; cfg.minb = spec_minb_for(h, 0); cfg.variant = 0; cfg.ahead = h->spec_ahead;
            static_slow = !spec_in_cache(spec_source(L, cfg));
        }
        h->spec_auto_ok = true;
        // Class-looped walk (bnbp_spec.cuh, BNBP_CLASSLOOP): networks the unrolled walk refuses for their SIZE -- or would
        // take minutes to compile -- whose nodes fall into few shape classes: one unrolled body per class, looped over the
        // class's nodes (cfg 3: the 10 000-node grid has 6 classes).  BNBP_CLASSLOOP=0 never, 1 (default) where the unrolled
        // walk is refused or slow to compile, 2 wherever possible (the tests run the small networks through both generators).
        {
            int mode = 1;
            if (const char* ev = getenv("BNBP_CLASSLOOP")) mode = atoi(ev);
            h->spec_classloop = false;
            h->spec_classes_n = 0;
            if (mode != 0 && (!static_ok || static_slow || mode >= 2)) {
                std::string why2 = "the dense contraction path is active for this network";
                if (h->TS == 0 && class_eligible(L, h->precision == BNBP_FP32, &why2)) {
                    h->spec_eligible_ = true;
                    h->spec_classloop = true;
                    h->spec_classes_n = (int)spec_classes(L).size();
                    h->spec_why.clear();
                    h->fuse_ok = false;            // K0 / K4 fused into the first / last sweep need the nodes in column order
                } else if (!h->spec_eligible_) {
                    h->spec_why += "; class-looped walk: " + why2;
                }
            }
            if (static_slow && !h->spec_classloop) {
                h->spec_auto_ok = false;
                h->spec_why = "an unrolled walk of " + std::to_string(h->N) + " nodes takes NVRTC minutes and is not in the cubin cache "
                              "(bnbp_precompile or specialize = ALWAYS compiles it once); AUTO keeps the generic kernel";
            }
        }
        // class-looped walks over SMALL nodes (the grid of cfg 3: 20 input values per node, 128 registers) keep one more
        // block per SM resident: 16 warps with a node's loads in flight each instead of 12, and the 512 tiles of the 65 536
        // cases of cfg 3 are ONE wave of 148 x 4 blocks instead of 1.15 waves of 148 x 3
        // Large node classes the other way round: the loop holds the inputs of two nodes, so above ~36 values per node the
        // 168-register cap of 3 blocks per SM spills (168-352 B of stack per thread on 3-4-state nodes with 3-4 parents); at
        // 2 blocks per SM the same classes fit the register file, and a node of that size keeps 40+ rows in flight per warp.
        if (h->spec_classloop) {
            const int inputs = class_max_inputs(L);
            if (inputs <= 24) h->spec_minb = h->precision == BNBP_FP32 ? 5 : 4;
            else if (inputs > 36) h->spec_minb = h->precision == BNBP_FP32 ? 3 : 2;
            env_knobs();
            // the same first-use rule for class-looped walks of MANY classes (~0.5 s of NVRTC per class and variant: 63 classes
            // 31 s): beyond 24 classes AUTO takes them from the cubin cache only
            constexpr int CLASS_FAST_COUNT = 24;
            if (h->spec_classes_n > CLASS_FAST_COUNT) {
                SpecConfig cfg;
                cfg.fp32 = h->precision == BNBP_FP32;
                cfg.vec = h->spec_vec; cfg.minb = spec_minb_for(h, 0); cfg.variant = 0; cfg.ahead = h->spec_ahead;
                cfg.classloop = true;
                if (!spec_in_cache(spec_source(L, cfg))) {
                    h->spec_auto_ok = false;
                    h->spec_why = "a class-looped walk of " + std::to_string(h->spec_classes_n) + " node classes takes NVRTC half a minute per "
                                  "variant and is not in the cubin cache (bnbp_precompile or specialize = ALWAYS compiles it once); "
                                  "AUTO keeps the generic kernel";
                }
            }
        }
        // ---- on-chip kernel: the state of a 32-case group (pi/lambda + both message buffers) must fit the
        //      shared memory of one CTA
        constexpr size_t SMEM_OPTIN = 227 * 1024;
        // warps per group: 6 in fp64 (1 439 M case-sweeps/s on alarm37 against 1 377 M with 4 and 1 398 M with 8, r02i: more
        // warps hide more of the instruction-fetch latency until the busiest role -- node 28 alone is a quarter of the
        // arithmetic -- sets the pace); 4 in fp32, where four groups per SM leave 128 registers per thread
        h->oc_roles = h->precision == BNBP_FP32 ? 4 : 6;
        if (const char* ev = getenv("BNBP_OC_ROLES")) h->oc_roles = std::min(16, std::max(1, atoi(ev)));
        h->oc_ahead = 1;
        if (const char* ev = getenv("BNBP_OC_AHEAD")) h->oc_ahead = std::min(4, std::max(0, atoi(ev)));
        h->oc_smem = onchip_smem_bytes(L, h->precision == BNBP_FP32, h->oc_roles);
        int max_children = 0;
        for (int x = 0; x < h->N; ++x) max_children = std::max(max_children, (int)h->nodes[x].m);
        h->oc_eligible = h->spec_eligible_ && !h->spec_classloop && max_children <= ONCHIP_MREG && h->oc_smem <= SMEM_OPTIN;
        if (!h->spec_eligible_) h->oc_why = h->spec_why;
        else if (h->spec_classloop) h->oc_why = "the network is walked class by class (the on-chip kernel unrolls the walk node by node)";
        else if (max_children > ONCHIP_MREG)
            h->oc_why = "a hub with more than " + std::to_string(ONCHIP_MREG) + " children: its inbox cannot be read before the sweep barrier";
        else if (!h->oc_eligible) h->oc_why = "the state of 32 cases (" + std::to_string(h->oc_smem) + " B) exceeds the shared memory of an SM";
        h->oc_minb = (int)std::max<size_t>(1, std::min<size_t>(8, (228 * 1024) / (h->oc_smem + 1024)));
        if (const char* ev = getenv("BNBP_OC_MINB")) h->oc_minb = std::min(16, std::max(1, atoi(ev)));
        spec_partition(L, h->oc_roles, &h->oc_imbalance);
        // the on-chip kernel is an unrolled walk too (64 nodes: 76 s of NVRTC): same first-use rule
        h->oc_auto_ok = true;
        if (h->oc_eligible && h->N > UNROLL_FAST_NODES) {
            SpecConfig cfg;
            cfg.fp32 = h->precision == BNBP_FP32;
            cfg.vec = 1; cfg.minb = h->oc_minb; cfg.variant = 8; cfg.ahead = h->oc_ahead;
            cfg.roles = h->oc_roles; cfg.out_double = false;
            h->oc_auto_ok = spec_in_cache(spec_source(L, cfg));
        }
    }
    return BNBP_OK;
}

// bnbp_run_batch on a group handle (bnbp_create_multi): contiguous case ranges, one host thread per device, every
// device copies its rows straight into the caller's buffers; then the convergence summary is all-reduced over the
// group's communicator (one grouped NCCL call from this thread).
int run_group(bnbp_handle* g, const bnbp_evidence* ev, const bnbp_run_params* prm, void* out_marginals, int32_t* out_sweeps,
              uint8_t* out_converged)
{
    if (ev->n_cases < 0) return fail(BNBP_ERR_INVALID, "n_cases < 0");
    if (ev->n_cases > 0 && !ev->ev_off) return fail(BNBP_ERR_INVALID, "ev_off is NULL");
    const int G = (int)g->members.size();
    std::vector<int32_t> q, belcol, colmap;
    int rc = query_columns(g, *prm, &q, &belcol, &colmap);
    if (rc) return rc;
    const size_t row_bytes = colmap.size() * (prm->out_precision == BNBP_OUT_FP32 ? 4 : 8);
    std::vector<int> rcs((size_t)G, BNBP_OK);
    std::vector<std::string> errs((size_t)G);
    std::vector<int64_t> lo((size_t)G), hi((size_t)G);
    for (int i = 0; i < G; ++i) shard_range(ev->n_cases, i, G, &lo[(size_t)i], &hi[(size_t)i]);
    auto work = [&](int i) {
        bnbp_evidence e = *ev;
        e.n_cases = hi[(size_t)i] - lo[(size_t)i];
        e.ev_off = ev->ev_off ? ev->ev_off + lo[(size_t)i] : nullptr;
        rcs[(size_t)i] = bnbp_run_batch(g->members[(size_t)i], &e, prm, (char*)out_marginals + (size_t)lo[(size_t)i] * row_bytes,
                                        out_sweeps ? out_sweeps + lo[(size_t)i] : nullptr,
                                        out_converged ? out_converged + lo[(size_t)i] : nullptr);
        if (rcs[(size_t)i]) errs[(size_t)i] = bnbp_last_error();      // the error channel is thread-local
    };
    std::vector<std::thread> threads;
    for (int i = 1; i < G; ++i) threads.emplace_back(work, i);
    work(0);
    for (std::thread& t : threads) t.join();
    for (int i = 0; i < G; ++i)
        if (rcs[(size_t)i]) return fail(rcs[(size_t)i], "device " + std::to_string(g->members[(size_t)i]->device) + ": " + errs[(size_t)i]);
    // summary: per-case counts are still on each device (whole-shard staging of bnbp_run_batch)
    NCCL_TRY(NCCL(GroupStart)());
    for (int i = 0; i < G; ++i) {
        bnbp_handle* m = g->members[(size_t)i];
        CU_TRY(cudaSetDevice(m->device));
        const int64_t n = hi[(size_t)i] - lo[(size_t)i];
        if ((rc = enqueue_summary(m, (const int32_t*)m->s_out_sweeps.p, (const uint8_t*)m->s_out_conv.p, n, m->stream))) {
            NCCL(GroupEnd)();
            return rc;
        }
    }
    NCCL_TRY(NCCL(GroupEnd)());
    for (int i = 0; i < G; ++i) {
        CU_TRY(cudaSetDevice(g->members[(size_t)i]->device));
        if ((rc = fetch_summary(g->members[(size_t)i], g->members[(size_t)i]->stream))) return rc;
        CU_TRY(wait_stream(g->members[(size_t)i]->stream));
    }
    read_summary(g->members[0], &g->last_summary);
    g->last_case_sweeps = g->last_summary.case_sweeps;
    return BNBP_OK;
}

} // namespace

// =================================================================================================
extern "C" {

const char* bnbp_last_error(void) { return g_err.c_str(); }

int bnbp_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int bnbp_create(const bnbp_flat_network* net, const bnbp_options* opt, bnbp_handle** out)
{
    if (!net || !out) return fail(BNBP_ERR_INVALID, "bnbp_create: NULL argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(BNBP_ERR_NO_DEVICE, "no CUDA device: libbnbp has no CPU fallback");
    }
    int dev = opt ? opt->device : -1;
    if (dev < 0) CU_TRY(cudaGetDevice(&dev));
    if (dev >= ndev) return fail(BNBP_ERR_INVALID, "bnbp_create: device ordinal out of range");
    CU_TRY(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10)
        return fail(BNBP_ERR_NO_DEVICE, std::string("device ") + prop.name + " is not sm_100: kernels are built for sm_100a only");

    // a failed create releases what it had allocated (device buffers, streams, events)
    struct Destroy { void operator()(bnbp_handle* p) const { bnbp_destroy(p); } };
    std::unique_ptr<bnbp_handle, Destroy> h(new bnbp_handle());
    h->device = dev;
    int rc = build_layout(net, opt, h.get());
    if (rc) return rc;
    const int N = h->N, E = h->E;
    const std::vector<int32_t>& e_card = h->e_card;
    const std::vector<int32_t>& e_lam_out = h->e_lam_out;
    const std::vector<int32_t>& c_pi_out = h->c_pi_out;
    const size_t smem = generic_smem(h.get());

    // ---- upload -------------------------------------------------------------------------------------
    if ((rc = h->d_nodes.ensure(sizeof(NodeMeta) * N))) return rc;
    CU_TRY(cudaMemcpy(h->d_nodes.p, h->nodes.data(), sizeof(NodeMeta) * N, cudaMemcpyHostToDevice));
    const size_t eb = sizeof(int32_t) * std::max(E, 1);
    if ((rc = h->d_e_card.ensure(eb)) || (rc = h->d_e_lam_out.ensure(eb)) || (rc = h->d_c_pi_out.ensure(eb))) return rc;
    CU_TRY(cudaMemcpy(h->d_e_card.p, e_card.data(), eb, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(h->d_e_lam_out.p, e_lam_out.data(), eb, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(h->d_c_pi_out.p, c_pi_out.data(), eb, cudaMemcpyHostToDevice));
    rc = h->precision == BNBP_FP32 ? upload_cpt<float>(h.get(), net->cpt, net->cpt_off[N])
                                   : upload_cpt<double>(h.get(), net->cpt, net->cpt_off[N]);
    if (rc) return rc;
    if (h->TS > 0) {
        if ((rc = h->d_djobs.ensure(h->djobs.size() * sizeof(DenseJob))) || (rc = h->d_dytab.ensure(h->dytab.size() * 4)) ||
            (rc = h->d_ddig.ensure(h->ddig.size() * 8)))
            return rc;
        CU_TRY(cudaMemcpy(h->d_djobs.p, h->djobs.data(), h->djobs.size() * sizeof(DenseJob), cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(h->d_dytab.p, h->dytab.data(), h->dytab.size() * 4, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(h->d_ddig.p, h->ddig.data(), h->ddig.size() * 8, cudaMemcpyHostToDevice));
        int max_rows = 0;
        for (const bnbp_handle::DenseGroup& g : h->dgroups) max_rows = std::max(max_rows, g.max_rows);
        const int bytes = (int)dense_smem_bytes(max_rows, 8, h->tsize);
        cudaError_t e = h->precision == BNBP_FP32 ? set_dense_smem<float>(bytes) : set_dense_smem<double>(bytes);
        if (e != cudaSuccess) return fail(BNBP_ERR_CUDA, std::string("dense shared-memory opt-in: ") + cudaGetErrorString(e));
        int tc_bytes = 0;
        for (const bnbp_handle::TcGroup& g : h->tcgroups) tc_bytes = std::max(tc_bytes, (int)tc_smem_bytes(g.max_rows, g.stages));
        if (tc_bytes > 0 && (e = set_dense_tc_smem(tc_bytes)) != cudaSuccess)
            return fail(BNBP_ERR_CUDA, std::string("tensor-core dense shared-memory opt-in: ") + cudaGetErrorString(e));
    }
    if ((rc = h->d_misc.ensure(64))) return rc;
    CU_TRY(cudaMemset(h->d_misc.p, 0, 64));
    CU_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        CU_TRY(cudaEventCreate(&h->ev_total[i]));
        CU_TRY(cudaEventCreateWithFlags(&h->ev_poll[i], cudaEventDisableTiming));
    }
    CU_TRY(cudaMallocHost((void**)&h->pinned_poll, 4 * sizeof(int32_t)));
    // opt in to the dynamic shared memory the scratch needs
    if (smem > 48 * 1024) {
        cudaError_t e = h->precision == BNBP_FP32 ? set_smem<float>(h.get(), (int)smem) : set_smem<double>(h.get(), (int)smem);
        if (e != cudaSuccess) return fail(BNBP_ERR_CUDA, std::string("shared-memory opt-in: ") + cudaGetErrorString(e));
    }
    {   // the default output layout (every node): device tables exist before any communicator does
        bnbp_run_params all_nodes;
        memset(&all_nodes, 0, sizeof all_nodes);
        if ((rc = set_query(h.get(), all_nodes))) return rc;
    }
    *out = h.release();
    return BNBP_OK;
}

void bnbp_destroy(bnbp_handle* h)
{
    if (!h) return;
    if (!h->members.empty()) {            // a group handle owns its members; it holds no device state itself
        for (bnbp_handle* m : h->members) bnbp_destroy(m);
        delete h;
        return;
    }
    cudaSetDevice(h->device);
    // ncclCommAbort, not ncclCommDestroy: destroying flushes the communicator WITH the peers and blocks until they join,
    // so a rank that leaves early (an error, an exception unwinding through the handle) would hang instead of exiting
    if (h->comm) { if (h->stream) cudaStreamSynchronize(h->stream); NCCL(CommAbort)(h->comm); h->comm = nullptr; }
    if (h->comm_stream) { cudaStreamSynchronize(h->comm_stream); cudaStreamDestroy(h->comm_stream); }
    for (cudaEvent_t e : h->ev_comm) cudaEventDestroy(e);
    if (h->pin_summary) cudaFreeHost(h->pin_summary);
    for (DevBuf* b : {&h->d_belcol, &h->d_colmap, &h->s_full, &h->d_summary}) b->release();
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (DevBuf* b : {&h->d_nodes, &h->d_e_card, &h->d_e_lam_out, &h->d_c_pi_out, &h->d_cpt, &h->d_pl_init, &h->d_pl,
                      &h->d_msg[0], &h->d_msg[1], &h->d_evbits, &h->d_delta, &h->d_status, &h->d_sweeps, &h->d_misc,
                      &h->d_pl2, &h->d_msg2[0], &h->d_msg2[1], &h->d_evbits2, &h->d_orig[0], &h->d_orig[1], &h->d_src_pos, &h->d_tile_count,
                      &h->d_evst, &h->d_lw_order, &h->d_lw_par, &h->d_lw_cpt, &h->d_lw_out, &h->d_lw_wsum, &h->d_djobs, &h->d_dytab, &h->d_ddig, &h->d_cpt_t, &h->d_tscr,
                      &h->s_ev_off, &h->s_ev_node, &h->s_ev_state, &h->s_ev_val_off, &h->s_ev_values, &h->s_out[0], &h->s_out[1], &h->s_out_all,
                      &h->s_out_sweeps, &h->s_out_conv})
        b->release();
    for (auto& kv : h->belief_plans) kv.second.groups.release();
    for (cudaEvent_t e : h->ev_chunk) cudaEventDestroy(e);
    if (h->copy_stream) { cudaStreamSynchronize(h->copy_stream); cudaStreamDestroy(h->copy_stream); }
    if (h->h2d_stream) { cudaStreamSynchronize(h->h2d_stream); cudaStreamDestroy(h->h2d_stream); }
    for (int v = 0; v < bnbp_handle::NSPEC; ++v) spec_unload(&h->spec[v]);
    for (int v = 0; v < 4; ++v) spec_unload(&h->oc[v]);
    for (cudaEvent_t e : h->ev_sweep) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_dense) cudaEventDestroy(e);
    for (int i = 0; i < 2; ++i) {
        if (h->ev_total[i]) cudaEventDestroy(h->ev_total[i]);
        if (h->ev_poll[i]) cudaEventDestroy(h->ev_poll[i]);
    }
    if (h->pinned_poll) cudaFreeHost(h->pinned_poll);
    if (h->pin_counts) cudaFreeHost(h->pin_counts);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int bnbp_refresh_cpt(bnbp_handle* h, const double* cpt, int64_t n_values)
{
    if (!h || !cpt) return fail(BNBP_ERR_INVALID, "bnbp_refresh_cpt: NULL argument");
    if (n_values != h->cpt_values) return fail(BNBP_ERR_INVALID, "bnbp_refresh_cpt: CPT size changed (topology edits need a new handle)");
    if (!h->members.empty()) {
        for (bnbp_handle* m : h->members) {
            const int rc = bnbp_refresh_cpt(m, cpt, n_values);
            if (rc) return rc;
        }
        return BNBP_OK;
    }
    CU_TRY(cudaSetDevice(h->device));
    CU_TRY(cudaDeviceSynchronize());          // runs may have been enqueued on caller streams
    h->cpt_host.assign(cpt, cpt + n_values);
    h->lw_ready = false;                      // the fp64 arena of the likelihood-weighting kernel is re-uploaded on next use
    for (int v = 0; v < bnbp_handle::NSPEC; ++v) {             // constant banks of the loaded specialised kernels
        if (h->spec_state[v] != 1) continue;
        std::string err;
        bool ok;
        if (h->precision == BNBP_FP32) {
            std::vector<float> tmp(h->cpt_host.begin(), h->cpt_host.end());
            ok = spec_upload_cpt(h->spec[v], tmp.data(), tmp.size() * 4, &err);
        } else {
            ok = spec_upload_cpt(h->spec[v], h->cpt_host.data(), h->cpt_host.size() * 8, &err);
        }
        if (!ok) return fail(BNBP_ERR_CUDA, err);
    }
    for (int v = 0; v < 4; ++v) {
        if (h->oc_state[v] != 1) continue;
        std::string err;
        bool ok;
        if (h->precision == BNBP_FP32) {
            std::vector<float> tmp(h->cpt_host.begin(), h->cpt_host.end());
            ok = spec_upload_cpt(h->oc[v], tmp.data(), tmp.size() * 4, &err);
        } else {
            ok = spec_upload_cpt(h->oc[v], h->cpt_host.data(), h->cpt_host.size() * 8, &err);
        }
        if (!ok) return fail(BNBP_ERR_CUDA, err);
    }
    return h->precision == BNBP_FP32 ? upload_cpt<float>(h, cpt, n_values) : upload_cpt<double>(h, cpt, n_values);
}

int bnbp_precompile(const bnbp_flat_network* net, const bnbp_options* opt, int32_t variant_mask)
{
    bnbp_handle h;
    int rc = build_layout(net, opt, &h);
    if (rc) return rc;
    if (!h.spec_eligible_) return fail(BNBP_ERR_INVALID, "network is not eligible for specialisation: " + h.spec_why);
    for (int idx = 0; idx < 4; ++idx) {                           // bits 8..11: the on-chip kernels
        if (!(variant_mask & (1 << (8 + idx)))) continue;
        if ((idx & 1) && h.precision != BNBP_FP32) continue;
        if (!h.oc_eligible) return fail(BNBP_ERR_INVALID, "network is not eligible for the on-chip kernel: " + h.oc_why);
        SpecConfig cfg;
        cfg.fp32 = h.precision == BNBP_FP32;
        cfg.vec = 1; cfg.minb = h.oc_minb; cfg.variant = 8 + (idx >> 1); cfg.ahead = h.oc_ahead;
        cfg.roles = h.oc_roles; cfg.out_double = (idx & 1) != 0;
        std::vector<char> cubin;
        std::string err;
        if (!spec_compile(spec_source(spec_layout(&h), cfg), &cubin, nullptr, nullptr, &err)) return fail(BNBP_ERR_CUDA, err);
    }
    for (int v = 0; v < bnbp_handle::NSPEC; ++v) {
        if (!(variant_mask & (1 << v))) continue;
        if (v == 7 && h.precision != BNBP_FP32) continue;     // marginals in double from a float kernel only
        if (v > 4 && h.spec_classloop) continue;              // no K0 / K4 fusion in a class-looped walk
        SpecConfig cfg;
        cfg.fp32 = h.precision == BNBP_FP32;
        cfg.vec = h.spec_vec; cfg.minb = spec_minb_for(&h, v); cfg.variant = v; cfg.ahead = h.spec_ahead;
        cfg.classloop = h.spec_classloop;
        std::vector<char> cubin;
        std::string err;
        if (!spec_compile(spec_source(spec_layout(&h), cfg), &cubin, nullptr, nullptr, &err)) return fail(BNBP_ERR_CUDA, err);
    }
    return BNBP_OK;
}

int bnbp_spec_source(const bnbp_flat_network* net, const bnbp_options* opt, int32_t variant, char* buf, int64_t cap,
                     int64_t* needed)
{
    if (variant < 0 || variant > 9) return fail(BNBP_ERR_INVALID, "variant must be 0..9");
    bnbp_handle h;
    int rc = build_layout(net, opt, &h);
    if (rc) return rc;
    if (!h.spec_eligible_) return fail(BNBP_ERR_INVALID, "network is not eligible for specialisation: " + h.spec_why);
    SpecConfig cfg;
    cfg.fp32 = h.precision == BNBP_FP32;
    cfg.vec = h.spec_vec; cfg.minb = spec_minb_for(&h, variant); cfg.variant = variant; cfg.ahead = h.spec_ahead;
    cfg.classloop = h.spec_classloop;
    if (cfg.classloop && variant > 4) return fail(BNBP_ERR_INVALID, "a class-looped walk has variants 0-4 only");
    if (variant >= 8) {
        if (!h.oc_eligible) return fail(BNBP_ERR_INVALID, "network is not eligible for the on-chip kernel: " + h.oc_why);
        cfg.vec = 1; cfg.minb = h.oc_minb; cfg.ahead = h.oc_ahead; cfg.roles = h.oc_roles;
    }
    const std::string src = spec_source(spec_layout(&h), cfg);
    if (needed) *needed = (int64_t)src.size() + 1;
    if (buf && cap > 0) {
        const size_t n = std::min<size_t>(src.size(), (size_t)cap - 1);
        memcpy(buf, src.data(), n);
        buf[n] = 0;
    }
    return BNBP_OK;
}

int bnbp_run_batch_device(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm, void* out_marginals,
                          int32_t* out_sweeps, uint8_t* out_converged, void* stream)
{
    if (!h || !ev || !out_marginals) return fail(BNBP_ERR_INVALID, "bnbp_run_batch_device: NULL argument");
    NvtxRange nvtx_call("bnbp_run_batch_device");
    int rc = validate_params(prm);
    if (rc) return rc;
    if (ev->n_cases < 0) return fail(BNBP_ERR_INVALID, "n_cases < 0");
    if (ev->n_cases > 0 && !ev->ev_off) return fail(BNBP_ERR_INVALID, "ev_off is NULL");
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    h->last_sweep_launches = h->last_kernel_launches = h->last_dense_launches = h->last_dense_tc_launches = 0;
    h->last_case_sweeps = 0;
    h->ev_sweep_used = 0;
    h->ev_dense_used = 0;
    h->last_compactions = 0;
    if (ev->n_cases == 0) return BNBP_OK;
    if (!h->members.empty()) return fail(BNBP_ERR_INVALID, "bnbp_run_batch_device: a group handle takes host buffers (bnbp_run_batch); the device path belongs to one device");
    if ((rc = set_query(h, *prm))) return rc;
    if ((rc = choose_kernels(h, ev->n_cases, *prm, ev->ev_values != nullptr, h->precision != BNBP_FP32))) return rc;
    if (!h->run_onchip && (rc = ensure_state(h, ev->n_cases))) return rc;
    // a flag left by an earlier (unchecked, asynchronous) run must not fail this one
    CU_TRY(cudaMemsetAsync(reinterpret_cast<int32_t*>(h->d_misc.p) + 1, 0, 4, st));
    CU_TRY(cudaEventRecord(h->ev_total[0], st));
    bool exact = true;
    const size_t row_bytes = (size_t)h->Vout * h->tsize;
    // gather (SURVEY 8e): out_marginals is [world][n_cases][row]; this rank's kernels write straight into its slot
    // and every chunk travels to the peers behind the kernels of the next chunk
    const bool gather = prm->gather != 0;
    if (gather && (!h->comm || h->comm_world < 1)) return fail(BNBP_ERR_INVALID, "gather needs a communicator (bnbp_comm_init)");
    const bool exchange = gather && h->comm_world > 1;
    // SMs left to the exchange while the on-chip grid runs: 8 per peer, at most 32 (N = 4: 18.2 ms per step with 0-12
    // SMs, 17.4 with 32, 15.8 without the exchange, r02g / r02h)
    h->reserve_sms = 0;
    if (exchange) {
        h->reserve_sms = std::min(32, 8 * (h->comm_world - 1));
        if (const char* e = getenv("BNBP_GATHER_SMS")) h->reserve_sms = std::max(0, atoi(e));
    }
    char* const base = (char*)out_marginals;
    char* const mine = base + (gather ? (size_t)h->comm_rank * (size_t)ev->n_cases * row_bytes : 0);
    int64_t step_cases = h->run_onchip ? ev->n_cases : h->cap;            // on chip: no resident state arena, one launch
    if (exchange) {
        // 8 chunks of >= 8 MB each when the batch allows it: the exchange of chunk i hides behind the kernels of chunk
        // i+1, so what stays exposed is the last chunk's -- 1/8 of (world-1)/world x the marginals over NVLink
        const int64_t min_cases = std::max<int64_t>(32, (int64_t)((8u << 20) / std::max<size_t>(1, row_bytes)));
        int64_t per = std::max(min_cases, (ev->n_cases + 7) / 8);
        per = (per + 31) / 32 * 32;
        step_cases = std::min(step_cases, per);
    }
    int n_chunk = 0;
    for (int64_t c0 = 0; c0 < ev->n_cases; c0 += step_cases, ++n_chunk) {
        const int64_t n = std::min<int64_t>(step_cases, ev->n_cases - c0);
        DevEvidence de{ev->ev_off + c0, 0, ev->ev_node, ev->ev_state, ev->ev_val_off, ev->ev_values, 0};
        int64_t planned = 0;
        char* const dst = mine + (size_t)c0 * row_bytes;
        if (h->precision == BNBP_FP32)
            rc = run_any<float, float>(h, n, de, *prm, (float*)dst, out_sweeps ? out_sweeps + c0 : nullptr,
                                       out_converged ? out_converged + c0 : nullptr, st, &planned);
        else
            rc = run_any<double, double>(h, n, de, *prm, (double*)dst, out_sweeps ? out_sweeps + c0 : nullptr,
                                         out_converged ? out_converged + c0 : nullptr, st, &planned);
        if (rc) return rc;
        if (planned < 0) exact = false; else h->last_case_sweeps += planned;
        if (exchange) {
            while ((int)h->ev_comm.size() < n_chunk + 2) {
                cudaEvent_t e;
                CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                h->ev_comm.push_back(e);
            }
            CU_TRY(cudaEventRecord(h->ev_comm[(size_t)n_chunk + 1], st));
        }
    }
    if (exchange) {
        // the collectives are enqueued AFTER all the kernels: an ncclGroupEnd costs the host ~0.1 ms, and issued between
        // two chunks it left the compute stream empty for that long, eight times per batch (r02g: the exchange cost its
        // full serial time whatever the SM split).  Each group waits for the event of its chunk on the library's own stream.
        int i = 0;
        for (int64_t c0 = 0; c0 < ev->n_cases; c0 += step_cases, ++i) {
            const int64_t n = std::min<int64_t>(step_cases, ev->n_cases - c0);
            CU_TRY(cudaStreamWaitEvent(h->comm_stream, h->ev_comm[(size_t)i + 1], 0));
            NCCL_TRY(NCCL(GroupStart)());
            for (int r = 0; r < h->comm_world; ++r) {
                char* const slot = base + ((size_t)r * (size_t)ev->n_cases + (size_t)c0) * row_bytes;
                NCCL_TRY(NCCL(Broadcast)(slot, slot, (size_t)n * h->Vout, h->tsize == 4 ? ncclFloat : ncclDouble, r, h->comm, h->comm_stream));
            }
            NCCL_TRY(NCCL(GroupEnd)());
        }
        // whatever follows on `st` sees every rank's rows
        CU_TRY(cudaEventRecord(h->ev_comm[0], h->comm_stream));
        CU_TRY(cudaStreamWaitEvent(st, h->ev_comm[0], 0));
    }
    if (!exact) h->last_case_sweeps = -1;
    CU_TRY(cudaEventRecord(h->ev_total[1], st));
    h->total_recorded = true;
    // epsilon mode has synchronised with the host already (termination census): report malformed evidence now.
    // Fixed-count runs stay asynchronous; the caller asks with bnbp_check_errors once it has synchronised.
    if (prm->epsilon > 0.0) return check_error_flag(h, st);
    return BNBP_OK;
}

int bnbp_check_errors(bnbp_handle* h, void* stream)
{
    if (!h) return fail(BNBP_ERR_INVALID, "bnbp_check_errors: NULL handle");
    if (!h->members.empty()) return fail(BNBP_ERR_INVALID, "bnbp_check_errors: a group handle has no device path");
    CU_TRY(cudaSetDevice(h->device));
    return check_error_flag(h, stream ? (cudaStream_t)stream : h->stream);
}

int bnbp_run_batch(bnbp_handle* h, const bnbp_evidence* ev, const bnbp_run_params* prm, void* out_marginals_v,
                   int32_t* out_sweeps, uint8_t* out_converged)
{
    if (!h || !ev || !out_marginals_v) return fail(BNBP_ERR_INVALID, "bnbp_run_batch: NULL argument");
    const auto t_entry = std::chrono::steady_clock::now();
    NvtxRange nvtx_call("bnbp_run_batch (host buffers: H2D evidence | kernels | D2H marginals, pipelined by chunk)");
    int rc = validate_params(prm);
    if (rc) return rc;
    if (!h->members.empty()) return run_group(h, ev, prm, out_marginals_v, out_sweeps, out_converged);
    const bool out_f32 = prm->out_precision == BNBP_OUT_FP32;
    if (out_f32 && h->precision != BNBP_FP32)
        return fail(BNBP_ERR_INVALID, "out_precision FP32 needs an fp32 handle (an fp64 handle returns the reference's doubles)");
    if (prm->out_precision < BNBP_OUT_DEFAULT || prm->out_precision > BNBP_OUT_FP32) return fail(BNBP_ERR_INVALID, "out_precision out of range");
    char* const out_marginals = (char*)out_marginals_v;
    if (ev->n_cases < 0) return fail(BNBP_ERR_INVALID, "n_cases < 0");
    if (ev->n_cases > 0 && !ev->ev_off) return fail(BNBP_ERR_INVALID, "ev_off is NULL");
    const int64_t nnz = ev->n_cases ? ev->ev_off[ev->n_cases] : 0;
    if (nnz > 0 && !ev->ev_node) return fail(BNBP_ERR_INVALID, "ev_node is NULL");
    const bool soft = ev->ev_values != nullptr;
    if (nnz > 0 && !soft && !ev->ev_state) return fail(BNBP_ERR_INVALID, "neither ev_state nor ev_values given");
    if (soft && !ev->ev_val_off) return fail(BNBP_ERR_INVALID, "ev_val_off is NULL");
    if (soft && ev->ev_val_off[nnz] < ev->ev_val_off[0]) return fail(BNBP_ERR_INVALID, "ev_val_off not monotone");
    if (ev->n_cases > 0 && (ev->ev_off[0] < 0 || nnz < ev->ev_off[0])) return fail(BNBP_ERR_INVALID, "ev_off not monotone");
    // (the per-case monotonicity check runs chunk by chunk below, while the device works on the chunk before)
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    h->last_sweep_launches = h->last_kernel_launches = h->last_dense_launches = h->last_dense_tc_launches = 0;
    h->last_case_sweeps = 0;
    h->ev_sweep_used = 0;
    h->ev_dense_used = 0;
    h->last_compactions = 0;
    if (ev->n_cases == 0) return BNBP_OK;
    h->reserve_sms = 0;
    if ((rc = set_query(h, *prm))) return rc;
    if ((rc = choose_kernels(h, ev->n_cases, *prm, soft, !out_f32))) return rc;
    if ((rc = measure_rates(h))) return rc;
    // Chunk pipeline on three streams: evidence of chunk i+1 goes up (h2d_stream) and the marginals of
    // chunk i-1 come down (copy_stream) while init/sweeps/beliefs of chunk i run.  Marginals are 8*V
    // bytes per case, so the copy is of the same order as the kernels.  plan_chunks() cuts the batch
    // in whole waves of the sweep grid (a 2.3-wave grid pays for 3, r01g/r01k traces): short chunks
    // first so the copy engine starts early, then chunks shrinking by 0.7 down to one wave so the
    // exposed tail copy is short.
    const int64_t wave = wave_cases(h, *prm);
    // copy over the host link vs the sweeps at the HBM floor (2*S*sizeof(T) bytes per case-sweep); both rates
    // are measured on this handle's device (measure_rates), not assumed
    const double sweeps_est = prm->epsilon > 0.0 ? (double)std::min(prm->max_sweeps > 0 ? prm->max_sweeps : 20, 20) : (double)prm->max_sweeps;
    const size_t out_elem = out_f32 ? 4 : 8;
    double rho = ((double)h->Vout * (double)out_elem / (h->link_gbs * 1e9)) /
                 std::max(1e-12, sweeps_est * 2.0 * (double)(h->PL + h->M) * (double)h->tsize / (h->hbm_gbs * 1e9));
    if (h->run_onchip) rho = 1.0;                          // the kernel moves ~1 KB per case: kernels and copy take about the same time
    std::vector<int64_t> plan;
    if (h->run_onchip) {
        // equal chunks (plan_chunks_balanced); BNBP_OC_PLAN=ramp (tuning knob): the copy-bound plan of the streaming kernels
        const char* mode = getenv("BNBP_OC_PLAN");
        plan = (mode && !strcmp(mode, "ramp")) ? plan_chunks(ev->n_cases, 2 * wave, 2.0) : plan_chunks_balanced(ev->n_cases, wave);
    } else {
        plan = plan_chunks(ev->n_cases, wave, rho);
    }
    if (prm->epsilon > 0.0 && plan.size() > 2 && !getenv("BNBP_CHUNKS") && !h->run_onchip) {
        // eps mode: the host waits inside every chunk (termination census), so chunks do not overlap each
        // other's kernels, only the copy of the chunk before; two chunks (~60/40 in whole waves) keep the
        // grids long and expose the copy of the smaller one only (4 chunks: 57.5 ms, r01fin)
        const int64_t W = ev->n_cases / wave;
        const int64_t first = std::max<int64_t>(1, (W * 3 + 2) / 5) * wave;
        plan = {first, ev->n_cases - first};
    }
    int64_t chunk = *std::max_element(plan.begin(), plan.end());
    if (!h->run_onchip && (rc = ensure_state(h, chunk))) return rc;
    if (!h->run_onchip && h->cap < chunk) {               // HBM cannot hold the planned chunk: equal resident chunks
        chunk = h->cap;
        plan.assign((size_t)((ev->n_cases + chunk - 1) / chunk), chunk);
    }
    // Output staging: the whole batch when HBM has the room (no chunk ever waits for a slot),
    // else a ring of two chunk-sized slots.
    const size_t row_bytes = (size_t)h->Vout * out_elem;
    bool whole = (size_t)ev->n_cases * row_bytes <= h->s_out_all.bytes;
    if (!whole && !getenv("BNBP_STAGING_RING")) {
        size_t free_b = 0, total_b = 0;
        CU_TRY(cudaMemGetInfo(&free_b, &total_b));
        whole = (double)ev->n_cases * (double)row_bytes <= 0.5 * (double)(free_b + h->s_out[0].bytes + h->s_out[1].bytes);
        if (whole) {
            h->s_out[0].release(); h->s_out[1].release();
            if ((rc = h->s_out_all.ensure((size_t)ev->n_cases * row_bytes))) return rc;
        }
    }
    if (!whole)
        for (int i = 0; i < 2; ++i)
            if ((rc = h->s_out[i].ensure((size_t)chunk * row_bytes))) return rc;
    // per-case sweep counts / flags stay on the device until the end: the caller's arrays are usually
    // pageable, and a pageable D2H per chunk would block the host and serialise the pipeline
    if ((rc = h->s_out_sweeps.ensure((size_t)ev->n_cases * 4))) return rc;
    if ((rc = h->s_out_conv.ensure((size_t)ev->n_cases))) return rc;
    if (h->pin_counts_bytes < (size_t)ev->n_cases * 5) {
        if (h->pin_counts) cudaFreeHost(h->pin_counts);
        h->pin_counts = nullptr;
        h->pin_counts_bytes = 0;
        CU_TRY(cudaMallocHost(&h->pin_counts, (size_t)ev->n_cases * 5));
        h->pin_counts_bytes = (size_t)ev->n_cases * 5;
    }
    int32_t* const pin_sweeps = (int32_t*)h->pin_counts;
    uint8_t* const pin_conv = (uint8_t*)h->pin_counts + (size_t)ev->n_cases * 4;
    // evidence staging for the whole batch (absolute offsets, like bnbp_run_batch_device)
    if ((rc = h->s_ev_off.ensure((size_t)(ev->n_cases + 1) * 8))) return rc;
    if ((rc = h->s_ev_node.ensure(std::max<size_t>(16, (size_t)nnz * 4)))) return rc;
    if (soft) {
        if ((rc = h->s_ev_val_off.ensure((size_t)(nnz + 1) * 8))) return rc;
        if ((rc = h->s_ev_values.ensure(std::max<size_t>(16, (size_t)(ev->ev_val_off[nnz] - ev->ev_val_off[0]) * 8)))) return rc;
    } else {
        if ((rc = h->s_ev_state.ensure(std::max<size_t>(16, (size_t)nnz * 4)))) return rc;
    }
    while (h->ev_chunk.size() < 3 * plan.size()) {       // per chunk: uploaded, computed, copied
        cudaEvent_t e;
        CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->ev_chunk.push_back(e);
    }
    const bool trace = getenv("BNBP_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto stamp = [&](const char* what, int i) {
        if (trace)
            fprintf(stderr, "[bnbp] %8.3f ms  %s %d\n",
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(), what, i);
    };
    if (trace) {
        fprintf(stderr, "[bnbp] wave %lld cases, copy/compute estimate %.2f, staging %s, chunks:", (long long)wave, rho,
                whole ? "whole batch" : "ring of 2");
        for (int64_t c : plan) fprintf(stderr, " %lld", (long long)c);
        fprintf(stderr, "\n");
    }
    CU_TRY(cudaMemsetAsync(reinterpret_cast<int32_t*>(h->d_misc.p) + 1, 0, 4, st));
    cudaStream_t cs = h->copy_stream, hs = h->h2d_stream;
    struct Drain {                       // no path leaves this call with copies from/to host memory in flight
        cudaStream_t a, b, c;
        ~Drain() { cudaStreamSynchronize(a); cudaStreamSynchronize(b); cudaStreamSynchronize(c); }
    } drain{hs, st, cs};
    CU_TRY(cudaEventRecord(h->ev_total[0], st));
    CU_TRY(cudaStreamWaitEvent(hs, h->ev_total[0], 0));   // uploads start with the call on the device timeline
    std::vector<cudaEvent_t> tev;                     // BNBP_TRACE: device timeline of the pipeline
    auto mark = [&](cudaStream_t s) {
        if (!trace) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, s);
        tev.push_back(e);
    };
    const int64_t val0 = soft ? ev->ev_val_off[0] : 0;
    int idx = 0;
    for (int64_t c0 = 0, n = 0; c0 < ev->n_cases; c0 += n, ++idx) {
        n = (size_t)idx + 1 >= plan.size() ? ev->n_cases - c0 : std::min<int64_t>(plan[(size_t)idx], ev->n_cases - c0);
        n = std::min<int64_t>(n, chunk);
        if ((size_t)(3 * idx + 2) >= h->ev_chunk.size()) {
            for (int k = 0; k < 3; ++k) {
                cudaEvent_t e;
                CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                h->ev_chunk.push_back(e);
            }
        }
        cudaEvent_t e_up = h->ev_chunk[3 * idx], e_done = h->ev_chunk[3 * idx + 1], e_copied = h->ev_chunk[3 * idx + 2];
        const int64_t a = ev->ev_off[c0], b = ev->ev_off[c0 + n];
        {
            bool mono = a >= 0 && b <= nnz;
            for (int64_t c = c0; c < c0 + n; ++c) mono &= ev->ev_off[c + 1] >= ev->ev_off[c];
            if (!mono) return fail(BNBP_ERR_INVALID, "ev_off not monotone");
        }
        // evidence of this chunk, into its place in the whole-batch arrays
        std::unique_ptr<NvtxRange> nvtx_h2d(new NvtxRange("bnbp: enqueue H2D evidence of a chunk"));
        CU_TRY(cudaMemcpyAsync((int64_t*)h->s_ev_off.p + c0, ev->ev_off + c0, (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, hs));
        if (b > a) CU_TRY(cudaMemcpyAsync((int32_t*)h->s_ev_node.p + a, ev->ev_node + a, (size_t)(b - a) * 4, cudaMemcpyHostToDevice, hs));
        DevEvidence de{(const int64_t*)h->s_ev_off.p + c0, 0, (const int32_t*)h->s_ev_node.p, nullptr, nullptr, nullptr, 0};
        if (soft) {
            const int64_t va = ev->ev_val_off[a], vb = ev->ev_val_off[b];
            {   // the offsets become memcpy ranges below: refuse anything not monotone inside [val0, end]
                bool mono = va >= val0 && vb <= ev->ev_val_off[nnz];
                for (int64_t e = a; e < b; ++e) mono &= ev->ev_val_off[e + 1] >= ev->ev_val_off[e];
                if (!mono) return fail(BNBP_ERR_INVALID, "ev_val_off not monotone");
            }
            CU_TRY(cudaMemcpyAsync((int64_t*)h->s_ev_val_off.p + a, ev->ev_val_off + a, (size_t)(b - a + 1) * 8, cudaMemcpyHostToDevice, hs));
            if (vb > va)
                CU_TRY(cudaMemcpyAsync((double*)h->s_ev_values.p + (va - val0), ev->ev_values + va, (size_t)(vb - va) * 8, cudaMemcpyHostToDevice, hs));
            de.ev_val_off = (const int64_t*)h->s_ev_val_off.p;
            de.ev_values = (const double*)h->s_ev_values.p;
            de.ev_val_base = val0;
        } else {
            if (b > a) CU_TRY(cudaMemcpyAsync((int32_t*)h->s_ev_state.p + a, ev->ev_state + a, (size_t)(b - a) * 4, cudaMemcpyHostToDevice, hs));
            de.ev_state = (const int32_t*)h->s_ev_state.p;
        }
        CU_TRY(cudaEventRecord(e_up, hs));
        nvtx_h2d.reset();
        CU_TRY(cudaStreamWaitEvent(st, e_up, 0));
        char* slot = whole ? (char*)h->s_out_all.p + (size_t)c0 * row_bytes : (char*)h->s_out[idx & 1].p;
        if (!whole && idx >= 2) CU_TRY(cudaStreamWaitEvent(st, h->ev_chunk[3 * (idx - 2) + 2], 0));   // ring slot is free again
        stamp("enqueue chunk", idx);
        mark(st);
        if (h->precision == BNBP_FP32 && out_f32)
            rc = run_any<float, float>(h, n, de, *prm, (float*)slot, (int32_t*)h->s_out_sweeps.p + c0, (uint8_t*)h->s_out_conv.p + c0, st, nullptr);
        else if (h->precision == BNBP_FP32)
            rc = run_any<float, double>(h, n, de, *prm, (double*)slot, (int32_t*)h->s_out_sweeps.p + c0, (uint8_t*)h->s_out_conv.p + c0, st, nullptr);
        else
            rc = run_any<double, double>(h, n, de, *prm, (double*)slot, (int32_t*)h->s_out_sweeps.p + c0, (uint8_t*)h->s_out_conv.p + c0, st, nullptr);
        if (rc) return rc;
        mark(st);
        CU_TRY(cudaEventRecord(e_done, st));
        CU_TRY(cudaStreamWaitEvent(cs, e_done, 0));
        mark(cs);
        NvtxRange nvtx_d2h("bnbp: enqueue D2H marginals of a chunk");
        CU_TRY(cudaMemcpyAsync(out_marginals + (size_t)c0 * row_bytes, slot, (size_t)n * row_bytes, cudaMemcpyDeviceToHost, cs));
        mark(cs);
        // per-case counts: into the library's pinned staging (the caller's arrays are usually pageable, and
        // a pageable D2H would block this thread until the chunk is done)
        if (out_sweeps)
            CU_TRY(cudaMemcpyAsync(pin_sweeps + c0, (const int32_t*)h->s_out_sweeps.p + c0, (size_t)n * 4, cudaMemcpyDeviceToHost, cs));
        if (out_converged)
            CU_TRY(cudaMemcpyAsync(pin_conv + c0, (const uint8_t*)h->s_out_conv.p + c0, (size_t)n, cudaMemcpyDeviceToHost, cs));
        CU_TRY(cudaEventRecord(e_copied, cs));
        stamp("enqueued copy", idx);
    }
    cudaEvent_t e_last = h->ev_chunk[3 * (idx - 1) + 2];
    // copy_stream is in order: everything before e_last has left when it fires
    stamp("all enqueued", idx);
    // the call returns with every result on the host
    CU_TRY(cudaStreamWaitEvent(st, e_last, 0));
    CU_TRY(cudaEventRecord(h->ev_total[1], st));
    h->total_recorded = true;
    const auto t_wait = std::chrono::steady_clock::now();
    NvtxRange nvtx_wait("bnbp: wait for the streams");
    if ((rc = check_error_flag(h, st))) return rc;
    CU_TRY(wait_stream(cs));
    h->last_host_wait_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_wait).count();
    stamp("done", idx);
    for (size_t i = 0; i + 3 < tev.size(); i += 4) {
        float a = 0, b = 0, c = 0, d = 0;
        cudaEventElapsedTime(&a, tev[0], tev[i]);
        cudaEventElapsedTime(&b, tev[0], tev[i + 1]);
        cudaEventElapsedTime(&c, tev[0], tev[i + 2]);
        cudaEventElapsedTime(&d, tev[0], tev[i + 3]);
        fprintf(stderr, "[bnbp] chunk %zu: compute %.3f..%.3f ms, copy %.3f..%.3f ms (device timeline)\n", i / 4, a, b, c, d);
    }
    for (cudaEvent_t e : tev) cudaEventDestroy(e);
    if (out_sweeps) memcpy(out_sweeps, pin_sweeps, (size_t)ev->n_cases * 4);
    if (out_converged) memcpy(out_converged, pin_conv, (size_t)ev->n_cases);
    if (!(prm->epsilon > 0.0)) {
        h->last_case_sweeps = ev->n_cases * (int64_t)prm->max_sweeps;     // fixed count: every case ran them all
    } else if (out_sweeps) {
        int64_t s = 0;
        for (int64_t c = 0; c < ev->n_cases; ++c) s += out_sweeps[c];
        h->last_case_sweeps = s;
    } else {
        h->last_case_sweeps = -1;
    }
    h->last_host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_entry).count();
    return BNBP_OK;
}

int bnbp_lw_run_batch(bnbp_handle* h, const bnbp_evidence* ev, int64_t n_samples, uint64_t seed, double* out_marginals,
                      double* out_weight_sum)
{
    if (!h || !ev || !out_marginals) return fail(BNBP_ERR_INVALID, "bnbp_lw_run_batch: NULL argument");
    if (!h->members.empty()) h = h->members[0];               // likelihood weighting is the cross-check: one device
    if (n_samples < 1) return fail(BNBP_ERR_INVALID, "bnbp_lw_run_batch: n_samples < 1");
    if (ev->n_cases < 0) return fail(BNBP_ERR_INVALID, "n_cases < 0");
    if (ev->ev_values) return fail(BNBP_ERR_INVALID, "likelihood weighting takes hard evidence (vertex -> state, likelihood_weighting.hpp:15)");
    if (ev->n_cases == 0) return BNBP_OK;
    if (!ev->ev_off) return fail(BNBP_ERR_INVALID, "ev_off is NULL");
    const int64_t nnz = ev->ev_off[ev->n_cases];
    if (nnz < 0 || ev->ev_off[0] < 0) return fail(BNBP_ERR_INVALID, "ev_off not monotone");
    if (nnz > 0 && (!ev->ev_node || !ev->ev_state)) return fail(BNBP_ERR_INVALID, "ev_node / ev_state is NULL");
    for (int64_t c = 0; c < ev->n_cases; ++c)
        if (ev->ev_off[c + 1] < ev->ev_off[c]) return fail(BNBP_ERR_INVALID, "ev_off not monotone");
    for (int x = 0; x < h->N; ++x)
        if (h->card[x] > 255) return fail(BNBP_ERR_INVALID, "likelihood weighting keeps states in bytes: cardinality > 255");
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t st = h->stream;
    int rc;
    if (!h->lw_ready) {
        // a topological order: parents first (weighted_sample resolves the parents recursively, :131-147)
        std::vector<int32_t> order, indeg(h->N), stack;
        std::vector<std::vector<int32_t>> ch(h->N);
        for (int x = h->N - 1; x >= 0; --x) {
            indeg[x] = h->nodes[x].k;
            for (int j = 0; j < h->nodes[x].k; ++j) ch[h->par_host[h->nodes[x].e0 + j]].push_back(x);
            if (!indeg[x]) stack.push_back(x);
        }
        while (!stack.empty()) {
            const int u = stack.back(); stack.pop_back();
            order.push_back(u);
            for (int c : ch[u]) if (--indeg[c] == 0) stack.push_back(c);
        }
        if ((rc = h->d_lw_order.ensure(std::max<size_t>(16, order.size() * 4)))) return rc;
        if ((rc = h->d_lw_par.ensure(std::max<size_t>(16, h->par_host.size() * 4)))) return rc;
        if ((rc = h->d_lw_cpt.ensure(std::max<size_t>(16, h->cpt_host.size() * 8)))) return rc;
        CU_TRY(cudaMemcpyAsync(h->d_lw_order.p, order.data(), order.size() * 4, cudaMemcpyHostToDevice, st));
        if (!h->par_host.empty())
            CU_TRY(cudaMemcpyAsync(h->d_lw_par.p, h->par_host.data(), h->par_host.size() * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(h->d_lw_cpt.p, h->cpt_host.data(), h->cpt_host.size() * 8, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaStreamSynchronize(st));          // the vectors above go out of scope
        h->lw_ready = true;
    }
    // block shape: one sample per thread; [node][thread] state bytes + the case's histogram in shared memory
    int threads = 128;
    auto smem_for = [&](int t) { return (size_t)h->V * 8 + (size_t)h->N * 4 + (size_t)h->N * t; };
    while (threads > 32 && smem_for(threads) > 200 * 1024) threads /= 2;
    const size_t smem = smem_for(threads);
    if (smem > 200 * 1024) return fail(BNBP_ERR_INVALID, "network too large for the likelihood-weighting kernel's shared-memory state");
    if (smem > 48 * 1024) CU_TRY(cudaFuncSetAttribute(lw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if ((rc = h->s_ev_off.ensure((size_t)(ev->n_cases + 1) * 8))) return rc;
    if ((rc = h->s_ev_node.ensure(std::max<size_t>(16, (size_t)nnz * 4)))) return rc;
    if ((rc = h->s_ev_state.ensure(std::max<size_t>(16, (size_t)nnz * 4)))) return rc;
    CU_TRY(cudaMemcpyAsync(h->s_ev_off.p, ev->ev_off, (size_t)(ev->n_cases + 1) * 8, cudaMemcpyHostToDevice, st));
    if (nnz > 0) {
        CU_TRY(cudaMemcpyAsync(h->s_ev_node.p, ev->ev_node, (size_t)nnz * 4, cudaMemcpyHostToDevice, st));
        CU_TRY(cudaMemcpyAsync(h->s_ev_state.p, ev->ev_state, (size_t)nnz * 4, cudaMemcpyHostToDevice, st));
    }
    const int64_t CH = 1 << 16;                     // cases per launch (bounds the device-side result buffer)
    if ((rc = h->d_lw_out.ensure((size_t)std::min(CH, ev->n_cases) * h->V * 8))) return rc;
    if ((rc = h->d_lw_wsum.ensure((size_t)std::min(CH, ev->n_cases) * 8))) return rc;
    int32_t* d_error = reinterpret_cast<int32_t*>(h->d_misc.p) + 1;
    CU_TRY(cudaMemsetAsync(d_error, 0, 4, st));
    h->last_kernel_launches = 0;
    for (int64_t c0 = 0; c0 < ev->n_cases; c0 += CH) {
        const int64_t n = std::min(CH, ev->n_cases - c0);
        LwArgs a;
        a.nodes = (const NodeMeta*)h->d_nodes.p;
        a.order = (const int32_t*)h->d_lw_order.p; a.par = (const int32_t*)h->d_lw_par.p;
        a.cpt = (const double*)h->d_lw_cpt.p;
        a.n_nodes = h->N; a.V = h->V;
        a.n_cases = n; a.case_base = c0;
        a.ev_off = (const int64_t*)h->s_ev_off.p + c0; a.ev_base = 0;
        a.ev_node = (const int32_t*)h->s_ev_node.p; a.ev_state = (const int32_t*)h->s_ev_state.p;
        a.n_samples = n_samples; a.seed = seed;
        a.out = (double*)h->d_lw_out.p; a.out_wsum = (double*)h->d_lw_wsum.p;
        a.error_flag = d_error;
        lw_kernel<<<(unsigned)n, threads, smem, st>>>(a);
        CU_TRY(cudaGetLastError());
        h->last_kernel_launches++;
        CU_TRY(cudaMemcpyAsync(out_marginals + (size_t)c0 * h->V, h->d_lw_out.p, (size_t)n * h->V * 8, cudaMemcpyDeviceToHost, st));
        if (out_weight_sum) CU_TRY(cudaMemcpyAsync(out_weight_sum + c0, h->d_lw_wsum.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    }
    return check_error_flag(h, st);
}

int bnbp_estimate_cpt(const bnbp_flat_network* net, const int32_t* samples, const int64_t* multiplicity, int64_t n_rows,
                      int32_t device, double* out_cpt)
{
    if (!net || !out_cpt || (n_rows > 0 && !samples)) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: NULL argument");
    if (n_rows < 0) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: n_rows < 0");
    const int N = net->n_nodes;
    if (N < 1 || !net->card || !net->parent_off || !net->cpt_off) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: malformed network");
    const int E = net->parent_off[N];
    if (E > 0 && !net->parents) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: parents is NULL");
    std::vector<NodeMeta> nodes((size_t)N);
    std::vector<int64_t> row_start((size_t)N + 1, 0);
    for (int x = 0; x < N; ++x) {
        NodeMeta& nd = nodes[(size_t)x];
        memset(&nd, 0, sizeof nd);
        nd.card = net->card[x];
        nd.k = net->parent_off[x + 1] - net->parent_off[x];
        nd.e0 = net->parent_off[x];
        nd.cpt_off = net->cpt_off[x];
        if (nd.card < 1 || nd.k < 0) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: bad cardinality / parent_off");
        int64_t Q = 1;
        for (int e = nd.e0; e < nd.e0 + nd.k; ++e) {
            const int u = net->parents[e];
            if (u < 0 || u >= N || u == x) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: bad parent id");
            Q *= net->card[u];
        }
        if (net->cpt_off[x + 1] - net->cpt_off[x] != Q * nd.card)
            return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: cpt_off does not match the parent configurations");
        row_start[(size_t)x + 1] = row_start[(size_t)x] + Q;
    }
    const int64_t n_values = net->cpt_off[N], n_cpt_rows = row_start[(size_t)N];
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
        cudaGetLastError();
        return fail(BNBP_ERR_NO_DEVICE, "no CUDA device: libbnbp has no CPU fallback");
    }
    if (device >= 0) CU_TRY(cudaSetDevice(device));
    DevBuf d_nodes, d_par, d_rows, d_samples, d_mult, d_counts, d_cpt, d_flag;
    struct Free { std::vector<DevBuf*> b; ~Free() { for (DevBuf* x : b) x->release(); } }
        guard{{&d_nodes, &d_par, &d_rows, &d_samples, &d_mult, &d_counts, &d_cpt, &d_flag}};
    int rc;
    if ((rc = d_nodes.ensure(nodes.size() * sizeof(NodeMeta)))) return rc;
    if ((rc = d_par.ensure(std::max<size_t>(16, (size_t)E * 4)))) return rc;
    if ((rc = d_rows.ensure(row_start.size() * 8))) return rc;
    if ((rc = d_counts.ensure(std::max<size_t>(16, (size_t)n_values * 8)))) return rc;
    if ((rc = d_cpt.ensure(std::max<size_t>(16, (size_t)n_values * 8)))) return rc;
    if ((rc = d_flag.ensure(16))) return rc;
    CU_TRY(cudaMemcpy(d_nodes.p, nodes.data(), nodes.size() * sizeof(NodeMeta), cudaMemcpyHostToDevice));
    if (E > 0) CU_TRY(cudaMemcpy(d_par.p, net->parents, (size_t)E * 4, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(d_rows.p, row_start.data(), row_start.size() * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(d_counts.p, 0, (size_t)n_values * 8));
    CU_TRY(cudaMemset(d_flag.p, 0, 16));
    // the sample table goes through HBM in slabs of <= 256 MB
    const int64_t slab = std::max<int64_t>(1, (int64_t)(256u << 20) / ((int64_t)N * 4));
    if (n_rows > 0) {
        if ((rc = d_samples.ensure((size_t)std::min(slab, n_rows) * N * 4))) return rc;
        if (multiplicity && (rc = d_mult.ensure((size_t)std::min(slab, n_rows) * 8))) return rc;
    }
    for (int64_t r0 = 0; r0 < n_rows; r0 += slab) {
        const int64_t n = std::min(slab, n_rows - r0);
        CU_TRY(cudaMemcpy(d_samples.p, samples + r0 * N, (size_t)n * N * 4, cudaMemcpyHostToDevice));
        if (multiplicity) CU_TRY(cudaMemcpy(d_mult.p, multiplicity + r0, (size_t)n * 8, cudaMemcpyHostToDevice));
        CountArgs a;
        a.nodes = (const NodeMeta*)d_nodes.p; a.par = (const int32_t*)d_par.p;
        a.samples = (const int32_t*)d_samples.p; a.mult = multiplicity ? (const int64_t*)d_mult.p : nullptr;
        a.n_rows = n; a.n_nodes = N;
        a.counts = (unsigned long long*)d_counts.p; a.error_flag = (int32_t*)d_flag.p;
        const int64_t work = n * N;
        const unsigned blocks = (unsigned)std::min<int64_t>((work + 255) / 256, 148 * 32);
        cpt_count_kernel<<<blocks, 256>>>(a);
        CU_TRY(cudaGetLastError());
    }
    cpt_normalize_kernel<<<(unsigned)((n_cpt_rows + 255) / 256), 256>>>((const NodeMeta*)d_nodes.p, (const int64_t*)d_rows.p, N, n_cpt_rows,
                                                                     (const unsigned long long*)d_counts.p, (double*)d_cpt.p);
    CU_TRY(cudaGetLastError());
    int32_t flag = 0;
    CU_TRY(cudaMemcpy(&flag, d_flag.p, 4, cudaMemcpyDeviceToHost));
    if (flag == 3) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: a sample holds a state outside [0, cardinality)");
    if (flag == 4) return fail(BNBP_ERR_INVALID, "bnbp_estimate_cpt: negative multiplicity");
    CU_TRY(cudaMemcpy(out_cpt, d_cpt.p, (size_t)n_values * 8, cudaMemcpyDeviceToHost));
    return BNBP_OK;
}

int bnbp_get_stats(const bnbp_handle* hc, bnbp_stats* out)
{
    if (!hc || !out) return fail(BNBP_ERR_INVALID, "bnbp_get_stats: NULL argument");
    bnbp_handle* h = const_cast<bnbp_handle*>(hc);
    if (!h->members.empty()) {            // group: the statistics of the first member, sweeps summed over the group
        const int rc = bnbp_get_stats(h->members[0], out);
        if (rc == BNBP_OK) out->last_case_sweeps = h->last_case_sweeps;
        return rc;
    }
    memset(out, 0, sizeof *out);
    out->state_values_per_case = (int64_t)h->PL + h->M;
    out->msg_values_per_case = h->M;
    out->belief_values_per_case = h->V;
    out->cpt_values = h->cpt_values;
    out->bytes_per_value = (int64_t)h->tsize;
    out->last_case_sweeps = h->last_case_sweeps;
    out->last_sweep_launches = h->last_sweep_launches;
    out->last_kernel_launches = h->last_kernel_launches;
    out->resident_cases = h->cap;
    out->last_specialised = h->last_specialised;
    out->spec_class_count = h->spec_classloop ? h->spec_classes_n : 0;
    out->cases_per_tile = h->tb;
    out->spec_compile_ms = h->spec_compile_ms;
    out->dense_nodes = h->dense_nodes;
    out->dense_values_per_case = h->TS;
    out->dense_flops_per_case_sweep = h->dense_flops_per_case;
    out->last_dense_launches = h->last_dense_launches;
    out->dense_tensor_jobs = h->dense_tc_jobs;
    out->dense_tensor_flops_per_case_sweep = h->dense_tc_flops_per_case;
    out->last_dense_tensor_launches = h->last_dense_tc_launches;
    out->last_fused = h->last_fused;
    out->last_compactions = h->last_compactions;
    out->last_onchip = h->last_onchip;
    out->onchip_roles = h->oc_eligible ? h->oc_roles : 0;
    out->onchip_smem_bytes = h->oc_eligible ? (int64_t)h->oc_smem : 0;
    out->onchip_role_imbalance = h->oc_imbalance;
    {
        int nb = 0;
        for (int i = 0; i < 4; ++i) if (h->oc_state[i] == 1) nb = std::max(nb, h->oc[i].blocks_per_sm);
        out->onchip_blocks_per_sm = nb;
    }
    out->last_host_ms = h->last_host_ms;
    out->last_host_wait_ms = h->last_host_wait_ms;
    out->last_dense_ms = -1.0;
    out->last_sweep_ms = -1.0;
    out->last_total_ms = -1.0;
    if (h->total_recorded) {
        cudaSetDevice(h->device);
        if (cudaEventSynchronize(h->ev_total[1]) == cudaSuccess) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, h->ev_total[0], h->ev_total[1]) == cudaSuccess) out->last_total_ms = ms;
            double sw = 0;
            bool ok = h->ev_sweep_used > 0;
            for (int i = 0; i < h->ev_sweep_used; ++i) {
                if (cudaEventElapsedTime(&ms, h->ev_sweep[2 * i], h->ev_sweep[2 * i + 1]) == cudaSuccess) sw += ms;
                else ok = false;
            }
            if (ok) out->last_sweep_ms = sw;
            double dn = 0;
            ok = h->ev_dense_used > 0;
            for (int i = 0; i < h->ev_dense_used; ++i) {
                if (cudaEventElapsedTime(&ms, h->ev_dense[2 * i], h->ev_dense[2 * i + 1]) == cudaSuccess) dn += ms;
                else ok = false;
            }
            if (ok) out->last_dense_ms = dn;
        }
        cudaGetLastError();
    }
    return BNBP_OK;
}

void* bnbp_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, std::max<size_t>(bytes, 1), cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        fail(BNBP_ERR_NOMEM, "bnbp_host_alloc: cudaHostAlloc failed");
        return nullptr;
    }
    return p;
}

void bnbp_host_free(void* p)
{
    if (p) cudaFreeHost(p);
}

int bnbp_create_multi(const bnbp_flat_network* net, const bnbp_options* opt, const int32_t* devices, int32_t n_devices,
                      bnbp_handle** out)
{
    if (!net || !out) return fail(BNBP_ERR_INVALID, "bnbp_create_multi: NULL argument");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(BNBP_ERR_NO_DEVICE, "no CUDA device: libbnbp has no CPU fallback");
    }
    std::vector<int> devs;
    if (n_devices <= 0) n_devices = ndev;
    for (int i = 0; i < n_devices; ++i) devs.push_back(devices ? devices[i] : i);
    for (size_t i = 0; i < devs.size(); ++i) {
        if (devs[i] < 0 || devs[i] >= ndev) return fail(BNBP_ERR_INVALID, "bnbp_create_multi: device ordinal out of range");
        for (size_t j = 0; j < i; ++j)
            if (devs[j] == devs[i]) return fail(BNBP_ERR_INVALID, "bnbp_create_multi: a device is listed twice");
    }
    struct Destroy { void operator()(bnbp_handle* p) const { bnbp_destroy(p); } };
    std::unique_ptr<bnbp_handle, Destroy> g(new bnbp_handle());
    int rc = build_layout(net, opt, g.get());              // host-side layout only: row widths, validation
    if (rc) return rc;
    g->device = devs[0];
    for (int d : devs) {
        bnbp_options o;
        memset(&o, 0, sizeof o);
        if (opt) o = *opt;
        o.device = d;
        bnbp_handle* m = nullptr;
        if ((rc = bnbp_create(net, &o, &m))) return rc;
        g->members.push_back(m);
        if ((rc = comm_resources(m))) return rc;
    }
    std::vector<ncclComm_t> comms(devs.size(), nullptr);
    NCCL_TRY(NCCL(CommInitAll)(comms.data(), (int)devs.size(), devs.data()));
    for (size_t i = 0; i < devs.size(); ++i) {
        g->members[i]->comm = comms[i];
        g->members[i]->comm_rank = (int)i;
        g->members[i]->comm_world = (int)devs.size();
    }
    *out = g.release();
    return BNBP_OK;
}

int bnbp_get_summary(const bnbp_handle* h, bnbp_summary* out)
{
    if (!h || !out) return fail(BNBP_ERR_INVALID, "bnbp_get_summary: NULL argument");
    *out = h->last_summary;
    return BNBP_OK;
}

int bnbp_comm_unique_id(void* id_out)
{
    if (!id_out) return fail(BNBP_ERR_INVALID, "bnbp_comm_unique_id: NULL argument");
    static_assert(sizeof(ncclUniqueId) <= BNBP_COMM_ID_BYTES, "ncclUniqueId larger than BNBP_COMM_ID_BYTES");
    ncclUniqueId id;
    NCCL_TRY(NCCL(GetUniqueId)(&id));
    memset(id_out, 0, BNBP_COMM_ID_BYTES);
    memcpy(id_out, &id, sizeof id);
    return BNBP_OK;
}

int bnbp_comm_init(bnbp_handle* h, int32_t world, int32_t rank, const void* id_in)
{
    if (!h || !id_in) return fail(BNBP_ERR_INVALID, "bnbp_comm_init: NULL argument");
    if (!h->members.empty()) return fail(BNBP_ERR_INVALID, "bnbp_comm_init: a group handle already owns its communicator");
    if (world < 1 || rank < 0 || rank >= world) return fail(BNBP_ERR_INVALID, "bnbp_comm_init: rank / world out of range");
    if (h->comm) return fail(BNBP_ERR_INVALID, "bnbp_comm_init: the handle already has a communicator");
    int rc = comm_resources(h);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(h->device));
    ncclUniqueId id;
    memcpy(&id, id_in, sizeof id);
    NCCL_TRY(NCCL(CommInitRank)(&h->comm, world, id, rank));
    h->comm_world = world;
    h->comm_rank = rank;
    return BNBP_OK;
}

int bnbp_comm_summary(bnbp_handle* h, const int32_t* d_sweeps, const uint8_t* d_converged, int64_t n_cases, bnbp_summary* out,
                      void* stream)
{
    if (!h || !out || (n_cases > 0 && (!d_sweeps || !d_converged))) return fail(BNBP_ERR_INVALID, "bnbp_comm_summary: NULL argument");
    if (!h->members.empty()) return fail(BNBP_ERR_INVALID, "bnbp_comm_summary: use bnbp_get_summary on a group handle");
    int rc = comm_resources(h);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(h->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if ((rc = enqueue_summary(h, d_sweeps, d_converged, n_cases, st))) return rc;
    if ((rc = fetch_summary(h, st))) return rc;
    CU_TRY(wait_stream(st));
    read_summary(h, out);
    h->last_summary = *out;
    return BNBP_OK;
}

} // extern "C"
