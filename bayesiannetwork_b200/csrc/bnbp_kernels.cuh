// bnbp_kernels.cuh — sm_100a kernels of the batched loopy-BP path.
//
// Work decomposition (DESIGN.md section 3): one thread owns VEC evidence cases and walks a
// contiguous range of nodes; a block owns one TILE of TB cases.  All per-case state lives in HBM
// as batch-minor SoA tiles  state[tile][slot][TB]  so that a warp reading one slot touches
// 32*VEC consecutive values (coalesced double2 / float4 accesses).  Everything that does not
// depend on the case (topology, cardinalities, CPT entries) is warp-uniform and is fetched
// through the read-only path as broadcast loads.
//
// One sweep = one launch of sweep_kernel = the whole body of the reference's while(true)
// (bayesian/inference/belief_propagation.hpp:75-148) for every resident case:
//   per node X (a "gather" formulation, every state slot is read once and written once):
//     reads   pi_X, lambda_X, pi-messages X<-parents, lambda-messages children->X   (time t)
//     writes  pi_X, lambda_X (in place: X is their only reader),
//             lambda-messages X->parents, pi-messages X->children                  (time t+1 buffer)
//   :202-218 calculate_pi_i, :240-266 calculate_lambda_k, :174-200 calculate_pi,
//   :220-238 calculate_lambda, :105-131 delta, :135-143 commit (= buffer swap), :298-311 normalize.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

namespace bnbp {

constexpr int KMAX = 8;        // max in-degree handled by the templated recursion
constexpr int MAX_CHUNKS = 192;

struct NodeMeta {              // 64 bytes, warp-uniform
    int32_t card;              // r_X
    int32_t k;                 // number of parents
    int32_t m;                 // number of children
    int32_t pl_off;            // slot of pi_X in the pi/lambda region (lambda_X at pl_off + card)
    int32_t pin_off;           // msg-buffer slot of the first pi-message into X (in-edge order)
    int32_t lin_off;           // msg-buffer slot of the first lambda-message into X (m blocks of r_X)
    int32_t e0;                // first in-edge index
    int32_t c0;                // first out-edge index
    int64_t cpt_off;           // offset into the device CPT arena
    int32_t bel_off;           // offset of X in a row of marginals
    int32_t scr_half;          // scratch values reserved for the outer parents' messages (accumulators follow)
    // dense contraction path (bnbp_dense.cuh): dense_s = 0 for ordinary nodes, else the split point s
    // (parents [0,s) form group A, [s,k) group B) and the slots of the per-case tables T1 / T2
    int32_t dense_s;
    int32_t t1_off;            // T1[(uB,x)], QB*r slots
    int32_t t2_off;            // T2[uA], QA slots
    int32_t pad_;
};

template <typename T> struct SweepArgs {
    const NodeMeta* nodes;
    const int32_t*  e_card;     // [E] cardinality of the parent of in-edge e
    const int32_t*  e_lam_out;  // [E] msg slot where the child writes lambda-msg (child->parent)
    const int32_t*  c_pi_out;   // [E] msg slot where the parent writes pi-msg (parent->child), out-edge order
    const T*        cpt;
    T*              pl;         // [tiles][PL][TB]
    const T*        msg_cur;    // [tiles][M][TB]
    T*              msg_nxt;
    const uint32_t* evbits;     // [tiles][W][TB]
    const T*        tscr;       // [tiles][TS][TB] per-case tables of the dense nodes (this sweep's GEMMs)
    int32_t PL, M, W, TS;
    int32_t n_chunks;
    int32_t chunk_off[MAX_CHUNKS + 1];
    // convergence bookkeeping (only touched when FREEZE / CHECK)
    const T* delta_prev;        // delta of the previous sweep (valid if prev_tested)
    T*       delta_cur;         // atomicMax target of this sweep (CHECK)
    T*       delta_next;        // reset to the :105 floor for the next sweep
    uint8_t* status;            // 0 active, 1 converged (frozen)
    int32_t* sweeps;            // sweeps executed when the case froze
    int32_t* last_active;       // largest sweep index that still had an active case (-1 at start)
    int32_t  sweep_index;       // t (0-based)
    int32_t  prev_tested;
    T eps;
    T damping;
    int32_t prefetch;           // 1: every node prefetches the inputs of the NEXT node of the walk into L2 (sweep_kernel)
};

template <typename T, int VEC> struct alignas(sizeof(T) * VEC) Pk { T v[VEC]; };

template <typename T, int VEC> __device__ __forceinline__ Pk<T, VEC> ldp(const T* p)
{
    return *reinterpret_cast<const Pk<T, VEC>*>(p);
}
template <typename T, int VEC> __device__ __forceinline__ void stp(T* p, const Pk<T, VEC>& x)
{
    *reinterpret_cast<Pk<T, VEC>*>(p) = x;
}

template <typename T> struct Lim;
template <> struct Lim<double> { static __device__ __forceinline__ double floor_() { return DBL_MIN; } };
template <> struct Lim<float>  { static __device__ __forceinline__ float floor_() { return FLT_MIN; } };

// max |new-old| with std::max(running, NaN) == running (:113-116): fmax ignores NaN.
__device__ __forceinline__ double absdiff_max(double run, double a, double b) { return fmax(run, fabs(a - b)); }
__device__ __forceinline__ float  absdiff_max(float run, float a, float b) { return fmaxf(run, fabsf(a - b)); }

// belief = (pi*lambda) / sum(pi*lambda) (:151-158): the sum is accumulated with explicit fused
// multiply-adds and the numerator is an explicitly rounded product, so that the compiler's choice of
// contraction cannot differ between the stand-alone belief kernels and the fused last sweep of
// bnbp_spec.cuh (which must agree bit for bit)
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float  mul_rn(float a, float b) { return __fmul_rn(a, b); }

// non-negative IEEE values order like their bit patterns
__device__ __forceinline__ void atomic_max_nonneg(double* p, double v)
{
    atomicMax(reinterpret_cast<unsigned long long*>(p), (unsigned long long)__double_as_longlong(v));
}
__device__ __forceinline__ void atomic_max_nonneg(float* p, float v)
{
    atomicMax(reinterpret_cast<unsigned int*>(p), __float_as_uint(v));
}

// Sweep launchers: defined in bnbp_sweep.cuh, explicitly instantiated one (T, VEC, RMAX) per
// translation unit (bnbp_sweep_inst.cu) so the build parallelises.
template <typename T, int VEC, int RMAX, int KNET>
cudaError_t launch_sweep_vr(const SweepArgs<T>& a, dim3 grid, size_t smem, bool freeze, bool check, cudaStream_t st, bool maxp);
template <typename T, int VEC, int RMAX, int KNET> cudaError_t set_sweep_smem(int bytes);

// ------------------------------------------------------------------------------------------------
// K0: initial state of one tile (belief_propagation.hpp:33-73).  One thread per case.
template <typename T> struct InitArgs {
    const NodeMeta* nodes;
    const T* pl_init;           // [PL] 1 everywhere, raw prior row for the pi of roots (:58-64)
    T* pl; T* msg0; uint32_t* evbits;
    int32_t PL, M, W, TB, n_nodes;
    int64_t n_valid;            // cases actually present in this chunk (rest is padding)
    const int64_t* ev_off;      // [n_valid+1], absolute offsets
    int64_t ev_base;            // ev_off value of the first case of the chunk in the arrays below
    const int32_t* ev_node; const int32_t* ev_state;
    const int64_t* ev_val_off; const double* ev_values; int64_t ev_val_base;
    T* delta; int64_t cap;      // delta[3][cap]
    uint8_t* status; int32_t* sweeps;
    int32_t* error_flag;
    int32_t write_msgs;         // 0: the first sweep will not read the time-0 messages (all ones)
};

template <typename T>
__global__ void __launch_bounds__(512) init_kernel(const InitArgs<T> a)
{
    const int tile = blockIdx.x, lane = threadIdx.x;
    const size_t TB = (size_t)a.TB;
    const int64_t c = (int64_t)tile * a.TB + lane;
    T* pl = a.pl + ((size_t)tile * a.PL) * TB + lane;
    T* msg = a.msg0 + ((size_t)tile * a.M) * TB + lane;
    uint32_t* evb = a.evbits + ((size_t)tile * a.W) * TB + lane;
    for (int s = 0; s < a.PL; ++s) pl[(size_t)s * TB] = __ldg(a.pl_init + s);
    if (a.write_msgs)
        for (int s = 0; s < a.M; ++s) msg[(size_t)s * TB] = T(1);
    for (int w = 0; w < a.W; ++w) evb[(size_t)w * TB] = 0u;
    for (int i = 0; i < 3; ++i) a.delta[(size_t)i * a.cap + c] = Lim<T>::floor_();
    a.sweeps[c] = 0;
    a.status[c] = (c < a.n_valid) ? 0 : 1;
    if (c >= a.n_valid) return;
    // evidence goes into BOTH pi and lambda (:69-73); the same thread wrote the defaults above
    const int64_t e0 = a.ev_off[c] - a.ev_base, e1 = a.ev_off[c + 1] - a.ev_base;
    for (int64_t e = e0; e < e1; ++e) {
        const int node = a.ev_node[e];
        if (node < 0 || node >= a.n_nodes) { *a.error_flag = 1; continue; }
        const NodeMeta nd = a.nodes[node];
        const int r = nd.card;
        if (a.ev_values) {
            const int64_t vo = a.ev_val_off[e] - a.ev_val_base;
            if (a.ev_val_off[e + 1] - a.ev_val_off[e] != r) { *a.error_flag = 2; continue; }
            for (int i = 0; i < r; ++i) {
                const T val = (T)a.ev_values[vo + i];
                pl[(size_t)(nd.pl_off + i) * TB] = val;
                pl[(size_t)(nd.pl_off + r + i) * TB] = val;
            }
        } else {
            const int st = a.ev_state[e];
            if (st < 0 || st >= r) { *a.error_flag = 3; continue; }
            for (int i = 0; i < r; ++i) {
                const T val = (i == st) ? T(1) : T(0);
                pl[(size_t)(nd.pl_off + i) * TB] = val;
                pl[(size_t)(nd.pl_off + r + i) * TB] = val;
            }
        }
        evb[(size_t)(node >> 5) * TB] |= 1u << (node & 31);
    }
}

// K0 of the fused launch sequence (specialised variants 5, 6/7 of bnbp_spec.cuh): the first sweep forms
// the time-0 pi/lambda itself, so all that is left of :33-73 is one state byte per (node, case)
// -- 0 not observed, s+1 observed in state s -- and the evidence bit masks the later sweeps read.
// Both arenas are zeroed by the caller; one thread per case scatters its observations.
struct EvidenceArgs {
    const NodeMeta* nodes;
    uint8_t* evst;              // [tiles][n_nodes][TB]
    uint32_t* evbits;           // [tiles][W][TB]
    int32_t W, TB, n_nodes;
    int64_t n_valid;
    const int64_t* ev_off; int64_t ev_base;
    const int32_t* ev_node; const int32_t* ev_state;
    int32_t* error_flag;
};

static __global__ void __launch_bounds__(512) evidence_kernel(const EvidenceArgs a)
{
    const int tile = blockIdx.x, lane = threadIdx.x;
    const size_t TB = (size_t)a.TB;
    const int64_t c = (int64_t)tile * a.TB + lane;
    if (c >= a.n_valid) return;
    uint8_t* est = a.evst + ((size_t)tile * a.n_nodes) * TB + lane;
    uint32_t* evb = a.evbits + ((size_t)tile * a.W) * TB + lane;
    const int64_t e0 = a.ev_off[c] - a.ev_base, e1 = a.ev_off[c + 1] - a.ev_base;
    for (int64_t e = e0; e < e1; ++e) {
        const int node = a.ev_node[e];
        if (node < 0 || node >= a.n_nodes) { *a.error_flag = 1; continue; }
        const int st = a.ev_state[e];
        if (st < 0 || st >= a.nodes[node].card) { *a.error_flag = 3; continue; }
        est[(size_t)node * TB] = (uint8_t)(st + 1);
        evb[(size_t)(node >> 5) * TB] |= 1u << (node & 31);
    }
}

// per-case sweep counts and converged flags of a chunk, when no belief kernel follows (fused sequence)
static __global__ void counts_kernel(const uint8_t* __restrict__ status, const int32_t* __restrict__ sweeps,
                              int32_t* __restrict__ out_sweeps, uint8_t* __restrict__ out_conv, int64_t n)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    if (out_sweeps) out_sweeps[c] = sweeps[c];
    if (out_conv) out_conv[c] = status[c];
}

// After the last sweep: cases still active get their sweep count and converged flag.
template <typename T>
__global__ void finalize_kernel(uint8_t* status, int32_t* sweeps, const T* delta_last, int last_tested,
                                T eps, int32_t total_sweeps, int64_t n)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    if (status[c] == 0) {
        sweeps[c] = total_sweeps;
        if (last_tested && delta_last[c] < eps) status[c] = 1;
    }
}

// K4: belief = normalize(pi .* lambda) (:151-158), written case-major [case][sum r].  The rows leave
// through shared memory so that global stores are coalesced: a thread writing its own 8*V-byte row
// would make every warp store touch 32 sectors with 8 valid bytes each.  Every WARP owns 32 cases and
// a private [32][W+1] tile: for a group of consecutive nodes (<= W columns of the marginal row) each
// lane normalises its case into its tile row (conflict-free: odd row stride), then the warp streams
// the 32 row segments to HBM, one 8*W-byte contiguous segment per store instruction.  Warps never
// wait for each other (no block barrier) and the tile is small enough for 24 resident warps per SM.
struct BeliefGroup { int32_t n0, n1, j0, j1; };   // nodes [n0, n1) = columns [j0, j1) of a marginal row

template <typename T, typename OUT>
__global__ void __launch_bounds__(512)
belief_tiled_kernel(const NodeMeta* __restrict__ nodes, const BeliefGroup* __restrict__ groups, int n_groups,
                    const T* __restrict__ pl_all, int PL, int TBi, int V, int stride, int64_t n_valid,
                    OUT* __restrict__ out, const uint8_t* __restrict__ status, const int32_t* __restrict__ sweeps,
                    int32_t* __restrict__ out_sweeps, uint8_t* __restrict__ out_conv,
                    const int32_t* __restrict__ orig = nullptr, int only_frozen = 0)
{
    // orig != nullptr: position p of the arena holds case orig[p] of the chunk (the arena was compacted,
    // see compact_* below); only_frozen = 1: write the cases whose status is set and leave the others alone,
    // 2: the opposite (the cases delta_retire_kernel has not written yet)
    extern __shared__ __align__(16) unsigned char belief_smem[];
    const int tile = blockIdx.x, lane = threadIdx.x;
    const int warp = lane >> 5, wl = lane & 31;
    OUT* const tile_buf = reinterpret_cast<OUT*>(belief_smem) + (size_t)warp * 32 * stride;
    const size_t TB = (size_t)TBi;
    const int64_t w0 = (int64_t)tile * TBi + warp * 32;     // first case of this warp
    const int64_t c = w0 + wl;
    if (w0 >= n_valid) return;                               // whole warp beyond the batch
    const int rows = (int)((n_valid - w0) < 32 ? (n_valid - w0) : 32);
    const T* const pl = pl_all + ((size_t)tile * PL) * TB + lane;
    OUT* const mine = tile_buf + (size_t)wl * stride;
    for (int g = 0; g < n_groups; ++g) {
        const BeliefGroup gr = groups[g];
        if (c < n_valid) {
            for (int X = gr.n0; X < gr.n1; ++X) {
                const NodeMeta nd = nodes[X];
                const int r = nd.card;
                const T* const p = pl + (size_t)nd.pl_off * TB;
                T s = T(0);
                for (int x = 0; x < r; ++x) s = fma(p[(size_t)x * TB], p[(size_t)(r + x) * TB], s);
                for (int x = 0; x < r; ++x)
                    mine[nd.bel_off - gr.j0 + x] = (OUT)(mul_rn(p[(size_t)x * TB], p[(size_t)(r + x) * TB]) / s);
            }
        }
        __syncwarp();
        const int w = gr.j1 - gr.j0;
        for (int row = 0; row < rows; ++row) {
            if (only_frozen && (status[w0 + row] == 0) == (only_frozen == 1)) continue;   // warp-uniform
            const int64_t dcase = orig ? (int64_t)orig[w0 + row] : w0 + row;
            OUT* const dst = out + (size_t)dcase * V + gr.j0;
            const OUT* const src = tile_buf + (size_t)row * stride;
            for (int j = wl; j < w; j += 32) dst[j] = src[j];
        }
        __syncwarp();
    }
    if (c < n_valid && !(only_frozen && (status[c] == 0) == (only_frozen == 1))) {
        const int64_t dcase = orig ? (int64_t)orig[c] : c;
        if (out_sweeps) out_sweeps[dcase] = sweeps[c];
        if (out_conv) out_conv[dcase] = status[c];
    }
}

// ------------------------------------------------------------------------------------------------
// Compaction of the still-active cases (eps mode).  The reference stops every case at its own sweep
// (:147); in a batch the sweep counts spread widely (alarm37, eps 1e-6: mean 13, max 40), and a warp keeps
// issuing the whole node walk as long as ONE of its 32 cases is active.  At a checkpoint the converged
// cases are retired (their beliefs are written, belief_tiled_kernel with only_frozen) and the active ones
// are gathered into dense tiles of a second arena, so the later sweeps launch a grid of the size of the
// work that is left.  A case's arithmetic does not depend on its position: results are bit-identical.
//
// census:  applies the freeze rule of the next sweep launch (status / sweeps, see the FREEZE prologue of
//          the sweep kernels) and counts the active cases per tile and in total.
template <typename T>
__global__ void compact_census_kernel(uint8_t* __restrict__ status, int32_t* __restrict__ sweeps, const T* __restrict__ delta_prev,
                                      int prev_tested, T eps, int32_t sweeps_done, int32_t* __restrict__ tile_count,
                                      int32_t* __restrict__ total)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;     // blockDim.x = cases per tile
    bool frozen = status[c] != 0;
    if (!frozen && prev_tested && delta_prev[c] < eps) {
        frozen = true;
        status[c] = 1;
        sweeps[c] = sweeps_done;
    }
    const int n = __syncthreads_count(!frozen);
    if (threadIdx.x == 0) {
        tile_count[blockIdx.x] = n;
        if (n) atomicAdd(total, n);
    }
}

// The convergence test as a kernel of its own (eps mode of the specialised family, no damping): the sweeps
// run as the PLAIN variant (no freeze / check logic: 1.09 instead of 2.6-2.9 ms per sweep on alarm37 fp64,
// r01v) and this kernel forms the reference's delta (:105-131) from the two message buffers:
//   delta = max(floor, max |new - old| over all message entries), NaN ignored; converged when delta < eps.
// A case that converges is RETIRED on the spot: the reference returns right after that sweep's commit
// (:135-158), so its belief is normalize(pi .* lambda) of the state as it is now -- written here, with
// its sweep count and flag.  Later sweeps may keep updating the retired case's state; nothing reads it.
// Also the census of the compaction (active cases per tile and in total).
template <typename T, typename OUT>
__global__ void delta_retire_kernel(const NodeMeta* __restrict__ nodes, int n_nodes, int PL, int M, int V,
                                    const T* __restrict__ pl_all, const T* __restrict__ msg_old, const T* __restrict__ msg_new,
                                    uint8_t* __restrict__ status, T eps, int32_t sweeps_done, int64_t n_valid,
                                    const int32_t* __restrict__ orig, OUT* __restrict__ out, int32_t* __restrict__ out_sweeps,
                                    uint8_t* __restrict__ out_conv, int32_t* __restrict__ tile_count, int32_t* __restrict__ total)
{
    const int tile = blockIdx.x, lane = threadIdx.x;
    const size_t TB = blockDim.x;
    const int64_t c = (int64_t)tile * blockDim.x + lane;
    bool active = status[c] == 0;
    if (active) {
        const T* const a = msg_old + ((size_t)tile * M) * TB + lane;
        const T* const b = msg_new + ((size_t)tile * M) * TB + lane;
        T d0 = Lim<T>::floor_(), d1 = Lim<T>::floor_();
        int s = 0;
        for (; s + 1 < M; s += 2) {
            d0 = absdiff_max(d0, b[(size_t)s * TB], a[(size_t)s * TB]);
            d1 = absdiff_max(d1, b[(size_t)(s + 1) * TB], a[(size_t)(s + 1) * TB]);
        }
        if (s < M) d0 = absdiff_max(d0, b[(size_t)s * TB], a[(size_t)s * TB]);
        const T d = d0 > d1 ? d0 : d1;
        if (d < eps) {
            active = false;
            status[c] = 1;
            if (c < n_valid) {
                const int64_t dcase = orig ? (int64_t)orig[c] : c;
                const T* const pl = pl_all + ((size_t)tile * PL) * TB + lane;
                OUT* const o = out + (size_t)dcase * V;
                for (int X = 0; X < n_nodes; ++X) {
                    const NodeMeta nd = nodes[X];
                    const int r = nd.card;
                    const T* const p = pl + (size_t)nd.pl_off * TB;
                    T sum = T(0);
                    for (int x = 0; x < r; ++x) sum = fma(p[(size_t)x * TB], p[(size_t)(r + x) * TB], sum);
                    for (int x = 0; x < r; ++x) o[nd.bel_off + x] = (OUT)(mul_rn(p[(size_t)x * TB], p[(size_t)(r + x) * TB]) / sum);
                }
                if (out_sweeps) out_sweeps[dcase] = sweeps_done;
                if (out_conv) out_conv[dcase] = 1;
            }
        }
    }
    const int n = __syncthreads_count(active);
    if (lane == 0) {
        tile_count[tile] = n;
        if (n) atomicAdd(total, n);
    }
}

// exclusive scan of the tile counts (one block; a batch has at most a few thousand tiles)
static __global__ void compact_scan_kernel(const int32_t* __restrict__ tile_count, int32_t* __restrict__ tile_off, int n_tiles)
{
    __shared__ int32_t part[1024];
    __shared__ int32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 1024) {
        const int i = base + threadIdx.x;
        const int32_t v = i < n_tiles ? tile_count[i] : 0;
        part[threadIdx.x] = v;
        __syncthreads();
        for (int d = 1; d < 1024; d <<= 1) {                                // Hillis-Steele inclusive scan
            const int32_t add = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
            __syncthreads();
            part[threadIdx.x] += add;
            __syncthreads();
        }
        if (i < n_tiles) tile_off[i] = carry + part[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += part[1023];
        __syncthreads();
    }
}

// new position -> old position, in the old order (stable), and the chunk-relative case index it holds
static __global__ void compact_index_kernel(const uint8_t* __restrict__ status, const int32_t* __restrict__ tile_off,
                                            const int32_t* __restrict__ orig_old, int32_t* __restrict__ src_pos,
                                            int32_t* __restrict__ orig_new)
{
    __shared__ int32_t warp_base[32];
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = status[c] == 0;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, active);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) warp_base[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t run = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { const int32_t n = warp_base[w]; warp_base[w] = run; run += n; }
    }
    __syncthreads();
    if (active) {
        const int32_t p = tile_off[blockIdx.x] + warp_base[warp] + __popc(m & ((1u << lane) - 1u));
        src_pos[p] = (int32_t)c;
        orig_new[p] = orig_old ? orig_old[c] : (int32_t)c;
    }
}

// gather pi/lambda, the current message buffer and the evidence masks of the active cases into dense
// tiles; reset the per-position bookkeeping (positions >= n_active of the last tile are padding: frozen)
template <typename T>
__global__ void compact_gather_kernel(const int32_t* __restrict__ src_pos, int32_t n_active, int TBi, int PL, int M, int W,
                                      const T* __restrict__ pl_src, const T* __restrict__ msg_src, const uint32_t* __restrict__ evb_src,
                                      T* __restrict__ pl_dst, T* __restrict__ msg_dst, uint32_t* __restrict__ evb_dst,
                                      uint8_t* __restrict__ status, T* __restrict__ delta, int64_t cap)
{
    const size_t TB = (size_t)TBi;
    const int tile = blockIdx.x, lane = threadIdx.x;
    const int64_t p = (int64_t)tile * TBi + lane;
    for (int i = 0; i < 3; ++i) delta[(size_t)i * cap + p] = Lim<T>::floor_();
    status[p] = p < n_active ? 0 : 1;
    if (p >= n_active) return;
    const int64_t q = src_pos[p];
    const size_t st = (size_t)(q / TBi), sl = (size_t)(q % TBi);
    const T* ps = pl_src + (st * PL) * TB + sl;
    T* pd = pl_dst + ((size_t)tile * PL) * TB + lane;
    for (int s = 0; s < PL; ++s) pd[(size_t)s * TB] = ps[(size_t)s * TB];
    const T* ms = msg_src + (st * M) * TB + sl;
    T* md = msg_dst + ((size_t)tile * M) * TB + lane;
    for (int s = 0; s < M; ++s) md[(size_t)s * TB] = ms[(size_t)s * TB];
    const uint32_t* es = evb_src + (st * W) * TB + sl;
    uint32_t* ed = evb_dst + ((size_t)tile * W) * TB + lane;
    for (int s = 0; s < W; ++s) ed[(size_t)s * TB] = es[(size_t)s * TB];
}

} // namespace bnbp
