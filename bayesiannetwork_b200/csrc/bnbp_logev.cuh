// bnbp_logev.cuh — per-case log-evidence: the Bethe estimate log Z_B of log P(e) from the state a run ends with.
//
// For one case after its last executed sweep T, per node X with parents U_1..U_k, m_X children and CPT P(x|u):
//   lambda_X   the row the state holds after sweep T (one-hot for an observed node)
//   pm_j(u)    the pi-message U_j -> X that sweep T READ (the committed messages of sweep T-1, damped if damping is on)
//   Z_X        = sum_{x,u} P(x|u) lambda_X(x) prod_j pm_j(u_j)
//   b_X(x,u)   = P(x|u) lambda_X(x) prod_j pm_j(u_j) / Z_X,  with marginals b_X(x) and b_X(u_j = u)
//   log Z_B    = sum_X [ ln Z_X - sum_x b_X(x) ln lambda_X(x) - sum_j sum_u b_X(u_j=u) ln pm_j(u) + m_X sum_x b_X(x) ln b_X(x) ]
// which is -F_Bethe; its family marginal over x is the library's node marginal, converged or not.  A term of weight 0
// contributes 0; a NaN Z_X makes the case NaN, otherwise a zero Z_X makes it -inf.  Sums are fp64 in both precisions.
//
// The kernel reads the batch-minor, tile-major arena of the streaming kernels (state[tile][slot][TB]) exactly as
// belief_tiled_kernel does, one case per thread.  A sweep with index t reads msg[t & 1], so the buffer the case's last
// sweep read is msg[(sweeps - 1) & 1]; in epsilon mode a frozen case's sweep count is its own.  The accumulators of b_X(x)
// and of one parent's b_X(u_j) live in a per-thread shared-memory column (cardinalities up to 128): the CPT is walked
// once per parent (once for a root), which keeps the scratch at r_X + max_j r_Uj values whatever the in-degree.
//
// Expected family counts (COUNTS = true, the E-step of EM): a case c of weight w_c whose score is finite also adds
//   counts[cpt_off[X] + q r_X + x] += w_c b_X(x, u_q)                                   for every X, q, x
// into the CPT-arena-shaped fp64 array `counts`; a NaN or -inf case adds nothing.  The topology is shared by all
// cases, so the block reduces each entry before one fp64 atomicAdd per entry and block.  Atomics leave the summation
// order open: counts agree between runs to rounding, not bit for bit.  With COUNTS = false the kernel is the plain
// log-evidence kernel.
#pragma once
#include "bnbp_kernels.cuh"

namespace bnbp {

template <typename T, bool COUNTS>
__global__ void __launch_bounds__(256)
log_evidence_kernel(const NodeMeta* __restrict__ nodes, int n_nodes, const int32_t* __restrict__ e_card,
                    const T* __restrict__ cpt, const T* __restrict__ pl_all, const T* __restrict__ msg0,
                    const T* __restrict__ msg1, int PL, int M, int TBi, int64_t n_valid,
                    const uint8_t* __restrict__ status, const int32_t* __restrict__ sweeps,
                    const int32_t* __restrict__ orig, int only_frozen, double* __restrict__ out,
                    int32_t* __restrict__ out_sweeps, uint8_t* __restrict__ out_conv,
                    const double* __restrict__ weights, double* __restrict__ counts)
{
    // orig / only_frozen: as belief_tiled_kernel (position p holds case orig[p] of the chunk; 1: only the retired
    // cases, whose state is final).  out_sweeps / out_conv: written here when no belief kernel runs (no marginals asked)
    // COUNTS: also the expected family counts (see the count pass below); out may then be NULL, weights is NULL or
    // indexed by the chunk's case.  Every thread of the block walks the count pass, with or without a case.
    extern __shared__ double logev_scr[];
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool has_case = true;
    if (!COUNTS) {
        if (p >= n_valid) return;
        if (only_frozen && (status[p] == 0) == (only_frozen == 1)) return;
    } else {
        has_case = p < n_valid && !(only_frozen && (status[p] == 0) == (only_frozen == 1));
    }
    const int nt = blockDim.x;
    // COUNTS: the block's reduction slots [nt / 32][32] come first
    double* const acc = logev_scr + (COUNTS ? nt : 0) + threadIdx.x;   // acc[i * nt]: b_X(x) at [0, r), b_X(u_j) at [r, r + r_j)
    const size_t TB = (size_t)TBi;
    const T* pl = nullptr;
    const T* msg = nullptr;
    double score = 0.0;
    int64_t dcase = 0;
    if (has_case) {
        const size_t tile = (size_t)(p / TBi), lane = (size_t)(p % TBi);
        pl = pl_all + tile * PL * TB + lane;
        msg = (((sweeps[p] - 1) & 1) ? msg1 : msg0) + tile * M * TB + lane;

        double total = 0.0;
        bool any_nan = false, any_zero = false;
        for (int X = 0; X < n_nodes; ++X) {
            const NodeMeta nd = nodes[X];
            const int r = nd.card, k = nd.k;
            const T* const lam = pl + (size_t)(nd.pl_off + r) * TB;
            const T* const P = cpt + nd.cpt_off;
            int rj[KMAX], slot[KMAX];
            int64_t Q = 1;
            for (int j = 0, s = nd.pin_off; j < k; ++j) {
                rj[j] = e_card[nd.e0 + j];
                slot[j] = s;
                s += rj[j];
                Q *= rj[j];
            }
            double Z = 0.0, t_par = 0.0;
            const int passes = k > 0 ? k : 1;
            for (int jp = 0; jp < passes; ++jp) {
                if (jp == 0)
                    for (int x = 0; x < r; ++x) acc[x * nt] = 0.0;
                if (k > 0)
                    for (int a = 0; a < rj[jp]; ++a) acc[(r + a) * nt] = 0.0;
                int cfg[KMAX];
                for (int j = 0; j < k; ++j) cfg[j] = 0;
                for (int64_t q = 0; q < Q; ++q) {
                    double pu = 1.0;
                    for (int j = 0; j < k; ++j) pu *= (double)msg[(size_t)(slot[j] + cfg[j]) * TB];
                    const T* const row = P + q * r;
                    double s = 0.0;
                    for (int x = 0; x < r; ++x) {
                        const double w = (double)__ldg(row + x) * (double)lam[(size_t)x * TB] * pu;
                        s += w;
                        if (jp == 0) acc[x * nt] += w;
                    }
                    if (k > 0) acc[(r + cfg[jp]) * nt] += s;
                    if (jp == 0) Z += s;
                    for (int j = k - 1; j >= 0; --j) {            // odometer, last parent fastest (the CPT's row order)
                        if (++cfg[j] < rj[j]) break;
                        cfg[j] = 0;
                    }
                }
                if (k > 0)
                    for (int a = 0; a < rj[jp]; ++a) {
                        const double b = acc[(r + a) * nt];
                        if (b > 0.0) t_par += b * log((double)msg[(size_t)(slot[jp] + a) * TB]);
                    }
            }
            if (isnan(Z)) { any_nan = true; continue; }
            if (Z == 0.0) { any_zero = true; continue; }
            const double iz = 1.0 / Z;
            double t = log(Z) - t_par * iz;
            for (int x = 0; x < r; ++x) {
                const double b = acc[x * nt] * iz;
                if (b > 0.0) t += b * ((double)nd.m * log(b) - log((double)lam[(size_t)x * TB]));
            }
            total += t;
        }
        dcase = orig ? (int64_t)orig[p] : p;
        score = any_nan ? (double)NAN : (any_zero ? -(double)INFINITY : total);
        if (!COUNTS || out) out[dcase] = score;
        if (out_sweeps) out_sweeps[dcase] = sweeps[p];
        if (out_conv) out_conv[dcase] = status[p];
    }
    if (!COUNTS) return;

    // Count pass: counts[cpt_off + q r + x] += w_c P(x|u_q) lambda_X(x) prod_j pm_j(u_qj) / Z_X for a case whose score is
    // finite (every Z_X is then finite and non-zero; Z_X is summed again in the score pass's order).  All threads walk the
    // same (X, q, x) sequence: each entry is summed over the warp with shuffles, the warp sums wait in shared memory for
    // 32 entries, and one thread per entry adds the block's sum with one fp64 atomicAdd (none when the sum is 0).
    const double wc = (has_case && isfinite(score)) ? (weights ? weights[dcase] : 1.0) : 0.0;
    const bool counted = wc != 0.0;
    const int warp = threadIdx.x >> 5, wl = threadIdx.x & 31, nw = nt >> 5;
    for (int X = 0; X < n_nodes; ++X) {
        const NodeMeta nd = nodes[X];
        const int r = nd.card, k = nd.k;
        const T* const lam = counted ? pl + (size_t)(nd.pl_off + r) * TB : nullptr;
        const T* const P = cpt + nd.cpt_off;
        int rj[KMAX], slot[KMAX], cfg[KMAX];
        int64_t Q = 1;
        for (int j = 0, s = nd.pin_off; j < k; ++j) {
            rj[j] = e_card[nd.e0 + j];
            slot[j] = s;
            s += rj[j];
            Q *= rj[j];
        }
        double scale = 0.0;
        if (counted) {
            double Z = 0.0;
            for (int j = 0; j < k; ++j) cfg[j] = 0;
            for (int64_t q = 0; q < Q; ++q) {
                double pu = 1.0;
                for (int j = 0; j < k; ++j) pu *= (double)msg[(size_t)(slot[j] + cfg[j]) * TB];
                const T* const row = P + q * r;
                double s = 0.0;
                for (int x = 0; x < r; ++x) s += (double)__ldg(row + x) * (double)lam[(size_t)x * TB] * pu;
                Z += s;
                for (int j = k - 1; j >= 0; --j) {
                    if (++cfg[j] < rj[j]) break;
                    cfg[j] = 0;
                }
            }
            scale = wc / Z;
        }
        for (int j = 0; j < k; ++j) cfg[j] = 0;
        int64_t base = nd.cpt_off;
        int fill = 0;
        for (int64_t q = 0; q < Q; ++q) {
            double pu = 1.0;
            if (counted)
                for (int j = 0; j < k; ++j) pu *= (double)msg[(size_t)(slot[j] + cfg[j]) * TB];
            const T* const row = P + q * r;
            for (int x = 0; x < r; ++x) {
                double v = counted ? (double)__ldg(row + x) * (double)lam[(size_t)x * TB] * pu * scale : 0.0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                if (wl == 0) logev_scr[warp * 32 + fill] = v;
                if (++fill == 32 || (q == Q - 1 && x == r - 1)) {
                    __syncthreads();
                    if (threadIdx.x < fill) {
                        double sum = 0.0;
                        for (int w = 0; w < nw; ++w) sum += logev_scr[w * 32 + threadIdx.x];
                        if (sum != 0.0) atomicAdd(counts + base + threadIdx.x, sum);
                    }
                    __syncthreads();
                    base += fill;
                    fill = 0;
                }
            }
            for (int j = k - 1; j >= 0; --j) {
                if (++cfg[j] < rj[j]) break;
                cfg[j] = 0;
            }
        }
    }
}

} // namespace bnbp
