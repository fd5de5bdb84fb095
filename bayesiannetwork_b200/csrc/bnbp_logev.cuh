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
#pragma once
#include "bnbp_kernels.cuh"

namespace bnbp {

template <typename T>
__global__ void __launch_bounds__(256)
log_evidence_kernel(const NodeMeta* __restrict__ nodes, int n_nodes, const int32_t* __restrict__ e_card,
                    const T* __restrict__ cpt, const T* __restrict__ pl_all, const T* __restrict__ msg0,
                    const T* __restrict__ msg1, int PL, int M, int TBi, int64_t n_valid,
                    const uint8_t* __restrict__ status, const int32_t* __restrict__ sweeps,
                    const int32_t* __restrict__ orig, int only_frozen, double* __restrict__ out,
                    int32_t* __restrict__ out_sweeps, uint8_t* __restrict__ out_conv)
{
    // orig / only_frozen: as belief_tiled_kernel (position p holds case orig[p] of the chunk; 1: only the retired
    // cases, whose state is final).  out_sweeps / out_conv: written here when no belief kernel runs (no marginals asked)
    extern __shared__ double logev_scr[];
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_valid) return;
    if (only_frozen && (status[p] == 0) == (only_frozen == 1)) return;
    const int nt = blockDim.x;
    double* const acc = logev_scr + threadIdx.x;          // acc[i * nt]: b_X(x) at [0, r), b_X(u_j) at [r, r + r_j)
    const size_t TB = (size_t)TBi;
    const size_t tile = (size_t)(p / TBi), lane = (size_t)(p % TBi);
    const T* const pl = pl_all + tile * PL * TB + lane;
    const T* const msg = (((sweeps[p] - 1) & 1) ? msg1 : msg0) + tile * M * TB + lane;

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
    const int64_t dcase = orig ? (int64_t)orig[p] : p;
    out[dcase] = any_nan ? (double)NAN : (any_zero ? -(double)INFINITY : total);
    if (out_sweeps) out_sweeps[dcase] = sweeps[p];
    if (out_conv) out_conv[dcase] = status[p];
}

} // namespace bnbp
