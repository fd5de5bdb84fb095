/* logev_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The reference computation the GPU log-evidence (csrc/bnbp_logev.cuh, bnbp_run_batch_log_evidence) is checked
 * against.  It runs oracle/bp_oracle.c's own run_case -- the pinned C restatement of the reference's loopy BP,
 * included here unchanged -- and scores each case from the state run_case leaves.  Built and loaded by
 * tests/logev_oracle.py. */
#include "../oracle/bp_oracle.c"

/* ------------------------------------------------------------------------------------------------
 * Log-evidence (extension, no reference counterpart): the Bethe estimate log Z_B of ln P(e) from run_case's state.
 * After the commit swap (:135-143) s->lam holds the rows of the last sweep T and s->npmsg the pi-messages that sweep
 * READ (the committed messages of sweep T-1, damped if damping is on; all ones for T = 1).  Per node X:
 *   Z_X = sum_{x,u} P(x|u) lam_X(x) prod_j pm_j(u_j),  b_X = that product / Z_X
 *   log Z_B = sum_X [ ln Z_X - sum_x b_X(x) ln lam_X(x) - sum_j sum_u b_X(u_j=u) ln pm_j(u) + m_X sum_x b_X(x) ln b_X(x) ]
 * Terms of weight 0 contribute 0; a NaN Z_X gives NaN, else a zero Z_X gives -inf. */
static double log_evidence(const net_t* g, state_t* s, double* bx, double* bu)
{
    double total = 0.0;
    int any_nan = 0, any_zero = 0;
    for (int32_t x = 0; x < g->n; ++x) {
        int32_t r = g->card[x], e0 = g->poff[x], k = g->poff[x + 1] - e0;
        int32_t m = g->choff[x + 1] - g->choff[x];
        const double* cpt = g->cpt + g->coff[x];
        const double* lam = s->lam + g->voff[x];
        int64_t Q = 1;
        for (int32_t j = 0; j < k; ++j) { Q *= g->card[g->par[e0 + j]]; s->cfg[j] = 0; }
        for (int32_t i = 0; i < r; ++i) bx[i] = 0.0;
        for (int64_t i = 0; i < g->moff[e0 + k] - g->moff[e0]; ++i) bu[i] = 0.0;
        double Z = 0.0;
        for (int64_t q = 0; q < Q; ++q) {
            double pu = 1.0;
            for (int32_t j = 0; j < k; ++j) pu *= s->npmsg[g->moff[e0 + j] + s->cfg[j]];
            double sq = 0.0;
            for (int32_t i = 0; i < r; ++i) {
                double w = cpt[q * r + i] * lam[i] * pu;
                bx[i] += w;
                sq += w;
            }
            for (int32_t j = 0; j < k; ++j) bu[g->moff[e0 + j] - g->moff[e0] + s->cfg[j]] += sq;
            Z += sq;
            for (int32_t j = k - 1; j >= 0; --j) {
                if (++s->cfg[j] < g->card[g->par[e0 + j]]) break;
                s->cfg[j] = 0;
            }
        }
        if (isnan(Z)) { any_nan = 1; continue; }
        if (Z == 0.0) { any_zero = 1; continue; }
        double t = log(Z);
        for (int32_t i = 0; i < r; ++i) {
            double b = bx[i] / Z;
            if (b > 0.0) t += (double)m * b * log(b) - b * log(lam[i]);
        }
        for (int32_t j = 0; j < k; ++j)
            for (int32_t u = 0; u < g->card[g->par[e0 + j]]; ++u) {
                double b = bu[g->moff[e0 + j] - g->moff[e0] + u] / Z;
                if (b > 0.0) t -= b * log(s->npmsg[g->moff[e0 + j] + u]);
            }
        total += t;
    }
    return any_nan ? NAN : (any_zero ? -INFINITY : total);
}

/* bp_oracle_run (sum-product) that also returns each case's log-evidence (log_evidence above) in out_log_evidence. */
int bp_oracle_run_log_evidence(int32_t n_nodes, const int32_t* card, const int32_t* parent_off,
                               const int32_t* parents, const int64_t* cpt_off, const double* cpt,
                               int64_t n_cases, const int64_t* ev_off, const int32_t* ev_node,
                               const int32_t* ev_state, double eps, int32_t max_sweeps, double damping,
                               int32_t check_interval, int32_t n_threads,
                               double* out_marginals, int32_t* out_sweeps, uint8_t* out_converged,
                               double* out_log_evidence)
{
    net_t g;
    memset(&g, 0, sizeof g);
    g.n = n_nodes; g.card = card; g.poff = parent_off; g.par = parents; g.coff = cpt_off; g.cpt = cpt;
    if (build_net(&g)) return -1;
    if (max_sweeps <= 0) max_sweeps = 1 << 30;
    if (check_interval <= 0) check_interval = 1;
    int64_t V = g.voff[n_nodes], M = g.moff[g.poff[n_nodes]];
    int err = 0;
#ifdef _OPENMP
    if (n_threads <= 0) n_threads = omp_get_max_threads();
#else
    n_threads = 1;
#endif
#pragma omp parallel num_threads(n_threads)
    {
        state_t s;
        memset(&s, 0, sizeof s);
        double* bx = (double*)malloc(sizeof(double) * ((size_t)V + 1));
        double* bu = (double*)malloc(sizeof(double) * ((size_t)M + 1));
        if (alloc_state(&g, &s) || !bx || !bu) {
#pragma omp atomic write
            err = -1;
        } else {
#pragma omp for schedule(dynamic, 4)
            for (int64_t c = 0; c < n_cases; ++c) {
                int64_t a = ev_off ? ev_off[c] : 0, b = ev_off ? ev_off[c + 1] : 0;
                run_case(&g, &s, b - a, ev_node + a, ev_state ? ev_state + a : NULL, NULL, NULL,
                         eps, max_sweeps, damping, check_interval,
                         out_marginals + c * V,
                         out_sweeps ? out_sweeps + c : NULL,
                         out_converged ? out_converged + c : NULL);
                out_log_evidence[c] = log_evidence(&g, &s, bx, bu);
            }
        }
        free(bx); free(bu);
        free_state(&s);
    }
    free_net(&g);
    return err;
}
