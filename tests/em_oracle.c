/* em_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The reference computation the GPU expected family counts (csrc/bnbp_logev.cuh with COUNTS, bnbp_run_batch_expected_counts)
 * are checked against.  It includes logev_oracle.c, which includes the pinned oracle/bp_oracle.c unchanged, runs that
 * restatement's own run_case per case, scores the case with logev_oracle.c's log_evidence and then adds the case's family
 * posteriors from the same state.  Cases are added serially in case order, so the result is deterministic.  Built and
 * loaded by tests/em_oracle.py. */
#include "logev_oracle.c"

/* counts[coff[X] + q r + x] += w P(x|u_q) lam_X(x) prod_j pm_j(u_qj) / Z_X for every node X, from the state run_case
 * leaves (s->lam: the rows of the last sweep; s->npmsg: the pi-messages that sweep read).  Z_X is summed in
 * log_evidence's order. */
static void add_family_posteriors(const net_t* g, state_t* s, double w, double* counts)
{
    for (int32_t x = 0; x < g->n; ++x) {
        int32_t r = g->card[x], e0 = g->poff[x], k = g->poff[x + 1] - e0;
        const double* cpt = g->cpt + g->coff[x];
        const double* lam = s->lam + g->voff[x];
        int64_t Q = 1;
        for (int32_t j = 0; j < k; ++j) { Q *= g->card[g->par[e0 + j]]; s->cfg[j] = 0; }
        double Z = 0.0;
        for (int64_t q = 0; q < Q; ++q) {
            double pu = 1.0;
            for (int32_t j = 0; j < k; ++j) pu *= s->npmsg[g->moff[e0 + j] + s->cfg[j]];
            double sq = 0.0;
            for (int32_t i = 0; i < r; ++i) sq += cpt[q * r + i] * lam[i] * pu;
            Z += sq;
            for (int32_t j = k - 1; j >= 0; --j) {
                if (++s->cfg[j] < g->card[g->par[e0 + j]]) break;
                s->cfg[j] = 0;
            }
        }
        for (int32_t j = 0; j < k; ++j) s->cfg[j] = 0;
        for (int64_t q = 0; q < Q; ++q) {
            double pu = 1.0;
            for (int32_t j = 0; j < k; ++j) pu *= s->npmsg[g->moff[e0 + j] + s->cfg[j]];
            for (int32_t i = 0; i < r; ++i) counts[g->coff[x] + q * r + i] += w * (cpt[q * r + i] * lam[i] * pu) / Z;
            for (int32_t j = k - 1; j >= 0; --j) {
                if (++s->cfg[j] < g->card[g->par[e0 + j]]) break;
                s->cfg[j] = 0;
            }
        }
    }
}

/* bp_oracle_run_log_evidence, serial, that also ADDS each case's family posteriors (weight weights[c], 1 when weights is
 * NULL) into counts [cpt_off[n_nodes]].  A case whose log-evidence is not finite adds nothing. */
int bp_oracle_run_expected_counts(int32_t n_nodes, const int32_t* card, const int32_t* parent_off,
                                  const int32_t* parents, const int64_t* cpt_off, const double* cpt,
                                  int64_t n_cases, const int64_t* ev_off, const int32_t* ev_node,
                                  const int32_t* ev_state, const double* weights, double eps, int32_t max_sweeps,
                                  double damping, int32_t check_interval, double* counts,
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
    state_t s;
    memset(&s, 0, sizeof s);
    double* bx = (double*)malloc(sizeof(double) * ((size_t)V + 1));
    double* bu = (double*)malloc(sizeof(double) * ((size_t)M + 1));
    int err = 0;
    if (alloc_state(&g, &s) || !bx || !bu) {
        err = -1;
    } else {
        for (int64_t c = 0; c < n_cases; ++c) {
            int64_t a = ev_off ? ev_off[c] : 0, b = ev_off ? ev_off[c + 1] : 0;
            run_case(&g, &s, b - a, ev_node + a, ev_state ? ev_state + a : NULL, NULL, NULL,
                     eps, max_sweeps, damping, check_interval,
                     out_marginals + c * V,
                     out_sweeps ? out_sweeps + c : NULL,
                     out_converged ? out_converged + c : NULL);
            double le = log_evidence(&g, &s, bx, bu);
            out_log_evidence[c] = le;
            double w = weights ? weights[c] : 1.0;
            if (isfinite(le) && w != 0.0) add_family_posteriors(&g, &s, w, counts);
        }
    }
    free(bx); free(bu);
    free_state(&s);
    free_net(&g);
    return err;
}
