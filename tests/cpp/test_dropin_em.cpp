// Three EM iterations through options::expected_counts and run_flat on the reference's chain A -> B -> C -> D
// (libs/bayesian/test/belief_propagation.cpp:127-182), starting from its CPTs: each M-step normalises the rows of
// flat_result::expected_counts and writes them back through the vertices' cpt_t, which the next run_flat picks up.
// Prints one line per iteration, "L <sum of the cases' log-evidence under the CPT going in %.17g>", then one line
// "CPT" followed by the final CPT arena (vertex_list() order).  Built and run by tests/test_gpu_em.py, which compares
// with BeliefPropagation.em of the Python binding.
#include <bayesian/graph.hpp>
#include <bayesian/inference/belief_propagation.hpp>

#include <cstdio>
#include <vector>

namespace {

// row q of a node's counts block, normalised (make_cpt's rule: an all-zero row becomes uniform)
std::vector<double> row(std::vector<double> const& counts, std::size_t off, int r, int q)
{
    std::vector<double> out(static_cast<std::size_t>(r));
    double tot = 0.0;
    for (int x = 0; x < r; ++x) tot += counts[off + static_cast<std::size_t>(q * r + x)];
    for (int x = 0; x < r; ++x)
        out[static_cast<std::size_t>(x)] = tot == 0.0 ? 1.0 / r : counts[off + static_cast<std::size_t>(q * r + x)] / tot;
    return out;
}

} // namespace

int main()
{
    bn::graph_t g;
    auto a = g.add_vertex(), b = g.add_vertex(), c = g.add_vertex(), d = g.add_vertex();
    g.add_edge(a, b); g.add_edge(b, c); g.add_edge(c, d);
    a->selectable_num = 3; b->selectable_num = 3; c->selectable_num = 2; d->selectable_num = 3;
    a->cpt.assign({}, a); a->cpt[bn::condition_t()].second = {0.30, 0.60, 0.10};
    b->cpt.assign({a}, b);
    b->cpt[{{a, 0}}].second = {0.20, 0.30, 0.50};
    b->cpt[{{a, 1}}].second = {0.30, 0.30, 0.40};
    b->cpt[{{a, 2}}].second = {0.80, 0.10, 0.10};
    c->cpt.assign({b}, c);
    c->cpt[{{b, 0}}].second = {0.50, 0.50};
    c->cpt[{{b, 1}}].second = {0.70, 0.30};
    c->cpt[{{b, 2}}].second = {0.40, 0.60};
    d->cpt.assign({c}, d);
    d->cpt[{{c, 0}}].second = {0.40, 0.30, 0.30};
    d->cpt[{{c, 1}}].second = {0.20, 0.60, 0.20};

    // cases over vertex_list() indices: {D=0}, {D=1}, {D=2}, {A=1, C=0}, {}, {A=0, B=2}, {B=1, D=2}, {A=2, C=1, D=0}
    std::vector<std::int64_t> ev_off = {0, 1, 2, 3, 5, 5, 7, 9, 12};
    std::vector<std::int32_t> ev_node = {3, 3, 3, 0, 2, 0, 1, 1, 3, 0, 2, 3};
    std::vector<std::int32_t> ev_state = {0, 1, 2, 1, 0, 0, 2, 1, 2, 2, 1, 0};
    bnbp_evidence ev;
    ev.n_cases = 8;
    ev.ev_off = ev_off.data();
    ev.ev_node = ev_node.data();
    ev.ev_state = ev_state.data();
    ev.ev_val_off = nullptr;
    ev.ev_values = nullptr;

    bn::inference::belief_propagation bp(g);
    bn::inference::belief_propagation::options opt;
    opt.epsilon = 0.0;
    opt.max_sweeps = 20;
    opt.log_evidence = true;
    opt.expected_counts = true;
    std::vector<double> cpt;
    for (int it = 0; it < 3; ++it) {
        auto const res = bp.run_flat(ev, opt);
        if (res.expected_counts.size() != 24 || res.log_evidence.size() != 8) return 1;
        double L = 0.0;
        for (double v : res.log_evidence) L += v;
        std::printf("L %.17g\n", L);
        std::vector<double> const& n = res.expected_counts;      // blocks: A 0..2, B 3..11, C 12..17, D 18..23
        a->cpt[bn::condition_t()].second = row(n, 0, 3, 0);
        for (int q = 0; q < 3; ++q) b->cpt[{{a, q}}].second = row(n, 3, 3, q);
        for (int q = 0; q < 3; ++q) c->cpt[{{b, q}}].second = row(n, 12, 2, q);
        for (int q = 0; q < 2; ++q) d->cpt[{{c, q}}].second = row(n, 18, 3, q);
        cpt.clear();
        for (double v : row(n, 0, 3, 0)) cpt.push_back(v);
        for (int q = 0; q < 3; ++q) for (double v : row(n, 3, 3, q)) cpt.push_back(v);
        for (int q = 0; q < 3; ++q) for (double v : row(n, 12, 2, q)) cpt.push_back(v);
        for (int q = 0; q < 2; ++q) for (double v : row(n, 18, 3, q)) cpt.push_back(v);
    }
    std::printf("CPT");
    for (double v : cpt) std::printf(" %.17g", v);
    std::printf("\n");
    return 0;
}
