// options::log_evidence through run_flat on the reference's chain A -> B -> C -> D (libs/bayesian/test/
// belief_propagation.cpp:127-182): prints one line per case, "<sweeps> <log-evidence %.17g>".  Built and run by
// tests/test_gpu_log_evidence.py, which compares the lines with the Python binding's result.
#include <bayesian/graph.hpp>
#include <bayesian/inference/belief_propagation.hpp>

#include <cstdio>
#include <vector>

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

    // cases over vertex_list() indices: {D=0}, {D=1}, {D=2}, {A=1, C=0}, {}
    std::vector<std::int64_t> ev_off = {0, 1, 2, 3, 5, 5};
    std::vector<std::int32_t> ev_node = {3, 3, 3, 0, 2};
    std::vector<std::int32_t> ev_state = {0, 1, 2, 1, 0};
    bnbp_evidence ev;
    ev.n_cases = 5;
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
    auto const res = bp.run_flat(ev, opt);
    if (res.log_evidence.size() != 5) return 1;
    for (std::size_t i = 0; i < res.n_cases; ++i) std::printf("%d %.17g\n", (int)res.sweeps[i], res.log_evidence[i]);
    return 0;
}
