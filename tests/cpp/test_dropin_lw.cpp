// Own tests of the drop-in likelihood_weighting.hpp and sampler.hpp (SURVEY 8 f2 / f3): the reference's
// call shapes, on the CUDA backend.  Runs on a B200 (calls libbnbp).
#define BOOST_TEST_MAIN
#include <boost/test/included/unit_test.hpp>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <fstream>

#include <unistd.h>

#include "bayesian/graph.hpp"
#include "bayesian/inference/belief_propagation.hpp"
#include "bayesian/inference/likelihood_weighting.hpp"
#include "bayesian/sampler.hpp"

namespace {

bn::graph_t pearl()
{
    bn::graph_t g;
    auto r = g.add_vertex(), s = g.add_vertex(), w = g.add_vertex(), h = g.add_vertex();
    g.add_edge(r, w); g.add_edge(r, h); g.add_edge(s, h);
    for (auto const& v : g.vertex_list()) v->selectable_num = 2;
    r->cpt.assign({}, r); r->cpt[bn::condition_t()].second = {0.2, 0.8};
    s->cpt.assign({}, s); s->cpt[bn::condition_t()].second = {0.1, 0.9};
    w->cpt.assign({r}, w);
    w->cpt[{{r, 0}}].second = {1.0, 0.0};
    w->cpt[{{r, 1}}].second = {0.2, 0.8};
    h->cpt.assign({r, s}, h);
    h->cpt[{{r, 0}, {s, 0}}].second = {1.0, 0.0};
    h->cpt[{{r, 0}, {s, 1}}].second = {1.0, 0.0};
    h->cpt[{{r, 1}, {s, 0}}].second = {0.9, 0.1};
    h->cpt[{{r, 1}, {s, 1}}].second = {0.0, 1.0};
    return g;
}

} // namespace

BOOST_AUTO_TEST_CASE(lw_lands_on_the_exact_posterior_of_a_polytree)
{
    bn::graph_t g = pearl();
    auto const& v = g.vertex_list();
    bn::inference::likelihood_weighting lw(g);
    lw.set_seed(7);
    bn::inference::likelihood_weighting::evidence_list ev;
    ev[v[3]] = 0;                                       // H = 0, the reference's own BP test case
    auto const res = lw(ev, 400000);
    // exact posterior (libs/bayesian/test/belief_propagation.cpp:92-121): R 0.7353/0.2647, S 0.3382/0.6618, W 0.7882/0.2118
    double const want[4][2] = {{0.7352941176470589, 0.2647058823529412}, {0.3382352941176471, 0.6617647058823529},
                               {0.7882352941176471, 0.21176470588235297}, {1.0, 0.0}};
    for (int i = 0; i < 4; ++i)
        for (int s = 0; s < 2; ++s) BOOST_CHECK(std::fabs(res.at(v[i])[0][s] - want[i][s]) < 0.01);
    // batched overload, and agreement with belief_propagation on the same evidence
    std::vector<bn::inference::likelihood_weighting::evidence_list> cases(3);
    cases[1][v[2]] = 1;
    cases[2][v[3]] = 1; cases[2][v[0]] = 1;
    auto const many = lw(cases, 200000);
    bn::inference::belief_propagation bp(g);
    bn::inference::belief_propagation::options opt;
    opt.epsilon = 1e-9;
    std::vector<bn::condition_t> conds(3);
    conds[1][v[2]] = 1;
    conds[2][v[3]] = 1; conds[2][v[0]] = 1;
    auto const exact = bp(conds, opt);
    for (std::size_t c = 0; c < 3; ++c)
        for (int i = 0; i < 4; ++i)
            for (int s = 0; s < 2; ++s) BOOST_CHECK(std::fabs(many[c].at(v[i])[0][s] - exact[c].at(v[i])[0][s]) < 0.01);
}

BOOST_AUTO_TEST_CASE(sampler_make_cpt_counts_on_the_device)
{
    bn::graph_t g;
    auto a = g.add_vertex(), b = g.add_vertex();
    g.add_edge(a, b);
    a->selectable_num = 2; b->selectable_num = 2;
    std::unordered_map<bn::condition_t, std::size_t> table;
    table[{{a, 0}, {b, 0}}] = 5;
    table[{{a, 0}, {b, 1}}] = 1;
    table[{{a, 1}, {b, 1}}] = 4;
    bn::sampler smp;
    BOOST_CHECK(!smp.make_cpt(g));                       // nothing loaded yet (sampler.hpp:84)
    BOOST_CHECK(smp.load_sample(table));
    BOOST_CHECK(smp.sampling_size() == 10);
    BOOST_CHECK(smp.make_cpt(g));
    BOOST_CHECK(a->cpt[bn::condition_t()].second == (std::vector<double>{0.6, 0.4}));
    BOOST_CHECK((b->cpt[{{a, 0}}].second == std::vector<double>{5.0 / 6.0, 1.0 / 6.0}));
    BOOST_CHECK((b->cpt[{{a, 1}}].second == std::vector<double>{0.0, 1.0}));
    // the reference's sample-file format: "count s_0 s_1" per line
    // (a file of its own: on a shared machine a fixed name under /tmp may belong to another user)
    char path[] = "/tmp/bnbp_test_samples_XXXXXX";
    const int fd = mkstemp(path);
    BOOST_CHECK(fd >= 0);
    if (fd >= 0) close(fd);
    { std::ofstream f(path); f << "3 0 0\n1 0 1\n"; }
    bn::sampler from_file(path);
    BOOST_CHECK(from_file.load_sample(g.vertex_list()));
    BOOST_CHECK(from_file.sampling_size() == 4);
    BOOST_CHECK(from_file.make_cpt(g));
    BOOST_CHECK((a->cpt[bn::condition_t()].second == std::vector<double>{1.0, 0.0}));
    BOOST_CHECK((b->cpt[{{a, 0}}].second == std::vector<double>{0.75, 0.25}));
    BOOST_CHECK((b->cpt[{{a, 1}}].second == std::vector<double>{0.5, 0.5}));     // never seen: uniform (:147-151)
    std::remove(path);
    // matrix_type helpers of the batched front ends
    bn::matrix_type const e = bn::matrix_type::row({0.3, 0.7});
    BOOST_CHECK(e.height() == 1 && e.width() == 2 && e.flat() == (std::vector<double>{0.3, 0.7}));
    BOOST_CHECK(std::fabs((e % e).normalized()[0][1] - 0.49 / 0.58) < 1e-15);     // belief of a soft-evidence node (SURVEY 0.4)
    BOOST_CHECK(e.same_shape(e.normalized()) && std::fabs(e.sum() - 1.0) < 1e-15);
}
