// bayesian/inference/belief_propagation.hpp — bn::inference::belief_propagation on B200.
//
// Drop-in for the reference class (godai0519/BayesianNetwork,
// bayesian/inference/belief_propagation.hpp:12-339): same constructor, same two operator()
// overloads, same return type, same numbers (Pearl pi/lambda loopy BP, synchronous schedule,
// stop when the largest message change is < epsilon).  Nothing is computed on the host: the
// network is flattened once (bn::flatten, graph.hpp) and every sweep runs in the CUDA kernels of
// libbnbp behind the C ABI of <bnbp.h>.  Link with -lbnbp.  There is no CPU fallback: without a
// B200 the constructor throws.
//
//   reference member (belief_propagation.hpp)              here
//   -----------------------------------------------------  -------------------------------------------
//   belief_propagation(graph_t const&)              :16-19  keeps a (shallow) graph copy like the
//                                                           reference; flattens + bnbp_create lazily
//   operator()(double eps = 0.001)                  :24-28  same
//   operator()(precondition map, double eps)        :31-159 one-case batch through bnbp_run_batch
//   return_type = unordered_map<vertex, matrix>     :14     same; every matrix is 1 x selectable_num
//   (state maps pi_, lambda_, pi_i_, lambda_k_ ...) :320-333 device arena inside libbnbp
//
// The reference reads vertex->cpt at call time, so CPT edits between calls are visible
// (graph.hpp:157-161).  That is preserved: every call re-flattens the (host) network, re-uploads
// the CPT arena when only values changed and rebuilds the device handle when the topology did.
//
// New, because the GPU wants batches (the reference takes one evidence set per call):
//   operator()(std::vector<precondition_type> const&, options)  -> std::vector<return_type>
//   operator()(std::vector<condition_t> const&, options)        hard evidence vertex -> state, the
//                                                               evidence type of likelihood_weighting
//                                                               (likelihood_weighting.hpp:15,28)
//   run_flat(bnbp_evidence const&, options)                     zero-copy CSR evidence in, flat
//                                                               marginals out (10^5-10^6 cases)
//   options::devices                                            several GPUs of the box behind one object: cases shard
//                                                               by contiguous ranges, NCCL inside libbnbp (SURVEY 8e)
//   options::query / float_marginals                            run_flat: only the asked-for vertices / floats leave the
//                                                               device; results land in page-locked memory (pinned_buffer)
//   loopy_belief_propagation                                    alias (the north-star name)
#ifndef BNB200_BAYESIAN_INFERENCE_BELIEF_PROPAGATION_HPP
#define BNB200_BAYESIAN_INFERENCE_BELIEF_PROPAGATION_HPP

#include <cstddef>
#include <cstdint>
#include <new>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <vector>

#include <bayesian/graph.hpp>
#include <bayesian/matrix.hpp>
#include <bnbp.h>

namespace bn {
namespace inference {

// Result storage of the flat call: page-locked host memory from libbnbp (bnbp_host_alloc), so the device-to-host
// copy of the marginals runs at the link rate and overlaps the kernels; a std::vector would be pageable (the copy
// goes through a driver bounce buffer at a fraction of the rate and blocks the calling thread) and zero-filled
// first (for 1M alarm37 cases a 0.9 GB memset).  The contents after resize() are unspecified.
template <class T> class pinned_buffer {
public:
    pinned_buffer() : data_(nullptr), size_(0), cap_(0) {}
    ~pinned_buffer() { bnbp_host_free(data_); }
    pinned_buffer(pinned_buffer&& o) : data_(o.data_), size_(o.size_), cap_(o.cap_) { o.data_ = nullptr; o.size_ = o.cap_ = 0; }
    pinned_buffer& operator=(pinned_buffer&& o)
    {
        if (this != &o) { bnbp_host_free(data_); data_ = o.data_; size_ = o.size_; cap_ = o.cap_; o.data_ = nullptr; o.size_ = o.cap_ = 0; }
        return *this;
    }
    pinned_buffer(pinned_buffer const&) = delete;
    pinned_buffer& operator=(pinned_buffer const&) = delete;
    void resize(std::size_t n)                         // contents are NOT preserved
    {
        if (n > cap_) {
            bnbp_host_free(data_);
            data_ = static_cast<T*>(bnbp_host_alloc(n * sizeof(T)));
            if (!data_) { size_ = cap_ = 0; throw std::bad_alloc(); }
            cap_ = n;
        }
        size_ = n;
    }
    T* data() { return data_; }
    T const* data() const { return data_; }
    std::size_t size() const { return size_; }
    bool empty() const { return size_ == 0; }
    T& operator[](std::size_t i) { return data_[i]; }
    T const& operator[](std::size_t i) const { return data_[i]; }
    T* begin() { return data_; }
    T* end() { return data_ + size_; }
    T const* begin() const { return data_; }
    T const* end() const { return data_ + size_; }
private:
    T* data_;
    std::size_t size_, cap_;
};

class belief_propagation {
public:
    typedef std::unordered_map<vertex_type, matrix_type> return_type;
    typedef std::unordered_map<vertex_type, matrix_type> precondition_type;

    // Run parameters of the batched overloads.  The defaults reproduce the reference: epsilon
    // 0.001 (:24), no sweep cap (:75 while(true)), no damping, delta tested after every sweep.
    struct options {
        double epsilon = 0.001;
        int max_sweeps = 0;          // 0 = unlimited, like the reference
        double damping = 0.0;        // extension; 0 = reference behaviour
        int check_interval = 1;      // extension; 1 = reference behaviour
        int precision = BNBP_FP64;   // the reference computes in double
        int device = -1;             // CUDA device ordinal, -1 = current
        int specialize = BNBP_SPEC_AUTO;
        int semiring = BNBP_SUM_PRODUCT;   // extension: BNBP_MAX_PRODUCT = max-marginals (the reference is sum-product)
        // several GPUs of this box (SURVEY 8e): a call shards its cases over these ordinals by contiguous ranges,
        // one host thread and stream set per device; {-1} = every visible device; empty = `device` alone.
        // Results do not depend on the sharding (bit for bit).
        std::vector<int> devices;
        // run_flat only -- what leaves the device (the map-returning overloads always return every vertex in double):
        std::vector<vertex_type> query;   // non-empty: only these vertices' marginals, in this order
        bool float_marginals = false;     // fp32 handles: marginals_f32 is filled instead of marginals (half the copy)
        bool log_evidence = false;        // flat_result::log_evidence: each case's Bethe estimate of ln P(e) (hard evidence)
        bool expected_counts = false;     // flat_result::expected_counts: the E-step of EM (bnbp_run_batch_expected_counts)
    };

    struct flat_result {
        std::size_t n_cases = 0;
        std::size_t values_per_case = 0;           // sum of selectable_num over the vertices of a row
        std::vector<std::size_t> vertex;           // vertex_list() index of the i-th vertex of a row (all, or the query)
        std::vector<std::size_t> offset;           // offset of that vertex inside one case's row
        pinned_buffer<double> marginals;           // [n_cases][values_per_case] (empty if float_marginals)
        pinned_buffer<float> marginals_f32;        // [n_cases][values_per_case] (only if float_marginals)
        pinned_buffer<std::int32_t> sweeps;        // sweeps executed per case
        pinned_buffer<std::uint8_t> converged;     // 1 if the case met delta < epsilon
        std::vector<double> log_evidence;          // options::log_evidence: per case (bnbp_run_batch_log_evidence), else empty
        // options::expected_counts: sum over the cases of P(x, u | e) per CPT entry, in the flat CPT arena of the graph
        // (vertex_list() order, rows by parent configuration, last parent fastest; each row normalised is the M-step,
        // written back through the vertices' cpt_t and picked up by the next call), else empty
        std::vector<double> expected_counts;
        bnbp_summary summary = bnbp_summary();     // totals over all devices (devices.size() > 1: all-reduced over NCCL)
    };

    explicit belief_propagation(graph_t const& graph) : graph_(graph) {}
    belief_propagation(graph_t const& graph, options const& opt) : graph_(graph), defaults_(opt) {}
    belief_propagation(belief_propagation const&) = delete;
    belief_propagation& operator=(belief_propagation const&) = delete;
    virtual ~belief_propagation() { release(); }

    // By-pass: no evidence (:24-28)
    inline return_type operator()(double const epsilon = 0.001)
    {
        precondition_type const none;
        return operator()(none, epsilon);
    }

    // Loopy belief propagation for one evidence set (:31-159).  precondition maps a vertex to its
    // 1 x selectable_num evidence row, which becomes both pi and lambda of that vertex (:69-73).
    return_type operator()(precondition_type const& precondition, double const epsilon = 0.001)
    {
        options opt = defaults_;
        opt.epsilon = epsilon;
        std::vector<precondition_type> const one(1, precondition);
        return std::move(operator()(one, opt).front());
    }

    // ---- batched overloads -------------------------------------------------------------------------
    std::vector<return_type> operator()(std::vector<precondition_type> const& cases, options const& opt)
    {
        sync_network(opt);
        std::vector<std::int64_t> ev_off(1, 0), ev_val_off(1, 0);
        std::vector<std::int32_t> ev_node;
        std::vector<double> ev_values;
        for (precondition_type const& one : cases) {
            for (auto const& entry : one) {
                std::size_t index = 0;
                if (!graph_.find_index(entry.first, index))
                    throw std::invalid_argument("belief_propagation: evidence on a vertex that is not in the graph");
                matrix_type const& row = entry.second;
                if (row.height() != 1 || row.width() != static_cast<std::size_t>(flat_.card[index]))
                    throw std::invalid_argument("belief_propagation: evidence must be a 1 x selectable_num matrix");
                ev_node.push_back(static_cast<std::int32_t>(index));
                ev_values.insert(ev_values.end(), row[0].begin(), row[0].end());
                ev_val_off.push_back(static_cast<std::int64_t>(ev_values.size()));
            }
            ev_off.push_back(static_cast<std::int64_t>(ev_node.size()));
        }
        bnbp_evidence ev;
        ev.n_cases = static_cast<std::int64_t>(cases.size());
        ev.ev_off = ev_off.data();
        ev.ev_node = ev_node.data();
        ev.ev_state = nullptr;
        ev.ev_val_off = ev_val_off.data();
        ev.ev_values = ev_values.empty() ? &zero_ : ev_values.data();   // non-NULL selects soft evidence
        return unpack(run_synced(ev, every_vertex_in_double(opt)));
    }

    std::vector<return_type> operator()(std::vector<condition_t> const& cases, options const& opt)
    {
        sync_network(opt);
        std::vector<std::int64_t> ev_off(1, 0);
        std::vector<std::int32_t> ev_node, ev_state;
        for (condition_t const& one : cases) {
            for (auto const& entry : one) {
                std::size_t index = 0;
                if (!graph_.find_index(entry.first, index))
                    throw std::invalid_argument("belief_propagation: evidence on a vertex that is not in the graph");
                ev_node.push_back(static_cast<std::int32_t>(index));
                ev_state.push_back(entry.second);
            }
            ev_off.push_back(static_cast<std::int64_t>(ev_node.size()));
        }
        bnbp_evidence ev;
        ev.n_cases = static_cast<std::int64_t>(cases.size());
        ev.ev_off = ev_off.data();
        ev.ev_node = ev_node.data();
        ev.ev_state = ev_state.data();
        ev.ev_val_off = nullptr;
        ev.ev_values = nullptr;
        return unpack(run_synced(ev, every_vertex_in_double(opt)));
    }

    // One hard-evidence case in the condition_t form (vertex -> state)
    return_type operator()(condition_t const& evidence, double const epsilon = 0.001)
    {
        options opt = defaults_;
        opt.epsilon = epsilon;
        std::vector<condition_t> const one(1, evidence);
        return std::move(operator()(one, opt).front());
    }

    // Zero-copy form: CSR evidence over vertex_list() indices (see bnbp_evidence in <bnbp.h>).
    flat_result run_flat(bnbp_evidence const& ev, options const& opt)
    {
        flat_result out;
        run_flat(ev, opt, out);
        return out;
    }

    // The same into a result the caller keeps between calls: its page-locked buffers are reused when they are large
    // enough (pinning 0.9 GB for 1M alarm37 cases costs a few hundred milliseconds -- more than ten calls).
    void run_flat(bnbp_evidence const& ev, options const& opt, flat_result& out)
    {
        sync_network(opt);
        run_synced(ev, opt, out);
    }

    // Statistics of the last run (device milliseconds, launches, bytes per case): bnbp_get_stats.
    bnbp_stats stats() const
    {
        bnbp_stats st;
        if (!handle_ || bnbp_get_stats(handle_, &st) != BNBP_OK) throw std::runtime_error(last_error("bnbp_get_stats"));
        return st;
    }

private:
    static std::string last_error(char const* what) { return std::string(what) + ": " + bnbp_last_error(); }

    void release()
    {
        if (handle_) bnbp_destroy(handle_);
        handle_ = nullptr;
    }

    // Bring the device arena in line with the host graph as it is NOW.
    void sync_network(options const& opt)
    {
        flat_network now = flatten(graph_);
        bool const same_handle = handle_ && opt.precision == precision_ && opt.device == device_ &&
                                 opt.specialize == specialize_ && opt.devices == devices_ && now.same_topology(flat_);
        if (same_handle) {
            if (now.cpt != flat_.cpt) {
                if (bnbp_refresh_cpt(handle_, now.cpt.data(), static_cast<std::int64_t>(now.cpt.size())) != BNBP_OK)
                    throw std::runtime_error(last_error("bnbp_refresh_cpt"));
                flat_.cpt.swap(now.cpt);
            }
            return;
        }
        release();
        flat_ = std::move(now);
        bnbp_flat_network net;
        net.n_nodes = static_cast<std::int32_t>(flat_.card.size());
        net.card = flat_.card.data();
        net.parent_off = flat_.parent_off.data();
        net.parents = flat_.parents.data();
        net.cpt_off = flat_.cpt_off.data();
        net.cpt = flat_.cpt.data();
        bnbp_options bo = bnbp_options();
        bo.precision = opt.precision;
        bo.device = opt.device;
        bo.specialize = opt.specialize;
        int rc;
        if (opt.devices.empty()) {
            rc = bnbp_create(&net, &bo, &handle_);
        } else {
            std::vector<std::int32_t> list(opt.devices.begin(), opt.devices.end());
            bool const all = list.size() == 1 && list[0] < 0;
            rc = bnbp_create_multi(&net, &bo, all ? nullptr : list.data(), all ? 0 : static_cast<std::int32_t>(list.size()), &handle_);
        }
        if (rc != BNBP_OK) {
            handle_ = nullptr;
            throw std::runtime_error(last_error(opt.devices.empty() ? "bnbp_create" : "bnbp_create_multi"));
        }
        precision_ = opt.precision;
        device_ = opt.device;
        specialize_ = opt.specialize;
        devices_ = opt.devices;
    }

    flat_result run_synced(bnbp_evidence const& ev, options const& opt)
    {
        flat_result out;
        run_synced(ev, opt, out);
        return out;
    }

    void run_synced(bnbp_evidence const& ev, options const& opt, flat_result& out)
    {
        out.n_cases = static_cast<std::size_t>(ev.n_cases);
        out.vertex.clear();
        std::vector<std::int32_t> query;
        for (vertex_type const& v : opt.query) {
            std::size_t index = 0;
            if (!graph_.find_index(v, index)) throw std::invalid_argument("belief_propagation: query vertex is not in the graph");
            query.push_back(static_cast<std::int32_t>(index));
            out.vertex.push_back(index);
        }
        if (query.empty())
            for (std::size_t i = 0; i < flat_.card.size(); ++i) out.vertex.push_back(i);
        out.offset.assign(out.vertex.size() + 1, 0);
        for (std::size_t i = 0; i < out.vertex.size(); ++i)
            out.offset[i + 1] = out.offset[i] + static_cast<std::size_t>(flat_.card[out.vertex[i]]);
        out.values_per_case = out.offset.back();
        void* dst;
        if (opt.float_marginals) { out.marginals.resize(0); out.marginals_f32.resize(out.n_cases * out.values_per_case); dst = out.marginals_f32.data(); }
        else { out.marginals_f32.resize(0); out.marginals.resize(out.n_cases * out.values_per_case); dst = out.marginals.data(); }
        out.sweeps.resize(out.n_cases);
        out.converged.resize(out.n_cases);
        bnbp_run_params prm = bnbp_run_params();
        prm.epsilon = opt.epsilon;
        prm.max_sweeps = opt.max_sweeps;
        prm.damping = opt.damping;
        prm.check_interval = opt.check_interval;
        prm.out_precision = opt.float_marginals ? BNBP_OUT_FP32 : BNBP_OUT_DEFAULT;
        prm.semiring = opt.semiring;
        prm.n_query = static_cast<std::int32_t>(query.size());
        prm.query_nodes = query.empty() ? nullptr : query.data();
        if (opt.log_evidence) out.log_evidence.resize(out.n_cases);
        else out.log_evidence.clear();
        if (opt.expected_counts) {
            out.expected_counts.assign(flat_.cpt.size(), 0.0);
            if (bnbp_run_batch_expected_counts(handle_, &ev, &prm, nullptr, out.expected_counts.data(), dst, out.sweeps.data(),
                                               out.converged.data(), opt.log_evidence ? out.log_evidence.data() : nullptr) != BNBP_OK)
                throw std::runtime_error(last_error("bnbp_run_batch_expected_counts"));
        } else if (opt.log_evidence) {
            out.expected_counts.clear();
            if (bnbp_run_batch_log_evidence(handle_, &ev, &prm, dst, out.sweeps.data(), out.converged.data(),
                                            out.log_evidence.data()) != BNBP_OK)
                throw std::runtime_error(last_error("bnbp_run_batch_log_evidence"));
        } else {
            out.expected_counts.clear();
            if (bnbp_run_batch(handle_, &ev, &prm, dst, out.sweeps.data(), out.converged.data()) != BNBP_OK)
                throw std::runtime_error(last_error("bnbp_run_batch"));
        }
        if (!opt.devices.empty()) bnbp_get_summary(handle_, &out.summary);
    }

    // the map-returning overloads keep the reference's result shape: every vertex, double
    static options every_vertex_in_double(options opt)
    {
        opt.query.clear();
        opt.float_marginals = false;
        opt.log_evidence = false;
        opt.expected_counts = false;
        return opt;
    }

    std::vector<return_type> unpack(flat_result const& flat) const
    {
        std::vector<vertex_type> const& nodes = graph_.vertex_list();
        std::vector<return_type> out(flat.n_cases);
        for (std::size_t c = 0; c < flat.n_cases; ++c) {
            double const* row = flat.marginals.data() + c * flat.values_per_case;
            for (std::size_t i = 0; i < nodes.size(); ++i) {
                matrix_type& m = out[c][nodes[i]];
                m.resize(1, static_cast<std::size_t>(flat_.card[i]));
                m.assign(row + flat.offset[i], row + flat.offset[i + 1]);
            }
        }
        return out;
    }

    graph_t const graph_;            // a copy, like the reference (:16-19,:320): vertices stay shared
    options defaults_;
    flat_network flat_;              // what the device arena currently holds
    bnbp_handle* handle_ = nullptr;
    int precision_ = BNBP_FP64, device_ = -1, specialize_ = BNBP_SPEC_AUTO;
    std::vector<int> devices_;
    double zero_ = 0.0;
};

// the name BASELINE.json's north star uses; the reference class is belief_propagation
typedef belief_propagation loopy_belief_propagation;

} // namespace inference
} // namespace bn

#endif // BNB200_BAYESIAN_INFERENCE_BELIEF_PROPAGATION_HPP
