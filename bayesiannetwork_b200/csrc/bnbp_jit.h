// bnbp_jit.h — run-time specialisation of the sweep kernel to one network ("network compiler").
//
// spec_source() turns the flat layout of a network into CUDA source: one trait struct per node in
// front of the hand-written templates of bnbp_spec.cuh.  SpecCompiler compiles it with NVRTC
// (dlopen'ed: the library loads without it and then only the generic kernel is available) to an
// sm_100a cubin, keeps cubins in an on-disk cache keyed by the source hash, and loads / launches
// them through the driver API (entry points fetched with cudaGetDriverEntryPoint, so libbnbp
// does not link libcuda either).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "bnbp_kernels.cuh"

namespace bnbp {

struct SpecLayout {                 // host view of the network the generator needs
    int N = 0, PL = 0, M = 0, W = 0, V = 0;
    int64_t cpt_values = 0;
    const NodeMeta* nodes = nullptr;
    const int32_t* e_card = nullptr;      // [E] parent cardinality per in-edge
    const int32_t* e_lam_out = nullptr;   // [E] slot of the lambda-message child -> parent
    const int32_t* c_pi_out = nullptr;    // [E] slot of the pi-message parent -> child (out-edge order)
};

struct SpecConfig {
    bool fp32 = false;
    int vec = 1;        // cases per thread
    int minb = 1;       // __launch_bounds__ min blocks per SM
    int variant = 0;    // 0 plain, 1 freeze, 2 freeze + check, 3 first, 4 last, 5 first + K0, 6/7 last + K4 (bnbp_spec.cuh)
    int ahead = 1;      // software-pipeline depth of the input loads
    bool classloop = false;     // one loop per node SHAPE class instead of one unrolled body per node (large networks)
    // on-chip variants (8 plain, 9 check: bnbp_onchip.cuh)
    int roles = 4;              // warps that share the node walk of a 32-case group
    bool out_double = false;    // marginals in double from a float kernel (the host-buffer call)
};

// cost of one node in one sweep as the role partition of the on-chip kernel sees it (multiply-adds + the
// normalisations it emits), and the longest-processing-time partition itself: owner[x] = role of node x
double spec_node_cost(const SpecLayout& L, int x);
std::vector<int> spec_partition(const SpecLayout& L, int roles, double* imbalance = nullptr);

// bytes of dynamic shared memory the on-chip kernel needs for one 32-case group
size_t onchip_smem_bytes(const SpecLayout& L, bool fp32, int roles);

// Children whose lambda-messages the on-chip kernel reads into registers in phase A, before the sweep barrier
// (bnbp_spec.cuh MREG; the generated on-chip source static_asserts that the two agree).  A node with more children
// would read its inbox in phase B, after other warps may have overwritten it with the next sweep's messages: such a
// network is not eligible for the on-chip kernel.
constexpr int ONCHIP_MREG = 64;

// Can (and should) this network be specialised?  why != nullptr receives the reason when not.
bool spec_eligible(const SpecLayout& L, bool fp32, std::string* why);

// Class-looped mode: a network too large to unroll node by node whose nodes fall into few shape classes
// (R, K, M, parent cardinalities) -- the grids of cfg 3.  spec_classes: members of every class in node order.
bool class_eligible(const SpecLayout& L, bool fp32, std::string* why);
std::vector<std::vector<int>> spec_classes(const SpecLayout& L);
int class_max_inputs(const SpecLayout& L);     // most input values per case any node's class loop holds (register pressure)

std::string spec_source(const SpecLayout& L, const SpecConfig& cfg);

// mirrors bnbp_spec::Aux (device side) for T = double / float
template <typename T> struct SpecAux {
    const T* delta_prev;
    T* delta_cur;
    T* delta_next;
    unsigned char* status;
    int* sweeps;
    int* last_active;
    int sweep_index;
    int prev_tested;
    T eps;
    T damping;
    int n_inner;                 // variant 0: sweeps per launch
    const unsigned char* evst;   // variant 5: evidence-state bytes [tiles][N][TBC]
    void* out;                   // variants 6/7: case-major marginals
    long long n_valid;
};

struct SpecKernel {                 // one loaded cubin
    void* module = nullptr;         // CUmodule
    void* function = nullptr;       // CUfunction
    uint64_t cpt_dptr = 0;          // address of bnbp_cpt in the module
    size_t cpt_bytes = 0;
    int blocks_per_sm = 0;          // resident 128-thread blocks per SM (0: unknown)
    bool from_cache = false;
    double compile_ms = 0.0;
};

// Compile (or fetch from the cache) without touching a GPU.  Returns false and fills err on failure.
// bypass_cache: compile even when the cache holds an entry (and overwrite it) -- the retry after a cached cubin
// failed to load.
bool spec_compile(const std::string& source, std::vector<char>* cubin, bool* from_cache, double* ms, std::string* err,
                  bool bypass_cache = false);

// Is the cubin of this source in the on-disk cache (so that using it costs no NVRTC time)?
bool spec_in_cache(const std::string& source);

// Load a cubin into the current context and resolve the kernel + the CPT constant.  threads / smem: the launch
// shape the occupancy is asked for (the on-chip kernel opts in to its dynamic shared memory here).
bool spec_load(const std::vector<char>& cubin, SpecKernel* out, std::string* err, const char* entry = "bnbp_spec_sweep",
               int threads = 128, size_t smem = 0);
void spec_unload(SpecKernel* k);
bool spec_upload_cpt(const SpecKernel& k, const void* host, size_t bytes, std::string* err);

// <<<(tiles, node_slices), 128, 0, st>>> bnbp_spec_sweep(pl, cur, nxt, evbits, aux)
// node_slices > 1: class-looped PLAIN variants only -- block (tile, y) walks the y-th slice of every node class (one sweep per launch)
bool spec_launch(const SpecKernel& k, unsigned tiles, cudaStream_t st, void* pl, const void* cur, void* nxt,
                 const void* evbits, const void* aux, std::string* err, unsigned node_slices = 1);

// mirrors bnbp_spec::OcArgs (device side) for T = double / float
template <typename T> struct OnchipArgs {
    const long long* ev_off;
    long long ev_base;
    const int* ev_node;
    const int* ev_state;
    long long n_cases;
    void* out;
    const int* bel_col;
    long long out_stride;
    int* out_sweeps;
    unsigned char* out_conv;
    unsigned long long* ticket;
    int* error_flag;
    T eps;
    T damping;
    int max_sweeps;
    int interval;
    int first_reserved_sm;
};

// <<<blocks, threads, smem, st>>> bnbp_onchip_run(args)
bool onchip_launch(const SpecKernel& k, unsigned blocks, unsigned threads, size_t smem, cudaStream_t st, const void* args,
                   std::string* err);

std::string spec_cache_dir();

} // namespace bnbp
