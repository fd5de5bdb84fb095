// bnbp_jit.cu — network compiler: source generation, NVRTC compilation, cubin cache, driver-API
// loading of the network-specialised sweep kernel (bnbp_spec.cuh).  See bnbp_jit.h.
#include "bnbp_jit.h"

#include <cuda.h>
#include <nvrtc.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <map>
#include <mutex>
#include <sstream>
#include <sys/stat.h>
#include <unistd.h>

namespace bnbp {

// the text of bnbp_spec.cuh, embedded by _build.py (a raw string literal)
static const char* const kSpecHeader =
#include "bnbp_spec_embed.inc"
    ;
// the text of bnbp_onchip.cuh (appended behind kSpecHeader for the on-chip variants)
static const char* const kOnchipHeader =
#include "bnbp_onchip_embed.inc"
    ;

// ---- eligibility ---------------------------------------------------------------------------------
bool spec_eligible(const SpecLayout& L, bool fp32, std::string* why)
{
    auto no = [&](const char* w) { if (why) *why = w; return false; };
    const size_t tsize = fp32 ? 4 : 8;
    if (L.N > 1024) return no("more than 1024 nodes: fully unrolled code would not fit the instruction caches");
    if ((size_t)L.cpt_values * tsize > 60 * 1024) return no("CPT arena larger than the 64 KB constant bank");
    double fma = 0;
    for (int x = 0; x < L.N; ++x) {
        const NodeMeta& nd = L.nodes[x];
        if (nd.k > 6) return no("in-degree > 6: accumulators would not fit the register file");
        if (nd.card > 16) return no("cardinality > 16: accumulators would not fit the register file");
        int sum_ru = 0;
        for (int j = 0; j < nd.k; ++j) {
            if (L.e_card[nd.e0 + j] > 16) return no("parent cardinality > 16");
            sum_ru += L.e_card[nd.e0 + j];
        }
        if (2 * nd.card + 2 * sum_ru > 96) return no("a node needs more than 96 live values per case");
        int64_t Q = 1;
        for (int j = 0; j < nd.k; ++j) Q *= L.e_card[nd.e0 + j];
        fma += 3.0 * (double)Q * nd.card;
    }
    // compile time grows faster than linearly with the unrolled body (alarm37, 1.8k multiply-adds: 17 s;
    // 17k: a quarter of an hour), so only small networks are worth a run-time compile
    if (fma > 6500) return no("unrolled sweep would exceed ~6.5k multiply-adds per case (NVRTC compile time)");
    return true;
}

// ---- class-looped walks (bnbp_spec.cuh, BNBP_CLASSLOOP) ------------------------------------------------
// The shape of a node is all its arithmetic depends on: (R, K, M, parent cardinalities).
static std::vector<int> node_shape(const SpecLayout& L, int x)
{
    const NodeMeta& nd = L.nodes[x];
    std::vector<int> key = {nd.card, nd.k, nd.m};
    for (int j = 0; j < nd.k; ++j) key.push_back(L.e_card[nd.e0 + j]);
    return key;
}

std::vector<std::vector<int>> spec_classes(const SpecLayout& L)
{
    std::map<std::vector<int>, size_t> index;            // shape -> class, classes numbered in order of first appearance
    std::vector<std::vector<int>> members;
    for (int x = 0; x < L.N; ++x) {
        const auto it = index.emplace(node_shape(L, x), members.size());
        if (it.second) members.emplace_back();
        members[it.first->second].push_back(x);
    }
    return members;
}

// input values per case of a node as the class loop holds them (pi, lambda, both inboxes, CPT entries in registers)
static int64_t class_inputs(const SpecLayout& L, int x)
{
    const NodeMeta& nd = L.nodes[x];
    int64_t sum_ru = 0, Q = 1;
    for (int j = 0; j < nd.k; ++j) { sum_ru += L.e_card[nd.e0 + j]; Q *= L.e_card[nd.e0 + j]; }
    const int64_t nq = Q * nd.card;
    return 2 * nd.card + sum_ru + (nd.m <= 4 ? nd.m * nd.card : 0) + (nq <= 32 ? nq : 0);
}

int class_max_inputs(const SpecLayout& L)
{
    int64_t mx = 0;
    for (int x = 0; x < L.N; ++x) mx = std::max(mx, class_inputs(L, x));
    return (int)mx;
}

bool class_eligible(const SpecLayout& L, bool fp32, std::string* why)
{
    (void)fp32;
    auto no = [&](const char* w) { if (why) *why = w; return false; };
    if (L.N < 1) return no("empty network");
    if (L.N > (1 << 18)) return no("more than 262 144 nodes: the record table is compiled into the kernel image");
    if (L.cpt_values > 0x7fffffffLL || (int64_t)L.PL + L.M > 0x7fffffffLL) return no("offsets beyond 32 bits (the record table holds ints)");
    const std::vector<std::vector<int>> cls = spec_classes(L);
    if (cls.size() > 96) return no("more than 96 node shape classes: one unrolled body per class would not fit the instruction caches");
    double fma = 0;
    for (const std::vector<int>& mem : cls) {
        const NodeMeta& nd = L.nodes[mem[0]];
        if (nd.k > 6) return no("in-degree > 6: accumulators would not fit the register file");
        if (nd.card > 16) return no("cardinality > 16: accumulators would not fit the register file");
        int64_t Q = 1;
        for (int j = 0; j < nd.k; ++j) {
            if (L.e_card[nd.e0 + j] > 16) return no("parent cardinality > 16");
            Q *= L.e_card[nd.e0 + j];
        }
        if (nd.m > 64) return no("a hub with more than 64 children: its class record would not stay in registers");
        // the loop holds the inputs of TWO nodes (the one computed and the one loaded ahead), CPT entries included
        const int64_t nq = Q * nd.card;
        // (bnbp_spec.cuh: CPT_REG_MAX = 32 entries ride along in registers, larger tables are read where they are used)
        const int64_t inputs = class_inputs(L, mem[0]);
        if (inputs > 64) return no("a node class needs more than 64 input values per case: two sets of them would not fit the register file");
        if (nq > 1024) return no("a CPT of more than 1024 entries in a looped class (the dense path is the one for it)");
        fma += 3.0 * (double)nq;
    }
    if (fma > 8000) return no("the class bodies together would exceed ~8k multiply-adds (NVRTC compile time)");
    return true;
}

static std::string class_source(const SpecLayout& L, const SpecConfig& cfg, std::ostringstream& s)
{
    const std::vector<std::vector<int>> cls = spec_classes(L);
    s << "#define BNBP_CLASSLOOP 1\n";
    std::ostringstream rec, walk;
    size_t n_rec = 0;
    for (size_t c = 0; c < cls.size(); ++c) {
        const NodeMeta& nd = L.nodes[cls[c][0]];
        int rumax = 0;
        for (int j = 0; j < nd.k; ++j) rumax = std::max(rumax, (int)L.e_card[nd.e0 + j]);
        // shape only; the per-node members of the unrolled mode exist (zeroed) so that both modes name them
        s << "struct C" << c << " { static constexpr int R=" << nd.card << ",K=" << nd.k << ",M=" << nd.m << ",RUMAX=" << rumax
          << ",X=0,PL=0,PIN=0,LIN=0,CPT=0,BEL=0,GJ0=0;";
        auto arr = [&](const char* name, int n, auto get) {
            s << " static constexpr int " << name << "[" << std::max(n, 1) << "]={";
            for (int j = 0; j < std::max(n, 1); ++j) s << (j ? "," : "") << (j < n ? get(j) : 0);
            s << "};";
        };
        arr("RU", nd.k, [&](int j) { return (int)L.e_card[nd.e0 + j]; });
        arr("LO", nd.k, [&](int) { return 0; });
        arr("PO", nd.m, [&](int) { return 0; });
        s << " };   // " << cls[c].size() << " nodes\n";
        walk << " BNBP_CLASS(C" << c << "," << n_rec << "," << cls[c].size() << ")";
        for (int x : cls[c]) {
            const NodeMeta& nx = L.nodes[x];
            rec << x << "," << nx.pl_off << "," << nx.pin_off << "," << nx.lin_off << "," << nx.cpt_off;
            for (int j = 0; j < nx.k; ++j) rec << "," << L.e_lam_out[nx.e0 + j];
            for (int j = 0; j < nx.m; ++j) rec << "," << L.c_pi_out[nx.c0 + j];
            rec << ",\n";
            n_rec += (size_t)(5 + nx.k + nx.m);
        }
    }
    s << "// per node, class by class: X, PL, PIN, LIN, CPT, LO[K], PO[M]\n";
    s << "__device__ const int bnbp_rec[" << n_rec + 1 << "] = {\n" << rec.str() << "0};\n";
    s << "#define BNBP_WALK" << walk.str() << "\n";
    (void)cfg;
    s << kSpecHeader;
    return s.str();
}

// ---- role partition of the on-chip kernel ------------------------------------------------------------
double spec_node_cost(const SpecLayout& L, int x)
{
    const NodeMeta& nd = L.nodes[x];
    double Q = 1.0, sum_ru = 0.0;
    for (int j = 0; j < nd.k; ++j) { Q *= L.e_card[nd.e0 + j]; sum_ru += L.e_card[nd.e0 + j]; }
    const double r = nd.card, k = nd.k, m = nd.m;
    const double walk = nd.k ? (2.0 * r + 2.0) * Q + 3.0 * Q * (k > 1 ? 1.5 : 1.0) : 0.0;   // leaf level: 2r+2 per row; upper levels
    const double child = m > 0 ? r * m * (m <= 4 ? m : 2.0) : 0.0;                        // leave-one-out products
    const double norms = 14.0 * (2.0 + k + m) + 2.0 * (2.0 * r + sum_ru + m * r);         // reciprocal + sum + scale per row emitted
    const double ldst = 2.0 * (2.0 * r + sum_ru + m * r);
    return walk + child + norms + ldst;
}

std::vector<int> spec_partition(const SpecLayout& L, int roles, double* imbalance)
{
    std::vector<int> order((size_t)L.N), owner((size_t)L.N, 0);
    std::vector<double> cost((size_t)L.N), load((size_t)roles, 0.0);
    for (int x = 0; x < L.N; ++x) { order[(size_t)x] = x; cost[(size_t)x] = spec_node_cost(L, x); }
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[(size_t)a] > cost[(size_t)b]; });
    double total = 0.0;
    for (int x : order) {
        int best = 0;
        for (int r = 1; r < roles; ++r) if (load[(size_t)r] < load[(size_t)best]) best = r;
        owner[(size_t)x] = best;
        load[(size_t)best] += cost[(size_t)x];
        total += cost[(size_t)x];
    }
    if (imbalance) {
        double mx = 0.0;
        for (double l : load) mx = std::max(mx, l);
        *imbalance = total > 0.0 ? mx * roles / total : 1.0;
    }
    return owner;
}

size_t onchip_smem_bytes(const SpecLayout& L, bool fp32, int roles)
{
    const size_t tsize = fp32 ? 4 : 8;
    return ((size_t)L.PL + (size_t)L.M) * 32 * tsize + (size_t)roles * 32 * tsize + 32 * 8;   // pi/lambda + ONE message buffer
}

// ---- source generation -----------------------------------------------------------------------------
// columns of the marginal group that ends with node x
static int nd_width(const SpecLayout& L, const std::vector<int>& gj0, int x)
{
    return L.nodes[x].bel_off + L.nodes[x].card - gj0[(size_t)x];
}

std::string spec_source(const SpecLayout& L, const SpecConfig& cfg)
{
    std::ostringstream s;
    s << "// generated by libbnbp spec_source(): network traits for bnbp_spec.cuh\n";
    s << "#define BNBP_T " << (cfg.fp32 ? "float" : "double") << "\n";
    s << "#define BNBP_VEC " << cfg.vec << "\n";
    s << "#define BNBP_MINB " << cfg.minb << "\n";
    s << "#define BNBP_VARIANT " << cfg.variant << "\n";
    s << "#define BNBP_AHEAD " << cfg.ahead << "\n";
    s << "#define BNBP_PL " << L.PL << "\n#define BNBP_M " << L.M << "\n#define BNBP_W " << L.W << "\n";
    s << "#define BNBP_NCPT " << L.cpt_values << "\n";
    s << "#define BNBP_N " << L.N << "\n#define BNBP_V " << L.V << "\n";
    const bool onchip = cfg.variant >= 8;
    if (cfg.classloop && cfg.variant > 4) return "#error \"class-looped walks exist for variants 0-4\"\n";
    s << "#define BNBP_OUT " << ((cfg.fp32 && cfg.variant != 7 && !(onchip && cfg.out_double)) ? "float" : "double") << "\n";
    if (cfg.classloop) return class_source(L, cfg, s);
    // groups of consecutive nodes whose marginals fit the 32-column tile of variants 6/7
    std::vector<int> gj0((size_t)L.N, 0), gend((size_t)L.N, 0);   // group start column per node, 1 = last node of its group
    for (int x = 0; x < L.N;) {
        const int j0 = L.nodes[x].bel_off;
        int w = 0, y = x;
        while (y < L.N && w + L.nodes[y].card <= 32) { gj0[(size_t)y] = j0; w += L.nodes[y].card; ++y; }
        if (y == x) { gj0[(size_t)y] = j0; ++y; }          // cardinality > 32: not eligible anyway
        gend[(size_t)y - 1] = 1;
        x = y;
    }
    for (int x = 0; x < L.N; ++x) {
        const NodeMeta& nd = L.nodes[x];
        int rumax = 0;
        for (int j = 0; j < nd.k; ++j) rumax = std::max(rumax, (int)L.e_card[nd.e0 + j]);
        s << "struct N" << x << " { static constexpr int X=" << x << ",R=" << nd.card << ",K=" << nd.k << ",M=" << nd.m
          << ",PL=" << nd.pl_off << ",PIN=" << nd.pin_off << ",LIN=" << nd.lin_off << ",CPT=" << nd.cpt_off
          << ",RUMAX=" << rumax << ",BEL=" << nd.bel_off << ",GJ0=" << gj0[(size_t)x] << ";";
        auto arr = [&](const char* name, int n, auto get) {
            s << " static constexpr int " << name << "[" << std::max(n, 1) << "]={";
            for (int j = 0; j < std::max(n, 1); ++j) s << (j ? "," : "") << (j < n ? get(j) : 0);
            s << "};";
        };
        arr("RU", nd.k, [&](int j) { return (int)L.e_card[nd.e0 + j]; });
        arr("LO", nd.k, [&](int j) { return (int)L.e_lam_out[nd.e0 + j]; });
        arr("PO", nd.m, [&](int j) { return (int)L.c_pi_out[nd.c0 + j]; });
        s << " };\n";
    }
    if (onchip) {
        // one walk per role (warp): the nodes the longest-processing-time partition gave it, in index order
        const int roles = std::max(1, cfg.roles);
        const std::vector<int> owner = spec_partition(L, roles, nullptr);
        s << "#define BNBP_ROLES " << roles << "\n#define BNBP_ROLE_LIST(OP)";
        for (int r = 0; r < roles; ++r) s << " OP(" << r << ")";
        s << "\n";
        for (int r = 0; r < roles; ++r) {
            std::vector<int> mine;
            for (int x = 0; x < L.N; ++x) if (owner[(size_t)x] == r) mine.push_back(x);
            s << "#define BNBP_NODES_" << r << "(OP)";
            for (int x : mine) s << " OP(N" << x << ")";
            // phase A: the inboxes of all its nodes into registers; barrier; phase B: compute and emit
            s << "\n#define BNBP_WALK_" << r;
            for (int x : mine) s << " BNBP_DECL(N" << x << ")";
            for (int x : mine) s << " BNBP_LOADM(N" << x << ")";
            s << " BNBP_SYNC";
            for (int x : mine) s << " BNBP_COMP(N" << x << ")";
            s << "\n";
        }
        auto table = [&](const char* type, const char* name, auto get) {
            s << "__device__ __constant__ " << type << " " << name << "[" << L.N << "] = {";
            for (int x = 0; x < L.N; ++x) s << (x ? "," : "") << get(x);
            s << "};\n";
        };
        table("unsigned char", "bnbp_owner", [&](int x) { return owner[(size_t)x]; });
        table("int", "bnbp_ploff", [&](int x) { return (int)L.nodes[x].pl_off; });
        table("unsigned char", "bnbp_cardn", [&](int x) { return (int)L.nodes[x].card; });
        s << "#define BNBP_WALK\n";
        s << kSpecHeader << "\n" << kOnchipHeader;
        s << "\nstatic_assert(bnbp_spec::MREG == " << ONCHIP_MREG << ", \"on-chip eligibility (ONCHIP_MREG) and the kernel's MREG disagree\");\n";
        return s.str();
    }
    // walk: declarations, then loads `ahead` nodes in front of the arithmetic
    s << "#define BNBP_WALK";
    for (int x = 0; x < L.N; ++x) s << " BNBP_DECL(N" << x << ")";
    const int ahead = std::max(0, cfg.ahead);
    for (int x = 0; x < std::min(ahead, L.N); ++x) s << " BNBP_LOAD(N" << x << ")";
    for (int x = 0; x < L.N; ++x) {
        if (x + ahead < L.N) s << " BNBP_LOAD(N" << (x + ahead) << ")";
        s << " BNBP_COMP(N" << x << ")";
        if ((cfg.variant == 6 || cfg.variant == 7) && gend[(size_t)x])
            s << " BNBP_FLUSH(" << gj0[(size_t)x] << "," << (nd_width(L, gj0, x)) << ")";
    }
    s << "\n";
    s << kSpecHeader;
    return s.str();
}

// ---- NVRTC (dlopen) -----------------------------------------------------------------------------------
namespace {

struct Nvrtc {
    void* so = nullptr;
    decltype(&nvrtcCreateProgram) createProgram = nullptr;
    decltype(&nvrtcCompileProgram) compileProgram = nullptr;
    decltype(&nvrtcDestroyProgram) destroyProgram = nullptr;
    decltype(&nvrtcGetProgramLogSize) getLogSize = nullptr;
    decltype(&nvrtcGetProgramLog) getLog = nullptr;
    decltype(&nvrtcGetCUBINSize) getCubinSize = nullptr;
    decltype(&nvrtcGetCUBIN) getCubin = nullptr;
    decltype(&nvrtcGetErrorString) errorString = nullptr;
    decltype(&nvrtcVersion) version = nullptr;
    std::string load_error;
};

Nvrtc& nvrtc()
{
    static Nvrtc n;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnvrtc.so.12", "libnvrtc.so", "/usr/local/cuda/lib64/libnvrtc.so.12",
                               "/usr/local/cuda/lib64/libnvrtc.so"};
        for (const char* nm : names) {
            n.so = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
            if (n.so) break;
        }
        if (!n.so) { n.load_error = std::string("libnvrtc not found: ") + dlerror(); return; }
#define BNBP_SYM(field, name)                                                        \
    n.field = reinterpret_cast<decltype(n.field)>(dlsym(n.so, name));                \
    if (!n.field) { n.load_error = std::string("libnvrtc lacks ") + name; return; }
        BNBP_SYM(createProgram, "nvrtcCreateProgram")
        BNBP_SYM(compileProgram, "nvrtcCompileProgram")
        BNBP_SYM(destroyProgram, "nvrtcDestroyProgram")
        BNBP_SYM(getLogSize, "nvrtcGetProgramLogSize")
        BNBP_SYM(getLog, "nvrtcGetProgramLog")
        BNBP_SYM(getCubinSize, "nvrtcGetCUBINSize")
        BNBP_SYM(getCubin, "nvrtcGetCUBIN")
        BNBP_SYM(errorString, "nvrtcGetErrorString")
        BNBP_SYM(version, "nvrtcVersion")
#undef BNBP_SYM
    });
    return n;
}

uint64_t fnv1a(const void* p, size_t n, uint64_t h)
{
    const unsigned char* b = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < n; ++i) { h ^= b[i]; h *= 0x100000001B3ull; }
    return h;
}

bool read_file(const std::string& path, std::vector<char>* out)
{
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    fseek(f, 0, SEEK_END);
    long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    if (n <= 0) { fclose(f); return false; }
    out->resize((size_t)n);
    const bool ok = fread(out->data(), 1, (size_t)n, f) == (size_t)n;
    fclose(f);
    return ok;
}

void write_file_atomic(const std::string& path, const std::vector<char>& data)
{
    const std::string tmp = path + ".tmp" + std::to_string((long)getpid());
    FILE* f = fopen(tmp.c_str(), "wb");
    if (!f) return;                                   // the cache is best effort
    const bool ok = fwrite(data.data(), 1, data.size(), f) == data.size();
    fclose(f);
    if (!ok || rename(tmp.c_str(), path.c_str()) != 0) unlink(tmp.c_str());
}

} // namespace

std::string spec_cache_dir()
{
    if (const char* e = getenv("BNBP_CACHE_DIR")) return e;
    Dl_info info;
    if (dladdr(reinterpret_cast<const void*>(&spec_cache_dir), &info) && info.dli_fname) {
        std::string p = info.dli_fname;
        const size_t slash = p.rfind('/');
        if (slash != std::string::npos) return p.substr(0, slash) + "/jitcache";
    }
    return "/tmp/bnbp_jitcache_" + std::to_string((long)geteuid());
}

static const char* const kNvrtcOpts[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", "-default-device"};
constexpr int kNvrtcOptCount = (int)(sizeof kNvrtcOpts / sizeof kNvrtcOpts[0]);

// file of the cubin of `source` in the cache (key: source text + compiler options)
static std::string cache_path(const std::string& source)
{
    uint64_t h1 = fnv1a(source.data(), source.size(), 0xcbf29ce484222325ull);
    uint64_t h2 = fnv1a(source.data(), source.size(), 0x84222325cbf29ce4ull);
    for (int i = 0; i < kNvrtcOptCount; ++i) {
        h1 = fnv1a(kNvrtcOpts[i], strlen(kNvrtcOpts[i]), h1);
        h2 = fnv1a(kNvrtcOpts[i], strlen(kNvrtcOpts[i]), h2);
    }
    char name[64];
    snprintf(name, sizeof name, "%016llx%016llx.cubin", (unsigned long long)h1, (unsigned long long)h2);
    return spec_cache_dir() + "/" + name;
}

bool spec_in_cache(const std::string& source)
{
    if (getenv("BNBP_NO_CACHE")) return false;
    struct stat sb;
    return stat(cache_path(source).c_str(), &sb) == 0 && sb.st_uid == geteuid() && sb.st_size > 0;
}

bool spec_compile(const std::string& source, std::vector<char>* cubin, bool* from_cache, double* ms, std::string* err,
                  bool bypass_cache)
{
    const char* const* opts = kNvrtcOpts;
    const int n_opts = kNvrtcOptCount;
    // (The compiler version is deliberately NOT part of the key.  It was for a while -- a cubin of another toolkit should
    //  not be picked up -- but a process that has PyTorch loaded resolves libnvrtc.so.12 to PyTorch's bundled copy (12.8
    //  against the toolkit's 12.9), so every kernel precompiled at build time missed the cache and the GPU test run paid
    //  15-80 s of NVRTC per kernel, r02o.  A cubin this driver cannot load is instead replaced on the spot: ensure_spec /
    //  ensure_onchip recompile with bypass_cache when cuModuleLoadData refuses a cached one.)
    const std::string dir = spec_cache_dir();
    const std::string path = cache_path(source);
    if (from_cache) *from_cache = false;
    if (ms) *ms = 0.0;
    if (!getenv("BNBP_NO_CACHE") && !bypass_cache) {
        // only files of the current user are trusted (the cubin is loaded into the GPU context as is)
        struct stat sb;
        if (stat(path.c_str(), &sb) == 0 && sb.st_uid == geteuid() && read_file(path, cubin)) {
            if (from_cache) *from_cache = true;
            return true;
        }
    }
    Nvrtc& n = nvrtc();
    if (!n.load_error.empty()) { if (err) *err = n.load_error; return false; }
    const auto t0 = std::chrono::steady_clock::now();
    nvrtcProgram prog = nullptr;
    nvrtcResult r = n.createProgram(&prog, source.c_str(), "bnbp_spec_net.cu", 0, nullptr, nullptr);
    if (r != NVRTC_SUCCESS) { if (err) *err = std::string("nvrtcCreateProgram: ") + n.errorString(r); return false; }
    r = n.compileProgram(prog, n_opts, opts);
    if (r != NVRTC_SUCCESS) {
        size_t ls = 0;
        n.getLogSize(prog, &ls);
        std::string log(ls, '\0');
        if (ls) n.getLog(prog, &log[0]);
        if (log.size() > 4000) log.resize(4000);
        if (err) *err = std::string("nvrtcCompileProgram: ") + n.errorString(r) + "\n" + log;
        n.destroyProgram(&prog);
        return false;
    }
    size_t cs = 0;
    r = n.getCubinSize(prog, &cs);
    if (r != NVRTC_SUCCESS || cs == 0) {
        if (err) *err = "nvrtcGetCUBINSize failed";
        n.destroyProgram(&prog);
        return false;
    }
    cubin->resize(cs);
    r = n.getCubin(prog, cubin->data());
    n.destroyProgram(&prog);
    if (r != NVRTC_SUCCESS) { if (err) *err = "nvrtcGetCUBIN failed"; return false; }
    if (ms) *ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (!getenv("BNBP_NO_CACHE")) {
        mkdir(dir.c_str(), 0700);
        write_file_atomic(path, *cubin);
        if (getenv("BNBP_KEEP_SOURCE")) {
            std::vector<char> src(source.begin(), source.end());
            write_file_atomic(path.substr(0, path.size() - 6) + ".cu", src);
        }
    }
    return true;
}

// ---- driver API through the runtime (no link-time dependency on libcuda) -------------------------------
namespace {

struct Driver {
    decltype(&cuModuleLoadData) moduleLoadData = nullptr;
    decltype(&cuModuleUnload) moduleUnload = nullptr;
    decltype(&cuModuleGetFunction) moduleGetFunction = nullptr;
    decltype(&cuModuleGetGlobal) moduleGetGlobal = nullptr;
    decltype(&cuLaunchKernel) launchKernel = nullptr;
    decltype(&cuMemcpyHtoD) memcpyHtoD = nullptr;
    decltype(&cuGetErrorString) getErrorString = nullptr;
    decltype(&cuFuncSetAttribute) funcSetAttribute = nullptr;
    decltype(&cuOccupancyMaxActiveBlocksPerMultiprocessor) occupancy = nullptr;   // optional
    std::string load_error;
};

Driver& driver()
{
    static Driver d;
    static std::once_flag once;
    std::call_once(once, [] {
        auto get = [&](const char* name, void** fn) {
            cudaDriverEntryPointQueryResult q;
            cudaError_t e = cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q);
            if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !*fn) {
                cudaGetLastError();
                d.load_error = std::string("driver entry point ") + name + " unavailable";
                return false;
            }
            return true;
        };
        if (!get("cuModuleLoadData", (void**)&d.moduleLoadData)) return;
        if (!get("cuModuleUnload", (void**)&d.moduleUnload)) return;
        if (!get("cuModuleGetFunction", (void**)&d.moduleGetFunction)) return;
        if (!get("cuModuleGetGlobal", (void**)&d.moduleGetGlobal)) return;
        if (!get("cuLaunchKernel", (void**)&d.launchKernel)) return;
        if (!get("cuMemcpyHtoD", (void**)&d.memcpyHtoD)) return;
        if (!get("cuGetErrorString", (void**)&d.getErrorString)) return;
        if (!get("cuFuncSetAttribute", (void**)&d.funcSetAttribute)) return;
        if (!get("cuOccupancyMaxActiveBlocksPerMultiprocessor", (void**)&d.occupancy)) {
            d.occupancy = nullptr;          // only the chunk planner uses it: not an error
            d.load_error.clear();
        }
    });
    return d;
}

std::string cu_err(Driver& d, const char* what, CUresult r)
{
    const char* s = nullptr;
    if (d.getErrorString) d.getErrorString(r, &s);
    return std::string(what) + ": " + (s ? s : "unknown driver error");
}

} // namespace

bool spec_load(const std::vector<char>& cubin, SpecKernel* out, std::string* err, const char* entry, int threads, size_t smem)
{
    Driver& d = driver();
    if (!d.load_error.empty()) { if (err) *err = d.load_error; return false; }
    CUmodule mod = nullptr;
    CUresult r = d.moduleLoadData(&mod, cubin.data());
    if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuModuleLoadData", r); return false; }
    CUfunction fn = nullptr;
    r = d.moduleGetFunction(&fn, mod, entry);
    if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuModuleGetFunction", r); d.moduleUnload(mod); return false; }
    CUdeviceptr p = 0;
    size_t bytes = 0;
    r = d.moduleGetGlobal(&p, &bytes, mod, "bnbp_cpt");
    if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuModuleGetGlobal(bnbp_cpt)", r); d.moduleUnload(mod); return false; }
    out->module = mod;
    out->function = fn;
    out->cpt_dptr = (uint64_t)p;
    out->cpt_bytes = bytes;
    out->blocks_per_sm = 0;
    if (smem > 48 * 1024) {
        r = d.funcSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)smem);
        if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuFuncSetAttribute(max dynamic shared memory)", r); d.moduleUnload(mod); return false; }
    }
    if (d.occupancy) {
        int nb = 0;
        if (d.occupancy(&nb, fn, threads, smem) == CUDA_SUCCESS) out->blocks_per_sm = nb;
    }
    return true;
}

void spec_unload(SpecKernel* k)
{
    if (k && k->module) {
        Driver& d = driver();
        if (d.moduleUnload) d.moduleUnload((CUmodule)k->module);
        k->module = nullptr;
        k->function = nullptr;
    }
}

bool spec_upload_cpt(const SpecKernel& k, const void* host, size_t bytes, std::string* err)
{
    Driver& d = driver();
    if (bytes > k.cpt_bytes) { if (err) *err = "CPT larger than the module's constant arena"; return false; }
    if (bytes == 0) return true;
    CUresult r = d.memcpyHtoD((CUdeviceptr)k.cpt_dptr, host, bytes);
    if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuMemcpyHtoD(bnbp_cpt)", r); return false; }
    return true;
}

bool spec_launch(const SpecKernel& k, unsigned tiles, cudaStream_t st, void* pl, const void* cur, void* nxt,
                 const void* evbits, const void* aux, std::string* err, unsigned node_slices)
{
    Driver& d = driver();
    void* params[5] = {&pl, (void*)&cur, &nxt, (void*)&evbits, const_cast<void*>(aux)};
    CUresult r = d.launchKernel((CUfunction)k.function, tiles, node_slices ? node_slices : 1, 1, 128, 1, 1, 0, (CUstream)st, params, nullptr);
    if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuLaunchKernel(bnbp_spec_sweep)", r); return false; }
    return true;
}

bool onchip_launch(const SpecKernel& k, unsigned blocks, unsigned threads, size_t smem, cudaStream_t st, const void* args,
                   std::string* err)
{
    Driver& d = driver();
    void* params[1] = {const_cast<void*>(args)};
    CUresult r = d.launchKernel((CUfunction)k.function, blocks, 1, 1, threads, 1, 1, (unsigned)smem, (CUstream)st, params, nullptr);
    if (r != CUDA_SUCCESS) { if (err) *err = cu_err(d, "cuLaunchKernel(bnbp_onchip_run)", r); return false; }
    return true;
}

} // namespace bnbp
