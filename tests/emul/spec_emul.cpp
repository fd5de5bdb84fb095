// spec_emul.cpp -- host emulation of ONE generated sweep kernel (see cuda_host_shim.h).  Built by
// tests/test_netcompiler_emul.py as   g++ -O0 -std=c++17 -ffp-contract=off -fvisibility=hidden -fno-gnu-unique
//                                         -DBNBP_GENERATED='"<file>"' -shared ...
// Hidden visibility / no unique symbols: a test process loads several of these objects, and every one of them defines
// trait structs of the same names (N0, C0, ...) with static data members -- they must not be unified across objects.
#include "cuda_host_shim.h"
#include BNBP_GENERATED

#pragma GCC visibility push(default)
extern "C" {

int emul_pl() { return BNBP_PL; }
int emul_m() { return BNBP_M; }
int emul_w() { return BNBP_W; }
int emul_tbc() { return (int)bnbp_spec::TBC; }
int emul_variant() { return BNBP_VARIANT; }
int emul_value_bytes() { return (int)sizeof(T); }

void emul_set_cpt(const T* cpt, long long n) { memcpy(bnbp_cpt, cpt, (size_t)n * sizeof(T)); }

// What the kernel keeps in registers, per node of the walk (unrolled) or per node class (class-looped), in walk order:
// children whose lambda-messages are loaded ahead (0: streamed where used) and CPT entries loaded ahead (0: read where
// used).  The generator's register budget (class_inputs in bnbp_jit.cu) assumes the same split.  Returns the count.
int emul_register_plan(int* children, int* cpt)
{
    int n = 0;
    auto rec = [&](int m, bool reg_children, bool reg_cpt, int nq) {
        children[n] = (m > 0 && reg_children) ? m : 0;
        cpt[n] = reg_cpt ? nq : 0;
        ++n;
    };
    (void)rec;
#define BNBP_PLAN(NN) rec(NN::M, NN::M <= bnbp_spec::MREG, bnbp_spec::In<NN>::CPT_REG, bnbp_spec::In<NN>::NQ);
#if BNBP_CLASSLOOP
#define BNBP_CLASS(CC, FIRST, COUNT) BNBP_PLAN(CC)
#else
#define BNBP_DECL(NN) BNBP_PLAN(NN)
#define BNBP_LOAD(NN)
#define BNBP_COMP(NN)
#define BNBP_FLUSH(J0, WW)
#endif
    BNBP_WALK
    return n;
}

// One launch of <<<(tiles, node_slices), 128>>> bnbp_spec_sweep(pl, cur, nxt, evbits, aux).  delta / status / sweeps / last_active: the
// per-case arrays of the freeze / check variants (ignored by the plain ones).  evst: variant 5 only.
void emul_launch(T* pl, const T* cur, T* nxt, const unsigned* evbits, int tiles, int n_inner, T eps, T damping,
                 int sweep_index, int prev_tested, const T* delta_prev, T* delta_cur, T* delta_next,
                 unsigned char* status, int* sweeps, int* last_active, int node_slices, const unsigned char* evst)
{
    bnbp_spec::Aux a;
    memset(&a, 0, sizeof a);
    a.evst = evst;                  // variant 5 (first sweep fused with K0): evidence-state bytes [tiles][N][TBC], 0 = not observed
    a.delta_prev = delta_prev; a.delta_cur = delta_cur; a.delta_next = delta_next;
    a.status = status; a.sweeps = sweeps; a.last_active = last_active;
    a.sweep_index = sweep_index; a.prev_tested = prev_tested;
    a.eps = eps; a.damping = damping; a.n_inner = n_inner;
    // grid (tiles, node_slices), slices outermost and in DESCENDING order: nothing may depend on the order of blocks
    gridDim.x = (unsigned)tiles;
    gridDim.y = (unsigned)(node_slices > 0 ? node_slices : 1);
    for (int y = (int)gridDim.y - 1; y >= 0; --y)
        for (int t = 0; t < tiles; ++t)
            for (int tid = 0; tid < 128; ++tid) {
                blockIdx.x = (unsigned)t;
                blockIdx.y = (unsigned)y;
                threadIdx.x = (unsigned)tid;
                bnbp_spec_sweep(pl, cur, nxt, evbits, a);
            }
}

}
#pragma GCC visibility pop
