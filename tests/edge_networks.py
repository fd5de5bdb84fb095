"""Small networks that sit on the shape boundaries where the generated kernels change their code (bnbp_jit.cu,
bnbp_spec.cuh, bnbp_onchip.cuh), each named after the boundary it pins:

    indeg5_6        nodes of 5 and 6 parents of mixed cardinality, as child and as parent (parent_rec<N, L> at depth
                    5 and 6, the deepest the network compiler accepts); loopy
    card16          cardinality 16 (root, inner node with parents (16, 4): 72 live values and 1 024 CPT entries,
                    a 16-state chain) with small leaves; pacc[R] / lacc[K][RUMAX] at their largest
    card1           cardinality-1 root, inner node and parents of a multi-parent node; loopy
    hub4, hub5      the streaming kernels' MREG = 4: children's lambda-messages in registers / streamed
    hub64, hub65    the on-chip kernel's MREG = 64 and the class-looped walk's limit of 64 children
    cpt32, cpt33    class mode: a CPT of 32 entries rides in registers (CPT_REG_MAX), one of 33 is read where used
    inputs64        class mode: a node class of exactly 64 input values per case (4 states, one 8-state parent, 4
                    children: 8 + 8 + 16 + 32)
    tile32          marginal groups of exactly 32 columns (16+16, 16+15+1) followed by more nodes (variants 6 / 7)
    edgeless        no edge at all (M = 0)
    single          one node
    w32, w33        32 and 33 nodes: evidence on node 31 / on node 32, the first bit of the second word of the
                    observed-node bits
    determ          exact 0 / 1 CPT rows (OR, AND, copy) and 1e-12 entries, a loopy and a polytree component;
                    random evidence contradicts them in some cases (all-zero rows: NaN where the oracle has NaN).
                    Its fp32 runs hold the plain fp32 bar: the 1e-12 entries and their products stay far above the
                    smallest normal float, so the subnormal flush of the on-chip reciprocal (DESIGN section 4) never
                    applies

and the shapes the compilers refuse (REFUSED: network, variant, environment, reason).  Every unrolled network stays
well below the 6 500 multiply-add cap of spec_eligible: NVRTC time grows like N^2.4.  The CPTs come from
synth._assemble (strictly positive rows) except where a boundary needs exact zeros (determ).
"""
from __future__ import annotations

import numpy as np

from bayesiannetwork_b200 import synth
from bayesiannetwork_b200.flat import FlatNetwork


def _with_rows(net: FlatNetwork, rows: dict) -> FlatNetwork:
    cpt = net.cpt.copy()
    for x, r in rows.items():
        r = np.asarray(r, dtype=np.float64).ravel()
        assert r.size == net.cpt_off[x + 1] - net.cpt_off[x]
        cpt[net.cpt_off[x]:net.cpt_off[x + 1]] = r
    return FlatNetwork(net.card, net.parent_off, net.parents, net.cpt_off, cpt, name=net.name)


def _hub(m: int, name: str) -> FlatNetwork:
    return synth._assemble([2] + [2 + (i % 2) for i in range(m)], [[]] + [[0]] * m, 40 + m, name)


def _determ() -> FlatNetwork:
    # loopy component: 2 = OR(0, 1), 3 = copy of 2 up to 1e-12 (and 0 -> 0 exactly), 4 = AND(2, 3)
    # polytree component: 6 = copy of 5, 7 = NOT 6 up to 1e-12
    card = [2, 2, 2, 2, 2, 2, 2, 2]
    par = [[], [], [0, 1], [0, 2], [2, 3], [], [5], [6]]
    net = synth._assemble(card, par, 11, "determ")
    eps = 1e-12
    return _with_rows(net, {
        2: [[1, 0], [0, 1], [0, 1], [0, 1]],
        3: [[1, 0], [eps, 1 - eps], [1, 0], [0, 1]],
        4: [[1, 0], [1, 0], [1, 0], [0, 1]],
        6: [[1, 0], [0, 1]],
        7: [[eps, 1 - eps], [1, 0]],
    })


def catalogue():
    """name -> FlatNetwork, in a fixed order."""
    nets = [
        synth._assemble([2, 3, 4, 2, 3, 2, 3, 2, 4, 2],
                        [[], [], [], [], [], [], [0, 1, 2, 3, 4], [0, 1, 2, 3, 4, 5], [1, 3, 5, 6, 7], [7]], 5, "indeg5_6"),
        synth._assemble([16, 4, 16, 16, 2, 3], [[], [], [0, 1], [2], [3], [2, 4]], 6, "card16"),
        synth._assemble([1, 2, 3, 1, 2, 1, 2], [[], [], [0, 1], [2], [3], [4], [0, 3, 5]], 7, "card1"),
        synth._assemble([3] + [2] * 4 + [2], [[]] + [[0]] * 4 + [[1, 2]], 8, "hub4"),
        synth._assemble([3] + [2] * 5 + [2], [[]] + [[0]] * 5 + [[1, 2]], 8, "hub5"),
        _hub(64, "hub64"),
        _hub(65, "hub65"),
        synth._assemble([4, 4, 2, 2, 3], [[], [], [0, 1], [2], [2, 3]], 9, "cpt32"),
        synth._assemble([11, 3, 2, 2], [[], [0], [1], [0, 2]], 10, "cpt33"),
        synth._assemble([8, 4, 2, 2, 3, 2], [[], [0], [1], [1], [1], [1, 2]], 12, "inputs64"),
        synth._assemble([16, 16, 16, 15, 1, 2, 3], [[], [0], [1], [], [3], [2, 4], [5]], 13, "tile32"),
        synth._assemble([2, 3, 4], [[], [], []], 14, "edgeless"),
        synth._assemble([3], [[]], 15, "single"),
        synth._assemble([2] * 32, [[]] + [[i] for i in range(31)], 16, "w32"),
        synth._assemble([2] * 33, [[]] + [[i] for i in range(32)], 17, "w33"),
        _determ(),
    ]
    return {n.name: n for n in nets}


NAMES = list(catalogue())

# What each generator does with a catalogue network: class-looped walk (BNBP_CLASSLOOP=2) and on-chip kernel accepted?
CLASSLOOP_REFUSED = {
    "card16": "a node class needs more than 64 input values per case",
    "hub65": "a hub with more than 64 children: its class record would not stay in registers",
}
ONCHIP_REFUSED = {
    "hub65": "a hub with more than 64 children: its inbox cannot be read before the sweep barrier",
}


def is_polytree(net: FlatNetwork) -> bool:
    """No cycle in the undirected skeleton (BP is exact there)."""
    comp = list(range(net.n_nodes))

    def find(v):
        while comp[v] != v:
            comp[v] = comp[comp[v]]
            v = comp[v]
        return v

    for x in range(net.n_nodes):
        for u in net.parents[net.parent_off[x]:net.parent_off[x + 1]]:
            a, b = find(int(u)), find(x)
            if a == b:
                return False
            comp[a] = b
    return True


def evidence(net: FlatNetwork, n_cases: int, seed: int = 3):
    """Hard evidence, every node with probability 1/4 (card-1 nodes included); on w32 / w33 every case also observes
    the last node, so the bit that opens (w33) or closes (w32) a word of observed-node bits is always set somewhere."""
    ev = synth.make_evidence(net, n_cases, seed=seed, p=0.25)
    if net.name not in ("w32", "w33"):
        return ev
    from bayesiannetwork_b200.flat import EvidenceBatch
    last = net.n_nodes - 1
    cases = []
    for c in range(n_cases):
        d = {int(ev.ev_node[e]): int(ev.ev_state[e]) for e in range(ev.ev_off[c], ev.ev_off[c + 1])}
        d.setdefault(last, c % 2)
        cases.append(d)
    return EvidenceBatch.from_cases(net, cases)


def _refused():
    """(network, variant, environment, reason) of shapes one side of a boundary refuses."""
    card = [2] * 8
    yield synth._assemble(card, [[]] * 7 + [list(range(7))], 20, "indeg7"), 0, {}, "in-degree > 6"
    yield synth._assemble([17, 2], [[], [0]], 21, "card17"), 0, {}, "cardinality > 16"
    # 65 8-state children of a 16-state root: a CPT arena too large to unroll (66 KB in double), CPTs too small for the
    # dense path (128 entries), and the class-looped walk refuses the hub
    yield (synth._assemble([16] + [8] * 65, [[]] + [[0]] * 65, 22, "hub65_wide"), 0, {"BNBP_CLASSLOOP": "2"},
           "class-looped walk: a hub with more than 64 children")
    # 100 node shapes (10 roots of 2 ... 11 states, each with children of 2 ... 11 states): too many multiply-adds to
    # unroll, and too many classes to loop
    card, par = list(range(2, 12)), [[] for _ in range(10)]
    for p in range(10):
        for r in range(2, 12):
            card.append(r)
            par.append([p])
    yield synth._assemble(card, par, 23, "classes100"), 0, {"BNBP_CLASSLOOP": "2"}, "more than 96 node shape classes"
    yield _hub(65, "hub65"), 8, {}, ONCHIP_REFUSED["hub65"]


REFUSED = list(_refused())
