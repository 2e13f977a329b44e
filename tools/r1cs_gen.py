"""Generated (graph, R1CS) pairs whose witnesses satisfy the R1CS by construction (no circom here to compile real ones).

Wire 0 is the constant 1 and wires 1 .. n_in are the graph's inputs (input signal "x").  Every further wire k comes with
one constraint  A * B = C' + g * w_k  over earlier wires, and the graph computes  w_k = (<A,w> * <B,w> - <C',w>) / g
from Mul / Add / Sub nodes and constants.  The witness list is the wires in order, so wire i is witness position i,
as for a circom circuit.

  random_pair(rnd, ...)    coefficients from {1, M - 1, 0, small, tests/util.py EDGE values, uniform}; linear
                           combinations of 0 to 100 terms, repeated wires, constant-only (wire 0) combinations, empty A/B
  poseidon_pair(rnd, ...)  what circom --O2 leaves of Poseidon: S-box constraints x*x = x2, x2*x2 = x4, x4*x = x5 where
                           x is a substituted mix-layer combination of the previous state plus a round constant

Both return (graph_bytes, r1cs) with r1cs in the layout of tests/r1cs_ref.py.
"""
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import pyoracle as po  # noqa: E402
from tests.util import EDGE  # noqa: E402

M = po.M


class _Builder:
    def __init__(self, n_in):
        self.nodes = [(po.K_INPUT, i) for i in range(n_in + 1)]
        self.wire_node = list(range(n_in + 1))          # wire -> graph node
        self.consts = {}
        self.cons = []
        self.lc_cache = {}

    def const(self, v):
        v %= M
        if v not in self.consts:
            self.nodes.append((po.K_CONST, v))
            self.consts[v] = len(self.nodes) - 1
        return self.consts[v]

    def duo(self, op, a, b):
        self.nodes.append((po.K_DUO, po.DUO[op], a, b))
        return len(self.nodes) - 1

    def lc_node(self, lc):
        key = tuple(lc)
        if key in self.lc_cache:
            return self.lc_cache[key]
        acc = None
        for w, c in lc:
            x = self.wire_node[w]
            t = x if c % M == 1 else self.duo("Mul", self.const(c), x)
            acc = t if acc is None else self.duo("Add", acc, t)
        n = self.const(0) if acc is None else acc
        self.lc_cache[key] = n
        return n

    def new_wire(self, a, b, c_rest, g=1):
        """adds wire k with A * B = C' + g * w_k; returns k"""
        k = len(self.wire_node)
        v = self.duo("Mul", self.lc_node(a), self.lc_node(b))
        if c_rest:
            v = self.duo("Sub", v, self.lc_node(c_rest))
        if g % M != 1:
            v = self.duo("Mul", v, self.const(pow(g, M - 2, M)))
        self.wire_node.append(v)
        self.cons.append((list(a), list(b), list(c_rest) + [(k, g % M)]))
        return k

    def result(self, n_in):
        r1cs = {"n_wires": len(self.wire_node), "n_pub_out": 0, "n_pub_in": 0, "n_prv_in": n_in,
                "n_labels": len(self.wire_node), "constraints": self.cons}
        return po.serialize_graph(self.nodes, self.wire_node, {"x": (1, n_in)}), r1cs


def random_coeff(rnd):
    r = rnd.random()
    if r < 0.25:
        return 1
    if r < 0.4:
        return M - 1
    if r < 0.45:
        return 0
    if r < 0.6:
        return rnd.randrange(2, 1000)
    if r < 0.75:
        return rnd.choice(EDGE) % M
    return rnd.randrange(M)


def random_lc(rnd, n_wires):
    r = rnd.random()
    if r < 0.08:
        return []
    if r < 0.15:
        return [(0, random_coeff(rnd))]                   # constant-only
    n = rnd.choice((1, 1, 2, 3, 4, 5, 8, 13, 21, 22, 23, 30, 50, 100))
    lc = [(rnd.randrange(n_wires) if rnd.random() < 0.7 else rnd.randrange(max(0, n_wires - 8), n_wires), random_coeff(rnd))
          for _ in range(n)]
    if n > 1 and rnd.random() < 0.3:
        lc[rnd.randrange(n)] = (lc[0][0], random_coeff(rnd))   # a repeated wire
    return lc


def random_pair(rnd: random.Random, n_in=6, n_constraints=120):
    b = _Builder(n_in)
    for _ in range(n_constraints):
        nw = len(b.wire_node)
        g = rnd.choice((1, M - 1, rnd.randrange(1, M)))
        b.new_wire(random_lc(rnd, nw), random_lc(rnd, nw), random_lc(rnd, nw) if rnd.random() < 0.7 else [], g)
    return b.result(n_in)


def _lc_add(acc, lc, c):
    for w, v in lc:
        acc[w] = (acc.get(w, 0) + c * v) % M


def poseidon_pair(rnd: random.Random, n_in=4, t=3, n_hashes=2, full_rounds=8, partial_rounds=57, max_terms=40):
    """A chain of Poseidon-like permutations; the state is kept as linear combinations of wires (substituted, as --O2
    does) and materialised by a linear constraint 1 * lc = w when one grows past max_terms."""
    b = _Builder(n_in)
    mix = [[rnd.randrange(1, M) for _ in range(t)] for _ in range(t)]
    state = [{1 + (i % n_in): 1} for i in range(t)]
    for _h in range(n_hashes):
        for r in range(full_rounds + partial_rounds):
            full = r < full_rounds // 2 or r >= full_rounds // 2 + partial_rounds
            for j in range(t if full else 1):
                x = dict(state[j])
                x[0] = (x.get(0, 0) + rnd.randrange(M)) % M         # round constant
                xl = sorted(x.items())
                x2 = b.new_wire(xl, xl, [])
                x4 = b.new_wire([(x2, 1)], [(x2, 1)], [])
                x5 = b.new_wire([(x4, 1)], xl, [])
                state[j] = {x5: 1}
            new = []
            for i in range(t):
                acc = {}
                for j in range(t):
                    _lc_add(acc, state[j].items(), mix[i][j])
                acc = {w: c for w, c in acc.items() if c}
                if len(acc) > max_terms:
                    acc = {b.new_wire([(0, 1)], sorted(acc.items()), []): 1}
                new.append(acc)
            state = new
    return b.result(n_in)
