"""Bit-sliced plan (csrc/bitplan.cpp) on the host simulator: typing (table domain, bit-vector domain with bit heaps),
LUT DAG, steps and plane slots, the bit contract on inputs.  The simulator (tests/csrc/plan_host_sim.cpp) executes the
same steps the device kernel does, on one group of 32 input sets."""
import random

import pytest

from tests import util
from tests.util import po

M = po.M


def boolean_graph(rnd: random.Random, n_inputs=24, n_gates=300):
    """Random graph in the shapes circomlib gives Boolean circuits: polynomial gates on bits (a*b, a+b-2ab,
    a*(1-2b-2c+4bc)+b+c-2bc, 1-a, multiplexers c*(a-b)+b), BinSum-style sums of shifted bits with (lin >> k) & 1
    extraction, and word arithmetic in the style of sha256compression_function.circom (Shl, Shr, Bor, Band, Bxor, Add,
    masks).  Witness: bits only.  Returns (nodes, witness_signals, input_map)."""
    nodes = [(po.K_INPUT, i) for i in range(n_inputs + 1)]
    cache = {}

    def const(v):
        if v % M not in cache:
            nodes.append((po.K_CONST, v % M))
            cache[v % M] = len(nodes) - 1
        return cache[v % M]

    def duo(op, a, b):
        nodes.append((po.K_DUO, po.DUO[op], a, b))
        return len(nodes) - 1
    bits = list(range(1, n_inputs + 1))
    wit = [0]
    words = []          # (node, width)
    for _ in range(n_gates):
        r = rnd.random()
        pick = lambda: rnd.choice(bits[-40:] if rnd.random() < 0.6 else bits)
        if r < 0.15:
            bits.append(duo("Mul", pick(), pick()))
        elif r < 0.3:                                # xor: a + b - 2ab
            a, b = pick(), pick()
            bits.append(duo("Sub", duo("Add", a, b), duo("Mul", const(2), duo("Mul", a, b))))
        elif r < 0.42:                               # xor3 as xor3.circom writes it
            a, b, c = pick(), pick(), pick()
            mid = duo("Mul", b, c)
            t = duo("Add", duo("Sub", duo("Sub", const(1), duo("Mul", const(2), b)), duo("Mul", const(2), c)), duo("Mul", const(4), mid))
            bits.append(duo("Sub", duo("Add", duo("Add", duo("Mul", a, t), b), c), duo("Mul", const(2), mid)))
            wit.append(mid)
        elif r < 0.5:                                # not, mux
            if rnd.random() < 0.5:
                bits.append(duo("Sub", const(1), pick()))
            else:
                c, a, b = pick(), pick(), pick()
                bits.append(duo("Add", duo("Mul", c, duo("Sub", a, b)), b))
        elif r < 0.62:                               # BinSum: lin = sum bits * 2^j over several operands, then extraction
            n, ops_ = rnd.choice([2, 4, 8, 32]), rnd.choice([2, 3, 5])
            lin = const(0)
            for _k in range(ops_):
                for j in range(n):
                    lin = duo("Add", lin, duo("Mul", pick(), const(1 << j)))
            nout = n + (ops_ - 1).bit_length()
            for k in range(nout):
                bits.append(duo("Band", duo("Shr", lin, const(k)), const(1)))
                if rnd.random() < 0.7:
                    wit.append(bits[-1])
        elif r < 0.7:                                # pack a word from bits (Shl + Add, or Mul by 2^j)
            n = rnd.choice([8, 24])                    # x << (n - k) must stay below 2^62 (like SHA-256's 32-bit rotations)
            w = const(0)
            for j in range(n):
                w = duo("Add", w, duo("Shl", pick(), const(j)) if rnd.random() < 0.5 else duo("Mul", pick(), const(1 << j)))
            words.append((w, n))
        elif r < 0.9 and words:                      # word ops
            (x, wx), (y, wy) = rnd.choice(words), rnd.choice(words)
            k = rnd.randrange(1, max(2, min(8, wx)))
            op = rnd.choice(["Bxor", "Band", "Bor", "rot", "add", "shr", "not"])
            if wx < 2 and op in ("rot", "shr"):
                op = "not"
            if op == "rot":
                mask = const((1 << wx) - 1)
                words.append((duo("Band", duo("Bor", duo("Shr", x, const(k)), duo("Shl", x, const(wx - k))), mask), wx))
            elif op == "add":
                words.append((duo("Band", duo("Add", x, y), const((1 << max(wx, wy)) - 1)), max(wx, wy)))
            elif op == "shr":
                words.append((duo("Shr", x, const(k)), max(wx - k, 1)))
            elif op == "not":
                words.append((duo("Bxor", x, const((1 << wx) - 1)), wx))
            else:
                words.append((duo(op, x, y), max(wx, wy)))
        elif words:                                  # unpack a word into bits again
            x, wx = rnd.choice(words)
            for k in range(min(wx, 6)):
                bits.append(duo("Band", duo("Shr", x, const(rnd.randrange(wx))), const(1)))
        wit.append(bits[-1])
    wit += bits[-8:] + [1, 1, const(1), const(0), const(7)]
    return nodes, wit, {"x": (1, n_inputs)}


@pytest.mark.parametrize("merge", [True, False])
def test_random_boolean_graphs(merge):
    rnd = random.Random(2024)
    luts = 0
    for t in range(12):
        nodes, wit, imap = boolean_graph(rnd, n_inputs=rnd.choice([5, 24, 70]), n_gates=rnd.choice([60, 300]))
        g = util.BitSimGraph(po.serialize_graph(nodes, wit, imap), merge=merge)
        assert g.info["eligible"], g.reason
        luts += g.info["n_luts"]
        n_in = g.I - 1
        rows = [[1] + [rnd.randrange(2) for _ in range(n_in)] for _ in range(rnd.choice([1, 7, 32]))]
        res, ok = g.eval(rows)
        assert ok == (1 << len(rows)) - 1
        for b, row in enumerate(rows):
            assert res[b] == po.evaluate(nodes, row, wit, "circom"), (t, b)
    assert luts > 1000


def test_contract_violations_are_detected_per_input_set():
    rnd = random.Random(7)
    nodes, wit, imap = boolean_graph(rnd, n_inputs=16, n_gates=120)
    g = util.BitSimGraph(po.serialize_graph(nodes, wit, imap))
    rows = [[1] + [rnd.randrange(2) for _ in range(16)] for _ in range(32)]
    bad = {3: 2, 8: M - 1, 17: 1 << 255, 31: 256}
    for b, v in bad.items():
        rows[b][1 + b % 16] = v
    res, ok = g.eval(rows)
    assert ok == ((1 << 32) - 1) & ~sum(1 << b for b in bad)
    for b, row in enumerate(rows):
        if b in bad:
            assert res[b] is None
        else:
            assert res[b] == po.evaluate(nodes, row, wit, "circom")


def test_sha256_is_all_bits_and_exact():
    data = util.golden_graph("circuit8_sha256_512")
    g = util.BitSimGraph(data)
    assert g.info["eligible"] and g.info["n_luts"] > 100000 and g.info["n_inputs_checked"] == 512
    nodes, wit, imap = po.deserialize_graph(data)
    buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs("circuit8_sha256_512")))
    rnd = random.Random(8)
    rows = [buf] + [[1] + [rnd.randrange(2) for _ in range(512)] for _ in range(3)]
    res, ok = g.eval(rows)
    assert ok == 15
    assert po.wtns_from_witness(res[0]) == util.golden_wtns("circuit8_sha256_512")
    for b in (1, 3):
        assert res[b] == po.evaluate(nodes, rows[b], wit)


@pytest.mark.parametrize("name", ["circuit5_poseidon", "circuit7_poseidon4", "poseidon2", "circuit9_authV2", "circuit11_key_expansion"])
def test_field_graphs_are_not_eligible(name):
    """field arithmetic on the inputs (Poseidon: every value would be a 254-bit table entry of a few "bit" inputs; authV2:
    sums that can reach the modulus; circuit11: comparisons of integers)"""
    g = util.BitSimGraph(util.golden_graph(name))
    assert not g.info["eligible"] and g.reason


def test_degenerate_plans_and_edge_graphs():
    # Num2Bits + Bits2Num of ONE field input: pure wiring (no LUTs), the input is taken apart into the bits of its canonical
    # value (no contract), `out` and the input itself are wide witness values
    g = util.BitSimGraph(util.golden_graph("circuit6_num2bits"))
    assert g.info["eligible"] and g.info["n_luts"] == 0 and g.info["has_field_inputs"] and g.info["n_wide"] == 2
    # a plane at several witness positions, an input that is a witness signal itself, constants, an input nobody reads
    nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_INPUT, 2), (po.K_INPUT, 3), (po.K_DUO, po.DUO["Mul"], 1, 2), (po.K_CONST, 5),
             (po.K_DUO, po.DUO["Mul"], 3, 3), (po.K_DUO, po.DUO["Sub"], 6, 3)]
    wit = [0, 4, 4, 1, 5, 4, 2, 7]
    g = util.BitSimGraph(po.serialize_graph(nodes, wit, {"x": (1, 3)}))
    assert g.info["eligible"] and g.info["n_inputs_checked"] == 3
    rows = [[1, a, b, c] for a in (0, 1) for b in (0, 1) for c in (0, 1)] + [[1, 1, 1, 5]]
    res, ok = g.eval(rows)
    assert ok == 0xFF                                 # x*x - x is 0 for bits only: the set with x = 5 must not take this path
    for b in range(8):
        assert res[b] == po.evaluate(nodes, rows[b], wit)
    # a witness signal that is a small integer, not a bit: a wide witness value
    nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_INPUT, 2), (po.K_DUO, po.DUO["Add"], 1, 2)]
    g = util.BitSimGraph(po.serialize_graph(nodes, [0, 3], {"x": (1, 2)}))
    assert g.info["eligible"] and g.info["n_wide"] == 1
    res, ok = g.eval([[1, 1, 1], [1, 0, 1], [1, 2, 0]])
    assert ok == 3 and res[0] == [1, 2] and res[1] == [1, 1]


def field_bits_graph(rnd: random.Random, n_field=3, n_bits=6, n_gates=80):
    """Field inputs that the graph only takes apart (Num2Bits: (x >> k) & 1, masks) next to contract bits: logic on the
    extracted bits, Bits2Num-style recomposition up to 250 bits (wide witness values), the inputs themselves as witness
    signals.  Returns (nodes, witness_signals, input_map)."""
    n_inputs = n_field + n_bits
    nodes = [(po.K_INPUT, i) for i in range(n_inputs + 1)]
    cache = {}

    def const(v):
        if v % M not in cache:
            nodes.append((po.K_CONST, v % M))
            cache[v % M] = len(nodes) - 1
        return cache[v % M]

    def duo(op, a, b):
        nodes.append((po.K_DUO, po.DUO[op], a, b))
        return len(nodes) - 1
    wit = [0] + list(range(1, n_inputs + 1))
    bits = list(range(n_field + 1, n_inputs + 1))
    for f in range(1, n_field + 1):
        ks = rnd.sample(range(0, 254), 40) + [0, 253, 254, 255, 300]
        for k in ks:
            bits.append(duo("Band", duo("Shr", f, const(k)), const(1)))
            if rnd.random() < 0.5:
                wit.append(bits[-1])
        wit.append(duo("Band", duo("Shr", f, const(rnd.randrange(200))), const((1 << rnd.randrange(2, 40)) - 1)))   # a masked slice: wide
    for _ in range(n_gates):
        r = rnd.random()
        pick = lambda: rnd.choice(bits)
        if r < 0.3:
            bits.append(duo("Mul", pick(), pick()))
        elif r < 0.6:
            a, b = pick(), pick()
            bits.append(duo("Sub", duo("Add", a, b), duo("Mul", const(2), duo("Mul", a, b))))
        elif r < 0.8:
            lc = const(0)
            for j in sorted(rnd.sample(range(250), rnd.choice([3, 40, 216]))):
                lc = duo("Add", lc, duo("Mul", pick(), const(1 << j)))
            wit.append(lc)                                 # Bits2Num: a wide witness value
            continue
        else:
            bits.append(duo("Sub", const(1), pick()))
        wit.append(bits[-1])
    return nodes, wit, {"x": (1, n_inputs)}


def test_field_inputs_taken_apart_into_bits_and_wide_outputs():
    rnd = random.Random(606)
    for t in range(8):
        n_field, n_bits = rnd.choice([1, 3]), rnd.choice([0, 6])
        nodes, wit, imap = field_bits_graph(rnd, n_field, n_bits)
        g = util.BitSimGraph(po.serialize_graph(nodes, wit, imap))
        assert g.info["eligible"] and g.info["has_field_inputs"] and g.info["n_wide"] >= n_field, g.reason
        rows = []
        for _ in range(32):
            fv = [rnd.choice([0, 1, M - 1, M, M + 5, (1 << 256) - 1, (1 << 253), rnd.randrange(M), rnd.randrange(1 << 256)]) for _ in range(n_field)]
            rows.append([1] + fv + [rnd.randrange(2) for _ in range(n_bits)])
        if n_bits:
            rows[7][n_field + 1] = 9                       # breaks the contract of a bit input; field inputs have none
        res, ok = g.eval(rows)
        assert ok == (0xFFFFFFFF & ~(1 << 7) if n_bits else 0xFFFFFFFF)
        for b, row in enumerate(rows):
            if res[b] is not None:
                assert res[b] == po.evaluate(nodes, row, wit, "circom"), (t, b)


def test_bit_corpus_coverage():
    """util.bit_corpus, the corpus of the GPU matrix (tests/test_gpu_bit_matrix.py), reaches everything util.bit_plan_coverage
    records, and its plans are exact on the simulator: every step residue mod 16, header rings of 1 .. 4 and >= 7 chunks,
    steps of 1, 2 .. 31 and 32 LUTs, copies, slot reuse, wide values of every plane-loop length, constants, unread contract
    inputs and field-input bits in every limb"""
    from oracle import cref
    import numpy as np
    rnd = random.Random(11)
    cov = None
    for name, data in util.bit_corpus():
        g = util.BitSimGraph(data)
        assert g.info["eligible"] and (g.info["n_luts"] or g.info["has_field_inputs"]), name
        c = util.bit_plan_coverage(g.plan())
        cov = c if cov is None else util.merge_coverage(cov, c)
        if g.W > 5000:
            continue                                   # SHA-256: test_sha256_is_all_bits_and_exact
        rows = [[1] + [rnd.choice([0, 1, 1, M - 1, (1 << 256) - 1]) if rnd.random() < 0.3 else rnd.randrange(2) for _ in range(g.I - 1)]
                for _ in range(32)]
        res, ok = g.eval(rows)
        want = cref.CGraph(data).evaluate_batch(np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(32, -1, 32), 4)
        for b in range(32):
            if (ok >> b) & 1:
                assert res[b] == util.unpack_u256(want[b].tobytes()), (name, b)
    util.assert_bit_coverage(cov)
