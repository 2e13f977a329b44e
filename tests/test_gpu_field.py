"""The field and integer primitives on the GPU, one primitive per kernel (tests/csrc/field_device_api.cu), against the
Python-integer reference of tests/field_ref.py.

The host tests (test_field_host.py) run the device formulations with an emulated carry flag; this runs what the GPU
runs: the PTX carry chains, carries kept between separate asm statements, the 64-bit pair accumulators and
__funnelshift_r.  Every primitive runs in two builds, roomy (no register limit) and register-starved (at most 32
registers: the carry chains spill), in one launch over the edge cross product of its operands, limb-pattern tuples and
uniform tuples.  The launch size is not a multiple of the block, rows past it are canaries that must come back as sent,
every output word and status word is compared exactly, and the two builds must return identical bytes."""
import ctypes
import random
import time

import numpy as np
import pytest

from tests import field_ref as fr
from tests import util
from tests.field_ref import M

pytestmark = pytest.mark.gpu

# tests/csrc/field_device_api.cu: enum Prim, in order
PRIMS = ["mul", "mul_wide", "sqr_wide", "sqr", "mul_lo", "mont_mul", "to_mont", "from_mont", "add", "sub", "neg", "reduce",
         "shr", "shl", "bitop", "bnot", "cmp", "divrem", "pow", "inv_fermat", "inv_safegcd", "mul_hi_trunc", "mont_reduce",
         "dot_eval", "mul2", "ntt_mul", "bfly_dif", "bfly_dit", "alu", "from_narrow"]
VARIANTS = ("roomy", "starved")
N_RANDOM, N_RANDOM_SLOW = 1 << 16, 1 << 14      # limb-pattern and uniform tuples each; pow, the inversions, divrem
CANARY_ROWS = 37
OUT_FILL, STATUS_FILL = 0xA5A5A5A5, 0x5A5A5A5A


def pair(x, y):
    return x | (y << 256)


# name -> (operand domains, random tuples, reference (a, b, c, op) -> (output integer, status), ops of a row or None).
# A row is (a, b, c, op): a, b, c are the integers the operand arrays hold (two values are packed low first), op the
# per-row word.  Rows whose operands take several op words are expanded over all of them on the edges.
SPECS = {
    "mul": ("cc", N_RANDOM, lambda a, b, c, op: (fr.mul(a, b), 0)),
    "mul_wide": ("ww", N_RANDOM, lambda a, b, c, op: (fr.mul_wide(a, b), 0)),
    "sqr_wide": ("w", N_RANDOM, lambda a, b, c, op: (fr.mul_wide(a, a), 0)),
    "sqr": ("c", N_RANDOM, lambda a, b, c, op: (fr.mul(a, a), 0)),
    "mul_lo": ("ww", N_RANDOM, lambda a, b, c, op: (fr.mul_lo(a, b), 0)),
    "mont_mul": ("cc", N_RANDOM, lambda a, b, c, op: (fr.mont_mul(a, b), 0)),
    "to_mont": ("c", N_RANDOM, lambda a, b, c, op: (fr.to_mont(a), 0)),
    "from_mont": ("c", N_RANDOM, lambda a, b, c, op: (fr.from_mont(a), 0)),
    "add": ("cc", N_RANDOM, lambda a, b, c, op: (fr.add(a, b), 0)),
    "sub": ("cc", N_RANDOM, lambda a, b, c, op: (fr.sub(a, b), 0)),
    "neg": ("c", N_RANDOM, lambda a, b, c, op: (fr.neg(a), 0)),
    "reduce": ("w", N_RANDOM, lambda a, b, c, op: (fr.reduce256(a), 0)),
    "shr": ("cs", N_RANDOM, lambda a, b, c, op: (fr.shr(a, b), 0)),
    "shl": ("cs", N_RANDOM, lambda a, b, c, op: fr.shl(a, b)),
    "bitop": ("cc", N_RANDOM, lambda a, b, c, op: fr.bitop(a, b, op), (0, 1, 2)),
    "bnot": ("w", N_RANDOM, lambda a, b, c, op: (fr.bnot(a), 0)),
    "cmp": ("cc", N_RANDOM, lambda a, b, c, op: (0, fr.cmp(a, b, op)), (0, 1, 2, 3)),
    "divrem": ("cc", N_RANDOM_SLOW, lambda a, b, c, op: (pair(*fr.divrem(a, b)), 0)),
    "pow": ("cc", N_RANDOM_SLOW, lambda a, b, c, op: (fr.fe_pow(a, b), 0)),
    "inv_fermat": ("c", N_RANDOM_SLOW, lambda a, b, c, op: (fr.inv(a), 0)),
    "inv_safegcd": ("c", N_RANDOM_SLOW, lambda a, b, c, op: (fr.inv(a), 0)),
    "mul_hi_trunc": ("ww", N_RANDOM, lambda a, b, c, op: (fr.mul_hi_trunc(a, b), 0)),
    "ntt_mul": ("cc", N_RANDOM, lambda a, b, c, op: (fr.ntt_mul(a, b), 0)),
    "bfly_dif": ("ccc", N_RANDOM, lambda a, b, c, op: (pair(*fr.bfly_dif(a, b, c)), 0)),
    "bfly_dit": ("ccc", N_RANDOM, lambda a, b, c, op: (pair(*fr.bfly_dit(a, b, c)), 0)),
    "alu": ("ccc", N_RANDOM, lambda a, b, c, op: fr.alu(op, a, b, c), tuple(fr.ALU_OPS)),
    "from_narrow": ("n", N_RANDOM, lambda a, b, c, op: (fr.from_narrow(a), 0)),
}


def generic_rows(name, seed):
    doms, n_random, _, *ops = SPECS[name]
    ops = ops[0] if ops else (0,)
    rnd = random.Random(seed)
    rows = []
    tuples = fr.operand_tuples(doms, n_random, seed)
    n_edge = len(fr.edge_tuples(doms))
    for i, t in enumerate(tuples):
        t = t + (0,) * (3 - len(t))
        for op in (ops if i < n_edge else (rnd.choice(ops),)):
            rows.append(t + (op,))
    if name == "divrem":
        rows = [r for r in rows if r[1]]
    return rows


def mont_reduce_rows(seed):
    """(P, 0, 0, n_cond_sub) for 512-bit P below the bound of every n_cond_sub: P's low half any 256-bit value, its high
    half below the limit (edges, limb patterns reduced into range, uniform)"""
    rnd = random.Random(seed)
    rows = []
    for ncs in (1, 2, 3):
        lim = fr.mont_reduce_limit(ncs)
        his = [0, 1, lim - 1, lim - 2, lim >> 1, (1 << 32) - 1, M - 1]
        for lo in fr.WIDE_EDGES:
            for hi in his:
                rows.append((lo | (hi % lim) << 256, 0, 0, ncs))
        for _ in range(N_RANDOM // 3):
            lo = fr.limb_pattern(rnd, "w") if rnd.random() < 0.5 else rnd.getrandbits(256)
            hi = fr.limb_pattern(rnd, "w") % lim if rnd.random() < 0.5 else rnd.randrange(lim)
            rows.append((lo | hi << 256, 0, 0, ncs))
    return rows


def dot_rows(seed):
    """(xs, cs, n_terms | n_cond_sub << 8, kinds) of OP_DOTs of 0 .. 16 terms of all four kinds in any order, within the
    plan compiler's bound; operands are edges, limb patterns or uniform, and every 8th row has all operands M - 1"""
    rnd = random.Random(seed)
    pick = lambda: (rnd.choice(fr.CANON_EDGES) if rnd.random() < 0.4 else
                    fr.limb_pattern(rnd) if rnd.random() < 0.5 else rnd.randrange(M))
    rows = []
    while len(rows) < N_RANDOM_SLOW:
        n_mac, n_hi = rnd.randrange(0, 17), rnd.randrange(0, 5)
        n_const = rnd.randrange(0, 2)
        ncs = fr.dot_ncs(n_mac, n_hi)
        if ncs is None or n_mac + n_hi + n_const > 16:
            continue
        kinds = [0] * n_mac + [rnd.choice((1, 2)) for _ in range(n_hi)] + [3] * n_const
        rnd.shuffle(kinds)
        worst = len(rows) % 8 == 0
        xs = [0 if k == 3 else M - 1 if worst else pick() for k in kinds]
        cs = [0 if k in (1, 2) else M - 1 if worst else pick() for k in kinds]
        if worst:       # a subtracted value of 0 adds M, the largest plain term
            xs = [0 if k == 2 else x for k, x in zip(kinds, xs)]
        a = sum(x << (256 * t) for t, x in enumerate(xs))
        b = sum(c << (256 * t) for t, c in enumerate(cs))
        rows.append((a, b, len(kinds) | ncs << 8, sum(k << (2 * t) for t, k in enumerate(kinds))))
    return rows


def mul2_rows(seed):
    """two independent products per row, each pair from the edge cross product, limb patterns or uniform values"""
    t = fr.operand_tuples("cc", N_RANDOM, seed)
    rnd = random.Random(seed + 1)
    rows = []
    for i, (x1, y1) in enumerate(t):
        x2, y2 = t[(i * 7 + 3) % len(t)] if rnd.random() < 0.5 else t[-1 - i]
        rows.append((pair(x1, x2), pair(y1, y2), 0, 0))
    return rows


def dot_ref(a, b, c, op):
    nt = c & 0xFF
    kinds = [(op >> (2 * t)) & 3 for t in range(nt)]
    mask = (1 << 256) - 1
    return fr.dot_eval(kinds, [(a >> (256 * t)) & mask for t in range(nt)], [(b >> (256 * t)) & mask for t in range(nt)]), 0


CUSTOM = {
    "mont_reduce": (mont_reduce_rows, lambda a, b, c, op: (fr.mont_reduce(a), 0)),
    "dot_eval": (dot_rows, dot_ref),
    "mul2": (mul2_rows, lambda a, b, c, op: (pair(fr.mul(a & fr.MASK256, b & fr.MASK256), fr.mul(a >> 256, b >> 256)), 0)),
}
assert set(SPECS) | set(CUSTOM) == set(PRIMS)


def to_words(vals, words):
    if words == 0:
        return np.zeros((len(vals), 0), np.uint32)
    return np.frombuffer(b"".join(int(v).to_bytes(4 * words, "little") for v in vals), dtype=np.uint32).reshape(len(vals), words).copy()


def from_words(row):
    return sum(int(w) << (32 * i) for i, w in enumerate(row))


@pytest.fixture(scope="module")
def lib():
    return util.field_device_lib()


def shape(lib, prim):
    w = (ctypes.c_int * 4)()
    assert lib.fd_shape(prim, w) == 0
    return list(w)


def launch(lib, prim, variant, n, a, b, c, op, out, status):
    p = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))
    return lib.fd_launch(prim, variant, n, len(op), p(a), p(b), p(c), p(op), p(out), p(status))


@pytest.mark.parametrize("name", PRIMS)
def test_primitive_on_device(lib, name):
    t0 = time.time()
    prim = PRIMS.index(name)
    seed = 0xF1E1D + prim
    if name in CUSTOM:
        rows, ref = CUSTOM[name][0](seed), CUSTOM[name][1]
    else:
        rows, ref = generic_rows(name, seed), SPECS[name][2]
    if len(rows) % 128 == 0:        # the last block is partial in both builds
        rows = rows[:-1]
    n = len(rows)
    want = [ref(*r) for r in rows]
    wa, wb, wc, wo = shape(lib, prim)
    pad = [(0, 0, 0, 0)] * CANARY_ROWS
    a = to_words([r[0] for r in rows + pad], wa)
    b = to_words([r[1] for r in rows + pad], wb)
    c = to_words([r[2] for r in rows + pad], wc)
    op = np.array([r[3] for r in rows + pad], dtype=np.uint32)
    exp_out = to_words([v for v, _ in want], wo)
    exp_st = np.array([s for _, s in want], dtype=np.uint32)
    t_ref = time.time() - t0
    results = []
    for variant, vname in enumerate(VARIANTS):
        t1 = time.time()
        out = np.full((n + CANARY_ROWS, wo), OUT_FILL, dtype=np.uint32)
        st = np.full(n + CANARY_ROWS, STATUS_FILL, dtype=np.uint32)
        rc = launch(lib, prim, variant, n, a, b, c, op, out, st)
        assert rc == 0, f"{name} [{vname}]: CUDA error {rc}"
        assert (out[n:] == OUT_FILL).all() and (st[n:] == STATUS_FILL).all(), f"{name} [{vname}]: a canary row past n = {n} was written"
        bad = np.nonzero((out[:n] != exp_out).any(axis=1) | (st[:n] != exp_st))[0]
        if len(bad):
            lines = []
            for i in bad[:6]:
                ra, rb, rc_, rop = rows[i]
                lines.append(f"  row {i}: a={ra:#x} b={rb:#x} c={rc_:#x} op={rop}: want {want[i][0]:#x} status {want[i][1]}, "
                             f"got {from_words(out[i]):#x} status {int(st[i])}")
            pytest.fail(f"{name} [{vname}]: {len(bad)} of {n} rows differ\n" + "\n".join(lines))
        results.append((out, st))
        print(f"{name} [{vname}]: {n} rows checked, {time.time() - t1:.2f} s")
    assert np.array_equal(results[0][0], results[1][0]) and np.array_equal(results[0][1], results[1][1]), \
        f"{name}: the roomy and the starved builds differ"
    print(f"{name}: reference {t_ref:.2f} s, total {time.time() - t0:.2f} s")
