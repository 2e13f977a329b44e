"""csrc/field.cuh (the algorithms the CUDA kernels run: Barrett multiplication, the Montgomery helpers and
reduction, shifts, bitwise ops, signed comparisons, long division, pow, inversion) against Python integers, twice:
the plain host path, and the DEVICE formulations (PTX carry chains on even/odd accumulators) compiled for the host
with an emulated carry flag (-DGW_EMULATE_PTX).  The expected values come from tests/field_ref.py, which
test_gpu_field.py checks the real PTX against on the GPU."""
import ctypes
import random

import numpy as np
import pytest

from tests import field_ref as fr
from tests import util
from tests.util import M

A8 = ctypes.c_uint32 * 8
A16 = ctypes.c_uint32 * 16


def enc(x):
    return A8(*[(x >> (32 * i)) & 0xFFFFFFFF for i in range(8)])


def dec(a):
    return sum(int(v) << (32 * i) for i, v in enumerate(a))


def call2(f, a, b):
    r = A8()
    f(enc(a), enc(b), r)
    return dec(r)


def call1(f, a):
    r = A8()
    f(enc(a), r)
    return dec(r)


@pytest.mark.parametrize("ptx", [False, True])
def test_field_and_integer_ops_random_and_edges(ptx):
    L = util.field_host_lib(ptx)
    assert bool(L.t_emulates_ptx()) == ptx
    rnd = random.Random(1)
    for t in range(6000):
        a, b = util.random_value(rnd), util.random_value(rnd)
        assert call2(L.t_mul, a, b) == fr.mul(a, b)
        r16 = A16(); L.t_mul_wide(enc(a), enc(b), r16); assert dec(r16) == fr.mul_wide(a, b)
        r16 = A16(); L.t_sqr_wide(enc(a), r16); assert dec(r16) == fr.mul_wide(a, a)
        assert call1(L.t_sqr, a) == fr.mul(a, a)
        r8 = A8(); L.t_mul_lo(enc(a), enc(b), r8); assert dec(r8) == fr.mul_lo(a, b)
        assert call2(L.t_mont_mul, a, b) == fr.mont_mul(a, b)
        assert call1(L.t_to_mont, a) == fr.to_mont(a) and call1(L.t_from_mont, a) == fr.from_mont(a)
        assert call2(L.t_add, a, b) == fr.add(a, b) and call2(L.t_sub, a, b) == fr.sub(a, b)
        assert call1(L.t_neg, a) == fr.neg(a)
        x = rnd.randrange(1 << 256)
        assert call1(L.t_reduce, x) == fr.reduce256(x)
        sh = rnd.choice([0, 1, 31, 32, 33, 63, 64, 100, 128, 200, 252, 253, 254, 255, 256, M - 1, rnd.randrange(300)])
        assert call2(L.t_shr, a, sh) == fr.shr(a, sh)
        r = A8(); ov = L.t_shl(enc(a), enc(sh), r)
        assert (dec(r), ov) == fr.shl(a, sh)
        for w in range(3):
            r = A8(); eq = L.t_bitop(enc(a), enc(b), w, r)
            assert (dec(r), eq) == fr.bitop(a, b, w)
        for w in range(4):
            assert L.t_cmp(enc(a), enc(b), w) == fr.cmp(a, b, w)
        assert call1(L.t_bnot, a) == fr.bnot(a)
        if t < 150:
            if b:
                q, rr = A8(), A8(); L.t_divrem(enc(a), enc(b), q, rr); assert (dec(q), dec(rr)) == fr.divrem(a, b)
            assert call2(L.t_pow, a, b) == fr.fe_pow(a, b)
            assert call1(L.t_inv, a) == fr.inv(a)


@pytest.mark.parametrize("ptx", [False, True])
def test_barrett_worst_cases(ptx):
    L = util.field_host_lib(ptx)
    for a in ((1 << 256) - 1, (1 << 256) - (1 << 32), 0xFFFFFFFF, ((1 << 256) - 1) // 3, 1 << 255, 0):
        r16 = A16(); L.t_sqr_wide(enc(a), r16); assert dec(r16) == a * a
    for a in fr.BARRETT_A:
        for b in fr.BARRETT_B:
            assert call2(L.t_mul, a, b) == a * b % M


@pytest.mark.parametrize("ptx", [False, True])
def test_montgomery_reduction_of_accumulated_terms(ptx):
    """OP_DOT: P = sum of terms (value x pre-scaled constant, +-value << 256, constant), then ONE reduction
    P * 2^-256 mod M with the number of conditional subtractions the plan compiler derives from the term mix."""
    L = util.field_host_lib(ptx)
    rnd = random.Random(2)
    R = 1 << 256
    edge = [0, 1, M - 1, M - 2, (1 << 253), (1 << 224) - 1, 0xFFFFFFFF, (1 << 32), (M >> 1)]
    pick = lambda: rnd.choice(edge) if rnd.random() < 0.4 else rnd.randrange(M)
    # raw 512-bit values: anything whose reduced value stays below 2^ncs * M and 2^256
    for t in range(3000):
        ncs = rnd.choice([1, 2, 3])
        lim = fr.mont_reduce_limit(ncs)         # (P + mM) / R < P / R + M must stay below the bound
        P = rnd.randrange(lim * R) if rnd.random() < 0.7 else rnd.choice([0, 1, R - 1, R, lim * R - 1, (lim - 1) * R, (1 << 32) - 1,
                                                                              ((1 << 256) - 1) << 32, (lim * R - 1) & ~((1 << 224) - 1)])
        P %= lim * R
        r = A8(); L.t_mont_reduce(A16(*[(P >> (32 * i)) & 0xFFFFFFFF for i in range(16)]), ncs, r)
        assert dec(r) == fr.mont_reduce(P), (t, ncs, hex(P))
    # term by term, like the kernel
    for t in range(1500):
        n_mac, n_hi = rnd.randrange(0, 9), rnd.randrange(0, 4)
        if n_mac + n_hi == 0:
            continue
        ncs = fr.dot_ncs(n_mac, n_hi)
        if ncs is None:
            continue
        kinds, xs, cs, want = [], [], [], 0
        def term(k, x, c):
            kinds.append(k); xs.extend(enc(x)); cs.extend(enc(c))
        for _ in range(n_mac):
            x, c = pick(), pick()
            term(0, x, fr.to_mont(c)); want += x * c
        for _ in range(n_hi):
            x = pick()
            if rnd.random() < 0.5:
                term(1, x, 0); want += x
            else:
                term(2, x, 0); want -= x
        if rnd.random() < 0.5:
            c = pick(); term(3, 0, fr.to_mont(c)); want += c
        rnd.shuffle(order := list(range(len(kinds))))
        kinds2 = [kinds[i] for i in order]
        xs2 = [v for i in order for v in xs[8 * i:8 * i + 8]]
        cs2 = [v for i in order for v in cs[8 * i:8 * i + 8]]
        n = len(kinds2)
        r = A8(); L.t_dot_eval((ctypes.c_uint32 * n)(*kinds2), (ctypes.c_uint32 * (8 * n))(*xs2), (ctypes.c_uint32 * (8 * n))(*cs2), n, ncs, r)
        assert dec(r) == want % M, (t, n_mac, n_hi)


@pytest.mark.parametrize("ptx", [False, True])
def test_safegcd_inverse(ptx):
    """fe_inv (Bernstein-Yang divsteps): what Div and the batched OP_INV run on the device"""
    L = util.field_host_lib(ptx)
    for (a,) in fr.operand_tuples("c", 1500, seed=7):
        assert call1(L.t_inv_safegcd, a) == fr.inv(a), hex(a)


@pytest.mark.parametrize("ptx", [False, True])
def test_mul_hi_trunc_is_the_exact_partial_sum(ptx):
    """u256_mul_hi_trunc: the whole 16-limb output is the sum of the partial products a_j b_i with i + j >= 6"""
    L = util.field_host_lib(ptx)
    rnd = random.Random(8)
    pairs = fr.edge_tuples("ww") + [(fr.limb_pattern(rnd, "w"), fr.limb_pattern(rnd, "w")) for _ in range(2000)]
    pairs += [(rnd.getrandbits(256), rnd.getrandbits(256)) for _ in range(2000)]
    for a, b in pairs:
        r16 = A16(); L.t_mul_hi_trunc(enc(a), enc(b), r16)
        assert dec(r16) == fr.mul_hi_trunc(a, b), (hex(a), hex(b))


def test_device_harness_without_a_device_returns_an_error():
    """tests/csrc/field_device_api.cu builds for sm_100a, rejects a bad primitive id, and on a machine without a usable
    device returns the CUDA error instead of crashing, leaving the output as it was"""
    L = util.field_device_lib()
    w = (ctypes.c_int * 4)()
    assert L.fd_shape(0, w) == 0 and list(w) == [8, 8, 0, 8]
    assert L.fd_shape(L.fd_n_prims(), w) == -1
    a8 = np.array([np.frombuffer(enc(v), np.uint32) for v in (M - 1, 2)], np.uint32)
    p = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32))
    out, st, op = np.full((2, 8), 7, np.uint32), np.full(2, 7, np.uint32), np.zeros(2, np.uint32)
    assert L.fd_launch(L.fd_n_prims(), 0, 1, 2, p(a8), p(a8), None, p(op), p(out), p(st)) == 1     # cudaErrorInvalidValue
    rc = L.fd_launch(0, 0, 1, 2, p(a8), p(a8), None, p(op), p(out), p(st))
    if rc == 0:
        pytest.skip("a GPU is present")
    assert rc > 0 and (out == 7).all() and (st == 7).all()
