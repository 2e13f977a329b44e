"""Groth16 quotient evaluations of witness rows (gw_r1cs_quotient_*) and the batched BN254 NTT (gw_fr_ntt_batch_device):
without a GPU the root constants, the host-built tables, the reference pinned against itself, the butterflies with
worst-case operands in both host arithmetic builds, the argument checks and the ABI declarations; on the GPU the NTT
against the reference (tests/r1cs_quotient_ref.py) for every k up to 12 and by round trips, closed forms and Horner
evaluations up to 2^24, and the quotient against the reference, between its entry points and at the benchmark size."""
import ctypes
import importlib
import os
import random
import re
import subprocess

import numpy as np
import pytest

from tests import r1cs_quotient_ref as qref
from tests import r1cs_ref as ref
from tests import util
from tests.test_r1cs import _inputs, _pair
from tests.test_r1cs_abc import _distinct, _public, _tiling, trivial
from tools import r1cs_gen

M = util.M
OK = 0xFFFFFFFF
INV, COSET = 1, 2
R = (1 << 256) % M


@pytest.fixture(scope="module")
def cwc():
    subprocess.check_call(["python", os.path.join(util.ROOT, "circom-witnesscalc_b200", "build.py")])
    return importlib.import_module("circom-witnesscalc_b200")


# ---- without a GPU ------------------------------------------------------------------------------------------------
def test_root_constants():
    t = (M - 1) >> 28
    assert (M - 1) == t << 28 and t % 2 == 1
    legendre = lambda a: pow(a, (M - 1) // 2, M)
    assert [legendre(a) for a in (2, 3, 4, 5)] == [1, 1, 1, M - 1]
    assert qref.W28 == pow(5, t, M) == 19103219067921713944291392827692070036145651957329286315305642004821462161904
    assert pow(qref.W28, 1 << 28, M) == 1 and pow(qref.W28, 1 << 27, M) == M - 1
    for k in (0, 1, 12, 24):
        assert pow(qref.coset_gen(k), 1 << k, M) == M - 1 and qref.coset_gen(k) == pow(qref.root(k + 1), 1, M)


@pytest.mark.parametrize("emulate_ptx", [False, True])
def test_host_tables_equal_the_python_ones(emulate_ptx):
    lib = qref.ntt_host_lib(emulate_ptx)
    nt = lib.ntt_host_n_tables()
    names = ["TW_LO", "TW_HI", "ITW_LO", "ITW_HI", "CG_LO", "CG_HI", "ICG_LO", "ICG_HI", "QG_LO", "QGR_LO", "ROOT", "IROOT",
             "NINV"]
    assert nt == len(names)
    for k in (0, 1, 2, 7, 12, 13, 20, 24):
        buf = ctypes.create_string_buffer(32 * 4096 * nt)
        lib.ntt_host_tables(k, buf)
        got = util.unpack_u256(buf.raw)
        n, w, wi, g = 1 << k, qref.root(k), qref.root(k, True), qref.coset_gen(k)
        gi, ninv, w12 = pow(g, M - 2, M), pow(1 << k, M - 2, M), qref.root(12)
        exp = {"TW_LO": lambda t: pow(w, t, M), "TW_HI": lambda t: pow(w, 4096 * t, M),
               "ITW_LO": lambda t: pow(wi, t, M), "ITW_HI": lambda t: pow(wi, 4096 * t, M),
               "CG_LO": lambda t: pow(g, t, M), "CG_HI": lambda t: pow(g, 4096 * t, M),
               "ICG_LO": lambda t: ninv * pow(gi, t, M), "ICG_HI": lambda t: pow(gi, 4096 * t, M),
               "QG_LO": lambda t: ninv * pow(g, t, M), "QGR_LO": lambda t: ninv * pow(g, t, M) * R,
               "ROOT": lambda t: pow(w12, t, M) if t < 2048 else None,
               "IROOT": lambda t: pow(w12, (M - 2) * t, M) if t < 2048 else None,
               "NINV": lambda t: ninv if t == 0 else None}
        for j, name in enumerate(names):
            for t in (0, 1, 2, 3, 100, 2047, 2048, 4095):
                e = exp[name](t)
                assert got[j * 4096 + t] == (0 if e is None else e * R % M), (k, name, t)
        assert n == 1 << k


@pytest.mark.parametrize("k", range(0, 7))
def test_fast_reference_equals_the_defining_sums(k):
    rnd = random.Random(k)
    x = [rnd.randrange(1 << 256) for _ in range(1 << k)] if k else [M + 5]
    for flags in range(4):
        assert qref.ntt(x, flags & INV, flags & COSET) == qref.ntt_naive(x, flags & INV, flags & COSET), (k, flags)
    assert qref.ntt(qref.ntt(x, coset=True), inverse=True, coset=True) == [v % M for v in x]


def _trivial_row(m, n_wires=8, n_pub_out=0, n_pub_in=0, seed=0):
    """the system of test_r1cs_abc.trivial (w_0 w_1 = w_1 for each constraint) and a satisfying row (w_0 = 1)"""
    r = trivial(m, n_wires, n_pub_out, n_pub_in)
    rnd = random.Random(seed)
    return r, [1] + [rnd.randrange(M) for _ in range(n_wires - 1)]


@pytest.mark.parametrize("m,n_pub_out,n_pub_in", [(0, 0, 0), (1, 0, 0), (3, 0, 0), (4, 0, 0), (5, 1, 1), (6, 1, 1),
                                                  (13, 1, 2), (14, 0, 2)])
def test_formula_quotient_equals_the_polynomial_division(m, n_pub_out, n_pub_in):
    r, w = _trivial_row(m, 8, n_pub_out, n_pub_in, seed=m)
    h = qref.quotient_ref(r, w)
    assert h == qref.quotient_by_division(r, w)
    assert qref.ntt(h, inverse=True, coset=True)[-1] == 0            # deg H <= n - 2


def test_formula_quotient_equals_the_polynomial_division_on_generated_pairs():
    for seed, m, n_pub in ((5, 20, 0), (6, 28, 2), (7, 30, 1)):
        g, r = r1cs_gen.random_pair(random.Random(seed), n_constraints=m)
        r = dict(r, n_pub_out=min(1, n_pub), n_pub_in=n_pub - min(1, n_pub))
        nodes, wit, _ = util.po.deserialize_graph(g)
        rnd = random.Random(seed)
        w = util.po.evaluate(nodes, [1] + [util.random_value(rnd) for _ in range(6)], wit)
        assert ref.check_r1cs(r, w) is None
        assert qref.quotient_ref(r, w) == qref.quotient_by_division(r, w), seed


@pytest.mark.parametrize("emulate_ptx", [False, True])
def test_butterflies_with_worst_case_operands(emulate_ptx):
    lib = qref.ntt_host_lib(emulate_ptx)
    vals = [0, 1, 2, M - 1, M - 2, (M - 1) // 2, (M + 1) // 2, R, M - R, 0xFFFFFFFF, 1 << 224]
    rnd = random.Random(9)
    vals += [rnd.randrange(M) for _ in range(6)]
    ws = [M - 1, 0, 1, R, (M - 1) * R % M, rnd.randrange(M)]           # pre-scaled twiddles, M - 1 the largest
    for a in vals:
        for b in vals:
            for w in ws:
                wv = w * pow(R, M - 2, M) % M                           # the twiddle value w stands for
                for which, exp in ((0, ((a + b) % M, (a - b) * wv % M)), (1, ((a + b * wv) % M, (a - b * wv) % M)),
                                   (2, (a * wv % M, b))):
                    A, B = ctypes.create_string_buffer(a.to_bytes(32, "little"), 32), \
                        ctypes.create_string_buffer(b.to_bytes(32, "little"), 32)
                    lib.ntt_host_bfly(which, A, B, w.to_bytes(32, "little"))
                    assert (int.from_bytes(A.raw, "little"), int.from_bytes(B.raw, "little")) == exp, (which, a, b, w)


def test_arguments_are_rejected_before_a_device_is_touched(cwc):
    r = trivial(5, n_pub_out=1)
    rc = cwc.R1cs(ref.serialize_r1cs(r))
    W, n = r["n_wires"], 8
    rows = np.zeros((2, W, 32), np.uint8)
    out = np.zeros(2 * 3 * n * 32 + 64, np.uint8)
    ff = np.zeros(2, np.uint32)
    L, st = cwc._L, cwc.gw_status_t()

    def host(witness=rows.ctypes.data, row_pitch=0, h=out.ctypes.data, h_pitch=0, n_sets=2):
        return L.gw_r1cs_quotient_batch(rc._h, witness, n_sets, row_pitch, h, h_pitch, ff.ctypes.data, 1, ctypes.byref(st))

    def device(witness=rows.ctypes.data, row_pitch=0, h=out.ctypes.data, h_pitch=0, n_sets=2):
        return L.gw_r1cs_quotient_batch_device(rc._h, 0, witness, n_sets, row_pitch, h, h_pitch, None, None,
                                               ctypes.byref(st))

    def ntt(data=out.ctypes.data, n_vectors=2, log_n=3, pitch=0, flags=0):
        return L.gw_fr_ntt_batch_device(0, data, n_vectors, log_n, pitch, flags, None, ctypes.byref(st))

    def rejected(call, match, **kw):
        with pytest.raises(cwc.WitnessCalcError, match=match):
            cwc._check(call(**kw), st)

    for call in (host, device):
        rejected(call, "row_pitch is smaller", row_pitch=W * 32 - 16)
        rejected(call, "null argument", witness=None)
        rejected(call, "null argument", h=None)
        assert call(witness=None, h=None, n_sets=0) == 0
        cwc._check(0, st)
    rejected(host, "h_pitch is smaller", h_pitch=n * 32 - 16)
    rejected(device, "work_pitch is smaller", h_pitch=3 * n * 32 - 16)
    rejected(device, "16-byte aligned", row_pitch=W * 32 + 8)
    rejected(device, "16-byte aligned", h_pitch=3 * n * 32 + 8)
    rejected(device, "16-byte aligned", witness=rows.ctypes.data + 8)
    rejected(device, "16-byte aligned", h=out.ctypes.data + 8)
    assert L.gw_r1cs_quotient_batch(None, None, 0, 0, None, 0, None, 1, ctypes.byref(st)) == 1
    cwc._check(0, st)
    assert L.gw_r1cs_quotient_batch_device(None, 0, None, 0, 0, None, 0, None, None, ctypes.byref(st)) == 1
    cwc._check(0, st)
    # a domain above 2^24: m + n_pub + 1 = 2^24 + 1
    big = cwc.R1cs(ref.serialize_r1cs({"n_wires": 2, "n_pub_out": 1, "n_pub_in": 0, "constraints": [([(0, 1)], [], [])] * (1 << 24)}))
    assert big.abc_len(groth16=True) == 1 << 25
    with pytest.raises(cwc.WitnessCalcError, match="larger than 2\\^24"):
        cwc._check(L.gw_r1cs_quotient_batch(big._h, rows.ctypes.data, 1, 64, out.ctypes.data, 0, None, 1, ctypes.byref(st)), st)
    with pytest.raises(cwc.WitnessCalcError, match="larger than 2\\^24"):
        cwc._check(L.gw_r1cs_quotient_batch_device(big._h, 0, rows.ctypes.data, 1, 64, out.ctypes.data, 0, None, None,
                                                   ctypes.byref(st)), st)
    # the NTT
    rejected(ntt, "unknown flag bits 4", flags=4)
    rejected(ntt, "unknown flag bits 8", flags=INV | 8)
    rejected(ntt, "log_n = 25 is larger than 24", log_n=25)
    rejected(ntt, "log_n = 40 is larger than 24", log_n=40)
    rejected(ntt, "pitch is smaller", pitch=8 * 32 - 16)
    rejected(ntt, "multiple of 16", pitch=8 * 32 + 8)
    rejected(ntt, "16-byte aligned", data=out.ctypes.data + 8)
    rejected(ntt, "null argument", data=None)
    assert ntt(data=None, n_vectors=0) == 0
    cwc._check(0, st)
    rejected(ntt, "larger than 24", data=None, n_vectors=0, log_n=25)


def test_quotient_and_ntt_without_a_device_fail_loudly(cwc):
    if cwc.device_count() > 0:
        pytest.skip("a GPU is present")
    rc = cwc.R1cs(ref.serialize_r1cs(trivial(3)))
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        rc.quotient_batch(np.zeros((1, 8, 32), np.uint8))
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        rc.quotient_batch(np.zeros((1, 8, 32), np.uint8), want_verdict=True)
    buf = np.zeros(4096, np.uint8)
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        rc.quotient_batch_device(0, buf.ctypes.data, 1, buf.ctypes.data + 512)
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        cwc.ntt_batch_device(0, buf.ctypes.data, 1, 3)


def test_abi_declarations_match_in_the_header_the_python_binding_and_the_rust_shim(cwc):
    hdr = open(os.path.join(util.ROOT, "include", "graph_witness.h")).read()
    rs = open(os.path.join(util.ROOT, "rust-shim", "src", "ffi.rs")).read()
    assert re.search(r"#define GW_NTT_INVERSE 1u\b", hdr) and re.search(r"#define GW_NTT_COSET 2u\b", hdr)
    assert "pub const GW_NTT_INVERSE: u32 = 1;" in rs and "pub const GW_NTT_COSET: u32 = 2;" in rs
    assert cwc.NTT_INVERSE == 1 and cwc.NTT_COSET == 2
    rs_type = {"uint64_t": "u64", "uint32_t": "u32", "size_t": "usize", "int": "c_int"}
    py_type = {"uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32, "size_t": ctypes.c_size_t, "int": ctypes.c_int}
    for name in ("gw_fr_ntt_batch_device", "gw_r1cs_quotient_batch", "gw_r1cs_quotient_batch_device"):
        assert name in cwc.EXPORTS
        c_ret, c_args = re.search(r"\n(\w+)\s+" + name + r"\(([^)]*)\);", hdr).groups()
        c_sig = []
        for a in c_args.split(","):
            t = re.fullmatch(r"(?:const\s+)?(\w+)\s*(\*?)\s*\w+", a.strip())
            c_sig.append("ptr" if t.group(2) else t.group(1))
        r_args, r_ret = re.search(r"pub fn " + name + r"\(([^)]*)\)(?: -> (\w+))?;", rs).groups()
        assert ["ptr" if "*" in a else a.split(":")[1].strip() for a in r_args.split(",")] == \
            ["ptr" if t == "ptr" else rs_type[t] for t in c_sig], name
        assert r_ret == rs_type[c_ret], name
        f = getattr(cwc._L, name)
        assert len(f.argtypes) == len(c_sig), name
        for t, c in zip(f.argtypes, c_sig):
            assert (t is not py_type.get(c)) if c == "ptr" else (t is py_type[c]), (name, t, c)
        assert (f.restype or ctypes.c_int) is py_type[c_ret], name


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.array(a)).cuda()


def _vectors(k, D, seed):
    """D distinct vectors of 2^k values: random, with M, M + 5, 2^256 - 1 and M - 1 placed in them"""
    rnd = random.Random(seed)
    n = 1 << k
    vs = [[rnd.randrange(1 << 256) if d % 2 else rnd.randrange(M) for _ in range(n)] for d in range(D)]
    special = [M, M + 5, (1 << 256) - 1, M - 1, 0]
    for d in range(D):
        for s, v in enumerate(special):
            vs[d][(s * 7 + d) % n] = v
    return vs


@pytest.mark.gpu
@pytest.mark.parametrize("k", range(0, 13))
def test_gpu_ntt_small_k_every_entry(cwc, k):
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n, D = 1 << k, 3
    vs = _vectors(k, D, k)
    src = np.frombuffer(util.pack_u256([v for x in vs for v in x]), np.uint8).reshape(D, n * 32)
    per_cta = max(1, 2048 >> k)
    wave = 2 * sms * per_cta + 5                      # more vectors than one wave of CTAs
    for flags in range(4):
        exp = np.frombuffer(util.pack_u256([v for x in vs for v in qref.ntt(x, flags & INV, flags & COSET)]),
                            np.uint8).reshape(D, n * 32)
        for B in (1, 33, wave):
            idx = np.arange(B) % D
            d = _dev(src[idx])
            cwc.ntt_batch_device(0, d.data_ptr(), B, k, flags=flags)
            torch.cuda.synchronize()
            assert torch.equal(d, _dev(exp[idx])), (k, flags, B)


def _horner(x, pt):
    acc = 0
    for v in reversed(x):
        acc = (acc * pt + v) % M
    return acc


@pytest.mark.gpu
@pytest.mark.parametrize("k", [13, 16, 17, 20, 24])
def test_gpu_ntt_large_k(cwc, k):
    import torch
    n = 1 << k
    rng = np.random.default_rng(k)
    x = util.random_field_batch(rng, (2, n)).view(np.uint8).reshape(2, n * 32)
    x[0, :32] = np.frombuffer(((1 << 256) - 1).to_bytes(32, "little"), np.uint8)      # a value >= M
    canon = _dev(x)
    first = util.unpack_u256(x[0, :32].tobytes())[0]
    canon[0, :32] = _dev(np.frombuffer((first % M).to_bytes(32, "little"), np.uint8))
    # round trips, plain and coset
    for coset in (0, COSET):
        d = _dev(x)
        cwc.ntt_batch_device(0, d.data_ptr(), 2, k, flags=coset)
        y = d.clone()
        cwc.ntt_batch_device(0, d.data_ptr(), 2, k, flags=coset | INV)
        torch.cuda.synchronize()
        assert torch.equal(d, canon), (k, coset)
        if k <= 20:                                   # Horner spot checks of the forward outputs
            xs = util.unpack_u256(x[1].tobytes())
            w, g = qref.root(k), qref.coset_gen(k) if coset else 1
            for j in (0, 1, n // 2 + 3, n - 1):
                got = util.unpack_u256(y[1, 32 * j:32 * j + 32].cpu().numpy().tobytes())[0]
                assert got == _horner(xs, g * pow(w, j, M) % M), (k, coset, j)
    # unit vectors against their closed form: forward e_s -> (g^s) w^(s j); inverse e_s -> n^-1 (g^-j) w^(-s j)
    s_list = [0, 1, n // 2 + 1]
    units = np.zeros((len(s_list), n * 32), np.uint8)
    for r, s in enumerate(s_list):
        units[r, 32 * s] = 1
    js = [0, 1, 2, n // 3, n - 1]
    for flags in range(4):
        d = _dev(units)
        cwc.ntt_batch_device(0, d.data_ptr(), len(s_list), k, flags=flags)
        torch.cuda.synchronize()
        w, g, ninv = qref.root(k, flags & INV), qref.coset_gen(k), pow(n, M - 2, M)
        for r, s in enumerate(s_list):
            for j in js:
                got = util.unpack_u256(d[r, 32 * j:32 * j + 32].cpu().numpy().tobytes())[0]
                if flags & INV:
                    exp = ninv * pow(w, s * j, M) * (pow(g, (M - 2) * j, M) if flags & COSET else 1) % M
                else:
                    exp = pow(w, s * j, M) * (pow(g, s, M) if flags & COSET else 1) % M
                assert got == exp, (k, flags, s, j)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 14])
def test_gpu_ntt_pitches_canaries_and_a_stream(cwc, k):
    import torch
    n, B = 1 << k, 5
    vs = _vectors(k, B, 100 + k)
    pitch = n * 32 + 48
    host = np.full((B, pitch), 0xA5, np.uint8)
    host[:, :n * 32] = np.frombuffer(util.pack_u256([v for x in vs for v in x]), np.uint8).reshape(B, n * 32)
    d = _dev(host)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    cwc.ntt_batch_device(0, d.data_ptr(), B, k, pitch=pitch, flags=COSET, stream=s.cuda_stream)
    s.synchronize()
    got = d.cpu().numpy()
    assert (got[:, n * 32:] == 0xA5).all()
    for b in range(B):
        assert util.unpack_u256(got[b, :n * 32].tobytes()) == qref.ntt(vs[b], coset=True), b


def _h_expected(r, rows):
    return np.stack([np.frombuffer(util.pack_u256(qref.quotient_ref(r, util.unpack_u256(x.tobytes()))), np.uint8)
                     .reshape(-1, 32) for x in rows])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_quotient_matches_the_reference(cwc, shape):
    import torch
    g, r, n_in = _pair(shape)
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    rows, verdict, _, _ = _distinct(graph, r, n_in, 131)
    exp = _h_expected(r, rows)
    n = rc.abc_len(groth16=True)
    assert exp.shape[1] == n
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    big = 2 * sms + 40                                # the small path runs one row per CTA
    picked = {0, 5, 31, 32, big - 1} | set(random.Random(132).sample(range(big), 20))
    for B in (1, 33, big):
        idx = _tiling(B, len(rows), picked)
        got, ff = rc.quotient_batch(rows[idx], want_verdict=True)
        assert got.shape == (B, n, 32)
        assert (got == exp[idx]).all(), (shape, B)
        assert (ff == verdict[idx]).all()
    # valid rows: deg H <= n - 2
    h = rc.quotient_batch(rows[:4])
    for b in range(4):
        assert qref.ntt(util.unpack_u256(h[b].tobytes()), inverse=True, coset=True)[-1] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("m,n_pub_out,n_pub_in", [(0, 0, 0), (2, 0, 1), (3, 0, 1), (60, 1, 2), (61, 1, 2), (4092, 1, 2),
                                                  (4093, 1, 2), (8188, 1, 2), (8189, 1, 2)])
def test_gpu_quotient_domain_sizes(cwc, m, n_pub_out, n_pub_in):
    """m + n_pub + 1 = 2^k and 2^k + 1; n = 1 (no constraint, no public signal); both kernel paths"""
    r = trivial(m, 8, n_pub_out, n_pub_in)
    rc = cwc.R1cs(ref.serialize_r1cs(r))
    rnd = random.Random(m)
    ws = [[1] + [rnd.randrange(M) for _ in range(7)], [rnd.randrange(M) for _ in range(8)]]   # valid, violating
    rows = np.stack([np.frombuffer(util.pack_u256(w), np.uint8).reshape(8, 32) for w in ws])
    got, ff = rc.quotient_batch(rows, want_verdict=True)
    exp = _h_expected(r, rows)
    assert got.shape == exp.shape and (got == exp).all()
    assert ff[0] == OK and (ff[1] != OK or m == 0)


@pytest.mark.gpu
def test_gpu_quotient_large_domain_against_the_reference(cwc):
    """a Poseidon-shaped pair with n = 8192 (the two-pass kernels) against the reference, valid and violating rows"""
    g, r = r1cs_gen.poseidon_pair(random.Random(11), n_hashes=30)
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    n = rc.abc_len(groth16=True)
    assert n > 4096
    rows, verdict, _, _ = _distinct(graph, r, 4, 141)
    sel = [0, 4, 5, 9]
    exp = _h_expected(r, rows[sel])
    idx = np.arange(37) % len(sel)
    got, ff = rc.quotient_batch(rows[sel][idx], want_verdict=True)
    assert (got == exp[idx]).all() and (ff == verdict[sel][idx]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_host_and_device_entry_points_agree(cwc, shape):
    import torch
    g, r, n_in = _pair(shape)
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    rows, verdict, _, _ = _distinct(graph, r, n_in, 151)
    B, W = 300, graph.n_witness
    idx = _tiling(B, len(rows), set(random.Random(152).sample(range(B), 40)))
    bad = rows[idx]
    n = rc.abc_len(groth16=True)
    host, hff = rc.quotient_batch(bad, want_verdict=True)
    assert (hff == verdict[idx]).all()
    # host rows with a pitch, h with a padded pitch: the padding keeps its canary
    pitch, hp = W * 32 + 40, n * 32 + 24
    src = np.zeros((B, pitch), np.uint8)
    src[:, :W * 32] = bad.reshape(B, -1)
    out = np.full((B, hp), 0xA5, np.uint8)
    ff = np.zeros(B, np.uint32)
    st = cwc.gw_status_t()
    cwc._check(cwc._L.gw_r1cs_quotient_batch(rc._h, src.ctypes.data, B, pitch, out.ctypes.data, hp, ff.ctypes.data, 1,
                                             ctypes.byref(st)), st)
    assert (out[:, :n * 32] == host.reshape(B, -1)).all() and (out[:, n * 32:] == 0xA5).all() and (ff == hff).all()
    # device rows with a pitch, padded work rows with a canary, on a non-default stream
    dpitch, wp = W * 32 + 48, 3 * n * 32 + 32
    dev = torch.zeros((B, dpitch), dtype=torch.uint8, device="cuda:0")
    dev[:, :W * 32] = _dev(bad.reshape(B, -1))
    d_work = torch.full((B, wp), 0xA5, dtype=torch.uint8, device="cuda:0")
    d_ff = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    rc.quotient_batch_device(0, dev.data_ptr(), B, d_work.data_ptr(), row_pitch=dpitch, work_pitch=wp,
                             d_first_failed_ptr=d_ff.data_ptr(), stream=s.cuda_stream)
    s.synchronize()
    got = d_work.cpu().numpy()
    assert (got[:, :n * 32] == host.reshape(B, -1)).all() and (got[:, 3 * n * 32:] == 0xA5).all()
    assert (d_ff.cpu().numpy().view(np.uint32) == hff).all()
    assert (hff == rc.check_batch(bad)).all()
    # .wtns images in place
    files = np.zeros((B, graph.wtns_file_size() + 20), np.uint8)
    fp = files.shape[1]
    files[:, 76:76 + W * 32] = bad.reshape(B, -1)
    assert (rc.quotient_batch(files.reshape(-1)[76:], row_pitch=fp, n_sets=B) == host).all()
    if cwc.device_count() >= 2:
        two, ff2 = rc.quotient_batch(bad, n_gpus=2, want_verdict=True)
        assert (two == host).all() and (ff2 == hff).all()


@pytest.mark.gpu
def test_gpu_evaluation_and_quotient_on_one_stream(cwc):
    import torch
    g, r, n_in = _pair("poseidon")
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    B, W = 700, graph.n_witness
    inputs = _inputs(np.random.default_rng(161), B, n_in)
    n = rc.abc_len(groth16=True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_in = torch.from_numpy(inputs.reshape(B, -1)).cuda()
        d_w = torch.empty((B, W * 32), dtype=torch.uint8, device="cuda:0")
        d_work = torch.empty((B, 3 * n * 32), dtype=torch.uint8, device="cuda:0")
        d_ff = torch.empty(B, dtype=torch.int32, device="cuda:0")
    graph.calc_witness_batch_device(0, d_in.data_ptr(), B, d_w.data_ptr(), stream=s.cuda_stream)
    rc.quotient_batch_device(0, d_w.data_ptr(), B, d_work.data_ptr(), d_first_failed_ptr=d_ff.data_ptr(),
                             stream=s.cuda_stream)
    s.synchronize()
    host, hff = rc.quotient_batch(graph.calc_witness_batch(inputs), want_verdict=True)
    assert (d_work[:, :n * 32].cpu().numpy() == host.reshape(B, -1)).all()
    assert (d_ff.cpu().numpy().view(np.uint32) == hff).all() and (hff == OK).all()


@pytest.mark.gpu
def test_gpu_deg_h_at_the_benchmark_size(cwc):
    """the n = 65 536 pair of tools/r1cs_bench.py: on valid rows the coset-inverse NTT of h has entry n - 1 equal to 0
    (on the GPU); a violating row matches the Python reference"""
    import torch
    g, r = r1cs_gen.poseidon_pair(random.Random(1), n_hashes=196)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    n = rc.abc_len(groth16=True)
    assert n == 65536
    B, W = 6, graph.n_witness
    rows = graph.calc_witness_batch(_inputs(np.random.default_rng(171), B, 4))
    bad = rows[0].copy()
    bad[1000] = np.frombuffer((M + 3).to_bytes(32, "little"), np.uint8)
    bad[5000] = np.frombuffer(random.Random(172).randrange(M).to_bytes(32, "little"), np.uint8)
    batch = np.concatenate([rows, bad[None]])
    h, ff = rc.quotient_batch(batch, want_verdict=True)
    assert (ff[:B] == OK).all() and ff[B] != OK
    d = _dev(h[:B].reshape(B, -1))
    cwc.ntt_batch_device(0, d.data_ptr(), B, 16, flags=INV | COSET)
    torch.cuda.synchronize()
    top = d[:, (n - 1) * 32:].cpu().numpy()
    assert not top.any()
    assert d[:, :(n - 2) * 32].any(dim=1).all()
    exp = qref.quotient_ref(r, util.unpack_u256(batch[B].tobytes()))
    assert util.unpack_u256(h[B].tobytes()) == exp
