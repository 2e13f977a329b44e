"""A, B and C of witness rows (gw_r1cs_abc_*): the vector lengths of both layouts, the per-constraint step on the host
with worst-case operands and values >= M, the argument checks and the ABI declarations without a GPU; on the GPU every
value of every row against the Python reference (tests/r1cs_abc_ref.py), the verdicts against the check, the
host and device entry points against each other, and `wtns-check --all`."""
import ctypes
import importlib
import os
import random
import re
import subprocess

import numpy as np
import pytest

from tests import r1cs_abc_ref as abc_ref
from tests import r1cs_ref as ref
from tests import util
from tests.test_r1cs import _inputs, _pair

M = util.M
OK = 0xFFFFFFFF
GROTH16 = 1


@pytest.fixture(scope="module")
def cwc():
    subprocess.check_call(["python", os.path.join(util.ROOT, "circom-witnesscalc_b200", "build.py")])
    return importlib.import_module("circom-witnesscalc_b200")


def trivial(m, n_wires=8, n_pub_out=0, n_pub_in=0):
    return {"n_wires": n_wires, "n_pub_out": n_pub_out, "n_pub_in": n_pub_in, "n_prv_in": 0,
            "constraints": [([(0, 1)], [(1, 1)], [(1, 1)])] * m}


# ---- without a GPU ------------------------------------------------------------------------------------------------
def test_abc_len_in_both_layouts(cwc):
    for m, n_pub_out, n_pub_in, groth in [(62, 0, 0, 64), (63, 0, 0, 64), (64, 0, 0, 128),     # m + n_pub + 1 = 63, 64, 65
                                          (60, 1, 1, 64), (61, 1, 1, 64), (62, 1, 1, 128),
                                          (0, 0, 0, 1), (0, 2, 3, 8), (1, 0, 0, 2), (5, 3, 4, 16)]:
        r = trivial(m, n_pub_out=n_pub_out, n_pub_in=n_pub_in)
        rc = cwc.R1cs(ref.serialize_r1cs(r))
        assert rc.abc_len() == m == abc_ref.abc_len(r)
        assert rc.abc_len(groth16=True) == groth == abc_ref.abc_len(r, groth16=True), (m, n_pub_out, n_pub_in)
    # the public signals (and wire 0) must be wires
    rc = cwc.R1cs(ref.serialize_r1cs(trivial(3, n_wires=4, n_pub_out=2, n_pub_in=2)))
    assert rc.abc_len() == 3 and rc.abc_len(groth16=True) == 0
    with pytest.raises(cwc.WitnessCalcError, match="4 public signals need more than the 4 wires"):
        rc.abc_batch(np.zeros((1, 4, 32), np.uint8), groth16=True)
    assert cwc._L.gw_r1cs_abc_len(rc._h, 2) == 0 and cwc._L.gw_r1cs_abc_len(None, 0) == 0


def _worst_case():
    """the operands of tests/test_r1cs.py::test_chunk_bound_with_worst_case_operands: wires 1 .. 119 hold M - 1,
    wires 120 .. 238 hold 0; linear combinations one term below, at and above the chunk bound and far above it"""
    half = 119
    wit = [1] + [M - 1] * half + [0] * half
    top = lambda i: 1 + (i % half)
    zero = lambda i: 1 + half + (i % half)
    c_worst = (M - 1) * pow(1 << 256, M - 2, M) % M
    cons = []
    for n in (3, 4, 5, 8, 9, 21, 22, 23, 44, 45, 100):
        for c, wire in ((c_worst, top), (M - 2, top), (M - 3, top), (1, top), (M - 1, zero), (M - 1, top)):
            lc = [(wire(i), c) for i in range(n)]
            cons.append((lc, lc, lc))
        mixed = [((zero if i % 3 == 2 else top)(i), (c_worst, 1, M - 1)[i % 3]) for i in range(n)]
        cons.append((mixed, [(0, M - 1)], mixed))
    return {"n_wires": 1 + 2 * half, "constraints": cons}, wit


@pytest.mark.parametrize("emulate_ptx", [False, True])
def test_per_constraint_abc_with_worst_case_operands_and_values_above_m(emulate_ptx):
    lib = abc_ref.abc_host_lib(emulate_ptx)
    r, wit = _worst_case()
    data = ref.serialize_r1cs(r)
    h = lib.r1cs_abc_host_load(data, len(data))
    assert h
    abc = ctypes.create_string_buffer(96)
    # the worst case itself, then wires 1, 2, 3 at M, M + 5 and 2^256 - 1 (top wires) and 120 at M (a zero wire)
    above = {1: M, 2: M + 5, 3: (1 << 256) - 1, 120: M}
    for w in (wit, [above.get(i, v) for i, v in enumerate(wit)]):
        row = util.pack_u256(w)
        exp = abc_ref.abc_ref(r, w)
        for k, con in enumerate(r["constraints"]):
            reduced = lib.r1cs_abc_host_eval(h, k, row, abc)
            assert util.unpack_u256(abc.raw) == [exp[0][k], exp[1][k], exp[2][k]], (k, len(con[0]))
            assert reduced == any(w[i] >= M for lc in con for i, c in lc), k
    lib.r1cs_abc_host_free(h)


def test_arguments_are_rejected_before_a_device_is_touched(cwc):
    r = trivial(5, n_pub_out=1)
    rc = cwc.R1cs(ref.serialize_r1cs(r))
    W, n = r["n_wires"], 5
    rows = np.zeros((2, W, 32), np.uint8)
    out = np.zeros(2 * 3 * 8 * 32 + 64, np.uint8)
    ff = np.zeros(2, np.uint32)
    L, st = cwc._L, cwc.gw_status_t()

    def host(witness=rows.ctypes.data, row_pitch=0, abc=out.ctypes.data, abc_pitch=0, options=0, n_sets=2):
        return L.gw_r1cs_abc_batch(rc._h, witness, n_sets, row_pitch, abc, abc_pitch, options, ff.ctypes.data, 1,
                                   ctypes.byref(st))

    def device(witness=rows.ctypes.data, row_pitch=0, abc=out.ctypes.data, abc_pitch=0, options=0, n_sets=2):
        return L.gw_r1cs_abc_batch_device(rc._h, 0, witness, n_sets, row_pitch, abc, abc_pitch, options, None, None,
                                          ctypes.byref(st))

    def rejected(call, match, **kw):
        with pytest.raises(cwc.WitnessCalcError, match=match):
            cwc._check(call(**kw), st)

    for call in (host, device):
        rejected(call, "unknown option bits 2", options=2)
        rejected(call, "unknown option bits 4", options=GROTH16 | 4)
        rejected(call, "row_pitch is smaller", row_pitch=W * 32 - 16)
        rejected(call, "abc_pitch is smaller", abc_pitch=3 * n * 32 - 16)
        rejected(call, "abc_pitch is smaller", abc_pitch=3 * n * 32, options=GROTH16)      # n = 8 there
        rejected(call, "null argument", witness=None)
        rejected(call, "null argument", abc=None)
        assert call(witness=None, abc=None, n_sets=0) == 0      # n_sets = 0: nothing to do, NULL buffers allowed
        cwc._check(0, st)
    assert rc._h and L.gw_r1cs_abc_batch(None, None, 0, 0, None, 0, 0, None, 1, ctypes.byref(st)) == 1
    cwc._check(0, st)
    # device buffers and pitches are 16-byte multiples
    rejected(device, "16-byte aligned", row_pitch=W * 32 + 8)
    rejected(device, "16-byte aligned", abc_pitch=3 * n * 32 + 8)
    rejected(device, "16-byte aligned", witness=rows.ctypes.data + 8)
    rejected(device, "16-byte aligned", abc=out.ctypes.data + 8)


def test_abc_without_a_device_fails_loudly(cwc):
    if cwc.device_count() > 0:
        pytest.skip("a GPU is present")
    rc = cwc.R1cs(ref.serialize_r1cs(trivial(3)))
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        rc.abc_batch(np.zeros((1, 8, 32), np.uint8))
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        rc.abc_batch(np.zeros((1, 8, 32), np.uint8), groth16=True, want_verdict=True)
    buf = np.zeros(4096, np.uint8)
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        rc.abc_batch_device(0, buf.ctypes.data, 1, buf.ctypes.data + 512)


def test_abi_declarations_match_in_the_header_the_python_binding_and_the_rust_shim(cwc):
    hdr = open(os.path.join(util.ROOT, "include", "graph_witness.h")).read()
    rs = open(os.path.join(util.ROOT, "rust-shim", "src", "ffi.rs")).read()
    assert re.search(r"#define GW_R1CS_ABC_GROTH16 1u\b", hdr)
    assert "pub const GW_R1CS_ABC_GROTH16: u32 = 1;" in rs and cwc.R1CS_ABC_GROTH16 == 1
    rs_type = {"uint64_t": "u64", "uint32_t": "u32", "size_t": "usize", "int": "c_int"}
    py_type = {"uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32, "size_t": ctypes.c_size_t, "int": ctypes.c_int}
    for name in ("gw_r1cs_abc_len", "gw_r1cs_abc_batch", "gw_r1cs_abc_batch_device"):
        assert name in cwc.EXPORTS
        c_ret, c_args = re.search(r"\n(\w+)\s+" + name + r"\(([^)]*)\);", hdr).groups()
        c_sig = []                                       # parameter types, "ptr" for every pointer
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
def _public(r):
    """the pair with three public signals (the generated pairs have none): the Groth16 input rows read w_0 .. w_3"""
    return dict(r, n_pub_out=1, n_pub_in=2)


def _expected(r, w, groth16):
    A, B, C = abc_ref.abc_ref(r, w, groth16)
    return np.frombuffer(util.pack_u256(A + B + C), np.uint8).reshape(3, len(A), 32)


def _distinct(graph, r, n_in, seed):
    """four valid rows and corrupted variants: a wrong value, values >= M (M, M + 5, 2^256 - 1; one in a public input
    wire), two wrong values.  Returns (rows [D, W, 32], verdict [D], expected plain [D, 3, m, 32], expected Groth16)"""
    rnd = random.Random(seed)
    valid = graph.calc_witness_batch(_inputs(np.random.default_rng(seed), 4, n_in))
    W = graph.n_witness
    rows = [valid[i].copy() for i in range(4)]
    for j, changes in enumerate(([(None, None)], [(None, M)], [(2, M + 5)], [(None, (1 << 256) - 1)], [(3, M)],
                                 [(None, None), (None, None)])):
        row = valid[j % 4].copy()
        for wire, v in changes:
            wire = rnd.randrange(1, W) if wire is None else wire
            v = rnd.randrange(M) if v is None else v
            row[wire] = np.frombuffer(v.to_bytes(32, "little"), np.uint8)
        rows.append(row)
    rows = np.stack(rows)
    ws = [util.unpack_u256(x.tobytes()) for x in rows]
    verdict = np.array([OK if ref.check_r1cs(r, w) is None else ref.check_r1cs(r, w) for w in ws], np.uint32)
    assert (verdict[:4] == OK).all() and (verdict[4:] != OK).any()
    return rows, verdict, np.stack([_expected(r, w, False) for w in ws]), np.stack([_expected(r, w, True) for w in ws])


def _tiling(B, n_distinct, picked):
    idx = np.arange(B) % 4
    for j, b in enumerate(sorted(p for p in picked if p < B)):
        idx[b] = 4 + j % (n_distinct - 4)
    return idx


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_every_value_of_every_row_matches_the_reference(cwc, shape):
    import torch
    g, r, n_in = _pair(shape)
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    rows, verdict, exp_plain, exp_groth = _distinct(graph, r, n_in, 31)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    big = 512 * sms + 1500
    picked = {0, 5, 31, 32, 33, 500, 999, 512 * sms - 1, 512 * sms, big - 1} | set(random.Random(32).sample(range(big), 40))
    for B in (1, 33, 1000):
        idx = _tiling(B, len(rows), picked)
        batch = rows[idx]
        assert (rc.check_batch(batch) == verdict[idx]).all()
        for groth16, exp in ((False, exp_plain), (True, exp_groth)):
            got, ff = rc.abc_batch(batch, groth16=groth16, want_verdict=True)
            assert got.shape == (B, 3, rc.abc_len(groth16), 32)
            bad = np.nonzero((got != exp[idx]).reshape(B, -1).any(axis=1))[0]
            assert len(bad) == 0, (B, groth16, bad[:5])
            assert (ff == verdict[idx]).all(), (B, groth16)
            assert (rc.abc_batch(batch, groth16=groth16) == got).all()
    # more rows than one wave of 512-thread CTAs, on the device: compared there, chunk by chunk
    idx = _tiling(big, len(rows), picked)
    d_rows = torch.from_numpy(rows[idx].reshape(big, -1)).cuda()
    d_idx = torch.from_numpy(idx).cuda()
    d_ff = torch.zeros(big, dtype=torch.int32, device="cuda:0")
    for groth16, exp in ((False, exp_plain), (True, exp_groth)):
        n = rc.abc_len(groth16)
        d_exp = torch.from_numpy(exp.reshape(len(rows), -1)).cuda()
        d_abc = torch.empty((big, 3 * n * 32), dtype=torch.uint8, device="cuda:0")
        rc.abc_batch_device(0, d_rows.data_ptr(), big, d_abc.data_ptr(), groth16=groth16, d_first_failed_ptr=d_ff.data_ptr())
        torch.cuda.synchronize()
        for c0 in range(0, big, 8192):
            assert torch.equal(d_abc[c0:c0 + 8192], d_exp[d_idx[c0:c0 + 8192]]), (groth16, c0)
        assert (d_ff.cpu().numpy().view(np.uint32) == verdict[idx]).all()
        del d_abc


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_valid_rows_in_the_groth16_layout(cwc, shape):
    g, r, n_in = _pair(shape)
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    rows = graph.calc_witness_batch(_inputs(np.random.default_rng(41), 64, n_in))
    got, ff = rc.abc_batch(rows, groth16=True, want_verdict=True)
    assert (ff == OK).all()
    m, n = len(r["constraints"]), rc.abc_len(groth16=True)
    assert n >= m + 4 and n & (n - 1) == 0 and n // 2 < m + 4
    for b in range(0, 64, 9):
        A, B, C = (util.unpack_u256(got[b, i].tobytes()) for i in range(3))
        assert all((a * bb - c) % M == 0 for a, bb, c in zip(A, B, C))          # A o B = C at all n points
        w = util.unpack_u256(rows[b].tobytes())
        assert A[m:m + 4] == w[:4] and A[m + 4:] == [0] * (n - m - 4) and B[m:] == C[m:] == [0] * (n - m)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_host_and_device_entry_points_agree(cwc, shape):
    import torch
    g, r, n_in = _pair(shape)
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    rows, verdict, _, _ = _distinct(graph, r, n_in, 51)
    B, W = 1000, graph.n_witness
    idx = _tiling(B, len(rows), set(random.Random(52).sample(range(B), 60)))
    bad = rows[idx]
    for groth16 in (False, True):
        n = rc.abc_len(groth16)
        host, hff = rc.abc_batch(bad, groth16=groth16, want_verdict=True)
        assert (hff == verdict[idx]).all()
        # host rows with a pitch, output with a padded pitch: the padding keeps its canary
        pitch, out_b = W * 32 + 40, 3 * n * 32
        opitch = out_b + 24
        src = np.zeros((B, pitch), np.uint8)
        src[:, :W * 32] = bad.reshape(B, -1)
        out = np.full((B, opitch), 0xA5, np.uint8)
        ff = np.zeros(B, np.uint32)
        st = cwc.gw_status_t()
        cwc._check(cwc._L.gw_r1cs_abc_batch(rc._h, src.ctypes.data, B, pitch, out.ctypes.data, opitch, int(groth16),
                                            ff.ctypes.data, 1, ctypes.byref(st)), st)
        assert (out[:, :out_b] == host.reshape(B, -1)).all() and (out[:, out_b:] == 0xA5).all() and (ff == hff).all()
        # device rows with a pitch, padded output with a canary, on a non-default stream
        dpitch = W * 32 + 48
        dev = torch.zeros((B, dpitch), dtype=torch.uint8, device="cuda:0")
        dev[:, :W * 32] = torch.from_numpy(bad.reshape(B, -1)).cuda()
        d_out = torch.full((B, out_b + 32), 0xA5, dtype=torch.uint8, device="cuda:0")
        d_ff = torch.zeros(B, dtype=torch.int32, device="cuda:0")
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        rc.abc_batch_device(0, dev.data_ptr(), B, d_out.data_ptr(), row_pitch=dpitch, abc_pitch=out_b + 32, groth16=groth16,
                            d_first_failed_ptr=d_ff.data_ptr(), stream=s.cuda_stream)
        s.synchronize()
        got = d_out.cpu().numpy()
        assert (got[:, :out_b] == host.reshape(B, -1)).all() and (got[:, out_b:] == 0xA5).all()
        assert (d_ff.cpu().numpy().view(np.uint32) == hff).all()
        # .wtns images in place
        files = np.zeros((B, graph.wtns_file_size() + 20), np.uint8)
        fp = files.shape[1]
        files[:, 76:76 + W * 32] = bad.reshape(B, -1)
        assert (rc.abc_batch(files.reshape(-1)[76:], groth16=groth16, row_pitch=fp, n_sets=B) == host).all()
        if cwc.device_count() >= 2:
            two, ff2 = rc.abc_batch(bad, groth16=groth16, n_gpus=2, want_verdict=True)
            assert (two == host).all() and (ff2 == hff).all()


@pytest.mark.gpu
def test_gpu_evaluation_and_abc_on_one_stream(cwc):
    import torch
    g, r, n_in = _pair("poseidon")
    r = _public(r)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    B, W = 3000, graph.n_witness
    inputs = _inputs(np.random.default_rng(61), B, n_in)
    n = rc.abc_len(groth16=True)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_in = torch.from_numpy(inputs.reshape(B, -1)).cuda()
        d_w = torch.empty((B, W * 32), dtype=torch.uint8, device="cuda:0")
        d_abc = torch.empty((B, 3 * n * 32), dtype=torch.uint8, device="cuda:0")
        d_ff = torch.empty(B, dtype=torch.int32, device="cuda:0")
    graph.calc_witness_batch_device(0, d_in.data_ptr(), B, d_w.data_ptr(), stream=s.cuda_stream)
    rc.abc_batch_device(0, d_w.data_ptr(), B, d_abc.data_ptr(), groth16=True, d_first_failed_ptr=d_ff.data_ptr(),
                        stream=s.cuda_stream)
    s.synchronize()
    host, hff = rc.abc_batch(graph.calc_witness_batch(inputs), groth16=True, want_verdict=True)
    assert (d_abc.cpu().numpy() == host.reshape(B, -1)).all()
    assert (d_ff.cpu().numpy().view(np.uint32) == hff).all() and (hff == OK).all()


@pytest.mark.gpu
def test_gpu_no_constraints(cwc):
    g, r, n_in = _pair("random")
    graph = cwc.Graph(g)
    empty = cwc.R1cs(ref.serialize_r1cs({"n_wires": graph.n_witness, "n_pub_out": 1, "n_pub_in": 2, "constraints": []}))
    rows = graph.calc_witness_batch(_inputs(np.random.default_rng(71), 70, n_in))
    rows[5, 2] = np.frombuffer((M + 9).to_bytes(32, "little"), np.uint8)
    plain, ff = empty.abc_batch(rows, want_verdict=True)
    assert plain.shape == (70, 3, 0, 32) and (ff == OK).all()
    groth, ff = empty.abc_batch(rows, groth16=True, want_verdict=True)
    assert groth.shape == (70, 3, 4, 32) and (ff == OK).all()
    for b in range(70):
        w = util.unpack_u256(rows[b].tobytes())
        assert util.unpack_u256(groth[b, 0].tobytes()) == [v % M for v in w[:4]]
    assert not groth[:, 1:].any()
    assert empty.abc_batch(rows[:0]).shape == (0, 3, 0, 32)


@pytest.mark.gpu
def test_gpu_wtns_check_all(cwc, tmp_path):
    g, r, n_in = _pair("poseidon")
    graph = cwc.Graph(g)
    (tmp_path / "c.r1cs").write_bytes(ref.serialize_r1cs(r))
    files = graph.calc_witness_batch_wtns(_inputs(np.random.default_rng(81), 2, n_in))
    (tmp_path / "good.wtns").write_bytes(files[0].tobytes())
    w = util.po.parse_wtns(files[1].tobytes())
    cons = r["constraints"]
    for k in (40, len(cons) - 1):                       # the wires constraints 40 and m - 1 define
        wire = cons[k][2][-1][0]
        w[wire] = (w[wire] + 1) % M
    high = cons[100][0][-1][0]                          # a wire constraint 100 reads, at its value + M
    w[high] += M
    (tmp_path / "bad.wtns").write_bytes(util.po.wtns_from_witness(w))
    A, B, C = abc_ref.abc_ref(r, w)
    broken = [k for k in range(len(cons)) if (A[k] * B[k] - C[k]) % M]
    assert len(broken) >= 2 and high != 0
    exe = os.path.join(util.ROOT, "circom-witnesscalc_b200", "bin", "wtns-check")
    good, bad = str(tmp_path / "good.wtns"), str(tmp_path / "bad.wtns")
    res = subprocess.run([exe, "--all", str(tmp_path / "c.r1cs"), good, bad], capture_output=True, text=True)
    exp = [f"{good}: OK", f"{bad}: constraint {ref.check_r1cs(r, w)} not satisfied"]
    exp += [f"  constraint {k}: {A[k]} * {B[k]} != {C[k]}" for k in broken]
    exp += [f"  wire {high}: {w[high]} >= M"]
    assert res.returncode == 1 and res.stdout.splitlines() == exp, res.stdout + res.stderr
    # without --all: the verdict lines only
    res = subprocess.run([exe, str(tmp_path / "c.r1cs"), good, bad], capture_output=True, text=True)
    assert res.returncode == 1 and res.stdout.splitlines() == exp[:2]
    res = subprocess.run([exe, "--all", str(tmp_path / "c.r1cs"), good], capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.splitlines() == exp[:1]
