"""R1CS check: the .r1cs codec (reference and library), the compiled program and its chunk bound on the host, and the
GPU entry points (host rows, device rows, fused evaluate-and-check, wtns-check) against the reference checker on
generated (graph, R1CS) pairs (tools/r1cs_gen.py)."""
import ctypes
import importlib
import os
import random
import struct
import subprocess

import numpy as np
import pytest

from tests import r1cs_ref as ref
from tests import util
from tools import r1cs_gen

M = util.M
OK = 0xFFFFFFFF


@pytest.fixture(scope="module")
def cwc():
    subprocess.check_call(["python", os.path.join(util.ROOT, "circom-witnesscalc_b200", "build.py")])
    return importlib.import_module("circom-witnesscalc_b200")


def two_constraints():
    # w = [1, x, y, z]:  x * y = z   and   (2 - x) * 1 = 0
    return {"n_wires": 4, "n_pub_out": 1, "n_pub_in": 1, "n_prv_in": 1, "n_labels": 4,
            "constraints": [([(1, 1)], [(2, 1)], [(3, 1)]),
                            ([(0, 2), (1, M - 1)], [(0, 1)], [])]}


# ---- codec --------------------------------------------------------------------------------------------------------
def test_reference_codec_golden_bytes_and_round_trip():
    data = ref.serialize_r1cs(two_constraints())
    le32 = lambda v: struct.pack("<I", v)
    hdr = le32(32) + M.to_bytes(32, "little") + le32(4) + le32(1) + le32(1) + le32(1) + struct.pack("<Q", 4) + le32(2)
    term = lambda w, c: le32(w) + c.to_bytes(32, "little")
    cons = (le32(1) + term(1, 1) + le32(1) + term(2, 1) + le32(1) + term(3, 1)
            + le32(2) + term(0, 2) + term(1, M - 1) + le32(1) + term(0, 1) + le32(0))
    labels = b"".join(struct.pack("<Q", i) for i in range(4))
    golden = (b"r1cs" + le32(1) + le32(3) + le32(1) + struct.pack("<Q", 64) + hdr + le32(2) + struct.pack("<Q", len(cons))
              + cons + le32(3) + struct.pack("<Q", 32) + labels)
    assert len(hdr) == 64 and data == golden
    back = ref.parse_r1cs(data)
    assert back["constraints"] == [tuple(c) for c in two_constraints()["constraints"]]
    assert ref.check_r1cs(back, [1, 3, 5, 15]) == 1          # 2 - 3 != 0
    assert ref.check_r1cs(back, [1, 2, 5, 10]) is None
    assert ref.check_r1cs(back, [1, 2, 5, 11]) == 0


def test_load_and_info_without_gpu(cwc):
    r = cwc.R1cs(ref.serialize_r1cs(two_constraints(), order=(3, 2, 1)))      # sections in any order
    info = r.info()
    assert (info["n_wires"], info["n_pub_out"], info["n_pub_in"], info["n_prv_in"], info["n_constraints"], info["n_labels"]) == (4, 1, 1, 1, 2, 4)
    # x*y=z: three T_ADDHI; 2*w0 (T_MAC) - x (T_SUBHI); 1*w0 (T_ADDHI)
    assert (info["n_terms"], info["n_mac_terms"], info["n_consts"], info["n_chunks"]) == (6, 1, 1, 5)


def _rejected(cwc, data, match):
    with pytest.raises(cwc.WitnessCalcError, match=match):
        cwc.R1cs(data)


def test_rejects_bad_magic_version_and_missing_sections(cwc):
    good = ref.serialize_r1cs(two_constraints())
    _rejected(cwc, b"r1cz" + good[4:], "magic")
    _rejected(cwc, good[:4] + struct.pack("<I", 2) + good[8:], "version 2")
    _rejected(cwc, ref.serialize_r1cs(two_constraints(), order=(2, 3)), r"header section \(1\) missing")
    _rejected(cwc, ref.serialize_r1cs(two_constraints(), order=(1, 3)), r"constraints section \(2\) missing")
    _rejected(cwc, b"", "magic")


def test_rejects_truncation_and_size_mismatch(cwc):
    good = ref.serialize_r1cs(two_constraints())
    for n in (3, 8, 11, 20, 80, len(good) - 1):
        _rejected(cwc, good[:n], "truncated|magic")
    _rejected(cwc, good + b"\0", "after the last section")
    # a constraints section one byte longer than its constraints, and one whose counts run past its end
    r = two_constraints()
    body = ref.serialize_r1cs(r, order=(2,), with_labels=False)[12:]
    t, size = struct.unpack_from("<IQ", body, 0)
    hdr_sec = ref.serialize_r1cs(r, order=(1,), with_labels=False)[12:]
    longer = b"r1cs" + struct.pack("<II", 1, 2) + hdr_sec + struct.pack("<IQ", 2, size + 1) + body[12:] + b"\0"
    _rejected(cwc, longer, "longer than its")
    r["constraints"] = r["constraints"] + [([(1, 1)], [], [])]
    hdr_more = ref.serialize_r1cs(r, order=(1,), with_labels=False)[12:]
    shorter = b"r1cs" + struct.pack("<II", 1, 2) + hdr_more + body
    _rejected(cwc, shorter, "truncated")
    _rejected(cwc, ref.serialize_r1cs(two_constraints(), extra_sections=[(1, b"\0" * 4)]), "twice|BN254")
    labels_short = ref.serialize_r1cs(two_constraints(), order=(1, 2), extra_sections=[(3, b"\0" * 24)])
    _rejected(cwc, labels_short, "wire2label")


def test_rejects_other_fields_wires_and_custom_gates(cwc):
    r = two_constraints()
    _rejected(cwc, ref.serialize_r1cs(r, n8=48, prime=M), "n8 = 48")
    _rejected(cwc, ref.serialize_r1cs(r, prime=M + 2), "this library evaluates BN254 graphs only")
    bad = two_constraints()
    bad["constraints"][1] = ([(4, 1)], [], [])
    _rejected(cwc, ref.serialize_r1cs(bad), "wire 4 >= n_wires = 4")
    for t in (4, 5):
        _rejected(cwc, ref.serialize_r1cs(r, extra_sections=[(t, b"\0" * 8)]), "custom gates")


def test_coefficients_at_or_above_m_are_reduced():
    lib = ref.host_lib()
    r = {"n_wires": 3, "constraints": [([(1, M + 1)], [(2, 2 * M + 5)], [(0, 3 * M + 7), (1, M)])]}
    data = ref.serialize_r1cs(r)
    h = lib.r1cs_host_load(data, len(data), None, 0)
    info = (ctypes.c_uint64 * 11)()
    lib.r1cs_host_info(h, info)
    assert info[6] == 3 and info[7] == 2          # M + 1 -> 1 (T_ADDHI); M -> 0 (dropped); 2M + 5, 3M + 7 -> T_MAC
    for w1, w2 in ((5, 7), (3, 1), (7 * pow(25, M - 2, M) % M, 5)):       # w1 * (5 w2) == 7
        assert lib.r1cs_host_check(h, util.pack_u256([1, w1, w2])) == (OK if (w1 * 5 * w2 - 7) % M == 0 else 0)
    assert lib.r1cs_host_check(h, util.pack_u256([1, 7 * pow(25, M - 2, M) % M, 5])) == OK
    lib.r1cs_host_free(h)


def test_check_batch_without_a_device_fails_loudly(cwc):
    if cwc.device_count() > 0:
        pytest.skip("a GPU is present")
    r = cwc.R1cs(ref.serialize_r1cs(two_constraints()))
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device"):
        r.check_batch(np.zeros((1, 4, 32), np.uint8))


def test_info_struct_is_the_same_in_the_header_the_python_binding_and_the_rust_shim(cwc):
    import re
    hdr = open(os.path.join(util.ROOT, "include", "graph_witness.h")).read()
    end = hdr.index("} gw_r1cs_info_t;")
    body = hdr[hdr.rindex("typedef struct", 0, end):end]
    c_fields = re.findall(r"^\s*(uint64_t|uint32_t)\s+(\w+);", body, re.M)
    py_fields = [(("uint64_t" if t is ctypes.c_uint64 else "uint32_t"), n) for n, t in cwc.gw_r1cs_info_t._fields_]
    assert c_fields == py_fields and len(c_fields) == 10
    rs = open(os.path.join(util.ROOT, "rust-shim", "src", "ffi.rs")).read()
    rbody = rs[rs.index("pub struct gw_r1cs_info_t"):]
    rbody = rbody[:rbody.index("}")]
    rs_fields = [(("uint64_t" if t == "u64" else "uint32_t"), n) for n, t in re.findall(r"pub (\w+): (u64|u32),", rbody)]
    assert rs_fields == c_fields


# ---- compiled program on the host: chunk bound with worst-case operands -------------------------------------------
@pytest.mark.parametrize("emulate_ptx", [False, True])
def test_chunk_bound_with_worst_case_operands(emulate_ptx):
    """the largest operand of each term kind, in linear combinations one term below, at and above the chunk bound
    (22 T_MAC or 4 T_ADDHI / T_SUBHI terms per reduction) and far above it:
      T_MAC   value M - 1 times the stored constant M - 1 (coefficient (M - 1) / 2^256 mod M), and two other constants;
      T_ADDHI value M - 1;  T_SUBHI value 0 (it adds (M - x) << 256, largest at x = 0) and value M - 1"""
    lib = ref.host_lib(emulate_ptx)
    half = 119
    n_w = 1 + 2 * half
    wit = [1] + [M - 1] * half + [0] * half                   # wires 1 .. 119 hold M - 1, wires 120 .. 238 hold 0
    top = lambda i: 1 + (i % half)
    zero = lambda i: 1 + half + (i % half)
    c_worst = (M - 1) * pow(1 << 256, M - 2, M) % M          # stored as c * 2^256 mod M = M - 1
    assert c_worst * (1 << 256) % M == M - 1
    cons = []
    for n in (3, 4, 5, 8, 9, 21, 22, 23, 44, 45, 100):
        for c, wire in ((c_worst, top), (M - 2, top), (M - 3, top), (1, top), (M - 1, zero), (M - 1, top)):
            lc = [(wire(i), c) for i in range(n)]
            cons.append((lc, lc, lc))
        mixed = [((zero if i % 3 == 2 else top)(i), (c_worst, 1, M - 1)[i % 3]) for i in range(n)]
        cons.append((mixed, [(0, M - 1)], mixed))
    r = {"n_wires": n_w, "constraints": cons}
    data = ref.serialize_r1cs(r)
    h = lib.r1cs_host_load(data, len(data), None, 0)
    abc = ctypes.create_string_buffer(96)
    row = util.pack_u256(wit)
    for k, con in enumerate(cons):
        st = lib.r1cs_host_eval(h, k, row, abc)
        got = util.unpack_u256(abc.raw)
        assert got == [ref.lc_value(lc, wit) for lc in con], (k, len(con[0]))
        a, b, c = got
        assert st == (1 if (a * b - c) % M == 0 else 0)
    exp = ref.check_r1cs(ref.parse_r1cs(data), wit)
    assert lib.r1cs_host_check(h, row) == (OK if exp is None else exp)
    lib.r1cs_host_free(h)


@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_compiled_program_matches_the_reference_on_the_host(shape):
    rnd = random.Random(11)
    g, r = r1cs_gen.random_pair(rnd, n_constraints=80) if shape == "random" else r1cs_gen.poseidon_pair(rnd, n_hashes=1)
    nodes, wit, _ = util.po.deserialize_graph(g)
    data = ref.serialize_r1cs(r)
    lib = ref.host_lib(emulate_ptx=True)
    h = lib.r1cs_host_load(data, len(data), None, 0)
    n_in = 6 if shape == "random" else 4
    for trial in range(6):
        w = util.po.evaluate(nodes, [1] + [util.random_value(rnd) for _ in range(n_in)], wit)
        assert ref.check_r1cs(r, w) is None
        if trial:
            for _ in range(trial):
                i = rnd.randrange(len(w))
                w[i] = rnd.choice((rnd.randrange(M), (w[i] + 1) % M, M + rnd.randrange(1 << 64)))
        exp = ref.check_r1cs(r, w)
        assert lib.r1cs_host_check(h, util.pack_u256(w)) == (OK if exp is None else exp)
    lib.r1cs_host_free(h)


# ---- GPU ----------------------------------------------------------------------------------------------------------
def _pair(shape):
    rnd = random.Random(3 if shape == "random" else 4)
    if shape == "random":
        g, r = r1cs_gen.random_pair(rnd, n_constraints=150)
        return g, r, 6
    g, r = r1cs_gen.poseidon_pair(rnd, n_hashes=2)
    return g, r, 4


def _inputs(rnd_np, B, n_in):
    vals = util.random_field_batch(rnd_np, (B, n_in + 1))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    return vals.view(np.uint8).reshape(B, n_in + 1, 32)


def _corrupt(rows, rnd, frac=0.7):
    """flips random witness entries in a copy; some rows stay valid.  Returns (rows, list of witness ints per row)"""
    rows = rows.copy()
    B, W, _ = rows.shape
    for b in range(B):
        if rnd.random() < frac:
            for _ in range(rnd.choice((1, 1, 2, 5))):
                i = rnd.randrange(W)
                v = rnd.choice((rnd.randrange(M), 0, 1, M - 1, M + rnd.randrange(1000), (1 << 256) - 1))
                rows[b, i] = np.frombuffer(v.to_bytes(32, "little"), np.uint8)
    return rows


def _expected(r, rows):
    out = []
    for b in range(rows.shape[0]):
        e = ref.check_r1cs(r, util.unpack_u256(rows[b].tobytes()))
        out.append(OK if e is None else e)
    return np.array(out, dtype=np.uint32)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_witnesses_pass_and_corrupted_rows_report_the_oracle_index(cwc, shape):
    g, r, n_in = _pair(shape)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    assert graph.n_witness == rc.info()["n_wires"]
    rnd_np, rnd = np.random.default_rng(7), random.Random(8)
    rows = graph.calc_witness_batch(_inputs(rnd_np, 4096, n_in))
    assert (rc.check_batch(rows) == OK).all()
    for B in (1, 33, 4096):
        bad = _corrupt(rows[:B], rnd)
        exp = _expected(r, bad)
        got = rc.check_batch(bad)
        assert (got == exp).all(), (B, np.nonzero(got != exp)[0][:5])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_batch_larger_than_one_wave_of_ctas(cwc, shape):
    """more rows than one wave of 512-thread CTAs covers: every CTA walks a second tile.  Whole warps of corrupted rows
    in the first tiles stop early; the next tile must restage its constraint stream from the start."""
    import torch
    g, r, n_in = _pair(shape)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    valid = graph.calc_witness_batch(_inputs(np.random.default_rng(21), 1024, n_in))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 512 * sms + 1500
    rows = np.ascontiguousarray(np.tile(valid, (B // len(valid) + 1, 1, 1))[:B])
    rnd = random.Random(22)
    picked = set(range(64)) | set(range(512 * sms - 40, 512 * sms + 70)) | set(rnd.sample(range(B), 300))
    picked = sorted(picked)
    rows[picked] = _corrupt(rows[picked], rnd, frac=1.0)
    exp = np.full(B, OK, dtype=np.uint32)
    exp[picked] = _expected(r, rows[picked])
    W = graph.n_witness
    d_rows = torch.from_numpy(rows.reshape(B, W * 32)).cuda()
    d_ff = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    rc.check_batch_device(0, d_rows.data_ptr(), B, d_ff.data_ptr())
    torch.cuda.synchronize()
    got = d_ff.cpu().numpy().view(np.uint32)
    assert (got == exp).all(), np.nonzero(got != exp)[0][:5]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["random", "poseidon"])
def test_gpu_entry_points_agree(cwc, shape):
    import torch
    g, r, n_in = _pair(shape)
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    rnd_np, rnd = np.random.default_rng(9), random.Random(10)
    B = 1000
    inputs = _inputs(rnd_np, B, n_in)
    rows, flags = graph.calc_witness_batch(inputs, want_flags=True)
    bad = _corrupt(rows, rnd, frac=0.5)
    exp = _expected(r, bad[:150])
    host = rc.check_batch(bad)
    assert (host[:150] == exp).all()
    # device rows on a non-default stream, with a pitch
    W = graph.n_witness
    pitch = W * 32 + 48
    dev = torch.zeros((B, pitch), dtype=torch.uint8, device="cuda:0")
    dev[:, :W * 32] = torch.from_numpy(bad.reshape(B, W * 32)).cuda()
    d_ff = torch.zeros(B, dtype=torch.int32, device="cuda:0")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    rc.check_batch_device(0, dev.data_ptr(), B, d_ff.data_ptr(), row_pitch=pitch, stream=s.cuda_stream)
    s.synchronize()
    assert (d_ff.cpu().numpy().view(np.uint32) == host).all()
    # host entry on .wtns images (pitched, 76-byte header in front of every row)
    files = graph.calc_witness_batch_wtns(inputs, file_pitch=graph.wtns_file_size() + 20)
    fp = files.shape[1]
    files[:, 76:76 + W * 32] = bad.reshape(B, W * 32)
    assert (rc.check_batch(files.reshape(-1)[76:], row_pitch=fp, n_sets=B) == host).all()
    # fused evaluate-and-check, with and without the witness
    w2, f2, ff2 = graph.calc_witness_batch_check(rc, inputs)
    assert (w2 == rows).all() and (f2 == flags).all() and (ff2 == OK).all()
    w3, f3, ff3 = graph.calc_witness_batch_check(rc, inputs, want_witness=False)
    assert w3 is None and (f3 == flags).all() and (ff3 == OK).all()


@pytest.mark.gpu
def test_gpu_two_devices_agree_with_one(cwc):
    if cwc.device_count() < 2:
        pytest.skip("one CUDA device")
    g, r, n_in = _pair("random")
    graph, rc = cwc.Graph(g), cwc.R1cs(ref.serialize_r1cs(r))
    inputs = _inputs(np.random.default_rng(12), 3001, n_in)
    bad = _corrupt(graph.calc_witness_batch(inputs), random.Random(13))
    assert (rc.check_batch(bad, n_gpus=2) == rc.check_batch(bad)).all()
    _, _, ff1 = graph.calc_witness_batch_check(rc, inputs)
    _, _, ff2 = graph.calc_witness_batch_check(rc, inputs, n_gpus=2, want_witness=False)
    assert (ff1 == ff2).all() and (ff1 == OK).all()


@pytest.mark.gpu
def test_gpu_no_constraints_and_wire_count_mismatch(cwc):
    g, r, n_in = _pair("random")
    graph = cwc.Graph(g)
    empty = cwc.R1cs(ref.serialize_r1cs({"n_wires": graph.n_witness, "constraints": []}))
    rows = graph.calc_witness_batch(_inputs(np.random.default_rng(1), 70, n_in))
    assert (empty.check_batch(rows) == OK).all()
    other = cwc.R1cs(ref.serialize_r1cs({"n_wires": graph.n_witness - 1, "constraints": []}))
    with pytest.raises(cwc.WitnessCalcError, match=f"{graph.n_witness} values but the R1CS has {graph.n_witness - 1} wires"):
        graph.calc_witness_batch_check(other, _inputs(np.random.default_rng(1), 4, n_in))
    sel = graph.select([0, 1, 2])
    rc = cwc.R1cs(ref.serialize_r1cs(r))
    with pytest.raises(cwc.WitnessCalcError, match="3 values"):
        sel.calc_witness_batch_check(rc, _inputs(np.random.default_rng(1), 4, n_in))


@pytest.mark.gpu
def test_gpu_wtns_check_cli(cwc, tmp_path):
    g, r, n_in = _pair("poseidon")
    graph = cwc.Graph(g)
    (tmp_path / "c.r1cs").write_bytes(ref.serialize_r1cs(r))
    files = graph.calc_witness_batch_wtns(_inputs(np.random.default_rng(2), 3, n_in))
    paths = []
    for i in range(3):
        p = tmp_path / f"w{i}.wtns"
        p.write_bytes(files[i].tobytes())
        paths.append(str(p))
    exe = os.path.join(util.ROOT, "circom-witnesscalc_b200", "bin", "wtns-check")
    # sections in any order: the witness section before the header section
    img = files[2].tobytes()
    (tmp_path / "swapped.wtns").write_bytes(img[:12] + img[64:] + img[12:64])
    paths.append(str(tmp_path / "swapped.wtns"))
    res = subprocess.run([exe, str(tmp_path / "c.r1cs")] + paths, capture_output=True, text=True)
    assert res.returncode == 0 and res.stdout.count(": OK") == 4, res.stdout + res.stderr
    w = util.po.parse_wtns(files[1].tobytes())
    k = r["constraints"][40][2][-1][0]                  # the wire constraint 40 defines
    w[k] = (w[k] + 1) % M
    (tmp_path / "bad.wtns").write_bytes(util.po.wtns_from_witness(w))
    exp = ref.check_r1cs(r, w)
    res = subprocess.run([exe, str(tmp_path / "c.r1cs"), paths[0], str(tmp_path / "bad.wtns")], capture_output=True, text=True)
    assert res.returncode == 1 and f"bad.wtns: constraint {exp} not satisfied" in res.stdout and ": OK" in res.stdout
    data = bytearray(files[0].tobytes())
    data[28] ^= 1                                        # the prime
    (tmp_path / "prime.wtns").write_bytes(bytes(data))
    short = util.po.wtns_from_witness(util.po.parse_wtns(files[0].tobytes())[:-1])
    (tmp_path / "short.wtns").write_bytes(short)
    res = subprocess.run([exe, str(tmp_path / "c.r1cs"), str(tmp_path / "prime.wtns"), str(tmp_path / "short.wtns")],
                         capture_output=True, text=True)
    assert res.returncode == 1 and "prime" in res.stdout and "wires" in res.stdout and "OK" not in res.stdout
