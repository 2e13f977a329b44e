"""GPU parity tests: the CUDA path, called through the C ABI, against the Python oracle and the
committed golden .wtns files.  Bit-exact comparison everywhere (integer arithmetic)."""
import importlib
import os
import random

import numpy as np
import pytest

from tests import util
from tests.util import po

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def cwc():
    mod = importlib.import_module("circom-witnesscalc_b200")
    assert mod.device_count() >= 1, "no CUDA device visible"
    return mod


GOLDEN = ["circuit1", "circuit2", "circuit3", "circuit4", "circuit5_poseidon", "circuit6_num2bits",
          "circuit7_poseidon4", "poseidon2", "poseidon3", "poseidon5", "circuit11_key_expansion", "circuit8_sha256_512",
          "circuit9_authV2", "authV2_32_32"]


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_wtns_drop_in(cwc, name):
    """gw_calc_witness(inputs.json, graph.bin) == committed .wtns, byte for byte (test_circuits.sh:81 `cmp`)."""
    got = cwc.calc_witness_wtns(util.golden_inputs(name), util.golden_graph(name))
    assert got == util.golden_wtns(name)


@pytest.mark.parametrize("name", ["circuit5_poseidon", "circuit2", "circuit6_num2bits", "circuit9_authV2"])
def test_drop_in_binaries_run_and_cmp(cwc, name, tmp_path):
    """The equivalent of test_circuits.sh:64,81: RUN `calc-witness <graph.bin> <inputs.json> <out.wtns>` and the
    plain-C embedding example (examples/calc_witness.c, argv order <inputs> <graph> <witness> as in the reference's
    example) and `cmp` what they write with the golden .wtns."""
    import os
    import subprocess
    gp, ip = tmp_path / "graph.bin", tmp_path / "inputs.json"
    gp.write_bytes(util.golden_graph(name))
    ip.write_text(util.golden_inputs(name))
    want = util.golden_wtns(name)
    out1 = tmp_path / "cli.wtns"
    r = subprocess.run([cwc.CLI_PATH, str(gp), str(ip), str(out1)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "Witness generated in:" in r.stdout and f"witness saved to {out1}" in r.stdout      # calc-witness.rs:41,48
    assert out1.read_bytes() == want
    assert os.path.exists(cwc.EXAMPLE_PATH), "bin/example-calc-witness missing: run circom-witnesscalc_b200/build.py"
    out2 = tmp_path / "example.wtns"
    r = subprocess.run([cwc.EXAMPLE_PATH, str(ip), str(gp), str(out2)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr + r.stdout
    assert out2.read_bytes() == want
    # error path of the CLI: a corrupt graph is an error message and a non-zero exit, not a crash
    bad = tmp_path / "bad.bin"
    bad.write_bytes(util.golden_graph(name)[:40])
    r = subprocess.run([cwc.CLI_PATH, str(bad), str(ip), str(tmp_path / "x.wtns")], capture_output=True, text=True, timeout=60)
    assert r.returncode not in (0, -11) and "Error" in r.stderr


def test_reference_held_known_answers_on_gpu(cwc):
    """tests/golden/kat.json (AuthV2(32,32) expOut incl. profileNonce = 10, Poseidon(3), t = 6, t = 3: vectors the
    reference tree holds) through gw_calc_witness (latency kernel) AND the throughput kernel (one batch of all cases)."""
    import json
    for name, cases in sorted(util.kat().items()):
        data = util.golden_graph(name)
        g = cwc.Graph(data)
        for case in cases:
            w = cwc.calc_witness(json.dumps(case["inputs"]), data)
            util.kat_check(w, g.input_signals, g.n_inputs, case, util.KAT_OUTPUTS[name])
        out = g.calc_witness_batch(g.pack_inputs([{k: (v if isinstance(v, list) else [v]) for k, v in c["inputs"].items()} for c in cases]))
        for b, case in enumerate(cases):
            util.kat_check(util.unpack_u256(out[b].tobytes()), g.input_signals, g.n_inputs, case, util.KAT_OUTPUTS[name])


def test_random_graphs_all_ops(cwc):
    rnd = random.Random(1234)
    for t in range(12):
        nodes, wit, imap = util.random_graph(rnd, n_ops=400)
        g = cwc.Graph(po.serialize_graph(nodes, wit, imap))
        B = 96 + t            # not a multiple of the CTA size: ragged last tile
        rows = [[1] + [util.random_value(rnd) if rnd.random() < 0.8 else rnd.randrange(1 << 256) for _ in range(6)]
                for _ in range(B)]
        inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(B, 7, 32)
        out = g.calc_witness_batch(inp)
        for b in range(0, B, 7):
            want = po.evaluate(nodes, rows[b], wit, "circom")
            assert util.unpack_u256(out[b].tobytes()) == want, (t, b)


def test_reference_undefined_flags(cwc):
    """cases where the reference panics get the circom value and a per-set flag"""
    nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_INPUT, 2),
             (po.K_DUO, po.DUO["Shl"], 1, 2), (po.K_DUO, po.DUO["Bxor"], 1, 2), (po.K_DUO, po.DUO["Pow"], 1, 2)]
    g = cwc.Graph(po.serialize_graph(nodes, [0, 3, 4, 5], {"a": (1, 1), "b": (2, 1)}))
    M = po.M
    rows = [[1, 5, 3], [1, M - 1, 200], [1, M, 0], [1, (1 << 253), (1 << 253) ^ M]]
    inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(4, 3, 32)
    out, flags = g.calc_witness_batch(inp, want_flags=True)
    for b, r in enumerate(rows):
        assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, r, [0, 3, 4, 5], "circom")
    assert flags[0] == 4 and flags[1] & 1 and flags[3] & 2


def test_uno_ops_id_lnot_bnot_and_flags(cwc):
    """UnoOperation beyond Neg (SURVEY 8a row 4): Id is unimplemented! in the reference (graph.rs:195), Lnot / Bnot are
    north_star's extensions (circom semantics: !a, (~a & (2^254 - 1)) mod M).  Values equal the oracle's circom mode and
    the per-set flag says which reference-undefined op ran (8 = Id, 16 = Lnot/Bnot)."""
    M = po.M
    for uno, flag in ((po.UNO["Neg"], 0), (po.UNO["Id"], 8), (po.UNO["Lnot"], 16), (po.UNO["Bnot"], 16)):
        nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_CONST, 5), (po.K_UNO, uno, 1), (po.K_UNO, uno, 2),
                 (po.K_DUO, po.DUO["Mul"], 3, 3), (po.K_UNO, uno, 5)]
        wit = [0, 3, 4, 6]
        g = cwc.Graph(po.serialize_graph(nodes, wit, {"a": (1, 1)}))
        vals = [0, 1, 2, M - 1, M >> 1, (M >> 1) + 1, (1 << 253) - 1, 1 << 253, (1 << 254) - 1 - M, (1 << 254) - M, M + 3, (1 << 256) - 1]
        rows = [[1, v] for v in vals]
        inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), 2, 32)
        out, flags = g.calc_witness_batch(inp, want_flags=True)
        for b, r in enumerate(rows):
            assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, r, wit, "circom"), (uno, b)
            assert flags[b] == flag, (uno, b, flags[b])
        # the same single witness through latency mode
        for r in rows[:6]:
            one = np.frombuffer(util.pack_u256(r), dtype=np.uint8).reshape(2, 32)
            got, fl = g.calc_witness_latency(one, want_flags=True)
            assert util.unpack_u256(got.tobytes()) == po.evaluate(nodes, r, wit, "circom") and fl == flag


def test_batch_matches_single_and_properties(cwc):
    """batch of random inputs on Poseidon(2): every row equals the oracle; duplicated rows give
    duplicated witnesses (purity); size-independent check on a larger batch via row sampling."""
    name = "poseidon2"
    data = util.golden_graph(name)
    nodes, wit, imap = po.deserialize_graph(data)
    g = cwc.Graph(data)
    rng = np.random.default_rng(7)
    B = 4096 + 37
    vals = util.random_field_batch(rng, (B, g.n_inputs))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    vals[B - 1] = vals[0]
    inp = vals.view(np.uint8).reshape(B, g.n_inputs, 32)
    out = g.calc_witness_batch(inp)
    assert (out[B - 1] == out[0]).all()
    for b in [0, 1, 31, 32, 127, 128, 4095, 4096, B - 2]:
        row = util.limbs_to_ints(vals[b])
        assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, row, wit)


def test_bad_inputs_return_errors(cwc):
    data = util.golden_graph("circuit1")
    with pytest.raises(cwc.WitnessCalcError):
        cwc.calc_witness_wtns('{"a": "1", "zzz": "2"}', data)          # unknown key (reference: panic)
    with pytest.raises(cwc.WitnessCalcError):
        cwc.calc_witness_wtns('{"a": ["1", "2"]}', data)                # wrong length (reference: panic)
    with pytest.raises(cwc.WitnessCalcError):
        cwc.calc_witness_wtns('{"a": -1}', data)                        # lib.rs:211-214
    with pytest.raises(cwc.WitnessCalcError):
        cwc.calc_witness_wtns('{"a": "1"', data)                        # invalid JSON (reference: panic)
    with pytest.raises(cwc.WitnessCalcError):
        cwc.calc_witness_wtns('{"a": "1"}', b"not a graph file at all....")


# GW_LAT_BIT=0: Boolean graphs (SHA-256, Num2Bits) also take the generic latency kernel instead of the bit-sliced plan
# GW_LAT_MODE=level: the level-synchronous kernel (eval_latency_kernel); default: the dataflow kernel (eval_dataflow_kernel)
LATENCY_ENVS = [{}, {"GW_LAT_MODE": "level"}, {"GW_LAT_BIT": "0"}, {"GW_LAT_MODE": "level", "GW_LAT_CHAIN": "0", "GW_LAT_BIT": "0"},
                {"GW_LAT_WARPS": "2", "GW_LAT_SLOW_WARPS": "1", "GW_LAT_D": "1"}, {"GW_LAT_MODE": "level", "GW_LAT_WARPS": "2", "GW_LAT_SLOW_WARPS": "1", "GW_LAT_D": "1"},
                {"GW_LAT_WARPS": "5", "GW_LAT_D": "60", "GW_LAT_SPLIT": "0", "GW_LAT_BIT": "0"},
                {"GW_LAT_MODE": "level", "GW_LAT_WARPS": "5", "GW_LAT_D": "60", "GW_LAT_SPLIT": "0", "GW_LAT_BIT": "0"}, {"GW_LAT_FUSE": "0"},
                {"GW_LAT_MODE": "level", "GW_LAT_FUSE": "0"}, {"GW_LAT_LINKS": "2"}, {"GW_LAT_LINKS": "0"}]


@pytest.mark.parametrize("env", LATENCY_ENVS)
def test_latency_mode_random_graphs_and_golden(cwc, monkeypatch, env):
    """single-witness latency mode (one CTA: level-synchronous main warps, asynchronous slow warps, lane chains):
    gw_calc_witness_latency.  The plan options are read when the latency plan of a graph is first built."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    rnd = random.Random(4321)
    for t in range(10):
        nodes, wit, imap = util.random_graph(rnd, n_ops=500)
        g = cwc.Graph(po.serialize_graph(nodes, wit, imap))
        for _ in range(2):
            row = [1] + [util.random_value(rnd) if rnd.random() < 0.8 else rnd.randrange(1 << 256) for _ in range(6)]
            out, ms = g.calc_witness_latency(np.frombuffer(util.pack_u256(row), dtype=np.uint8).reshape(7, 32))
            assert util.unpack_u256(out.tobytes()) == po.evaluate(nodes, row, wit, "circom"), t
    for name in ("circuit5_poseidon", "circuit6_num2bits", "circuit8_sha256_512", "circuit9_authV2"):
        data = util.golden_graph(name)
        nodes, wit, imap = po.deserialize_graph(data)
        g = cwc.Graph(data)
        buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs(name)))
        if env.get("GW_LAT_FUSE") == "0" and name == "circuit9_authV2":
            # one instruction per graph node keeps more values alive than the shared-memory value file holds: the
            # latency entry point says so, and the drop-in gw_calc_witness falls back to the throughput kernel
            with pytest.raises(cwc.WitnessCalcError, match="too wide"):
                g.calc_witness_latency(np.frombuffer(util.pack_u256(buf), dtype=np.uint8).reshape(g.n_inputs, 32))
            assert cwc.calc_witness_wtns(util.golden_inputs(name), data) == util.golden_wtns(name)
            continue
        for _ in range(3):                                   # repeated launches reuse the uploaded plan
            out, ms = g.calc_witness_latency(np.frombuffer(util.pack_u256(buf), dtype=np.uint8).reshape(g.n_inputs, 32))
            assert po.wtns_from_witness(util.unpack_u256(out.tobytes())) == util.golden_wtns(name)
        print(f"latency mode {name} {env}: {ms:.2f} ms kernel")


def test_poseidon_like_graphs_batch_and_latency(cwc):
    """random graphs with Poseidon's shapes (OP_POW5, straight-line OP_DOT shapes, chains, divisions) on the device:
    a small batch through the throughput kernel and single witnesses through the latency kernel"""
    for seed in range(24):
        rnd = random.Random(5000 + seed)
        nodes, wit, imap = util.poseidon_like_graph(rnd, rnd.choice([2, 3, 5]), rnd.choice([3, 8, 20]))
        g = cwc.Graph(po.serialize_graph(nodes, wit, imap))
        rows = [[1] + [util.random_value(rnd) if rnd.random() < 0.8 else rnd.randrange(1 << 256) for _ in range(6)] for _ in range(5)]
        inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), 7, 32)
        out = g.calc_witness_batch(inp)
        for b, row in enumerate(rows):
            want = po.evaluate(nodes, row, wit, "circom")
            assert util.unpack_u256(out[b].tobytes()) == want, (seed, b)
            if b < 2:
                lat, _ = g.calc_witness_latency(inp[b])
                assert util.unpack_u256(lat.tobytes()) == want, (seed, b, "latency")


def test_single_witness_through_batch_kernel(cwc, monkeypatch):
    monkeypatch.setenv("GW_SINGLE_MODE", "batch")
    for name in ("circuit2", "circuit5_poseidon", "circuit9_authV2"):
        assert cwc.calc_witness_wtns(util.golden_inputs(name), util.golden_graph(name)) == util.golden_wtns(name)


def test_multi_gpu_shards_host_api(cwc):
    """gw_calc_witness_batch(..., n_gpus = all visible): contiguous shards, one host thread per GPU, no collective.
    With one visible GPU this still exercises the sharding entry point (n_gpus = 1)."""
    n = cwc.device_count()
    name = "circuit7_poseidon4"
    data = util.golden_graph(name)
    nodes, wit, imap = po.deserialize_graph(data)
    g = cwc.Graph(data)
    rng = np.random.default_rng(77)
    B = 5000 + 13
    vals = util.random_field_batch(rng, (B, g.n_inputs))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    inp = vals.view(np.uint8).reshape(B, g.n_inputs, 32)
    one = g.calc_witness_batch(inp, n_gpus=1)
    many = g.calc_witness_batch(inp, n_gpus=n)
    assert (one == many).all()
    for b in sorted({0, B // n - 1, min(B // n, B - 1), B - 1}):
        assert util.unpack_u256(many[b].tobytes()) == po.evaluate(nodes, util.limbs_to_ints(vals[b]), wit)
    print(f"sharded over {n} GPU(s)")
    # gw_calc_witness_batch_on: the same call on an explicit device range (one process per GPU passes its own device)
    out = np.empty_like(one)
    g.calc_witness_batch_ptr(inp.ctypes.data, B, out.ctypes.data, n_gpus=1, first_device=n - 1)
    assert (out == one).all()
    with pytest.raises(cwc.WitnessCalcError, match="device range"):
        g.calc_witness_batch_ptr(inp.ctypes.data, B, out.ctypes.data, n_gpus=1, first_device=n)
    with pytest.raises(cwc.WitnessCalcError, match="exceeds"):
        g.calc_witness_batch(inp, n_gpus=n + 1)


def test_batch_wtns_framing_select_and_batch_cli(cwc, tmp_path):
    """SURVEY 8f: JSON Lines -> packed inputs -> .wtns images framed by the pitched D2H copy (byte-identical to the
    single-witness entry point); selected-signals graphs return exactly those witness positions; the batch CLI
    writes the same files."""
    import json
    import subprocess
    name = "circuit7_poseidon4"
    data = util.golden_graph(name)
    nodes, wit, imap = po.deserialize_graph(data)
    g = cwc.Graph(data)
    rnd = random.Random(11)
    recs = [json.loads(util.golden_inputs(name))] + [{"a": [str(rnd.randrange(po.M)) for _ in range(4)]} for _ in range(300)]
    text = "\n".join(json.dumps(r) for r in recs)
    inp = g.parse_inputs_batch(text)
    fsz = g.wtns_file_size()
    for pitch in (fsz, fsz + 52):
        files = g.calc_witness_batch_wtns(inp, pitch)
        assert files[0, :fsz].tobytes() == util.golden_wtns(name)
        for i in (1, 150, 300):
            assert files[i, :fsz].tobytes() == cwc.calc_witness_wtns(json.dumps(recs[i]), data)
        assert (files[:, fsz:] == 0).all()
    full = g.calc_witness_batch(inp)
    pos = [5, 0, g.n_witness - 1, 5, 17]
    sel = g.select(pos)
    part = sel.calc_witness_batch(inp)
    assert part.shape == (301, 5, 32) and (part == full[:, pos, :]).all()
    assert sel.calc_witness_wtns(json.dumps(recs[3]))[76:] == full[3, pos, :].tobytes()
    # batch CLI
    gp, ip, od = tmp_path / "g.bin", tmp_path / "in.jsonl", tmp_path / "out"
    gp.write_bytes(data); ip.write_text(text)
    cli = cwc.CLI_PATH + "-batch"
    r = subprocess.run([cli, str(gp), str(ip), str(od)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "301 input sets parsed" in r.stdout and "Witnesses generated in:" in r.stdout
    assert (od / "00000000.wtns").read_bytes() == util.golden_wtns(name)
    assert (od / "00000300.wtns").read_bytes() == files[300, :fsz].tobytes()
    r = subprocess.run([cli], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage:" in r.stderr


def test_stream_api_chunks_order_and_stop(cwc):
    """gw_calc_witness_batch_stream (SURVEY 8f-2 streaming D2H): the chunks handed to the consumer, reassembled, equal the
    dense host-buffer call; chunks of one GPU arrive in order and cover the batch exactly once (ragged last chunk);
    a consumer that returns nonzero stops the call with an error."""
    name = "poseidon2"
    data = util.golden_graph(name)
    g = cwc.Graph(data)
    rng = np.random.default_rng(21)
    B = 5 * 512 + 77
    vals = util.random_field_batch(rng, (B, g.n_inputs))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    inp = np.ascontiguousarray(vals.view(np.uint8).reshape(B, g.n_inputs, 32))
    dense = g.calc_witness_batch(inp)
    for chunk in (512, 0, 1, B + 5):
        if chunk == 1:
            n, src = 40, inp[:40]
        else:
            n, src = B, inp
        got = np.zeros((n, g.n_witness, 32), dtype=np.uint8)
        seen = []

        def consumer(device, first, rows, flags):
            seen.append((first, rows.shape[0]))
            got[first:first + rows.shape[0]] = rows
            assert (flags == 0).all()
            return 0
        g.calc_witness_batch_stream(src.ctypes.data, n, consumer, chunk_sets=chunk)
        assert (got == dense[:n]).all()
        assert [s[0] for s in seen] == sorted(s[0] for s in seen) and sum(s[1] for s in seen) == n
        if chunk == 512:
            assert [s[1] for s in seen] == [512] * 5 + [77]
    calls = []
    with pytest.raises(cwc.WitnessCalcError, match="stopped by the consumer"):
        g.calc_witness_batch_stream(inp.ctypes.data, B, lambda d, f, r, fl: calls.append(f) or len(calls) >= 2, chunk_sets=512)
    assert len(calls) == 2
    # all visible GPUs: every set is delivered exactly once whichever GPU computed it
    n_dev = cwc.device_count()
    if n_dev > 1:
        import threading
        lock = threading.Lock()
        got = np.zeros_like(dense)
        cover = np.zeros(B, dtype=np.int32)

        def consumer2(device, first, rows, flags):
            with lock:
                got[first:first + rows.shape[0]] = rows
                cover[first:first + rows.shape[0]] += 1
            return 0
        g.calc_witness_batch_stream(inp.ctypes.data, B, consumer2, n_gpus=n_dev, chunk_sets=256)
        assert (cover == 1).all() and (got == dense).all()


def test_device_entry_point_on_two_streams(cwc, monkeypatch):
    """gw_calc_witness_batch_device from two CUDA streams at once: the kernels of one graph share the per-device spill
    area, so the library chains them (VERDICT r01 weak 8 / ADVICE: silent corruption when they overlapped).  A tiny
    register file (GW_REGS=4) makes every launch spill heavily."""
    torch = pytest.importorskip("torch")
    monkeypatch.setenv("GW_REGS", "4")
    rnd = random.Random(77)
    nodes, wit, imap = util.random_graph(rnd, n_ops=600, ops=[0, 2, 3, 7, 8, 16, 18])
    g = cwc.Graph(po.serialize_graph(nodes, wit, imap))
    assert g.info["n_spill"] > 0
    B = 148 * 64
    rows = [[1] + [util.random_value(rnd) for _ in range(6)] for _ in range(64)]
    base = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(64, 7 * 32)
    ins = [torch.from_numpy(np.tile(np.roll(base, k, axis=0), (B // 64, 1))).cuda() for k in range(2)]
    outs = [torch.empty((B, g.n_witness * 32), dtype=torch.uint8, device="cuda") for _ in range(2)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    torch.cuda.synchronize()
    for rep in range(3):
        for k in range(2):
            g.calc_witness_batch_device(0, ins[k].data_ptr(), B, outs[k].data_ptr(), None, streams[k].cuda_stream)
    torch.cuda.synchronize()
    want = [po.evaluate(nodes, r, wit, "circom") for r in rows]
    for k in range(2):
        got = outs[k].cpu().numpy().reshape(B, g.n_witness, 32)
        order = np.roll(np.arange(64), k)
        for b in list(range(64)) + [B - 1, B - 33, 4097]:
            assert util.unpack_u256(got[b].tobytes()) == want[order[b % 64]], (k, b)
        # every tile of 64 rows is identical: a corrupted spill slot anywhere shows up
        assert (got.reshape(B // 64, 64, -1) == got[:64].reshape(1, 64, -1)).all()


def test_set_device_and_graph_cache(cwc):
    """gw_set_device selects the GPU of the single-witness entry points; the graph cache of gw_calc_witness compares
    bytes, so two graphs of equal length never alias."""
    n = cwc.device_count()
    with pytest.raises(cwc.WitnessCalcError):
        cwc.set_device(n)
    cwc.set_device(n - 1)
    try:
        assert cwc.calc_witness_wtns(util.golden_inputs("circuit1"), util.golden_graph("circuit1")) == util.golden_wtns("circuit1")
    finally:
        cwc.set_device(0)
    a = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_CONST, 7), (po.K_DUO, po.DUO["Add"], 1, 2)]
    b = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_CONST, 9), (po.K_DUO, po.DUO["Add"], 1, 2)]
    ga, gb = (po.serialize_graph(x, [0, 3], {"a": (1, 1)}) for x in (a, b))
    assert len(ga) == len(gb)
    for _ in range(2):
        assert cwc.calc_witness('{"a": "5"}', ga) == [1, 12]
        assert cwc.calc_witness('{"a": "5"}', gb) == [1, 14]


def test_bitsliced_path_boolean_graphs_and_fallback(cwc, monkeypatch):
    """Boolean graphs run bit-sliced (csrc/bitplan.cpp: 32 input sets per word, lane = LUT instruction); the plan is typed
    under the contract "inputs are bits", which the kernel checks per input set: the sets that break it are evaluated by
    the generic kernel in the same call.  Every row must equal the oracle whichever path produced it, flags included."""
    from tests.test_bitplan import boolean_graph
    rnd = random.Random(99)
    for t in range(6):
        n_in = rnd.choice([5, 24, 70])
        nodes, wit, imap = boolean_graph(rnd, n_inputs=n_in, n_gates=rnd.choice([60, 300]))
        data = po.serialize_graph(nodes, wit, imap)
        g = cwc.Graph(data)
        B = rnd.choice([1, 31, 32, 33, 200, 1029])
        rows = [[1] + [rnd.randrange(2) for _ in range(n_in)] for _ in range(B)]
        bad = set(rnd.sample(range(B), min(B, rnd.choice([0, 1, 9])))) if t else set()
        for b in bad:
            rows[b][1 + rnd.randrange(n_in)] = rnd.choice([2, po.M - 1, rnd.randrange(po.M), 1 << 255])
        inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(B, n_in + 1, 32)
        out, flags = g.calc_witness_batch(inp, want_flags=True)
        for b in sorted(set(range(0, B, max(1, B // 24))) | bad | {B - 1}):
            assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, rows[b], wit, "circom"), (t, b, b in bad)
        assert (flags[[b for b in range(B) if b not in bad]] == 0).all()
        # the generic kernel alone gives the same bytes
        monkeypatch.setenv("GW_BITSLICE", "0")
        g0 = cwc.Graph(data)
        monkeypatch.delenv("GW_BITSLICE")
        assert (g0.calc_witness_batch(inp) == out).all(), t


def test_bitsliced_sha256_bits_and_field_inputs(cwc):
    """SHA-256(512) through the bit-sliced path: digests against hashlib, rows with non-bit inputs (the generic kernel
    takes them) against the C oracle, all in one batch with a ragged last group."""
    import hashlib
    from oracle import cref
    name = "circuit8_sha256_512"
    data = util.golden_graph(name)
    g = cwc.Graph(data)
    rng = np.random.default_rng(88)
    B = 32 * 9 + 5
    inp = np.zeros((B, g.n_inputs, 32), dtype=np.uint8)
    inp[:, :, 0] = rng.integers(0, 2, size=(B, g.n_inputs), dtype=np.uint8)
    inp[:, 0, 0] = 1
    field_rows = [7, 64, 65, B - 1]
    vals = util.random_field_batch(rng, (len(field_rows), g.n_inputs)).view(np.uint8).reshape(len(field_rows), g.n_inputs, 32)
    for k, b in enumerate(field_rows):
        inp[b, 1:] = vals[k, 1:]
    out = g.calc_witness_batch(inp)
    for b in (0, 1, 31, 32, 100, B - 2):
        bits = inp[b, 1:513, 0]
        msg = bytes(int("".join(str(int(x)) for x in bits[8 * i:8 * i + 8]), 2) for i in range(64))
        dg = out[b, 1:257, 0]
        assert bytes(int("".join(str(int(x)) for x in dg[8 * i:8 * i + 8]), 2) for i in range(32)) == hashlib.sha256(msg).digest(), b
    rows = field_rows + [0, 8, 63, 66]
    want = cref.CGraph(data).evaluate_batch(inp[rows], 4)
    assert (out[rows] == want).all()


def test_bitsliced_field_inputs_wide_values_and_num2bits(cwc, monkeypatch):
    """Field inputs that a graph only takes apart (Num2Bits: Shr + Band) carry no contract on the bit-sliced path: their
    planes are the bits of the value reduced mod M (Fr::new, graph.rs:376), whatever the caller passes (0, M - 1, M,
    2^256 - 1 ...); witness values that are integers of several bits (Bits2Num sums, the inputs themselves) are assembled
    from their planes by bit_expand_wide_kernel.  Every row against the oracle, and against the generic kernel."""
    from tests.test_bitplan import field_bits_graph
    rnd = random.Random(707)
    M = po.M
    for t in range(6):
        n_field, n_bits = rnd.choice([1, 3]), rnd.choice([0, 6])
        nodes, wit, imap = field_bits_graph(rnd, n_field, n_bits)
        data = po.serialize_graph(nodes, wit, imap)
        g = cwc.Graph(data)
        B = rnd.choice([1, 33, 200, 1029])
        rows = []
        for _ in range(B):
            fv = [rnd.choice([0, 1, M - 1, M, M + 5, (1 << 256) - 1, 1 << 253, rnd.randrange(M), rnd.randrange(1 << 256)]) for _ in range(n_field)]
            rows.append([1] + fv + [rnd.randrange(2) for _ in range(n_bits)])
        bad = set()
        if n_bits and B > 8:
            bad = {7, B - 1}
            for b in bad:
                rows[b][n_field + 1] = rnd.choice([9, M - 1])
        inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(B, len(rows[0]), 32)
        out, flags = g.calc_witness_batch(inp, want_flags=True)
        for b in sorted(set(range(0, B, max(1, B // 24))) | bad | {B - 1}):
            assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, rows[b], wit, "circom"), (t, b, b in bad)
        assert (flags[[b for b in range(B) if b not in bad]] == 0).all()
        monkeypatch.setenv("GW_BITSLICE", "0")
        g0 = cwc.Graph(data)
        monkeypatch.delenv("GW_BITSLICE")
        assert (g0.calc_witness_batch(inp) == out).all(), t
    # circuit6 (Num2Bits(256)... of one field input + Bits2Num): pure wiring on the bit path; arbitrary 256-bit inputs
    name = "circuit6_num2bits"
    data = util.golden_graph(name)
    nodes, wit, _ = po.deserialize_graph(data)
    g = cwc.Graph(data)
    rng = np.random.default_rng(66)
    B = 32 * 41 + 3
    vals = rng.integers(0, 1 << 64, size=(B, g.n_inputs, 4), dtype=np.uint64)     # arbitrary 256-bit values, mostly >= M
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    vals[0, 1:, :] = 0
    vals[1, 1:, :] = np.uint64(0xFFFFFFFFFFFFFFFF)
    vals[2::3, 1:, 3] &= np.uint64((1 << 61) - 1)                                    # a third of them below M
    inp = vals.view(np.uint8).reshape(B, g.n_inputs, 32)
    out = g.calc_witness_batch(inp)
    for b in list(range(0, B, 97)) + [1, B - 1]:
        assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, util.limbs_to_ints(vals[b]), wit, "circom"), b
    monkeypatch.setenv("GW_BITSLICE", "0")
    g0 = cwc.Graph(data)
    monkeypatch.delenv("GW_BITSLICE")
    assert (g0.calc_witness_batch(inp) == out).all()


def test_bit_contract_speculation_is_dropped_when_inputs_are_field_elements(cwc):
    """A Boolean graph fed field elements: every set breaks the contract and is evaluated by the generic kernel; after the
    first such launch the engine stops speculating for this graph (both paths would be paid).  Results stay exact."""
    from tests.test_bitplan import boolean_graph
    rnd = random.Random(11)
    nodes, wit, imap = boolean_graph(rnd, n_inputs=24, n_gates=300)
    g = cwc.Graph(po.serialize_graph(nodes, wit, imap))
    B = 256
    for rep in range(3):
        rows = [[1] + [rnd.randrange(po.M) for _ in range(24)] for _ in range(B)]
        inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(B, 25, 32)
        out = g.calc_witness_batch(inp)
        for b in range(0, B, 37):
            assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, rows[b], wit, "circom"), (rep, b)
    rows = [[1] + [rnd.randrange(2) for _ in range(24)] for _ in range(B)]
    inp = np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(B, 25, 32)
    out = g.calc_witness_batch(inp)
    for b in range(0, B, 37):
        assert util.unpack_u256(out[b].tobytes()) == po.evaluate(nodes, rows[b], wit, "circom"), b


def test_latency_mode_boolean_graph_uses_bit_plan_and_falls_back(cwc):
    """Single witness of a Boolean graph: the bit-sliced plan is the level-parallel plan (one LUT node per lane); an input
    set that breaks the bit contract is evaluated by the generic latency kernel in the same call.  Flags included."""
    from tests.test_bitplan import boolean_graph
    rnd = random.Random(515)
    for t in range(4):
        n_in = rnd.choice([5, 24])
        nodes, wit, imap = boolean_graph(rnd, n_inputs=n_in, n_gates=200)
        g = cwc.Graph(po.serialize_graph(nodes, wit, imap))
        assert g.info["bit_eligible"] == 1
        for broken in (False, True, False):
            row = [1] + [rnd.randrange(2) for _ in range(n_in)]
            if broken:
                row[1 + rnd.randrange(n_in)] = rnd.choice([2, po.M - 1, rnd.randrange(po.M)])
            out, ms = g.calc_witness_latency(np.frombuffer(util.pack_u256(row), dtype=np.uint8).reshape(n_in + 1, 32))
            assert util.unpack_u256(out.tobytes()) == po.evaluate(nodes, row, wit, "circom"), (t, broken)


def test_dataflow_watchdog_turns_a_stuck_wait_into_an_error_and_a_fallback(tmp_path):
    """A wait that no packet satisfies (injected in the -DGW_PROFILING build of the library: GW_LAT_DBG=8) must not hang the
    GPU: the kernel's watchdog ends it, gw_calc_witness_latency reports it, and the drop-in gw_calc_witness falls back to
    the throughput kernel and still returns the right .wtns."""
    import subprocess
    import sys
    prof = os.path.join(util.ROOT, "circom-witnesscalc_b200", "lib_variants", "libcwc_prof.so")
    if not os.path.exists(prof):
        pytest.skip("profiling build of the library not present")
    code = r'''
import importlib, sys
sys.path.insert(0, %r)
import numpy as np
from tests import util
from tests.util import po
cwc = importlib.import_module("circom-witnesscalc_b200")
name = "circuit5_poseidon"
data = util.golden_graph(name)
nodes, wit, imap = po.deserialize_graph(data)
g = cwc.Graph(data)
buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs(name)))
try:
    g.calc_witness_latency(np.frombuffer(util.pack_u256(buf), dtype=np.uint8).reshape(g.n_inputs, 32))
    print("NO-ERROR")
except cwc.WitnessCalcError as e:
    print("ERR", e)
print("WTNS-OK" if cwc.calc_witness_wtns(util.golden_inputs(name), data) == util.golden_wtns(name) else "WTNS-BAD")
''' % util.ROOT
    env = dict(os.environ, GW_LIB_PATH=prof, GW_LAT_DBG="8", GW_LAT_WATCHDOG="262144", GW_LAT_WARPS="3")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert "ERR" in r.stdout and "watchdog" in r.stdout, r.stdout + r.stderr
    assert "WTNS-OK" in r.stdout, r.stdout + r.stderr
