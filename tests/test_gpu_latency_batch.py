"""The latency kernels in batch form (gw_calc_witness_latency_batch, _device): one latency CTA per input set, row by row
against the C oracle and the single-witness call.

CTA b of a batch launch evaluates input set b (or row_map[b] for the sets a Boolean graph's bit-sliced launch hands back)
and offsets its input row, witness row and flag word by it; nothing else differs from the single call.  So the tests look for
what only a batch can get wrong: a CTA that reads or writes its neighbour's row (batches of pairwise different rows at one
and two resident CTAs per SM and with a tail wave), flag words that are not cleared or land on the wrong set, the
Boolean-graph fallback rows at the edges of a 32-set group, the host staging split into whole waves, and the ordering of a
device call behind the caller's stream."""
import ctypes
import importlib
import os
import random
import re

import numpy as np
import pytest

from oracle import cref
from tests import r1cs_ref, util
from tests.util import po
from tools import r1cs_gen

pytestmark = pytest.mark.gpu

ENV_KEYS = util.LATENCY_ENV_KEYS + ("GW_BITSLICE", "GW_DEVICE", "GW_CHUNK_MB", "GW_TRACE_HOST")
TRACE = re.compile(r"\[gw trace\] device (\d+): (\d+) sets, chunk (\d+):")


@pytest.fixture(scope="module")
def cwc():
    mod = importlib.import_module("circom-witnesscalc_b200")
    assert mod.device_count() >= 1, "no CUDA device visible"
    return mod


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture
def env(monkeypatch):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)

    def set_env(d):
        for k in ENV_KEYS:
            monkeypatch.delenv(k, raising=False)
        for k, v in d.items():
            monkeypatch.setenv(k, v)
    return set_env


def _pack(rows):
    return np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32)


def _oracle(data, inp):
    return cref.CGraph(data).evaluate_batch(np.ascontiguousarray(inp), os.cpu_count() or 4).reshape(len(inp), -1, 32)


def _assert_rows(name, got, want, what=""):
    got, want = got.reshape(len(want), -1, 32), want.reshape(len(want), -1, 32)
    bad = np.nonzero((got != want).any(axis=2).any(axis=1))[0]
    assert len(bad) == 0, f"{name} {what}: {len(bad)} wrong rows of {len(want)}, first {bad[:8].tolist()}"


def _sms(torch):
    return int(torch.cuda.get_device_properties(0).multi_processor_count)


# ---- 1. the latency corpus under every latency option, all rows in one batch call -------------------------------------
@pytest.fixture(scope="module")
def corpus():
    out = []
    for name, nodes, wit, imap, rows in util.latency_corpus():
        data = po.serialize_graph(nodes, wit, imap)
        inp = _pack(rows)
        sim = util.SimGraph(data, **util.sim_options({}))
        out.append((name, data, rows, inp, _oracle(data, inp), [sim.eval(r)[1] for r in rows], sim))
    return out


@pytest.mark.parametrize("variant", [name for name, _ in util.LATENCY_VARIANTS])
def test_corpus_under_latency_option(cwc, env, corpus, variant):
    """every graph of the latency corpus in one batch call under one latency option: witness rows equal the oracle's, flag
    words the simulator's, and both what the single call gives row by row; a graph the simulator finds too wide gets the
    single call's error"""
    e = dict(util.LATENCY_VARIANTS)[variant]
    opts = util.latency_sim_options(e)
    for name, data, rows, inp, want, want_flags, sim in corpus:
        env(e)
        try:
            sim.eval_latency(rows[0], **opts)
            wide = False
        except ValueError as err:
            assert "too wide" in str(err), (name, str(err))
            wide = True
        g = cwc.Graph(data)
        if wide:
            with pytest.raises(cwc.WitnessCalcError, match="latency plan: graph is too wide"):
                g.calc_witness_latency_batch(inp)
            g.close()
            continue
        out, flags = g.calc_witness_latency_batch(inp, want_flags=True)
        _assert_rows(name, out, want, variant)
        assert flags.tolist() == want_flags, f"{name} {variant}: flags {flags.tolist()} != {want_flags}"
        for b in range(len(rows)):
            one, fl = g.calc_witness_latency(inp[b], want_flags=True)
            assert np.array_equal(one, out[b]) and fl == int(flags[b]), f"{name} {variant} row {b}: batch != single call"
        g.close()


# ---- 2. batch sizes around one and two resident CTAs per SM and a tail wave --------------------------------------------
@pytest.mark.parametrize("mode", ["dataflow", "level"])
def test_batch_size_edges(cwc, env, torch, mode):
    """a small graph (two CTAs fit an SM) at n = 1, S - 1, S, S + 1, 2 S + 1 and 4 S + 3 for S SMs, on pairwise different
    rows: a CTA that read or wrote its neighbour's row would show"""
    env({"GW_LAT_MODE": "level"} if mode == "level" else {})
    rnd = random.Random(1701)
    nodes, wit, imap = util.poseidon_like_graph(rnd, t=3, rounds=8, n_inputs=6)
    data = po.serialize_graph(nodes, wit, imap)
    S = _sms(torch)
    n_max = 4 * S + 3
    rows = [[1] + [rnd.randrange(util.M) for _ in range(6)] for _ in range(n_max)]
    inp = _pack(rows)
    want = _oracle(data, inp)
    assert len({w.tobytes() for w in want}) == n_max, "rows must give pairwise different witnesses"
    sim = util.SimGraph(data, **util.sim_options({}))
    want_flags = [sim.eval(r)[1] for r in rows]
    g = cwc.Graph(data)
    for n in (1, S - 1, S, S + 1, 2 * S + 1, 4 * S + 3):
        lo = (n * 7) % (n_max - n + 1)                 # a different stretch of rows for every n
        out, flags = g.calc_witness_latency_batch(inp[lo:lo + n], want_flags=True)
        _assert_rows("poseidon_like", out, want[lo:lo + n], f"{mode} n={n}")
        assert flags.tolist() == want_flags[lo:lo + n], f"{mode} n={n}: flags"
    g.close()


# ---- 3. Boolean graphs: the bit-sliced launch and its fallback rows ------------------------------------------------------
def _bit_graphs():
    out = [("sha256_512", util.golden_graph("circuit8_sha256_512"))]
    for name, data in util.bit_corpus():
        if name != "sha256_512" and util.BitSimGraph(data).info["n_luts"] > 0:
            out.append((name, data))
    return out


@pytest.mark.parametrize("lat_bit", ["1", "0"])
def test_boolean_graphs(cwc, env, lat_bit):
    """Boolean graphs with LUTs under GW_LAT_BIT = 1 (bit-sliced, then the contract-breaking sets through the latency kernels
    via row_map) and 0 (latency kernels throughout): breaking sets at 0, 31, 32 and the last set, then all, then none"""
    env({"GW_LAT_BIT": lat_bit})
    rnd = random.Random(88)
    n = 70
    for name, data in _bit_graphs():
        bs = util.BitSimGraph(data)
        contract = [int(i) for i, _, b in bs.plan()["inputs"] if b == util.BIT_CONTRACT]
        field = sorted({int(i) for i, _, b in bs.plan()["inputs"] if b != util.BIT_CONTRACT})
        base = []
        for _ in range(n):
            r = [1] + [rnd.randrange(2) for _ in range(bs.I - 1)]
            for i in field:
                r[i] = util.random_value(rnd)
            base.append(r)
        patterns = [("none", [])]
        if contract:
            patterns = [("edges", [0, 31, 32, n - 1]), ("all", list(range(n)))] + patterns
        g = cwc.Graph(data)
        sim = util.SimGraph(data, **util.sim_options({}))
        for what, breaking in patterns:
            rows = [list(r) for r in base]
            for b in breaking:
                rows[b][contract[b % len(contract)]] = rnd.choice([2, util.M - 1, (1 << 256) - 1])
            inp = _pack(rows)
            out, flags = g.calc_witness_latency_batch(inp, want_flags=True)
            _assert_rows(name, out, _oracle(data, inp), f"GW_LAT_BIT={lat_bit} {what}")
            assert flags.tolist() == [sim.eval(r)[1] for r in rows], f"{name} GW_LAT_BIT={lat_bit} {what}: flags"
        g.close()


# ---- 4. golden graphs --------------------------------------------------------------------------------------------------
def test_golden_graphs(cwc, env):
    """every golden graph with its golden input, five times in one batch: each row is the golden .wtns payload"""
    names = sorted(f[:-len(".bin.xz")] for f in os.listdir(os.path.join(util.GOLDEN, "graphs")) if f.endswith(".bin.xz"))
    assert len(names) == 14, names
    for name in names:
        g = cwc.Graph(util.golden_graph(name))
        row = g.parse_inputs_batch("[" + util.golden_inputs(name) + "]")
        inp = np.repeat(row, 5, axis=0)
        out = g.calc_witness_latency_batch(inp)
        payload = util.golden_wtns(name)[76:]
        for b in range(5):
            assert out[b].tobytes() == payload, f"{name} row {b}"
        g.close()


def test_authv2_more_than_a_wave(cwc, env, torch):
    """authV2 (one CTA per SM) on S + 5 seeded rows: more than one wave, every row against the C oracle"""
    data = util.golden_graph("circuit9_authV2")
    g = cwc.Graph(data)
    rng = np.random.default_rng(9)
    n = _sms(torch) + 5
    vals = util.random_field_batch(rng, (n, g.n_inputs))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    inp = vals.view(np.uint8).reshape(n, g.n_inputs, 32)
    _assert_rows("authV2", g.calc_witness_latency_batch(inp), _oracle(data, inp), "seeded rows")
    g.close()


# ---- 5. device buffers -------------------------------------------------------------------------------------------------
def test_device_stream_and_r1cs(cwc, env, torch):
    """on a non-default stream right behind a kernel that writes the inputs there, with and without d_flags; the witness
    rows are checked on the same stream by gw_r1cs_check_batch_device"""
    rnd = random.Random(31)
    gb, r = r1cs_gen.poseidon_pair(rnd, n_hashes=1)
    g, rc = cwc.Graph(gb), cwc.R1cs(r1cs_ref.serialize_r1cs(r))
    n = 300
    rows = [[1] + [rnd.randrange(util.M) for _ in range(g.n_inputs - 1)] for _ in range(n)]
    inp = _pack(rows)
    want = _oracle(gb, inp)
    want_ff = rc.check_batch(want)
    src = torch.from_numpy(inp.reshape(-1).copy()).cuda()
    s = torch.cuda.Stream()
    for with_flags in (True, False):
        d_in = torch.zeros(n * g.n_inputs * 32, dtype=torch.uint8, device="cuda")
        d_w = torch.full((n, g.n_witness * 32), 0xA5, dtype=torch.uint8, device="cuda")
        d_fl = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        d_ff = torch.zeros(n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(20_000_000)                  # the inputs land late on s: the call must wait for them
            d_in.copy_(src)
            g.calc_witness_latency_batch_device(0, d_in.data_ptr(), n, d_w.data_ptr(), d_fl.data_ptr() if with_flags else None,
                                                s.cuda_stream)
            rc.check_batch_device(0, d_w.data_ptr(), n, d_ff.data_ptr(), 0, s.cuda_stream)
        s.synchronize()
        _assert_rows("poseidon_pair", d_w.cpu().numpy(), want, f"device, flags={with_flags}")
        assert np.array_equal(d_ff.cpu().numpy().view(np.uint32), want_ff)
        fl = d_fl.cpu().numpy().view(np.uint32)
        assert (fl == 0).all() if with_flags else (fl == 0xFFFFFFFF).all()
    g.close()
    rc.close()


# ---- 6. call sequences, selections, chunks and devices -----------------------------------------------------------------
def _small_case(seed=4):
    rnd = random.Random(seed)
    nodes, wit, imap = util.poseidon_like_graph(rnd, t=3, rounds=8, n_inputs=6)
    data = po.serialize_graph(nodes, wit, imap)
    inp = _pack([util.matrix_row(rnd, 6) for _ in range(601)])
    return data, inp, _oracle(data, inp)


def test_call_sequence(cwc, env):
    """single latency call, latency batch, throughput batch and latency batch again on one Graph"""
    data, inp, want = _small_case()
    g = cwc.Graph(data)
    one, _ = g.calc_witness_latency(inp[0])
    _assert_rows("seq", one[None], want[:1], "single call")
    _assert_rows("seq", g.calc_witness_latency_batch(inp[:300]), want[:300], "latency batch")
    _assert_rows("seq", g.calc_witness_batch(inp[100:]), want[100:], "throughput batch")
    _assert_rows("seq", g.calc_witness_latency_batch(inp[1:]), want[1:], "latency batch again")
    g.close()


def test_selection_chunks_and_devices(cwc, env, capfd):
    """a gw_graph_select handle (some positions, none), a host call split into several chunks by a small GW_CHUNK_MB, an empty
    batch, and n_gpus = 2 / the second device"""
    data, inp, want = _small_case(5)
    g = cwc.Graph(data)
    pos = [3, 0, 7, 7, g.n_witness - 1]
    sel = g.select(pos)
    _assert_rows("select", sel.calc_witness_latency_batch(inp[:200]), want[:200, pos], "selection")
    empty = g.select([])
    out, flags = empty.calc_witness_latency_batch(inp[:50], want_flags=True)
    assert out.shape == (50, 0, 32) and (flags == 0).all()
    assert g.calc_witness_latency_batch(inp[:0]).shape == (0, g.n_witness, 32)
    env({"GW_CHUNK_MB": "1", "GW_TRACE_HOST": "1"})
    capfd.readouterr()
    _assert_rows("chunks", g.calc_witness_latency_batch(inp), want, "GW_CHUNK_MB=1")
    tr = [tuple(int(x) for x in m) for m in TRACE.findall(capfd.readouterr().err)]
    assert len(tr) == 1 and tr[0][1] == len(inp) and tr[0][2] < len(inp), f"meant several chunks: {tr}"
    env({})
    if cwc.device_count() >= 2:
        _assert_rows("shards", g.calc_witness_latency_batch(inp, n_gpus=2), want, "n_gpus=2")
        _assert_rows("device 1", g.calc_witness_latency_batch(inp[:77], first_device=1), want[:77], "first_device=1")
    for h in (sel, empty, g):
        h.close()


def test_cabi_arguments(cwc):
    """null arguments are refused before any device is touched; n_sets = 0 does nothing"""
    st = cwc.gw_status_t()
    assert cwc._L.gw_calc_witness_latency_batch(None, 0, 1, None, 0, None, None, ctypes.byref(st)) == 1
    cwc._check(0, st)
    g = cwc.Graph(util.golden_graph("circuit5_poseidon"))
    assert cwc._L.gw_calc_witness_latency_batch(g._h, 0, 1, None, 0, None, None, ctypes.byref(st)) == 0
    assert cwc._L.gw_calc_witness_latency_batch_device(g._h, 0, None, 0, None, None, None, ctypes.byref(st)) == 0
    assert cwc._L.gw_calc_witness_latency_batch_device(g._h, 0, None, 3, None, None, None, ctypes.byref(st)) == 1
    cwc._check(0, st)
    g.close()
