"""The host-memory entry points on the GPU: the orchestration around the kernels, row by row against plain references.

gw_calc_witness_batch / _on / _wtns / _check / _stream and gw_r1cs_check_batch / _abc_batch / _quotient_batch cut a batch
into chunks, stage them through two device buffers on two streams (and a three-slot pinned ring for the stream), copy
results to per-chunk offsets of the caller's buffers (2-D copies where a pitch is given), shard the batch over GPUs and
reuse or regrow their staging from call to call.  A mistake there puts right bytes in the wrong row or takes verdicts and
flags from the other buffer, so every batch here is tiled from a pool of distinct rows whose results differ (flagged
sets, sets that break the bit contract, sets that fail the R1CS), with such rows on the first and last set of every chunk
and every shard, and the expected results are computed once per distinct row: witness rows by the C oracle, flags by
the plan simulator, verdicts by tests/r1cs_ref.check_r1cs, A/B/C and h by tests/r1cs_abc_ref and r1cs_quotient_ref.
Output padding is filled with canary bytes that must survive.  The chunk schedule each call used is read back from
GW_TRACE_HOST and compared with the one the test meant to run."""
import ctypes
import importlib
import math
import os
import random
import re
import struct
import threading
import time

import numpy as np
import pytest

from oracle import cref
from tests import r1cs_abc_ref as abc_ref
from tests import r1cs_quotient_ref as qref
from tests import r1cs_ref as ref
from tests import util
from tests.test_bitplan import boolean_graph
from tests.test_gpu_bit_matrix import BAD_VALUES, contract_inputs
from tests.test_gpu_plan_matrix import _flag_graph
from tests.util import po
from tools import r1cs_gen

pytestmark = pytest.mark.gpu

M = util.M
OK = 0xFFFFFFFF
CANARY = 0xA5
FLAG_CANARY = 0xDEADBEEF
ENV_KEYS = ("GW_CHUNK_MB", "GW_TRACE_HOST", "GW_STREAM_CHUNK_MB", "GW_THREADS", "GW_BITSLICE", "GW_BIT_MIN_SETS", "GW_SINGLE_MODE",
            "GW_LAT_BIT", "GW_DEVICE")
TRACE = re.compile(r"\[gw trace\] device (\d+): (\d+) sets, chunk (\d+)")
BIT_TRACE = re.compile(r"\[gw bit\] variant")
SCHEDULES = ("0", "1", "default")          # GW_CHUNK_MB: one set per chunk, 1 MiB per staging buffer, unset
R1CS_B = 4101                              # >= 4096 sets: R1cs::host_rows_on cuts four chunks, the last one ragged


@pytest.fixture(scope="module")
def cwc():
    mod = importlib.import_module("circom-witnesscalc_b200")
    assert mod.device_count() >= 1, "no CUDA device visible"
    return mod


@pytest.fixture
def env(monkeypatch):
    for k in ENV_KEYS:
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setenv("GW_TRACE_HOST", "1")

    def set_env(**kv):
        for k, v in kv.items():
            if v is None:
                monkeypatch.delenv(k, raising=False)
            else:
                monkeypatch.setenv(k, str(v))
    return set_env


def _pack(rows):
    return np.frombuffer(b"".join(util.pack_u256(r) for r in rows), dtype=np.uint8).reshape(len(rows), -1, 32)


def _wtns_header(W):
    """the 76 bytes in front of a .wtns v2 file's values: magic, version, 2 sections, header section (n8, prime, W), values"""
    return (b"wtns" + struct.pack("<II", 2, 2) + struct.pack("<IQ", 1, 40) + struct.pack("<I", 32) + M.to_bytes(32, "little")
            + struct.pack("<I", W) + struct.pack("<IQ", 2, 32 * W))


def _traces(capfd):
    """(chunk traces (device, sets, chunk), number of bit-sliced launches) of the calls since the last read"""
    err = capfd.readouterr().err
    return [tuple(int(x) for x in m) for m in TRACE.findall(err)], len(BIT_TRACE.findall(err))


def chunk_edges(B, chunk_of, n_gpus=1):
    """the first and the last set of every chunk of every shard; shard g is [B g / n, B (g + 1) / n) and is cut into chunks
    of chunk_of(shard size) sets"""
    e = set()
    for g in range(n_gpus):
        lo, hi = B * g // n_gpus, B * (g + 1) // n_gpus
        if hi == lo:
            continue
        c = chunk_of(hi - lo)
        for off in range(lo, hi, c):
            e |= {off, min(off + c, hi) - 1}
    return e


class Kind:
    """a graph, a pool of distinct input rows, the oracle's witness rows and the simulator's flags of the pool, and the
    pool rows that go on chunk and shard edges (`marked`: flagged, failing the R1CS, or breaking the bit contract)"""

    def __init__(self, name, data, rows, marked=None, r1cs=None):
        self.name, self.data, self.r1cs = name, data, r1cs
        self.inp = _pack(rows)
        self.P, self.I = self.inp.shape[0], self.inp.shape[1]
        want = cref.CGraph(data).evaluate_batch(self.inp, os.cpu_count() or 4)
        self.W = want.size // (self.P * 32)
        self.want = want.reshape(self.P, self.W * 32)
        sim = util.SimGraph(data, **util.sim_options({}))
        self.flags = np.array([sim.eval(r)[1] for r in rows], dtype=np.uint32)
        if r1cs is not None:
            self.verdict = np.array([_verdict(r1cs, util.unpack_u256(w.tobytes())) for w in self.want], dtype=np.uint32)
        if marked is None:
            marked = np.nonzero(self.verdict != OK)[0] if r1cs is not None else np.nonzero(self.flags)[0]
        self.marked = np.asarray(marked)
        assert 0 < len(self.marked) < self.P, self.name

    def tile(self, B, edges=()):
        """pool row of every set: (7 b + 3) mod P, and marked rows on the given sets"""
        idx = (np.arange(B, dtype=np.int64) * 7 + 3) % self.P
        for j, b in enumerate(sorted(e for e in edges if 0 <= e < B)):
            idx[b] = self.marked[j % len(self.marked)]
        return idx

    def host_chunk(self, B, mb):
        """the chunk Engine::run_host_on cuts a batch of B sets into under GW_CHUNK_MB = mb (a device with room to spare)"""
        if mb == "0":
            return 1
        c = (1 << 20) // ((self.I + self.W) * 32) if mb == "1" else B
        if B >= 4 * 2048:
            c = min(c, (B + 3) // 4)
        return max(min(c, B), 1)

    def check_rows(self, idx, rows, flags=None, what=""):
        B = len(idx)
        rows = rows.reshape(B, self.W * 32)
        bad = np.nonzero((rows != self.want[idx]).any(axis=1))[0]
        assert len(bad) == 0, f"{self.name} {what} B={B}: {len(bad)} wrong witness rows, first {bad[:8].tolist()}"
        if flags is not None:
            badf = np.nonzero(flags != self.flags[idx])[0]
            assert len(badf) == 0, f"{self.name} {what} B={B}: wrong flags in sets {badf[:8].tolist()}: {flags[badf[:4]]} != {self.flags[idx][badf[:4]]}"

    def check_files(self, idx, files, pitch, flags=None, what=""):
        """.wtns files at the given pitch: header, values, then canary bytes up to the pitch"""
        B, end = len(idx), 76 + self.W * 32
        assert files.shape == (B, pitch)
        hb = np.nonzero((files[:, :76] != np.frombuffer(_wtns_header(self.W), np.uint8)).any(axis=1))[0]
        assert len(hb) == 0, f"{self.name} {what} pitch {pitch}: wrong .wtns header in files {hb[:8].tolist()}"
        self.check_rows(idx, np.ascontiguousarray(files[:, 76:end]), flags, f"{what} pitch {pitch}")
        cb = np.nonzero((files[:, end:] != CANARY).any(axis=1))[0]
        assert len(cb) == 0, f"{self.name} {what} pitch {pitch}: padding overwritten in files {cb[:8].tolist()}"


def _verdict(r1cs, w):
    k = ref.check_r1cs(r1cs, w)
    return OK if k is None else k


def _bool_kind(rnd):
    """a Boolean graph the bit-sliced path runs; one pool row in eight breaks the bit contract on one input (those sets go
    to the generic kernel in the same launch)"""
    for _ in range(20):
        nodes, wit, imap = boolean_graph(rnd, n_inputs=24, n_gates=300)
        data = po.serialize_graph(nodes, wit, imap)
        s = util.BitSimGraph(data)
        if s.info["eligible"] and s.info["n_luts"]:
            break
    else:
        raise AssertionError("no bit-eligible graph")
    con, fld, n_in = contract_inputs(data)
    assert con and not fld
    rows, bad = [], []
    for b in range(509):
        r = [1] + [rnd.randrange(2) for _ in range(n_in - 1)]
        if b % 8 == 5:
            r[con[(b * 5) % len(con)]] = BAD_VALUES[len(bad) % len(BAD_VALUES)]
            bad.append(b)
        rows.append(r)
    return Kind("boolean", data, rows, marked=bad)


def _r1cs_kind(name, pair, n_in, rnd, pool=127):
    """a generated (graph, R1CS) pair with x1 (x1 - 1) = 0 and x2 (x2 - 1) = 0 appended on two graph inputs, and three public
    signals: a set fails exactly when x1 or x2 is not a bit"""
    g, r = pair
    cons = list(r["constraints"]) + [([(w, 1)], [(w, 1), (0, M - 1)], []) for w in (1, 2)]
    r = dict(r, constraints=cons, n_pub_out=1, n_pub_in=2)
    rows = []
    for b in range(pool):
        x = [rnd.randrange(M) for _ in range(n_in)]
        x[0], x[1] = rnd.randrange(2), rnd.randrange(2)
        if b % 3 == 1:
            x[b % 2] = rnd.choice([2, M - 1, rnd.randrange(M)])
        rows.append([1] + x)
    k = Kind(name, g, rows, r1cs=r)
    assert set(k.verdict[k.marked].tolist()) <= {len(cons) - 2, len(cons) - 1}
    return k


@pytest.fixture(scope="module")
def kinds():
    rnd = random.Random(606)                   # the flag graph of test_gpu_plan_matrix's launch shapes
    nodes, wit, imap = _flag_graph(rnd)
    flags = Kind("flags", po.serialize_graph(nodes, wit, imap), [util.matrix_row(rnd, 6) for _ in range(509)])
    rnd = random.Random(7321)
    assert len(set(flags.flags.tolist())) > 2, "the flag graph must flag some sets and not others"
    out = {"flags": flags, "boolean": _bool_kind(rnd),
           "random": _r1cs_kind("random", r1cs_gen.random_pair(rnd, n_constraints=120), 6, rnd),
           "poseidon": _r1cs_kind("poseidon", r1cs_gen.poseidon_pair(rnd, n_hashes=1), 4, rnd)}
    out["flags"].nodes = (nodes, wit, imap)
    return out


def _batch(B, schedule):
    """batch sizes of a schedule: 1, 2, 3, chunk - 1, chunk + 1 and four chunks and a ragged tail"""
    if schedule == "default":
        return (1, 2, 3, 4 * 2048 - 1, 4 * 2048 + 3)       # one chunk; then chunks of 2049, 2049, 2049, 2048
    c = B
    return tuple(sorted({b for b in (1, 2, 3, c - 1, c + 1, 4 * c + c // 3 + 1) if b >= 1}))


def _schedule_sizes(kind, schedule):
    c = kind.host_chunk(1 << 12, schedule) if schedule == "1" else 1
    assert math.gcd(c, kind.P) == 1 or c == 1
    return _batch(c, schedule)


def _host(cwc, g, inp, entry, n_gpus=1, pitch=0, first_device=0):
    """one host-buffer call with canary-filled outputs: gw_calc_witness_batch ("batch"), _on ("on") or _wtns ("wtns");
    returns (rows or files, flags)"""
    B = inp.shape[0]
    flags = np.full(B, FLAG_CANARY, dtype=np.uint32)
    st = cwc.gw_status_t()
    if entry == "wtns":
        out = np.full((B, pitch), CANARY, dtype=np.uint8)
        rc = cwc._L.gw_calc_witness_batch_wtns(g._h, inp.ctypes.data, B, out.ctypes.data, pitch, flags.ctypes.data, n_gpus,
                                               ctypes.byref(st))
    else:
        out = np.full((B, g.n_witness * 32), CANARY, dtype=np.uint8)
        if entry == "batch":
            rc = cwc._L.gw_calc_witness_batch(g._h, inp.ctypes.data, B, out.ctypes.data, flags.ctypes.data, n_gpus, ctypes.byref(st))
        else:
            rc = cwc._L.gw_calc_witness_batch_on(g._h, first_device, inp.ctypes.data, B, out.ctypes.data, flags.ctypes.data, n_gpus,
                                                 ctypes.byref(st))
    cwc._check(rc, st)
    return out, flags


def _check_call(cwc, g, rc1, inp, witness=True, flags=True, n_gpus=1):
    """gw_calc_witness_batch_check with canary-filled outputs -> (rows or None, flags or None, first_failed)"""
    B = inp.shape[0]
    out = np.full((B, g.n_witness * 32), CANARY, dtype=np.uint8) if witness else None
    fl = np.full(B, FLAG_CANARY, dtype=np.uint32) if flags else None
    ff = np.full(B, 0x5A5A5A5A, dtype=np.uint32)
    st = cwc.gw_status_t()
    rc = cwc._L.gw_calc_witness_batch_check(g._h, rc1._h, 0, n_gpus, inp.ctypes.data, B, out.ctypes.data if witness else None,
                                            fl.ctypes.data if flags else None, ff.ctypes.data, ctypes.byref(st))
    cwc._check(rc, st)
    return out, fl, ff


def _expect_trace(capfd, B, chunk, n_calls=1, bit=False, what=""):
    tr, n_bit = _traces(capfd)
    assert tr == [(0, B, chunk)] * n_calls, f"{what}: meant {n_calls} x {B} sets in chunks of {chunk}, ran {tr}"
    if bit:
        assert n_bit >= n_calls, f"{what}: the bit-sliced kernels did not run"


# ---- witness rows through the host-buffer entry points -----------------------------------------------------------------
@pytest.mark.parametrize("schedule", SCHEDULES)
@pytest.mark.parametrize("kind_name", ["flags", "boolean", "random"])
def test_host_entry_points(cwc, env, capfd, kinds, kind_name, schedule):
    """gw_calc_witness_batch, _on and _wtns (file pitch = file size, + 52, + 1) under one chunk schedule at B = 1, 2, 3, chunk
    +- 1 and four chunks + a ragged tail: every row, flag, header and padding byte"""
    kind = kinds[kind_name]
    env(GW_CHUNK_MB=None if schedule == "default" else schedule)
    g = cwc.Graph(kind.data)
    if kind_name == "boolean":
        assert g.info["bit_eligible"] == 1
    size = g.wtns_file_size()
    assert size == 76 + kind.W * 32
    for B in _schedule_sizes(kind, schedule):
        chunk = kind.host_chunk(B, schedule)
        idx = kind.tile(B, chunk_edges(B, lambda n: kind.host_chunk(n, schedule)))
        inp = np.ascontiguousarray(kind.inp[idx])
        capfd.readouterr()
        for entry in ("batch", "on"):
            out, flags = _host(cwc, g, inp, entry)
            kind.check_rows(idx, out, flags, f"{schedule} {entry}")
        for pitch in (size, size + 52, size + 1):
            files, flags = _host(cwc, g, inp, "wtns", pitch=pitch)
            kind.check_files(idx, files, pitch, flags, f"{schedule} wtns")
        _expect_trace(capfd, B, chunk, 5, kind_name == "boolean", f"{kind_name} {schedule}")
    g.close()


@pytest.mark.parametrize("schedule", SCHEDULES)
@pytest.mark.parametrize("kind_name", ["random", "poseidon"])
def test_fused_check(cwc, env, capfd, kinds, kind_name, schedule):
    """gw_calc_witness_batch_check with and without the witness and the flags: the verdicts of sets that fail the appended
    bit constraints cross chunk boundaries, and each chunk's verdicts must come from its own buffer"""
    kind = kinds[kind_name]
    env(GW_CHUNK_MB=None if schedule == "default" else schedule)
    g, rc1 = cwc.Graph(kind.data), cwc.R1cs(ref.serialize_r1cs(kind.r1cs))
    for B in _schedule_sizes(kind, schedule):
        chunk = kind.host_chunk(B, schedule)
        idx = kind.tile(B, chunk_edges(B, lambda n: kind.host_chunk(n, schedule)))
        if B > 5:                               # (smaller batches are all chunk edges: every set fails)
            assert (kind.verdict[idx] == OK).any() and (kind.verdict[idx] != OK).any()
        inp = np.ascontiguousarray(kind.inp[idx])
        capfd.readouterr()
        for witness, flags in ((True, True), (False, True), (True, False)):
            out, fl, ff = _check_call(cwc, g, rc1, inp, witness, flags)
            what = f"{schedule} check witness={witness} flags={flags}"
            bad = np.nonzero(ff != kind.verdict[idx])[0]
            assert len(bad) == 0, f"{kind_name} {what} B={B}: wrong verdicts in sets {bad[:8].tolist()}"
            if witness:
                kind.check_rows(idx, out, fl, what)
            elif flags:
                assert (fl == kind.flags[idx]).all(), what
        _expect_trace(capfd, B, chunk, 3, what=f"{kind_name} {schedule}")
    g.close()
    rc1.close()


# ---- the stream ---------------------------------------------------------------------------------------------------------
class Consumer:
    """checks every chunk against the oracle and the simulator when it arrives (after `sleep` seconds: a delivered slot must
    not be overwritten meanwhile); returns nonzero at chunk `stop`"""

    def __init__(self, kind, idx, sleep=0.0, stop=None):
        self.kind, self.idx, self.sleep, self.stop = kind, idx, sleep, stop
        self.seen, self.lock, self.error = [], threading.Lock(), None

    def __call__(self, device, first, rows, flags):
        if self.sleep:
            time.sleep(self.sleep)
        n = rows.shape[0]
        try:
            self.kind.check_rows(self.idx[first:first + n], np.ascontiguousarray(rows), np.array(flags), f"stream chunk at {first}")
        except AssertionError as e:
            self.error = self.error or e
            return 1
        with self.lock:
            self.seen.append((device, first, n))
            return 1 if self.stop is not None and len(self.seen) == self.stop + 1 else 0

    def run(self, g, inp, B, **kw):
        """the stream over the whole batch; a wrong chunk fails with the consumer's message"""
        try:
            g.calc_witness_batch_stream(inp.ctypes.data, B, self, **kw)
        finally:
            if self.error:
                raise self.error

    def assert_cover(self, B, chunk, n_gpus=1):
        want = []
        for g in range(n_gpus):
            lo, hi = B * g // n_gpus, B * (g + 1) // n_gpus
            want += [(g, o, min(chunk(hi - lo), hi - o)) for o in range(lo, hi, chunk(hi - lo))]
        assert sorted(self.seen, key=lambda s: s[1]) == want, (self.seen[:6], want[:6])


def _stream_chunk(chunk_sets, B, auto):
    return max(min(chunk_sets or auto, B), 1)


@pytest.mark.parametrize("chunk_sets", [1, 31, 32, 33, 0])
@pytest.mark.parametrize("kind_name", ["flags", "boolean", "random"])
def test_stream(cwc, env, capfd, kinds, kind_name, chunk_sets):
    """gw_calc_witness_batch_stream with chunk_sets 1, 31, 32, 33 and 0 (auto: one wave of 32-thread CTAs): rows and flags
    checked on arrival, by a fast and by a slow consumer; stops at the first, second and last chunk"""
    torch = pytest.importorskip("torch")
    kind = kinds[kind_name]
    env(GW_THREADS=32 if chunk_sets == 0 else None)
    auto = torch.cuda.get_device_properties(0).multi_processor_count * 32
    g = cwc.Graph(kind.data)
    B = {1: 40, 31: 300, 32: 300, 33: 300, 0: 2 * auto + 77}[chunk_sets]
    chunk = _stream_chunk(chunk_sets, B, auto)
    idx = kind.tile(B, chunk_edges(B, lambda n: chunk))
    inp = np.ascontiguousarray(kind.inp[idx])
    n_chunks = -(-B // chunk)
    capfd.readouterr()
    for sleep in (0.0, 0.02):
        c = Consumer(kind, idx, sleep=sleep)
        c.run(g, inp, B, chunk_sets=chunk_sets)
        c.assert_cover(B, lambda n: chunk)
    _expect_trace(capfd, B, chunk, 2, kind_name == "boolean", f"{kind_name} stream {chunk_sets}")
    for stop in sorted({0, 1, n_chunks - 1}):
        c = Consumer(kind, idx, stop=stop)
        with pytest.raises(cwc.WitnessCalcError, match="stopped by the consumer"):
            g.calc_witness_batch_stream(inp.ctypes.data, B, c, chunk_sets=chunk_sets)
        assert c.error is None, c.error
        assert [s[1] for s in c.seen] == [k * chunk for k in range(stop + 1)], (stop, c.seen)
    g.close()


# ---- the R1CS host entry points -----------------------------------------------------------------------------------------
class R1csRows:
    """distinct witness rows of an R1CS kind: valid rows, rows failing the appended constraints, rows with a wrong value,
    values M, M + 5 and 2^256 - 1; their verdicts, A/B/C in both layouts and h"""

    def __init__(self, kind, r1cs=None, n=61, quotient=True, abc=True):
        self.r = r1cs or kind.r1cs
        rnd = random.Random(n)
        ws = [util.unpack_u256(w.tobytes()) for w in kind.want[:n]]
        for j, v in enumerate((None, M, M + 5, (1 << 256) - 1, None, M)):
            w = list(ws[j % n])
            wire = rnd.randrange(1, kind.W)
            w[wire] = rnd.randrange(M) if v is None else v
            ws.append(w)
        self.D, self.W = len(ws), kind.W
        self.rows = _pack(ws).reshape(self.D, -1)
        self.verdict = np.array([_verdict(self.r, w) for w in ws], dtype=np.uint32)
        self.marked = np.nonzero(self.verdict != OK)[0]
        assert 0 < len(self.marked) < self.D
        if abc:
            self.abc = {gr: np.stack([np.frombuffer(util.pack_u256(sum(abc_ref.abc_ref(self.r, w, gr), [])), np.uint8) for w in ws])
                        for gr in (False, True)}
        if quotient:
            self.h = np.stack([np.frombuffer(util.pack_u256(qref.quotient_ref(self.r, w)), np.uint8) for w in ws])

    def tile(self, B, edges):
        idx = (np.arange(B, dtype=np.int64) * 5 + 1) % self.D
        for j, b in enumerate(sorted(e for e in edges if 0 <= e < B)):
            idx[b] = self.marked[j % len(self.marked)]
        return idx

    def layout(self, idx, pitch, off):
        """the rows of idx in a canary-filled buffer: row b at b * pitch + off -> (buffer, pointer)"""
        B = len(idx)
        buf = np.full((B, pitch), CANARY, dtype=np.uint8)
        if off:
            buf[:, :76] = np.frombuffer(_wtns_header(self.W), np.uint8)
        buf[:, off:off + self.W * 32] = self.rows[idx]
        return buf, buf.ctypes.data + off


@pytest.fixture(scope="module")
def r1cs_rows(kinds):
    return {name: R1csRows(kinds[name]) for name in ("random", "poseidon")}


def _r1cs_check(cwc, rc1, ptr, B, pitch, n_gpus=1):
    ff = np.full(B, 0x5A5A5A5A, dtype=np.uint32)
    st = cwc.gw_status_t()
    cwc._check(cwc._L.gw_r1cs_check_batch(rc1._h, ptr, B, pitch, ff.ctypes.data, n_gpus, ctypes.byref(st)), st)
    return ff


def _r1cs_abc(cwc, rc1, ptr, B, pitch, out_pitch, groth16, n_gpus=1):
    out = np.full((B, out_pitch), CANARY, dtype=np.uint8)
    ff = np.full(B, 0x5A5A5A5A, dtype=np.uint32)
    st = cwc.gw_status_t()
    cwc._check(cwc._L.gw_r1cs_abc_batch(rc1._h, ptr, B, pitch, out.ctypes.data, out_pitch, cwc.R1CS_ABC_GROTH16 if groth16 else 0,
                                        ff.ctypes.data, n_gpus, ctypes.byref(st)), st)
    return out, ff


def _r1cs_quotient(cwc, rc1, ptr, B, pitch, h_pitch, n_gpus=1):
    out = np.full((B, h_pitch), CANARY, dtype=np.uint8)
    ff = np.full(B, 0x5A5A5A5A, dtype=np.uint32)
    st = cwc.gw_status_t()
    cwc._check(cwc._L.gw_r1cs_quotient_batch(rc1._h, ptr, B, pitch, out.ctypes.data, h_pitch, ff.ctypes.data, n_gpus,
                                             ctypes.byref(st)), st)
    return out, ff


def _assert_out(out, exp, idx, what, block=512):
    """out [B, pitch]: exp[idx] in front of every row, canary bytes behind; compared in blocks of rows"""
    n = exp.shape[1]
    for b0 in range(0, len(idx), block):
        o = out[b0:b0 + block]
        bad = np.nonzero((o[:, :n] != exp[idx[b0:b0 + block]]).any(axis=1))[0]
        assert len(bad) == 0, f"{what}: wrong results in rows {(bad[:8] + b0).tolist()}"
        cb = np.nonzero((o[:, n:] != CANARY).any(axis=1))[0]
        assert len(cb) == 0, f"{what}: padding overwritten in rows {(cb[:8] + b0).tolist()}"


def _assert_ff(ff, exp, what):
    bad = np.nonzero(ff != exp)[0]
    assert len(bad) == 0, f"{what}: wrong verdicts in rows {bad[:8].tolist()}: {ff[bad[:4]]} != {exp[bad[:4]]}"


def _run_r1cs_entry_points(cwc, rc1, rr, B, n_gpus=1):
    """check, plain and Groth16 A/B/C, and h, each under input layouts dense, + 48 bytes, .wtns images in place and .wtns
    images at an odd pitch, and outputs dense and pitched; h at a pitch >= 3 n x 32 first"""
    chunk = lambda n: (n + 3) // 4 if n >= 4 * 1024 else n
    idx = rr.tile(B, chunk_edges(B, chunk, n_gpus))
    row_b, wtns = rr.W * 32, 76 + rr.W * 32
    n_plain, n_groth = rc1.abc_len(), rc1.abc_len(groth16=True)
    outs = [(3 * 32 * n_plain, 32 * (3 * n_groth + 1)), (3 * 32 * n_plain + 40, 32 * n_groth), (3 * 32 * n_plain, 32 * n_groth + 24),
            (3 * 32 * n_plain + 40, 32 * n_groth)]
    for (pitch, off), (abc_pitch, h_pitch) in zip(((row_b, 0), (row_b + 48, 0), (wtns, 76), (wtns + 1, 76)), outs):
        what = f"B={B} n_gpus={n_gpus} row pitch {pitch} +{off}"
        buf, ptr = rr.layout(idx, pitch, off)
        h, ff = _r1cs_quotient(cwc, rc1, ptr, B, pitch, h_pitch, n_gpus)
        _assert_out(h, rr.h, idx, f"quotient h pitch {h_pitch} {what}")
        _assert_ff(ff, rr.verdict[idx], f"quotient {what}")
        _assert_ff(_r1cs_check(cwc, rc1, ptr, B, pitch, n_gpus), rr.verdict[idx], f"check {what}")
        for groth16 in (False, True):
            ap = abc_pitch if not groth16 else 3 * 32 * n_groth + (abc_pitch - 3 * 32 * n_plain)
            abc, ff = _r1cs_abc(cwc, rc1, ptr, B, pitch, ap, groth16, n_gpus)
            _assert_out(abc, rr.abc[groth16], idx, f"abc groth16={groth16} pitch {ap} {what}")
            _assert_ff(ff, rr.verdict[idx], f"abc groth16={groth16} {what}")
        assert (buf[:, off + row_b:] == CANARY).all() and (off == 0 or (buf[:, :76] == np.frombuffer(_wtns_header(rr.W), np.uint8)).all())


@pytest.mark.parametrize("kind_name", ["random", "poseidon"])
def test_r1cs_host_entry_points(cwc, kinds, r1cs_rows, kind_name):
    """gw_r1cs_check_batch, _abc_batch (plain and Groth16) and _quotient_batch on 4101 rows (four chunks, the last ragged)
    with valid, violating and >= M rows on every chunk edge, pitched inputs and outputs with canaries"""
    rr = r1cs_rows[kind_name]
    rc1 = cwc.R1cs(ref.serialize_r1cs(rr.r))
    _run_r1cs_entry_points(cwc, rc1, rr, R1CS_B)
    rc1.close()


def test_r1cs_quotient_two_pass_domain(cwc, kinds):
    """h of 4101 rows in four chunks for a pair whose Groth16 domain is 8192 (the two-pass NTT), dense and pitched h"""
    kind = kinds["random"]
    cons = kind.r1cs["constraints"]
    big = dict(kind.r1cs, constraints=[cons[i % len(cons)] for i in range(4200)])
    rr = R1csRows(kind, big, n=3, abc=False)
    rc1 = cwc.R1cs(ref.serialize_r1cs(big))
    n = rc1.abc_len(groth16=True)
    assert n == 8192 and rr.h.shape[1] == n * 32
    B = R1CS_B
    idx = rr.tile(B, chunk_edges(B, lambda m: (m + 3) // 4))
    buf, ptr = rr.layout(idx, rr.W * 32, 0)
    for h_pitch in (n * 32, n * 32 + 24):
        h, ff = _r1cs_quotient(cwc, rc1, ptr, B, rr.W * 32, h_pitch)
        _assert_out(h, rr.h, idx, f"two-pass quotient h pitch {h_pitch}")
        _assert_ff(ff, rr.verdict[idx], "two-pass quotient")
        del h
    rc1.close()


# ---- several GPUs -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_gpus", [2, 3])
def test_shards(cwc, env, capfd, kinds, r1cs_rows, n_gpus):
    """the host, .wtns, check, stream and R1CS entry points sharded over n_gpus GPUs, with flagged and failing sets on the
    shard boundaries B g / n_gpus and on every chunk edge of every shard"""
    if cwc.device_count() < n_gpus:
        pytest.skip(f"{cwc.device_count()} GPU(s) visible, {n_gpus} needed")
    env(GW_CHUNK_MB="1")
    for kind_name in ("flags", "random"):
        kind = kinds[kind_name]
        g = cwc.Graph(kind.data)
        size = g.wtns_file_size()
        for B in (n_gpus, 4 * kind.host_chunk(1 << 12, "1") + 5):
            idx = kind.tile(B, chunk_edges(B, lambda m: kind.host_chunk(m, "1"), n_gpus))
            inp = np.ascontiguousarray(kind.inp[idx])
            out, flags = _host(cwc, g, inp, "batch", n_gpus)
            kind.check_rows(idx, out, flags, f"{n_gpus} GPUs")
            files, flags = _host(cwc, g, inp, "wtns", n_gpus, pitch=size + 52)
            kind.check_files(idx, files, size + 52, flags, f"{n_gpus} GPUs")
            if cwc.device_count() > n_gpus:
                out, flags = _host(cwc, g, inp, "on", n_gpus, first_device=1)
                kind.check_rows(idx, out, flags, f"{n_gpus} GPUs from device 1")
            if kind.r1cs is not None:
                rc1 = cwc.R1cs(ref.serialize_r1cs(kind.r1cs))
                out, fl, ff = _check_call(cwc, g, rc1, inp, n_gpus=n_gpus)
                _assert_ff(ff, kind.verdict[idx], f"check {n_gpus} GPUs")
                kind.check_rows(idx, out, fl, f"check {n_gpus} GPUs")
                rc1.close()
            c = Consumer(kind, idx)
            c.run(g, inp, B, n_gpus=n_gpus, chunk_sets=33)
            c.assert_cover(B, lambda m: min(33, m), n_gpus)
        g.close()
    rr = r1cs_rows["poseidon"]
    rc1 = cwc.R1cs(ref.serialize_r1cs(rr.r))
    _run_r1cs_entry_points(cwc, rc1, rr, n_gpus * R1CS_B, n_gpus)
    rc1.close()


# ---- call sequences on one handle ---------------------------------------------------------------------------------------
def test_graph_call_sequence(cwc, env, capfd, kinds):
    """one graph handle: host -> stream -> check -> host -> host, with chunks that grow, shrink and grow again (the staging
    buffers, the verdict buffers and the pinned ring are regrown or reused between the calls)"""
    kind = kinds["random"]
    g, rc1 = cwc.Graph(kind.data), cwc.R1cs(ref.serialize_r1cs(kind.r1cs))
    c1 = kind.host_chunk(1 << 12, "1")
    steps = [("host", "1", 4 * c1 + 7), ("stream", 33, 1000), ("check", "default", 4 * 2048 + 3), ("host", "0", 5),
             ("check", "1", 2 * c1 + 1), ("host", "default", 4 * 2048 + 41), ("stream", 0, 3001), ("check", "default", 4 * 2048 + 3)]
    for what, sched, B in steps:
        if what == "stream":
            chunk = _stream_chunk(sched, B, B)
            idx = kind.tile(B, chunk_edges(B, lambda n: chunk))
            inp = np.ascontiguousarray(kind.inp[idx])
            c = Consumer(kind, idx)
            c.run(g, inp, B, chunk_sets=sched)
            c.assert_cover(B, lambda n: chunk)
            _traces(capfd)
            continue
        env(GW_CHUNK_MB=None if sched == "default" else sched)
        chunk = kind.host_chunk(B, sched)
        idx = kind.tile(B, chunk_edges(B, lambda n: kind.host_chunk(n, sched)))
        inp = np.ascontiguousarray(kind.inp[idx])
        capfd.readouterr()
        if what == "host":
            out, flags = _host(cwc, g, inp, "batch")
            kind.check_rows(idx, out, flags, f"sequence host {sched}")
        else:
            out, fl, ff = _check_call(cwc, g, rc1, inp)
            _assert_ff(ff, kind.verdict[idx], f"sequence check {sched}")
            kind.check_rows(idx, out, fl, f"sequence check {sched}")
        _expect_trace(capfd, B, chunk, what=f"sequence {what} {sched}")
    g.close()
    rc1.close()


def test_r1cs_call_sequence(cwc, r1cs_rows):
    """one R1CS handle: check -> plain A/B/C -> Groth16 A/B/C -> quotient -> check at different B (the staging is
    reallocated when the chunk or the output row grows, and reused otherwise)"""
    rr = r1cs_rows["random"]
    rc1 = cwc.R1cs(ref.serialize_r1cs(rr.r))
    row_b = rr.W * 32
    for what, B in (("check", 4101), ("plain", 1000), ("groth16", 5003), ("quotient", 4099), ("plain", 4500), ("check", 9001)):
        idx = rr.tile(B, chunk_edges(B, lambda n: (n + 3) // 4 if n >= 4096 else n))
        buf, ptr = rr.layout(idx, row_b, 0)
        if what == "check":
            ff = _r1cs_check(cwc, rc1, ptr, B, row_b)
        elif what == "quotient":
            n = rc1.abc_len(groth16=True)
            out, ff = _r1cs_quotient(cwc, rc1, ptr, B, row_b, 32 * n + 8)
            _assert_out(out, rr.h, idx, f"sequence quotient B={B}")
        else:
            groth16 = what == "groth16"
            out, ff = _r1cs_abc(cwc, rc1, ptr, B, row_b, 3 * 32 * rc1.abc_len(groth16), groth16)
            _assert_out(out, rr.abc[groth16], idx, f"sequence {what} B={B}")
        _assert_ff(ff, rr.verdict[idx], f"sequence {what} B={B}")
    rc1.close()


def test_two_threads_one_graph(cwc, env, kinds):
    """two host threads on one graph handle and one device at once, different batches and chunk schedules (ctypes releases
    the GIL: the calls overlap in the library)"""
    env(GW_TRACE_HOST=None, GW_CHUNK_MB="1")
    kind = kinds["flags"]
    g = cwc.Graph(kind.data)
    errors = []

    def work(seed, sizes):
        try:
            for B in sizes:
                idx = kind.tile(B, chunk_edges(B, lambda n: kind.host_chunk(n, "1")))
                idx = (idx + seed) % kind.P
                out, flags = _host(cwc, g, np.ascontiguousarray(kind.inp[idx]), "batch")
                kind.check_rows(idx, out, flags, f"thread {seed}")
        except Exception as e:          # noqa: BLE001 -- reported by the main thread
            errors.append(e)
    th = [threading.Thread(target=work, args=(1, (3001, 777, 5003, 64))), threading.Thread(target=work, args=(2, (4999, 1, 2500, 9000)))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    g.close()
    assert not errors, errors


# ---- small and empty selections -----------------------------------------------------------------------------------------
def _selection_r1cs(n):
    """an R1CS over the n selected values: (w0 - wj)^2 = 0 for j = 1 .. n - 1, and w0^2 = w0 when n == 1 (holds where the
    values are equal, or w0 a bit)"""
    if n == 1:
        cons = [([(0, 1)], [(0, 1)], [(0, 1)])]
    else:
        cons = [([(0, 1), (j, M - 1)], [(0, 1), (j, M - 1)], []) for j in range(1, n)]
    return {"n_wires": n, "n_pub_out": 0, "n_pub_in": 0, "n_prv_in": 0, "constraints": cons}


@pytest.mark.parametrize("which", ["one", "repeated", "empty"])
def test_selections(cwc, env, capfd, kinds, which):
    """gw_graph_select of 1 position, of repeated positions and of none, through the host, _on, .wtns, check, stream,
    latency and device entry points: the selected values of the oracle's rows, and the simulator's flags of the selected
    graph (0 for every set when the program is empty; the device entry point's flags are pre-filled with 0xFFFFFFFF)"""
    torch = pytest.importorskip("torch")
    base = kinds["flags"]
    nodes, wit, imap = base.nodes
    pos = {"one": [5], "repeated": [5, 5, 11, 5], "empty": []}[which]
    data = po.serialize_graph(nodes, [wit[p] for p in pos], imap)
    sim = util.SimGraph(data, **util.sim_options({}))
    assert (sim.info["n_instrs"] == 0) == (which == "empty")
    kind = Kind.__new__(Kind)
    kind.name, kind.data, kind.P, kind.I, kind.W = f"select {pos}", data, base.P, base.I, len(pos)
    kind.inp = base.inp
    kind.want = np.ascontiguousarray(base.want.reshape(base.P, -1, 32)[:, pos].reshape(base.P, 32 * len(pos)))
    kind.flags = np.array([sim.eval(util.unpack_u256(r.tobytes()))[1] for r in base.inp], dtype=np.uint32)
    kind.marked = np.nonzero(kind.flags)[0] if kind.flags.any() else np.arange(1)
    r1 = _selection_r1cs(len(pos))
    kind.verdict = np.array([_verdict(r1, util.unpack_u256(w.tobytes())) for w in kind.want], dtype=np.uint32)
    sel = cwc.Graph(base.data).select(pos)
    assert sel.n_witness == len(pos) and sel.wtns_file_size() == 76 + 32 * len(pos)
    rc1 = cwc.R1cs(ref.serialize_r1cs(r1))
    size = sel.wtns_file_size()
    for B in (1, 33, 1000):
        idx = kind.tile(B, ())
        d_in = torch.from_numpy(np.ascontiguousarray(kind.inp[idx])).cuda()
        d_out = torch.full((B, max(kind.W, 1) * 32), CANARY, dtype=torch.uint8, device="cuda")
        d_flags = torch.full((B,), -1, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        sel.calc_witness_batch_device(0, d_in.data_ptr(), B, d_out.data_ptr(), d_flags.data_ptr())
        torch.cuda.synchronize()
        out, flags = d_out.cpu().numpy(), d_flags.cpu().numpy().view(np.uint32)
        kind.check_rows(idx, np.ascontiguousarray(out[:, :kind.W * 32]), flags, f"device B={B}")
        if kind.W == 0:
            assert (out == CANARY).all()
    for sched in ("0", "default"):
        env(GW_CHUNK_MB=None if sched == "default" else sched)
        for B in ((1, 2, 7) if sched == "0" else (1, 3, 4 * 2048 + 3)):
            idx = kind.tile(B, chunk_edges(B, lambda n: kind.host_chunk(n, sched)))
            inp = np.ascontiguousarray(kind.inp[idx])
            for entry in ("batch", "on"):
                out, flags = _host(cwc, sel, inp, entry)
                kind.check_rows(idx, out, flags, f"{sched} {entry}")
            for pitch in (size, size + 52, size + 1):
                files, flags = _host(cwc, sel, inp, "wtns", pitch=pitch)
                kind.check_files(idx, files, pitch, flags, f"{sched} wtns")
            out, fl, ff = _check_call(cwc, sel, rc1, inp)
            kind.check_rows(idx, out, fl, f"{sched} check")
            _assert_ff(ff, kind.verdict[idx], f"{kind.name} {sched} check")
    env(GW_CHUNK_MB=None)
    B = 300
    idx = kind.tile(B, chunk_edges(B, lambda n: 31))
    inp = np.ascontiguousarray(kind.inp[idx])
    c = Consumer(kind, idx)
    c.run(sel, inp, B, chunk_sets=31)
    c.assert_cover(B, lambda n: 31)
    for b in (0, 1, int(kind.marked[0])):
        w, fl = sel.calc_witness_latency(kind.inp[b], want_flags=True)
        assert w.tobytes() == kind.want[b].tobytes() and fl == kind.flags[b], (kind.name, "latency", b)
    capfd.readouterr()
    sel.close()
    rc1.close()
