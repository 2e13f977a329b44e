"""gw_inputs_parse_batch_device: JSON Lines / JSON array text -> device rows.  The host parser gw_inputs_parse_batch is
the oracle throughout: rows are compared byte for byte, errors string for string."""
import ctypes
import importlib
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from tests import util
from tests.util import M, po
from tests.test_inputs_json import _graph as small_graph_bytes   # key1: 3 values, key2: 1, key3: 1
from tools import r1cs_gen

AUTHV2 = "circuit9_authV2"


@pytest.fixture(scope="module")
def cwc():
    subprocess.check_call([sys.executable, os.path.join(util.ROOT, "circom-witnesscalc_b200", "build.py")])
    return importlib.import_module("circom-witnesscalc_b200")


# ---- without a GPU ------------------------------------------------------------------------------------------------
def _raw(cwc):
    lib = ctypes.CDLL(cwc.LIB_PATH)
    f = lib.gw_inputs_parse_batch_device
    f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t,
                  ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p, ctypes.POINTER(cwc.gw_status_t)]
    return f


def test_argument_rejections_touch_no_device(cwc):
    f = _raw(cwc)
    g = cwc.Graph(small_graph_bytes())
    n, st = ctypes.c_size_t(7), cwc.gw_status_t()
    for args in ((None, 0, b"{}", 2, None, 0, ctypes.byref(n)),          # no graph
                 (g._h, 0, b"{}", 2, None, 0, None),                    # no n_sets
                 (g._h, 0, None, 2, None, 0, ctypes.byref(n)),          # no text, nonzero length
                 (g._h, 0, b"{}", 2, None, 4, ctypes.byref(n))):        # no rows, max_sets > 0
        assert f(*args, None, ctypes.byref(st)) == 1
        assert st.code == 1 and ctypes.string_at(st.error_msg) == b"null argument"


def test_no_device_is_a_loud_error(cwc):
    """with no visible device, even an empty text fails with the library's usual message"""
    code = ("import importlib, sys; sys.path.insert(0, %r); from tests.test_inputs_json import _graph\n"
            "cwc = importlib.import_module('circom-witnesscalc_b200'); g = cwc.Graph(_graph())\n"
            "for t in (b'', b'{}'):\n"
            "    try: g.parse_inputs_batch_device(t, 0, None, 0); print('no error')\n"
            "    except cwc.WitnessCalcError as e: print(e)\n") % util.ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=util.ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), check=True).stdout
    assert out.splitlines() == ["no CUDA device available: this library has no CPU fallback"] * 2


def test_rust_declaration_matches_the_header():
    rs = open(os.path.join(util.ROOT, "rust-shim", "src", "ffi.rs")).read()
    decl = rs[rs.index("pub fn gw_inputs_parse_batch_device("):]
    decl = decl[:decl.index(";")]
    assert [p.split(":")[0].strip() for p in decl[decl.index("(") + 1:decl.rindex(")")].split(",")] == \
        ["graph", "device", "text", "text_len", "d_inputs", "max_sets", "n_sets", "cuda_stream", "status"]


# ---- record generators --------------------------------------------------------------------------------------------
EDGES = [0, 1, M - 1, M, (1 << 256) - 1, (1 << 64) - 1, 1 << 64, 10 ** 9, 10 ** 9 - 1, 10 ** 18]


def _ws(rnd, array_form):
    return "".join(rnd.choice(" \t\r\n" if array_form else " \t\r") for _ in range(rnd.choice((0, 0, 0, 1, 2))))


def _value(rnd, v, array_form):
    if v < (1 << 64) and rnd.random() < 0.3:
        return str(v)
    return '"' + "0" * rnd.choice((0, 0, 0, 1, 5)) + str(v) + '"'


def good_record(rnd, signals, array_form=False):
    """a record in the device grammar: known keys in any order, some missing, whitespace around every token"""
    names = [k for k in signals if rnd.random() < 0.85]
    rnd.shuffle(names)
    w = lambda: _ws(rnd, array_form)   # noqa: E731
    members = []
    for k in names:
        ln = signals[k][1]
        vals = [rnd.choice(EDGES) if rnd.random() < 0.3 else rnd.randrange(M) for _ in range(ln)]
        if ln == 1 and rnd.random() < 0.5:
            body = _value(rnd, vals[0], array_form)
        else:
            body = "[" + w() + ("," + w()).join(_value(rnd, v, array_form) + w() for v in vals) + "]"
        members.append(w() + '"' + k + '"' + w() + ":" + w() + body + w())
    return w() + "{" + ",".join(members) + (w() if not members else "") + "}" + w()


def marked_record(rnd, signals):
    """records the device leaves to the host: escapes, underscores, repeated keys, "" """
    keys = list(signals)
    k = rnd.choice(keys)
    ln = signals[k][1]
    kind = rnd.randrange(5)
    if kind == 0:                                   # \\u escape in a key
        esc = "".join("\\u%04x" % ord(c) if rnd.random() < 0.5 else c for c in k)
        return '{"%s": %s}' % (esc, json.dumps([str(rnd.randrange(M)) for _ in range(ln)]))
    if kind == 1:                                   # escapes in values
        return '{"%s": [%s]}' % (k, ",".join('"\\u003%d%d"' % (rnd.randrange(10), rnd.randrange(10)) for _ in range(ln)))
    if kind == 2:                                   # underscores
        return '{"%s": [%s]}' % (k, ",".join('"1_%03d"' % rnd.randrange(1000) for _ in range(ln)))
    if kind == 3:                                   # a repeated key, first with another length: the last one wins
        return '{"%s": ["5"], "%s": %s}' % (k, k, json.dumps([str(i) for i in range(ln)]))
    return '{"%s": [%s]}' % (k, ",".join(['""'] * ln))


def jsonl(recs, rnd, crlf=False):
    nl = "\r\n" if crlf else "\n"
    out = []
    for r in recs:
        out.append(r)
        if rnd.random() < 0.05:
            out.append(rnd.choice(("", "  ", "\t \r")))
    return nl.join(out) + rnd.choice(("", nl))


def array_text(recs, indent):
    sep = ",\n  " if indent else ","
    return "[" + ("\n  " if indent else "") + sep.join(recs) + ("\n" if indent else "") + "]"


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    t = pytest.importorskip("torch")
    assert t.cuda.is_available()
    return t


def device_parse(cwc, torch, g, text, max_sets=None, stream=None):
    """-> ("ok", uint8 [n, I, 32]) or ("err", message), through the device parser"""
    if isinstance(text, str):
        text = text.encode()
    if max_sets is None:
        # the count-only call: more records than max_sets = 0 is an error that leaves the count in *n_sets
        cnt, st = ctypes.c_size_t(0), cwc.gw_status_t()
        _raw(cwc)(g._h, 0, text, len(text), None, 0, ctypes.byref(cnt), None, ctypes.byref(st))
        cwc._check(0, st)                # frees the message
        max_sets = cnt.value
    buf =torch.empty(max(max_sets, 1) * g.n_inputs * 32, dtype=torch.uint8, device="cuda")
    try:
        n = g.parse_inputs_batch_device(text, 0, buf.data_ptr(), max_sets, stream)
    except cwc.WitnessCalcError as e:
        return "err", str(e)
    return "ok", buf[:n * g.n_inputs * 32].cpu().numpy().reshape(n, g.n_inputs, 32)


def host_parse(cwc, g, text):
    try:
        return "ok", g.parse_inputs_batch(text, 0)
    except cwc.WitnessCalcError as e:
        return "err", str(e)


def assert_same(cwc, torch, g, text):
    want, got = host_parse(cwc, g, text), device_parse(cwc, torch, g, text)
    assert want[0] == got[0], (want[0], got[0], want[1] if want[0] == "err" else got[1], text[:300])
    if want[0] == "err":
        assert got[1] == want[1]
    else:
        assert want[1].shape == got[1].shape and np.array_equal(want[1], got[1])
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(util.manifest()))
def test_golden_graphs(cwc, torch, name):
    g = cwc.Graph(util.golden_graph(name))
    base = util.golden_inputs(name)
    base_line = json.dumps(json.loads(base))
    rnd = random.Random(name)
    want_w = np.frombuffer(util.golden_wtns(name)[76:], np.uint8).reshape(g.n_witness, 32)
    for n in (1, 33, 5000):
        recs = [base_line] + [good_record(rnd, g.input_signals) for _ in range(n - 1)]
        for text in (jsonl(recs, rnd), jsonl(recs, rnd, crlf=True), array_text(recs, False), array_text(recs, True)):
            st, rows = assert_same(cwc, torch, g, text)
            assert st == "ok" and rows.shape[0] == n
        # the unmodified record's row gives the golden witness
        d_in = torch.from_numpy(rows.reshape(n, -1)).cuda()
        d_w = torch.empty((1, g.n_witness * 32), dtype=torch.uint8, device="cuda")
        g.calc_witness_batch_device(0, d_in.data_ptr(), 1, d_w.data_ptr(), None, None)
        torch.cuda.synchronize()
        assert np.array_equal(d_w.cpu().numpy().reshape(g.n_witness, 32), want_w)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small", AUTHV2])
def test_grammar(cwc, torch, name):
    g = cwc.Graph(small_graph_bytes() if name == "small" else util.golden_graph(AUTHV2))
    rnd = random.Random(5)
    n = 10000 if name == "small" else 2000
    for array_form in (False, True):
        recs = [marked_record(rnd, g.input_signals) if rnd.random() < 0.1 else good_record(rnd, g.input_signals, array_form)
                for _ in range(n)]
        text = array_text(recs, False) if array_form else jsonl(recs, rnd)
        st, rows = assert_same(cwc, torch, g, text)
        assert st == "ok" and rows.shape[0] == n


@pytest.mark.gpu
def test_array_form_quirks(cwc, torch):
    g = cwc.Graph(small_graph_bytes())
    texts = [
        '[{"key2": "1"}, 5, {"key2": "2"}]',
        '[{"key2": "1"}, "a{[}\\"\\\\", {"key2": "2"}, ["}", {"x": "{"}], null, {"key3": 3}]',
        '[{"key2": "1"}, [5}, {"key2": "2"}]',                # a '}' closing a '[': the host's pairing
        '[{"key2": "1"} {"key2": "2"}]', '[}', '[ ]', '[]', '  \n [{}]  \n', '[{"key2": "1"}]\n\t ',
        '[{"key2": "1"}, {"key2": "2"}', '[{"key2": "1"}] x', '[{"key2": "1"}]]', '[{"key2": "1}]',
        '[{"key2": "1"}, {"key2": "\\"}"}, {"key2": "3"}]', '', ' \n\n ', '{}', '{}\n{}\n', '{"key2": "1"}',
    ]
    for t in texts:
        assert_same(cwc, torch, g, t)


BAD = ['[1, 2]', '{"key2": -1}', '{"key2": 1.5}', '{"key1": [["1"], "2", "3"]}', '{"key2": true}', '{"key2": null}',
       '{"key2": {"a": 1}}', '{"key2": "12x"}', '{"key2": "-5"}', '{"key2": "%d"}' % (1 << 256), '{"key2": "1"',
       '{"key2" "1"}', '{"nope": "1"}', '{"key1": ["1", "2"]}', '{"key2": 18446744073709551616}', '{"key2": 1e3}',
       '{"key2": "1",}', '{"key2": "1"} x', '{"key2": "1"}}', '{"key1": ["1", "2", "3", "4"]}', '{"key2": ["1", ]}']


@pytest.mark.gpu
def test_errors_name_the_host_record(cwc, torch):
    g = cwc.Graph(small_graph_bytes())
    rnd = random.Random(9)
    good = [good_record(rnd, g.input_signals) for _ in range(99)]
    for bad in BAD:
        for at in (0, 70, 99):
            recs = good[:at] + [bad] + good[at:]
            st, msg = assert_same(cwc, torch, g, jsonl(recs, rnd))
            assert st == "err"
            # in array form some of these are not records: the host's split skips depth-1 elements that are not objects,
            # so '[..., {"key2": "1"} x, ...]' and '[..., [1, 2], ...]' are accepted; device and host must still agree
            assert_same(cwc, torch, g, array_text(recs, rnd.random() < 0.5))
    # two bad records: the lower one is named
    recs = good[:10] + [BAD[1]] + good[10:50] + [BAD[12]] + good[50:]
    st, msg = assert_same(cwc, torch, g, jsonl(recs, rnd))
    assert msg.startswith("input set 11: ")
    recs = good[:10] + [BAD[12]] + good[10:50] + [BAD[1]] + good[50:]
    st, msg = assert_same(cwc, torch, g, array_text(recs, False))
    assert msg.startswith("input set 11: ")


@pytest.mark.gpu
def test_mutation_fuzz(cwc, torch):
    g = cwc.Graph(small_graph_bytes())
    rnd = random.Random(11)
    special = '"{}[],:\\'
    for i in range(2000):
        recs = [good_record(rnd, g.input_signals, i % 2 == 1) for _ in range(4)]
        t = list(array_text(recs, False) if i % 2 else jsonl(recs, rnd))
        for _ in range(rnd.choice((1, 1, 2, 3))):
            p = rnd.randrange(len(t) + 1)
            c = rnd.choice(special) if rnd.random() < 0.7 else chr(rnd.randrange(32, 127))
            op = rnd.randrange(3)
            if op == 0:
                t.insert(p, c)
            elif p < len(t):
                if op == 1:
                    del t[p]
                else:
                    t[p] = c
        assert_same(cwc, torch, g, "".join(t))


@pytest.mark.gpu
def test_sizes_and_shapes(cwc, torch):
    g = cwc.Graph(small_graph_bytes())
    rnd = random.Random(13)
    for t in ("", "[]", '{"key2": "1"}'):
        assert_same(cwc, torch, g, t)
    # text lengths around the 16-byte loads and the 16 KiB split tiles
    for target in list(range(1, 70)) + [16383, 16384, 16385, 32767, 32769, 65536 + 13]:
        recs, text = [], ""
        while len(text) < target:
            recs.append(good_record(rnd, g.input_signals))
            text = jsonl(recs, rnd)
        assert_same(cwc, torch, g, text[:target])
        assert_same(cwc, torch, g, array_text(recs, True)[:target])
        assert_same(cwc, torch, g, array_text(recs, True))


@pytest.mark.gpu
def test_max_sets_and_count_only(cwc, torch):
    g = cwc.Graph(small_graph_bytes())
    rnd = random.Random(17)
    text = jsonl([good_record(rnd, g.input_signals) for _ in range(100)], rnd).encode()
    assert g.parse_inputs_batch_device(b"", 0, None, 0) == 0
    with pytest.raises(cwc.WitnessCalcError, match="100 input sets.*max_sets = 0"):
        g.parse_inputs_batch_device(text, 0, None, 0)
    f = _raw(cwc)
    row = g.n_inputs * 32
    buf = torch.full((100 * row,), 0xA5, dtype=torch.uint8, device="cuda")
    n, st = ctypes.c_size_t(0), cwc.gw_status_t()
    assert f(g._h, 0, text, len(text), buf.data_ptr(), 60, ctypes.byref(n), None, ctypes.byref(st)) == 1
    msg = ctypes.string_at(st.error_msg).decode()
    assert n.value == 100 and "100 input sets" in msg and "max_sets = 60" in msg
    assert bool((buf == 0xA5).all())                 # nothing written, not even below max_sets
    assert g.parse_inputs_batch_device(text, 0, buf.data_ptr(), 100) == 100
    assert np.array_equal(buf.cpu().numpy().reshape(100, g.n_inputs, 32), g.parse_inputs_batch(text))
    buf2 = torch.full((101 * row,), 0x5A, dtype=torch.uint8, device="cuda")
    assert g.parse_inputs_batch_device(text, 0, buf2.data_ptr(), 101) == 100
    assert bool((buf2[100 * row:] == 0x5A).all())    # canary row past the last set


@pytest.mark.gpu
def test_one_record_of_megabytes(cwc, torch):
    L = 60000
    data = po.serialize_graph([(po.K_INPUT, i) for i in range(L + 2)], [0, 1, L + 1], {"big": (1, L), "x": (L + 1, 1)})
    g = cwc.Graph(data)
    rnd = random.Random(19)
    rec = '{"x": "7", "big": [' + ", ".join('"%d"' % rnd.randrange(1 << 256) for _ in range(L)) + "]}"
    assert len(rec) > 4_000_000
    for text in (rec, rec + "\n" + '{"x": 1}', "[" + rec + ", " + rec + "]"):
        st, rows = assert_same(cwc, torch, g, text)
        assert st == "ok"


@pytest.mark.gpu
def test_authv2_full_batch(cwc, torch):
    """262 144 authV2 records, one batch as bench.py sizes it, pinned text"""
    g = cwc.Graph(util.golden_graph(AUTHV2))
    rnd = random.Random(23)
    recs = [good_record(rnd, g.input_signals) for _ in range(256)]
    n = 262144
    text = ("\n".join(recs[i % 256] if i % 4099 else recs[(i * 7) % 256] for i in range(n)) + "\n").encode()
    pinned = torch.empty(len(text), dtype=torch.uint8).pin_memory()
    pinned.numpy()[:] = np.frombuffer(text, np.uint8)
    want = torch.from_numpy(g.parse_inputs_batch(text, 0).reshape(n, -1)).cuda()
    buf = torch.empty(n * g.n_inputs * 32, dtype=torch.uint8, device="cuda")
    f = _raw(cwc)
    f.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p] + f.argtypes[3:]
    cnt, st = ctypes.c_size_t(0), cwc.gw_status_t()
    assert f(g._h, 0, pinned.data_ptr(), len(text), buf.data_ptr(), n, ctypes.byref(cnt), None, ctypes.byref(st)) == 0
    assert cnt.value == n and torch.equal(buf.view(n, -1), want)


@pytest.mark.gpu
def test_stream_pipeline(cwc, torch):
    """parse, evaluate and check on one non-default stream with no host sync in between; compare with the host route"""
    rnd = random.Random(29)
    gb, r = r1cs_gen.poseidon_pair(rnd, n_hashes=2)
    from tests import r1cs_ref
    g, rc = cwc.Graph(gb), cwc.R1cs(r1cs_ref.serialize_r1cs(r))
    recs = [good_record(rnd, g.input_signals) for _ in range(3000)]
    text = jsonl(recs, rnd)
    n = len(recs)
    s = torch.cuda.Stream()
    d_in = torch.empty(n * g.n_inputs * 32, dtype=torch.uint8, device="cuda")
    d_w = torch.empty((n, g.n_witness * 32), dtype=torch.uint8, device="cuda")
    d_ff = torch.empty(n, dtype=torch.int32, device="cuda")
    with torch.cuda.stream(s):
        assert g.parse_inputs_batch_device(text, 0, d_in.data_ptr(), n, s.cuda_stream) == n
        g.calc_witness_batch_device(0, d_in.data_ptr(), n, d_w.data_ptr(), None, s.cuda_stream)
        rc.check_batch_device(0, d_w.data_ptr(), n, d_ff.data_ptr(), 0, s.cuda_stream)
    s.synchronize()
    want_w = g.calc_witness_batch(g.parse_inputs_batch(text))
    assert np.array_equal(d_w.cpu().numpy().reshape(want_w.shape), want_w)
    assert np.array_equal(d_ff.cpu().numpy().view(np.uint32), rc.check_batch(want_w))
