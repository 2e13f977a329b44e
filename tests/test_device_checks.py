"""Device checks of every host and device entry point: which device counts, ranges and indices each one rejects, with
which message, and in which order against its null-argument, pitch and wire-count checks and its early return for an
empty batch.  Table-driven over the C ABI: every case asserts the return code and error_msg exactly.

Without a GPU every entry point that would touch a device fails with the no-device message (the library has no CPU
fallback); the entry points that return early for an empty batch succeed without asking for one.  With a GPU, device
ranges past the visible devices fail with the message of the entry point's family, and device indices past them with
"CUDA device index out of range"; no kernel runs in either case."""
import ctypes
import importlib
import os
import subprocess

import numpy as np
import pytest

from tests import r1cs_ref, util

NO_DEVICE = "no CUDA device available: this library has no CPU fallback"
RANGE = "device range exceeds the visible CUDA devices"          # host entry points that take a first_device
N_GPUS = "n_gpus exceeds the number of visible CUDA devices"     # host entry points that start at device 0
INDEX = "CUDA device index out of range"                          # device entry points


@pytest.fixture(scope="module")
def cwc():
    subprocess.check_call(["python", os.path.join(util.ROOT, "circom-witnesscalc_b200", "build.py")])
    return importlib.import_module("circom-witnesscalc_b200")


class Api:
    """the graph, an R1CS of as many wires as the graph has witness values (the fused check compares them first) and
    host buffers of every argument, so that no entry point stops at a null argument or a pitch"""

    def __init__(self, cwc):
        self.cwc, self.L = cwc, cwc._L
        self.g = cwc.Graph(util.golden_graph("circuit1"))
        W, I = self.g.n_witness, self.g.n_inputs
        self.r = cwc.R1cs(r1cs_ref.serialize_r1cs({"n_wires": W, "constraints": [([(0, 1)], [(0, 1)], [(0, 1)])]}))
        n = 4
        self.inputs = np.zeros((n, I * 32), np.uint8)
        self.witness = np.zeros((n, W * 32), np.uint8)
        self.flags = np.zeros(n, np.uint32)
        self.files = np.zeros((n, self.L.gw_wtns_file_size(self.g._h)), np.uint8)
        abc_n = self.r.abc_len(groth16=True)
        self.abc = np.zeros((n, 3 * 32 * abc_n), np.uint8)
        self.text = b'{"main.a": "1"}\n' * n
        self.n_out = ctypes.c_size_t()
        self.stream_fn = cwc.CHUNK_FN(lambda *a: 0)
        self.st = cwc.gw_status_t()

    def p(self, a):
        return a.ctypes.data

    def call(self, name, n_sets=1, first_device=0, n_gpus=1, device=0):
        """rc and error_msg of entry point `name` over n_sets sets"""
        L, g, r, st, p = self.L, self.g._h, self.r._h, ctypes.byref(self.st), self.p
        ins, wit, fl = p(self.inputs), p(self.witness), p(self.flags)
        calls = {
            "gw_calc_witness_batch": lambda: L.gw_calc_witness_batch(g, ins, n_sets, wit, fl, n_gpus, st),
            "gw_calc_witness_batch_on": lambda: L.gw_calc_witness_batch_on(g, first_device, ins, n_sets, wit, fl, n_gpus, st),
            "gw_calc_witness_batch_wtns": lambda: L.gw_calc_witness_batch_wtns(g, ins, n_sets, p(self.files), self.files.shape[1],
                                                                               fl, n_gpus, st),
            "gw_calc_witness_batch_stream": lambda: L.gw_calc_witness_batch_stream(g, first_device, n_gpus, ins, n_sets, 0,
                                                                                   self.stream_fn, None, st),
            "gw_calc_witness_batch_check": lambda: L.gw_calc_witness_batch_check(g, r, first_device, n_gpus, ins, n_sets, wit, fl,
                                                                                 p(self.flags), st),
            "gw_calc_witness_latency_batch": lambda: L.gw_calc_witness_latency_batch(g, first_device, n_gpus, ins, n_sets, wit, fl, st),
            "gw_r1cs_check_batch": lambda: L.gw_r1cs_check_batch(r, wit, n_sets, 0, fl, n_gpus, st),
            "gw_r1cs_abc_batch": lambda: L.gw_r1cs_abc_batch(r, wit, n_sets, 0, p(self.abc), 0, self.cwc.R1CS_ABC_GROTH16, fl,
                                                             n_gpus, st),
            "gw_r1cs_quotient_batch": lambda: L.gw_r1cs_quotient_batch(r, wit, n_sets, 0, p(self.abc), 0, fl, n_gpus, st),
            # device entry points: the buffers are never read, the call fails before any device work
            "gw_inputs_parse_batch_device": lambda: L.gw_inputs_parse_batch_device(g, device, self.text, len(self.text) if n_sets else 0,
                                                                                   ins, n_sets, ctypes.byref(self.n_out), None, st),
            "gw_calc_witness_batch_device": lambda: L.gw_calc_witness_batch_device(g, device, ins, n_sets, wit, fl, None, st),
            "gw_calc_witness_latency": lambda: L.gw_calc_witness_latency(g, device, ins, wit, fl, None, st),
            "gw_calc_witness_latency_batch_device": lambda: L.gw_calc_witness_latency_batch_device(g, device, ins, n_sets, wit, fl,
                                                                                                   None, st),
            "gw_r1cs_check_batch_device": lambda: L.gw_r1cs_check_batch_device(r, device, wit, n_sets, 0, fl, None, st),
            "gw_r1cs_abc_batch_device": lambda: L.gw_r1cs_abc_batch_device(r, device, wit, n_sets, 0, p(self.abc), 0,
                                                                           self.cwc.R1CS_ABC_GROTH16, fl, None, st),
            "gw_r1cs_quotient_batch_device": lambda: L.gw_r1cs_quotient_batch_device(r, device, wit, n_sets, 0, p(self.abc), 0, fl,
                                                                                     None, st),
            "gw_fr_ntt_batch_device": lambda: L.gw_fr_ntt_batch_device(device, p(self.abc), n_sets, 4, 0, 0, None, st),
        }
        self.st.code, self.st.error_msg = 0, None
        rc = calls[name]()
        msg = ctypes.string_at(self.st.error_msg).decode() if self.st.error_msg else None
        if self.st.error_msg:
            ctypes.CDLL(None).free(ctypes.c_void_p(self.st.error_msg))
        return rc, msg


HOST_FIRST = ["gw_calc_witness_batch_on", "gw_calc_witness_batch_stream", "gw_calc_witness_batch_check",
              "gw_calc_witness_latency_batch"]
HOST_ZERO = ["gw_calc_witness_batch", "gw_calc_witness_batch_wtns", "gw_r1cs_check_batch", "gw_r1cs_abc_batch",
             "gw_r1cs_quotient_batch"]
DEVICE = ["gw_inputs_parse_batch_device", "gw_calc_witness_batch_device", "gw_calc_witness_latency",
          "gw_calc_witness_latency_batch_device", "gw_r1cs_check_batch_device", "gw_r1cs_abc_batch_device",
          "gw_r1cs_quotient_batch_device", "gw_fr_ntt_batch_device"]
# an empty batch returns before any device is asked for (after the arguments are checked)
EMPTY_OK = {"gw_calc_witness_latency_batch", "gw_calc_witness_latency_batch_device", "gw_r1cs_abc_batch",
            "gw_r1cs_quotient_batch", "gw_r1cs_abc_batch_device", "gw_r1cs_quotient_batch_device", "gw_fr_ntt_batch_device"}


@pytest.fixture(scope="module")
def api(cwc):
    return Api(cwc)


@pytest.mark.parametrize("n_sets", [1, 0])
@pytest.mark.parametrize("name", HOST_FIRST + HOST_ZERO + DEVICE)
def test_without_a_device(cwc, api, name, n_sets):
    if cwc.device_count() > 0:
        pytest.skip("a GPU is present")
    want = (0, None) if n_sets == 0 and name in EMPTY_OK else (1, NO_DEVICE)
    assert api.call(name, n_sets=n_sets, first_device=0, n_gpus=2, device=0) == want
    assert api.call(name, n_sets=n_sets, first_device=0, n_gpus=0, device=0) == want


def test_set_device_without_a_device(cwc):
    if cwc.device_count() > 0:
        pytest.skip("a GPU is present")
    assert cwc._L.gw_set_device(0) == 1 and cwc._L.gw_set_device(-1) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("name", HOST_FIRST)
def test_device_range(cwc, api, name):
    n = cwc.device_count()
    assert n >= 1, "no CUDA device visible"
    for first, n_gpus in ((0, n + 1), (-1, 1), (n, 1), (n, 0), (n - 1, 2)):
        assert api.call(name, first_device=first, n_gpus=n_gpus) == (1, RANGE), (first, n_gpus)


@pytest.mark.gpu
@pytest.mark.parametrize("name", HOST_ZERO)
def test_n_gpus(cwc, api, name):
    n = cwc.device_count()
    assert n >= 1, "no CUDA device visible"
    assert api.call(name, n_gpus=n + 1) == (1, N_GPUS)


@pytest.mark.gpu
@pytest.mark.parametrize("name", DEVICE)
def test_device_index(cwc, api, name):
    n = cwc.device_count()
    assert n >= 1, "no CUDA device visible"
    for device in (n, -1):
        assert api.call(name, device=device) == (1, INDEX), device


@pytest.mark.gpu
def test_set_device(cwc):
    n = cwc.device_count()
    assert n >= 1, "no CUDA device visible"
    assert cwc._L.gw_set_device(n) == 1 and cwc._L.gw_set_device(-1) == 1
