"""Python binding (ctypes) of the B200 witness evaluator's C ABI (include/graph_witness.h).

Mirrors the reference crate's public surface for the hot path (names from
/root/reference/src/lib.rs): ``calc_witness(inputs_json, graph_data)`` (lib.rs:125),
``wtns_from_witness`` (lib.rs:114), plus the pre-loaded ``Graph`` with the batch entry points.
All arithmetic happens in the CUDA library; this module only moves pointers.  There is no CPU
fallback: if ``lib/libcircom_witnesscalc.so`` is missing, importing fails loudly.

The directory name contains a hyphen, so import it with
``importlib.import_module("circom-witnesscalc_b200")``.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GW_LIB_PATH") or os.path.join(_HERE, "lib", "libcircom_witnesscalc.so")   # GW_LIB_PATH: kernel-variant experiments (tools/)
CLI_PATH = os.path.join(_HERE, "bin", "calc-witness")
CLI_BATCH_PATH = os.path.join(_HERE, "bin", "calc-witness-batch")
EXAMPLE_PATH = os.path.join(_HERE, "bin", "example-calc-witness")   # examples/calc_witness.c, the plain-C embedding example

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python circom-witnesscalc_b200/build.py` "
        "(there is no Python/CPU fallback for the witness evaluator)")

_L = ctypes.CDLL(LIB_PATH)

M = 21888242871839275222246405745257275088548364400416034343698204186575808495617


class gw_status_t(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int), ("error_msg", ctypes.c_void_p)]


class gw_graph_info_t(ctypes.Structure):
    _fields_ = [("n_nodes", ctypes.c_uint64), ("n_ops", ctypes.c_uint64), ("n_inputs", ctypes.c_uint32),
                ("n_witness", ctypes.c_uint32), ("n_input_signals", ctypes.c_uint32), ("n_instrs", ctypes.c_uint32),
                ("n_regs", ctypes.c_uint32), ("n_spill", ctypes.c_uint32), ("n_mul", ctypes.c_uint64),
                ("n_div", ctypes.c_uint64), ("n_spill_ld", ctypes.c_uint64), ("n_spill_st", ctypes.c_uint64),
                ("n_slots", ctypes.c_uint32), ("n_dot", ctypes.c_uint32), ("n_dot_mac", ctypes.c_uint32),
                ("n_mul_instr", ctypes.c_uint32), ("n_inversions", ctypes.c_uint32), ("threads", ctypes.c_uint32),
                ("sets_per_thread", ctypes.c_uint32), ("n_narrow_instr", ctypes.c_uint32),
                ("bit_eligible", ctypes.c_uint32), ("bit_luts", ctypes.c_uint32), ("bit_steps", ctypes.c_uint32),
                ("bit_wide", ctypes.c_uint32)]


class gw_r1cs_info_t(ctypes.Structure):
    _fields_ = [("n_wires", ctypes.c_uint32), ("n_pub_out", ctypes.c_uint32), ("n_pub_in", ctypes.c_uint32),
                ("n_prv_in", ctypes.c_uint32), ("n_constraints", ctypes.c_uint32), ("n_consts", ctypes.c_uint32),
                ("n_labels", ctypes.c_uint64), ("n_terms", ctypes.c_uint64), ("n_mac_terms", ctypes.c_uint64),
                ("n_chunks", ctypes.c_uint64)]


R1CS_OK = 0xFFFFFFFF    # GW_R1CS_OK: every constraint holds
R1CS_ABC_GROTH16 = 1    # GW_R1CS_ABC_GROTH16: ABC vectors in the Groth16 domain layout
NTT_INVERSE = 1         # GW_NTT_INVERSE
NTT_COSET = 2           # GW_NTT_COSET

_libc = ctypes.CDLL(None)
_libc.free.argtypes = [ctypes.c_void_p]

_vp, _sz = ctypes.c_void_p, ctypes.c_size_t
_L.gw_calc_witness.argtypes = [ctypes.c_char_p, _vp, _sz, ctypes.POINTER(_vp), ctypes.POINTER(_sz), ctypes.POINTER(gw_status_t)]
_L.gw_graph_load.argtypes = [_vp, _sz, ctypes.POINTER(_vp), ctypes.POINTER(gw_status_t)]
_L.gw_graph_free.argtypes = [_vp]
_L.gw_graph_info.argtypes = [_vp, ctypes.POINTER(gw_graph_info_t)]
_L.gw_graph_input_signal.argtypes = [_vp, ctypes.c_uint32, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint32)]
_L.gw_graph_calc_witness.argtypes = [_vp, ctypes.c_char_p, ctypes.POINTER(_vp), ctypes.POINTER(_sz), ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_batch.argtypes = [_vp, _vp, _sz, _vp, _vp, ctypes.c_int, ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_batch_on.argtypes = [_vp, ctypes.c_int, _vp, _sz, _vp, _vp, ctypes.c_int, ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_batch_device.argtypes = [_vp, ctypes.c_int, _vp, _sz, _vp, _vp, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_latency.argtypes = [_vp, ctypes.c_int, _vp, _vp, _vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_latency_batch.argtypes = [_vp, ctypes.c_int, ctypes.c_int, _vp, _sz, _vp, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_latency_batch_device.argtypes = [_vp, ctypes.c_int, _vp, _sz, _vp, _vp, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_wtns_header.argtypes = [ctypes.c_uint32, _vp]
_L.gw_inputs_parse_batch.argtypes = [_vp, ctypes.c_char_p, _sz, ctypes.c_int, ctypes.POINTER(_vp), ctypes.POINTER(_sz), ctypes.POINTER(gw_status_t)]
_L.gw_inputs_parse_batch_device.argtypes = [_vp, ctypes.c_int, ctypes.c_char_p, _sz, _vp, _sz, ctypes.POINTER(_sz), _vp,
                                             ctypes.POINTER(gw_status_t)]
_L.gw_wtns_file_size.restype = _sz
_L.gw_wtns_file_size.argtypes = [_vp]
_L.gw_calc_witness_batch_wtns.argtypes = [_vp, _vp, _sz, _vp, _sz, _vp, ctypes.c_int, ctypes.POINTER(gw_status_t)]
_L.gw_graph_select.argtypes = [_vp, _vp, _sz, ctypes.POINTER(_vp), ctypes.POINTER(gw_status_t)]
CHUNK_FN = ctypes.CFUNCTYPE(ctypes.c_int, _vp, ctypes.c_int, _sz, _sz, _vp, _sz, _vp)
_L.gw_calc_witness_batch_stream.argtypes = [_vp, ctypes.c_int, ctypes.c_int, _vp, _sz, _sz, CHUNK_FN, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_load.argtypes = [_vp, _sz, ctypes.POINTER(_vp), ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_free.argtypes = [_vp]
_L.gw_r1cs_info.argtypes = [_vp, ctypes.POINTER(gw_r1cs_info_t)]
_L.gw_r1cs_check_batch.argtypes = [_vp, _vp, _sz, _sz, _vp, ctypes.c_int, ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_check_batch_device.argtypes = [_vp, ctypes.c_int, _vp, _sz, _sz, _vp, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_abc_len.restype = ctypes.c_uint64
_L.gw_r1cs_abc_len.argtypes = [_vp, ctypes.c_uint32]
_L.gw_r1cs_abc_batch.argtypes = [_vp, _vp, _sz, _sz, _vp, _sz, ctypes.c_uint32, _vp, ctypes.c_int, ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_abc_batch_device.argtypes = [_vp, ctypes.c_int, _vp, _sz, _sz, _vp, _sz, ctypes.c_uint32, _vp, _vp,
                                        ctypes.POINTER(gw_status_t)]
_L.gw_fr_ntt_batch_device.argtypes = [ctypes.c_int, _vp, _sz, ctypes.c_uint32, _sz, ctypes.c_uint32, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_quotient_batch.argtypes = [_vp, _vp, _sz, _sz, _vp, _sz, _vp, ctypes.c_int, ctypes.POINTER(gw_status_t)]
_L.gw_r1cs_quotient_batch_device.argtypes = [_vp, ctypes.c_int, _vp, _sz, _sz, _vp, _sz, _vp, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_calc_witness_batch_check.argtypes = [_vp, _vp, ctypes.c_int, ctypes.c_int, _vp, _sz, _vp, _vp, _vp, ctypes.POINTER(gw_status_t)]
_L.gw_set_device.argtypes = [ctypes.c_int]
_L.gw_device_count.restype = ctypes.c_int
_L.gw_microbench_imad.restype = ctypes.c_double
_L.gw_microbench_imad.argtypes = [ctypes.c_int, ctypes.c_int]

EXPORTS = ["gw_calc_witness", "gw_graph_load", "gw_graph_free", "gw_graph_info", "gw_graph_input_signal",
           "gw_graph_calc_witness", "gw_calc_witness_batch", "gw_calc_witness_batch_on", "gw_calc_witness_batch_device", "gw_calc_witness_latency", "gw_wtns_header",
           "gw_device_count", "gw_microbench_imad", "gw_inputs_parse_batch", "gw_wtns_file_size", "gw_calc_witness_batch_wtns",
           "gw_graph_select", "gw_calc_witness_batch_stream", "gw_set_device", "gw_r1cs_load", "gw_r1cs_free", "gw_r1cs_info",
           "gw_r1cs_check_batch", "gw_r1cs_check_batch_device", "gw_calc_witness_batch_check", "gw_r1cs_abc_len",
           "gw_r1cs_abc_batch", "gw_r1cs_abc_batch_device", "gw_fr_ntt_batch_device", "gw_r1cs_quotient_batch",
           "gw_r1cs_quotient_batch_device", "gw_inputs_parse_batch_device", "gw_calc_witness_latency_batch",
           "gw_calc_witness_latency_batch_device"]


class WitnessCalcError(RuntimeError):
    pass


def _check(rc, st):
    msg = None
    if st.error_msg:
        msg = ctypes.string_at(st.error_msg).decode("utf-8", "replace")
        _libc.free(st.error_msg)
        st.error_msg = None
    if rc != 0:
        raise WitnessCalcError(msg or "unknown error")


def _take_malloced(ptr, n) -> bytes:
    data = ctypes.string_at(ptr.value, n.value)
    _libc.free(ptr)
    return data


def calc_witness_wtns(inputs_json, graph_data: bytes) -> bytes:
    """gw_calc_witness: inputs JSON + graph file bytes -> .wtns file bytes (the drop-in entry point)."""
    if isinstance(inputs_json, str):
        inputs_json = inputs_json.encode("utf-8")
    out, n, st = _vp(), _sz(), gw_status_t()
    rc = _L.gw_calc_witness(inputs_json, graph_data, len(graph_data), ctypes.byref(out), ctypes.byref(n), ctypes.byref(st))
    _check(rc, st)
    return _take_malloced(out, n)


def calc_witness(inputs_json, graph_data: bytes):
    """calc_witness (lib.rs:125): the witness as a list of ints."""
    w = calc_witness_wtns(inputs_json, graph_data)
    return [int.from_bytes(w[76 + 32 * i:108 + 32 * i], "little") for i in range((len(w) - 76) // 32)]


def wtns_from_witness(witness) -> bytes:
    """wtns_from_witness (lib.rs:114): frame canonical values as a .wtns v2 file."""
    hdr = ctypes.create_string_buffer(76)
    _L.gw_wtns_header(len(witness), hdr)
    return hdr.raw + b"".join(int(v).to_bytes(32, "little") for v in witness)


def set_device(device: int):
    """gw_set_device: CUDA device of the single-witness entry points"""
    if _L.gw_set_device(device) != 0:
        raise WitnessCalcError(f"CUDA device {device} does not exist")


def device_count() -> int:
    return _L.gw_device_count()


def ntt_batch_device(device, d_data_ptr, n_vectors, log_n, pitch=0, flags=0, stream=None):
    """DEVICE pointer: n_vectors transforms of 2^log_n 32-byte entries in place, vector v at d_data_ptr + v * pitch
    (pitch 0 = dense); flags NTT_INVERSE | NTT_COSET; asynchronous on `stream` (gw_fr_ntt_batch_device)."""
    st = gw_status_t()
    rc = _L.gw_fr_ntt_batch_device(device, d_data_ptr, n_vectors, log_n, pitch, flags, stream, ctypes.byref(st))
    _check(rc, st)


def microbench_imad(device=0, which=0) -> float:
    return _L.gw_microbench_imad(device, which)


class Graph:
    """A graph parsed, planned and (lazily) uploaded once: gw_graph_load."""

    def __init__(self, graph_data: bytes = None, _handle=None):
        self._h = _vp()
        if _handle is not None:
            self._h = _handle
        else:
            st = gw_status_t()
            rc = _L.gw_graph_load(graph_data, len(graph_data), ctypes.byref(self._h), ctypes.byref(st))
            _check(rc, st)
        info = gw_graph_info_t()
        _L.gw_graph_info(self._h, ctypes.byref(info))
        self.info = {k: int(getattr(info, k)) for k, _ in gw_graph_info_t._fields_}
        self.n_inputs = self.info["n_inputs"]
        self.n_witness = self.info["n_witness"]
        self.input_signals = {}
        for i in range(self.info["n_input_signals"]):
            nm, off, ln = ctypes.c_char_p(), ctypes.c_uint32(), ctypes.c_uint32()
            _L.gw_graph_input_signal(self._h, i, ctypes.byref(nm), ctypes.byref(off), ctypes.byref(ln))
            self.input_signals[nm.value.decode()] = (off.value, ln.value)

    def close(self):
        if self._h:
            _L.gw_graph_free(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def calc_witness_wtns(self, inputs_json) -> bytes:
        if isinstance(inputs_json, str):
            inputs_json = inputs_json.encode("utf-8")
        out, n, st = _vp(), _sz(), gw_status_t()
        rc = _L.gw_graph_calc_witness(self._h, inputs_json, ctypes.byref(out), ctypes.byref(n), ctypes.byref(st))
        _check(rc, st)
        return _take_malloced(out, n)

    def pack_inputs(self, input_sets) -> np.ndarray:
        """list of {name: [ints]} -> uint8 array [B, I, 32] (slot 0 = 1)"""
        buf = np.zeros((len(input_sets), self.n_inputs, 32), dtype=np.uint8)
        buf[:, 0, 0] = 1
        for b, s in enumerate(input_sets):
            for k, vals in s.items():
                off, ln = self.input_signals[k]
                assert ln == len(vals), f"input {k}: expected {ln} values"
                for i, v in enumerate(vals):
                    buf[b, off + i] = np.frombuffer(int(v).to_bytes(32, "little"), dtype=np.uint8)
        return buf

    def calc_witness_batch(self, inputs: np.ndarray, n_gpus=1, want_flags=False):
        """HOST buffers: inputs uint8 [B, I, 32] -> witness uint8 [B, W, 32] (gw_calc_witness_batch)."""
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        B = inputs.shape[0]
        assert inputs.shape[1:] == (self.n_inputs, 32), inputs.shape
        out = np.empty((B, self.n_witness, 32), dtype=np.uint8)
        flags = np.zeros(B, dtype=np.uint32) if want_flags else None
        st = gw_status_t()
        rc = _L.gw_calc_witness_batch(self._h, inputs.ctypes.data, B, out.ctypes.data,
                                      flags.ctypes.data if want_flags else None, n_gpus, ctypes.byref(st))
        _check(rc, st)
        return (out, flags) if want_flags else out

    def parse_inputs_batch(self, text, n_threads=0) -> np.ndarray:
        """JSON Lines (or a JSON array of objects) -> uint8 [B, I, 32] (gw_inputs_parse_batch, multi-threaded)."""
        if isinstance(text, str):
            text = text.encode("utf-8")
        out, n, st = _vp(), _sz(), gw_status_t()
        rc = _L.gw_inputs_parse_batch(self._h, text, len(text), n_threads, ctypes.byref(out), ctypes.byref(n), ctypes.byref(st))
        _check(rc, st)
        nbytes = n.value * self.n_inputs * 32
        arr = np.ctypeslib.as_array(ctypes.cast(out, ctypes.POINTER(ctypes.c_uint8)), shape=(max(nbytes, 1),))[:nbytes]
        arr = arr.reshape(n.value, self.n_inputs, 32).copy()           # one copy out of the malloc'ed buffer
        _libc.free(out)
        return arr

    def parse_inputs_batch_device(self, text, device, d_inputs_ptr, max_sets, stream=None) -> int:
        """JSON Lines (or a JSON array of objects) -> DEVICE rows: row r (n_inputs x 32 B) at d_inputs_ptr + r * n_inputs * 32,
        the same bytes as parse_inputs_batch.  Returns the number of input sets; more than max_sets is an error whose
        message names the count (max_sets=0 with d_inputs_ptr=None only counts).  Ordered on `stream` (a cudaStream_t
        as int, None = default stream); returns when the rows are complete (gw_inputs_parse_batch_device)."""
        if isinstance(text, str):
            text = text.encode("utf-8")
        n, st = _sz(), gw_status_t()
        rc = _L.gw_inputs_parse_batch_device(self._h, device, text, len(text), d_inputs_ptr, max_sets, ctypes.byref(n), stream,
                                             ctypes.byref(st))
        _check(rc, st)
        return n.value

    def wtns_file_size(self) -> int:
        return int(_L.gw_wtns_file_size(self._h))

    def calc_witness_batch_wtns(self, inputs: np.ndarray, file_pitch=0, n_gpus=1) -> np.ndarray:
        """HOST buffers: inputs uint8 [B, I, 32] -> uint8 [B, file_pitch]: row i starts with set i's complete .wtns
        file (gw_calc_witness_batch_wtns)."""
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        B = inputs.shape[0]
        pitch = file_pitch or self.wtns_file_size()
        out = np.zeros((B, pitch), dtype=np.uint8)
        st = gw_status_t()
        rc = _L.gw_calc_witness_batch_wtns(self._h, inputs.ctypes.data, B, out.ctypes.data, pitch, None, n_gpus, ctypes.byref(st))
        _check(rc, st)
        return out

    def select(self, positions) -> "Graph":
        """gw_graph_select: a graph whose witness is the given witness positions of this one."""
        pos = np.ascontiguousarray(positions, dtype=np.uint32)
        h, st = _vp(), gw_status_t()
        rc = _L.gw_graph_select(self._h, pos.ctypes.data, len(pos), ctypes.byref(h), ctypes.byref(st))
        _check(rc, st)
        return Graph(_handle=h)

    def calc_witness_latency(self, inputs_row: np.ndarray, device=0, want_flags=False):
        """ONE input set uint8 [I, 32] -> (witness uint8 [W, 32], kernel milliseconds): gw_calc_witness_latency.
        want_flags=True returns (witness, flags) instead, flags = the set's reference-undefined bits."""
        inputs_row = np.ascontiguousarray(inputs_row, dtype=np.uint8)
        assert inputs_row.shape == (self.n_inputs, 32), inputs_row.shape
        out = np.empty((self.n_witness, 32), dtype=np.uint8)
        ms = ctypes.c_float(0)
        fl = ctypes.c_uint32(0)
        st = gw_status_t()
        rc = _L.gw_calc_witness_latency(self._h, device, inputs_row.ctypes.data, out.ctypes.data,
                                        ctypes.addressof(fl) if want_flags else None, ctypes.byref(ms), ctypes.byref(st))
        _check(rc, st)
        return (out, int(fl.value)) if want_flags else (out, float(ms.value))

    def calc_witness_latency_batch(self, inputs: np.ndarray, n_gpus=1, first_device=0, want_flags=False):
        """HOST buffers: inputs uint8 [B, I, 32] -> witness uint8 [B, W, 32], one latency-mode CTA per set; row r equals
        calc_witness_latency(inputs[r]) (gw_calc_witness_latency_batch).  want_flags=True returns (witness, flags)."""
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        B = inputs.shape[0]
        assert inputs.shape[1:] == (self.n_inputs, 32), inputs.shape
        out = np.empty((B, self.n_witness, 32), dtype=np.uint8)
        flags = np.zeros(B, dtype=np.uint32) if want_flags else None
        st = gw_status_t()
        rc = _L.gw_calc_witness_latency_batch(self._h, first_device, n_gpus, inputs.ctypes.data, B, out.ctypes.data,
                                              flags.ctypes.data if want_flags else None, ctypes.byref(st))
        _check(rc, st)
        return (out, flags) if want_flags else out

    def calc_witness_latency_batch_device(self, device, d_inputs_ptr, n_sets, d_witness_ptr, d_flags_ptr=None, stream=None):
        """DEVICE pointers, one latency-mode CTA per set; ordered on `stream` (a cudaStream_t as int, None = default
        stream); returns when the rows are complete (gw_calc_witness_latency_batch_device)."""
        st = gw_status_t()
        rc = _L.gw_calc_witness_latency_batch_device(self._h, device, d_inputs_ptr, n_sets, d_witness_ptr, d_flags_ptr,
                                                     stream, ctypes.byref(st))
        _check(rc, st)

    def calc_witness_batch_ptr(self, inputs_ptr, n_sets, witness_ptr, flags_ptr=None, n_gpus=1, first_device=0):
        """HOST pointers (e.g. pinned torch tensors): no allocation, no copies besides the DMA.  The sets are sharded
        over devices first_device .. first_device + n_gpus - 1 (gw_calc_witness_batch_on)."""
        st = gw_status_t()
        rc = _L.gw_calc_witness_batch_on(self._h, first_device, inputs_ptr, n_sets, witness_ptr, flags_ptr, n_gpus, ctypes.byref(st))
        _check(rc, st)

    def calc_witness_batch_stream(self, inputs_ptr, n_sets, consumer, n_gpus=1, first_device=0, chunk_sets=0):
        """gw_calc_witness_batch_stream: HOST input pointer; `consumer(device, first_set, rows, flags)` is called per chunk with
        rows = uint8 [n, W, 32] and flags = uint32 [n] VIEWS of the library's pinned ring (valid during the call only);
        a truthy return value stops the stream."""
        W = self.n_witness

        def tramp(_user, device, first, n, rows, row_bytes, flags):
            r = np.ctypeslib.as_array(ctypes.cast(rows, ctypes.POINTER(ctypes.c_uint8)), shape=(n, W, 32)) if W else np.empty((n, 0, 32), np.uint8)
            f = np.ctypeslib.as_array(ctypes.cast(flags, ctypes.POINTER(ctypes.c_uint32)), shape=(n,))
            try:
                return 1 if consumer(device, first, r, f) else 0
            except Exception:          # nothing may unwind through the C frames
                import traceback
                traceback.print_exc()
                return 1
        cb = CHUNK_FN(tramp)
        st = gw_status_t()
        rc = _L.gw_calc_witness_batch_stream(self._h, first_device, n_gpus, inputs_ptr, n_sets, chunk_sets, cb, None, ctypes.byref(st))
        _check(rc, st)

    def calc_witness_batch_check(self, r1cs: "R1cs", inputs: np.ndarray, n_gpus=1, want_witness=True, first_device=0):
        """HOST buffers: evaluate and check against `r1cs` on the device in one pass (gw_calc_witness_batch_check).
        Returns (witness uint8 [B, W, 32] or None, flags uint32 [B], first_failed uint32 [B]); first_failed[b] is the
        lowest violated constraint of set b or R1CS_OK.  want_witness=False keeps the witnesses on the device."""
        inputs = np.ascontiguousarray(inputs, dtype=np.uint8)
        B = inputs.shape[0]
        assert inputs.shape[1:] == (self.n_inputs, 32), inputs.shape
        out = np.empty((B, self.n_witness, 32), dtype=np.uint8) if want_witness else None
        flags = np.zeros(B, dtype=np.uint32)
        first = np.zeros(B, dtype=np.uint32)
        st = gw_status_t()
        rc = _L.gw_calc_witness_batch_check(self._h, r1cs._h, first_device, n_gpus, inputs.ctypes.data, B,
                                            out.ctypes.data if want_witness else None, flags.ctypes.data, first.ctypes.data,
                                            ctypes.byref(st))
        _check(rc, st)
        return out, flags, first

    def calc_witness_batch_device(self, device, d_inputs_ptr, n_sets, d_witness_ptr, d_flags_ptr=None, stream=None):
        """DEVICE pointers; asynchronous on `stream` (a cudaStream_t as int, None = default stream)."""
        st = gw_status_t()
        rc = _L.gw_calc_witness_batch_device(self._h, device, d_inputs_ptr, n_sets, d_witness_ptr, d_flags_ptr,
                                             stream, ctypes.byref(st))
        _check(rc, st)


class R1cs:
    """A circuit's .r1cs file parsed and compiled once: gw_r1cs_load.  Checks witness rows against its constraints."""

    def __init__(self, data: bytes):
        self._h = _vp()
        st = gw_status_t()
        rc = _L.gw_r1cs_load(data, len(data), ctypes.byref(self._h), ctypes.byref(st))
        _check(rc, st)

    def info(self) -> dict:
        info = gw_r1cs_info_t()
        _L.gw_r1cs_info(self._h, ctypes.byref(info))
        return {k: int(getattr(info, k)) for k, _ in gw_r1cs_info_t._fields_}

    def close(self):
        if self._h:
            _L.gw_r1cs_free(self._h)
            self._h = _vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check_batch(self, rows, row_pitch=0, n_gpus=1, n_sets=None) -> np.ndarray:
        """HOST rows: a uint8 array whose row r starts at byte r * row_pitch (row_pitch 0: dense rows of n_wires x 32 B,
        e.g. a [B, W, 32] witness array) -> uint32 [B]: lowest violated constraint per row, or R1CS_OK
        (gw_r1cs_check_batch).  n_sets defaults to what the array holds."""
        rows = np.ascontiguousarray(rows, dtype=np.uint8)
        pitch = row_pitch or self.info()["n_wires"] * 32
        if n_sets is None:
            n_sets = rows.shape[0] if rows.ndim > 1 and not row_pitch else (rows.size // pitch if pitch else 0)
        assert n_sets == 0 or (n_sets - 1) * pitch + self.info()["n_wires"] * 32 <= rows.size, "rows too short"
        first = np.zeros(n_sets, dtype=np.uint32)
        st = gw_status_t()
        rc = _L.gw_r1cs_check_batch(self._h, rows.ctypes.data, n_sets, pitch, first.ctypes.data, n_gpus, ctypes.byref(st))
        _check(rc, st)
        return first

    def check_batch_device(self, device, d_witness_ptr, n_sets, d_first_failed_ptr, row_pitch=0, stream=None):
        """DEVICE pointers; asynchronous on `stream` (a cudaStream_t as int, None = default stream)
        (gw_r1cs_check_batch_device)."""
        st = gw_status_t()
        rc = _L.gw_r1cs_check_batch_device(self._h, device, d_witness_ptr, n_sets, row_pitch, d_first_failed_ptr, stream,
                                           ctypes.byref(st))
        _check(rc, st)

    def abc_len(self, groth16=False) -> int:
        """entries per vector of one ABC row (gw_r1cs_abc_len): n_constraints, or the Groth16 domain size"""
        return int(_L.gw_r1cs_abc_len(self._h, R1CS_ABC_GROTH16 if groth16 else 0))

    def abc_batch(self, rows, groth16=False, row_pitch=0, n_gpus=1, n_sets=None, want_verdict=False):
        """HOST rows as for check_batch -> uint8 [B, 3, n, 32]: <A_k,w>, <B_k,w>, <C_k,w> of every row (gw_r1cs_abc_batch);
        with want_verdict also the uint32 [B] verdicts of check_batch, from the same pass."""
        rows = np.ascontiguousarray(rows, dtype=np.uint8)
        n_wires = self.info()["n_wires"]
        pitch = row_pitch or n_wires * 32
        if n_sets is None:
            n_sets = rows.shape[0] if rows.ndim > 1 and not row_pitch else (rows.size // pitch if pitch else 0)
        assert n_sets == 0 or (n_sets - 1) * pitch + n_wires * 32 <= rows.size, "rows too short"
        n = self.abc_len(groth16)
        out = np.empty((n_sets, 3, n, 32), dtype=np.uint8)
        first = np.zeros(n_sets, dtype=np.uint32) if want_verdict else None
        st = gw_status_t()
        rc = _L.gw_r1cs_abc_batch(self._h, rows.ctypes.data, n_sets, pitch, out.ctypes.data, 0,
                                  R1CS_ABC_GROTH16 if groth16 else 0, first.ctypes.data if want_verdict else None, n_gpus,
                                  ctypes.byref(st))
        _check(rc, st)
        return (out, first) if want_verdict else out

    def abc_batch_device(self, device, d_witness_ptr, n_sets, d_abc_ptr, row_pitch=0, abc_pitch=0, groth16=False,
                         d_first_failed_ptr=None, stream=None):
        """DEVICE pointers; asynchronous on `stream` (a cudaStream_t as int, None = default stream)
        (gw_r1cs_abc_batch_device)."""
        st = gw_status_t()
        rc = _L.gw_r1cs_abc_batch_device(self._h, device, d_witness_ptr, n_sets, row_pitch, d_abc_ptr, abc_pitch,
                                         R1CS_ABC_GROTH16 if groth16 else 0, d_first_failed_ptr, stream, ctypes.byref(st))
        _check(rc, st)

    def quotient_batch(self, rows, row_pitch=0, n_gpus=1, n_sets=None, want_verdict=False):
        """HOST rows as for check_batch -> uint8 [B, n, 32] (n = abc_len(groth16=True)): the Groth16 quotient evaluations
        h = A_odd * B_odd - C_odd of every row (gw_r1cs_quotient_batch); with want_verdict also the uint32 [B] verdicts
        of check_batch, from the same pass."""
        rows = np.ascontiguousarray(rows, dtype=np.uint8)
        n_wires = self.info()["n_wires"]
        pitch = row_pitch or n_wires * 32
        if n_sets is None:
            n_sets = rows.shape[0] if rows.ndim > 1 and not row_pitch else (rows.size // pitch if pitch else 0)
        assert n_sets == 0 or (n_sets - 1) * pitch + n_wires * 32 <= rows.size, "rows too short"
        out = np.empty((n_sets, self.abc_len(groth16=True), 32), dtype=np.uint8)
        first = np.zeros(n_sets, dtype=np.uint32) if want_verdict else None
        st = gw_status_t()
        rc = _L.gw_r1cs_quotient_batch(self._h, rows.ctypes.data, n_sets, pitch, out.ctypes.data, 0,
                                       first.ctypes.data if want_verdict else None, n_gpus, ctypes.byref(st))
        _check(rc, st)
        return (out, first) if want_verdict else out

    def quotient_batch_device(self, device, d_witness_ptr, n_sets, d_work_ptr, row_pitch=0, work_pitch=0,
                              d_first_failed_ptr=None, stream=None):
        """DEVICE pointers; work rows of at least 3 x n x 32 bytes, h left in the first n x 32 bytes of each;
        asynchronous on `stream` (gw_r1cs_quotient_batch_device)."""
        st = gw_status_t()
        rc = _L.gw_r1cs_quotient_batch_device(self._h, device, d_witness_ptr, n_sets, row_pitch, d_work_ptr, work_pitch,
                                              d_first_failed_ptr, stream, ctypes.byref(st))
        _check(rc, st)
