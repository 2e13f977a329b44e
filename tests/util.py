"""Shared helpers of the test-suite: golden fixtures, random graphs, ctypes bindings of the
test-only host libraries (tests/csrc) and of the product library."""
import ctypes
import json
import lzma
import os
import random
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
BUILD = os.path.join(ROOT, "tests", "_build")
CSRC = os.path.join(ROOT, "circom-witnesscalc_b200", "csrc")

from oracle import pyoracle as po  # noqa: E402

M = po.M


# ---- fixtures -------------------------------------------------------------------------------------
def manifest():
    return json.load(open(os.path.join(GOLDEN, "manifest.json")))


def golden_graph(name) -> bytes:
    return lzma.decompress(open(os.path.join(GOLDEN, "graphs", name + ".bin.xz"), "rb").read())


def golden_inputs(name) -> str:
    return open(os.path.join(GOLDEN, "inputs", name + "_inputs.json")).read()


def golden_wtns(name) -> bytes:
    return lzma.decompress(open(os.path.join(GOLDEN, "wtns", name + ".wtns.xz"), "rb").read())


def kat():
    """reference-held known answers per golden graph (tests/golden/kat.json, written by tools/gen_graphs.py):
    [{inputs: {name: value | [values]}, expOut: {main signal: value}, source}]"""
    return json.load(open(os.path.join(GOLDEN, "kat.json")))


def kat_cases():
    return [(g, i) for g, v in sorted(kat().items()) for i in range(len(v))]


def kat_check(witness, input_map, n_inputs_row, case, out_names):
    """expOut of a circom_tester assertOut: main OUTPUT signals sit at witness positions 1.. in declaration order
    (out_names), main INPUT signals after them in input-buffer order."""
    n_out = len(out_names)
    for k, v in case["expOut"].items():
        if k in out_names:
            assert witness[1 + out_names.index(k)] == int(v), (k, case.get("desc"))
        else:
            off, ln = input_map[k]
            assert ln == 1 and witness[n_out + off] == int(v), (k, case.get("desc"))


KAT_OUTPUTS = {"authV2_32_32": ["userID"], "poseidon2": ["out"], "poseidon3": ["out"], "poseidon5": ["out"]}


# ---- packing ----------------------------------------------------------------------------------------
def pack_u256(vals) -> bytes:
    return b"".join(int(v).to_bytes(32, "little") for v in vals)


def unpack_u256(buf) -> list:
    buf = bytes(buf)
    return [int.from_bytes(buf[i:i + 32], "little") for i in range(0, len(buf), 32)]


def random_field_batch(rng: np.random.Generator, shape):
    """uniform values in [0, M) as a uint64 array [..., 4] (little-endian limbs) by rejection sampling"""
    n = int(np.prod(shape))
    out = np.empty((n, 4), dtype=np.uint64)
    top = M >> 192
    filled = 0
    while filled < n:
        cand = rng.integers(0, 1 << 64, size=(2 * (n - filled) + 16, 4), dtype=np.uint64)
        cand[:, 3] &= np.uint64((1 << 62) - 1)      # 254 bits
        hi = cand[:, 3]
        ok = hi < np.uint64(top)                      # strictly below the top limb of M: always < M
        eq = hi == np.uint64(top)
        if eq.any():
            for i in np.nonzero(eq)[0]:
                v = sum(int(cand[i, k]) << (64 * k) for k in range(4))
                ok[i] = v < M
        good = cand[ok]
        take = min(len(good), n - filled)
        out[filled:filled + take] = good[:take]
        filled += take
    return out.reshape(tuple(shape) + (4,))


def limbs_to_ints(a):
    a = np.asarray(a, dtype=np.uint64).reshape(-1, 4)
    return [int(r[0]) | (int(r[1]) << 64) | (int(r[2]) << 128) | (int(r[3]) << 192) for r in a]


# ---- random graphs ----------------------------------------------------------------------------------
EDGE = [0, 1, 2, 3, M - 1, M - 2, M >> 1, (M >> 1) + 1, (M >> 1) - 1, 1 << 253, (1 << 253) - 1, (1 << 254) - 1 - M,
        0xFFFFFFFF, 1 << 32, (1 << 64) - 1, 1 << 64, (1 << 128) - 1, 253, 254, 255, 256, 31, 32, 33, 64]


def random_value(rnd: random.Random):
    r = rnd.random()
    if r < 0.3:
        return rnd.choice(EDGE) % M
    if r < 0.45:
        return rnd.randrange(1 << rnd.randrange(1, 254))
    return rnd.randrange(M)


def random_graph(rnd: random.Random, n_inputs=6, n_ops=200, ops=None, n_consts=12, uno_ext=True):
    """A graph in the layout build-circuit produces: Input run first, then constants and ops.
    Returns (nodes, witness_signals, input_map)."""
    duo = ops if ops is not None else list(range(20))
    nodes = [(po.K_INPUT, i) for i in range(n_inputs + 1)]
    for _ in range(n_consts):
        nodes.append((po.K_CONST, random_value(rnd)))
    small = [len(nodes) + i for i in range(6)]
    for v in (0, 1, 5, 31, 32, 200):
        nodes.append((po.K_CONST, v))
    for _ in range(n_ops):
        n = len(nodes)
        pick = lambda: rnd.randrange(n) if rnd.random() < 0.7 else rnd.randrange(max(0, n - 8), n)
        r = rnd.random()
        if r < 0.08:
            # Neg mostly; Id / Lnot / Bnot (north_star's unary ops; the reference snapshot has Neg and Id only,
            # graph.rs:175-178, and Id is unimplemented! at run time) are drawn too when `uno_ext`
            nodes.append((po.K_UNO, rnd.choice((0, 0, 1, 2, 3)) if uno_ext else 0, pick()))
        elif r < 0.16:
            nodes.append((po.K_TRES, 0, pick(), pick(), pick()))
        else:
            op = rnd.choice(duo)
            a, b = pick(), pick()
            if op in (15, 16) and rnd.random() < 0.7:
                b = rnd.choice(small)
            if op == 0 and rnd.random() < 0.2:
                b = a
            nodes.append((po.K_DUO, op, a, b))
    n = len(nodes)
    wit = [0] + [rnd.randrange(n) for _ in range(min(n, 40))] + list(range(n - 10, n))
    return nodes, wit, {"x": (1, n_inputs)}


def poseidon_like_graph(rnd: random.Random, t=3, rounds=8, n_inputs=6):
    """Random graph with the shapes of circomlib's Poseidon (poseidon.circom: Ark, Sigma, Mix, MixS) and an occasional
    division: S-box chains x^2, x^4, x^5 (operand order and witness order varied), `lc += c * in[j]` sums,
    `in[i] + in[0] * c` updates, constants added before the S-box.  Exercises OP_POW5, the OP_DOT shapes, the
    Mul(const, x + c) folding, lane chains and split linear combinations.  Returns (nodes, witness_signals, input_map)."""
    nodes = [(po.K_INPUT, i) for i in range(n_inputs + 1)]

    def const(v):
        nodes.append((po.K_CONST, v))
        return len(nodes) - 1

    def duo(op, a, b):
        nodes.append((po.K_DUO, po.DUO[op], a, b))
        return len(nodes) - 1

    st = [1 + rnd.randrange(n_inputs) for _ in range(t)]
    wit = [0]
    for _ in range(rounds):
        full = rnd.random() < 0.3
        st = [duo("Add", s, const(rnd.randrange(M))) if rnd.random() < 0.8 else s for s in st]
        for j in range(t if full else 1):
            x = st[j]
            x2 = duo("Mul", x, x)
            x4 = duo("Mul", x2, x2)
            x5 = duo("Mul", x4, x) if rnd.random() < 0.8 else duo("Mul", x, x4)
            outs = [x2, x4, x5]
            if rnd.random() < 0.3:
                rnd.shuffle(outs)
            wit += [o for o in outs if rnd.random() < 0.9]
            st[j] = x5
        new = []
        if full or rnd.random() < 0.3:
            for _i in range(t):
                lc = None
                for j in range(t):
                    c = const(rnd.randrange(M))
                    term = duo("Mul", c, st[j]) if rnd.random() < 0.5 else duo("Mul", st[j], c)
                    lc = term if lc is None else duo("Add", lc, term)
                new.append(lc)
        else:
            lc = None
            for j in range(t):
                term = duo("Mul", const(rnd.randrange(M)), st[j])
                lc = term if lc is None else duo("Add", lc, term)
            new.append(lc)
            for i in range(1, t):
                new.append(duo("Add" if rnd.random() < 0.8 else "Sub", st[i], duo("Mul", st[0], const(rnd.randrange(M)))))
        st = new
        wit += [s for s in st if rnd.random() < 0.8]
        if rnd.random() < 0.15:
            d = duo("Div", st[0], st[-1])
            wit.append(d)
            st[0] = d
    wit += st
    return nodes, wit, {"x": (1, n_inputs)}


# ---- test-only host libraries -------------------------------------------------------------------------
def _build(name, sources, extra=()):
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, name)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [s for s in sources]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", out,
                               *sources, *extra])
    return out


_libs = {}


def field_host_lib(emulate_ptx=False):
    """csrc/field.cuh on the host.  emulate_ptx=True compiles the DEVICE formulations (PTX carry chains, even/odd
    accumulators) with an emulated carry flag instead of the plain host loops."""
    key = "field_ptx" if emulate_ptx else "field"
    if key not in _libs:
        _libs[key] = ctypes.CDLL(_build("libfieldhost_ptx.so" if emulate_ptx else "libfieldhost.so",
                                        [os.path.join(ROOT, "tests/csrc/field_host_api.cpp")],
                                        extra=("-DGW_EMULATE_PTX",) if emulate_ptx else ()))
    return _libs[key]


def sim_lib():
    if "sim" not in _libs:
        src = [os.path.join(ROOT, "tests/csrc/plan_host_sim.cpp")] + [os.path.join(CSRC, f) for f in
                                                                      ("graph.cpp", "plan.cpp", "bitplan.cpp", "inputs.cpp", "wtns.cpp")]
        L = ctypes.CDLL(_build("libgwsim.so", src))
        L.sim_load.restype = ctypes.c_void_p
        L.sim_load.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_size_t]
        L.sim_load2.restype = ctypes.c_void_p
        L.sim_load2.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]
        L.sim_free.argtypes = [ctypes.c_void_p]
        L.sim_code.restype = ctypes.c_size_t
        L.sim_code.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint32), ctypes.c_size_t]
        L.sim_info.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
        L.sim_info2.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
        L.sim_eval.restype = ctypes.c_int64
        L.sim_eval.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p]
        L.sim_eval_latency.restype = ctypes.c_int64
        L.sim_eval_latency.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64)]
        L.sim_eval_latency2.restype = ctypes.c_int64
        L.sim_eval_latency2.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.c_int,
                                        ctypes.POINTER(ctypes.c_uint32)]
        L.sim_eval_latency3.restype = ctypes.c_int64
        L.sim_eval_latency3.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_uint64), ctypes.c_int,
                                        ctypes.POINTER(ctypes.c_uint32), ctypes.POINTER(ctypes.c_uint64)]
        L.sim_error.restype = ctypes.c_char_p
        L.sim_error.argtypes = [ctypes.c_void_p]
        L.sim_inputs.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_size_t]
        L.sim_reserialize.restype = ctypes.c_size_t
        L.sim_reserialize.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t]
        L.sim_bit_load.restype = ctypes.c_void_p
        L.sim_bit_load.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t]
        L.sim_bit_load2.restype = ctypes.c_void_p
        L.sim_bit_load2.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_int, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_size_t]
        L.sim_bit_plan.restype = ctypes.c_size_t
        L.sim_bit_plan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_uint32), ctypes.c_size_t]
        L.sim_bit_free.argtypes = [ctypes.c_void_p]
        L.sim_bit_info.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
        L.sim_bit_eval.restype = ctypes.c_int64
        L.sim_bit_eval.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p]
        _libs["sim"] = L
    return _libs["sim"]


class BitSimGraph:
    """bit-sliced plan (csrc/bitplan.cpp) on the host simulator: groups of up to 32 input sets"""

    def __init__(self, data: bytes, max_support=0, merge=True, max_slots=0):
        self.L = sim_lib()
        err = ctypes.create_string_buffer(512)
        self.h = self.L.sim_bit_load2(data, len(data), max_support, int(merge), max_slots, err, 512)
        if not self.h:
            raise ValueError(err.value.decode())
        info = (ctypes.c_uint64 * 15)()
        self.L.sim_bit_info(self.h, info)
        keys = ["eligible", "n_steps", "n_slots", "n_luts", "n_levels", "n_bit", "n_tt", "n_bv", "n_full_adders", "n_merged", "n_inputs_checked", "n_consts",
                "has_field_inputs", "n_wide", "plane_stride"]
        self.info = dict(zip(keys, [int(x) for x in info]))
        self.reason = err.value.decode()
        nodes, wit, _ = po.deserialize_graph(data)
        self.I = 1 + max([n[1] for n in nodes if n[0] == po.K_INPUT] + [0])
        self.W = len(wit)

    def eval(self, rows):
        """rows: list (<= 32) of input lists -> (list of witness lists or None where the bit contract fails, ok mask)"""
        n = len(rows)
        out = ctypes.create_string_buffer(32 * self.W * n)
        ok = self.L.sim_bit_eval(self.h, b"".join(pack_u256(r) for r in rows), n, out)
        assert ok >= 0, "malformed bit plan"
        res = [unpack_u256(out.raw[32 * self.W * b:32 * self.W * (b + 1)]) if (ok >> b) & 1 else None for b in range(n)]
        return res, int(ok)

    def plan(self) -> dict:
        """the compiled plan: code [n_steps, 32, 4] (x, y, z, w of every lane), inputs [n, 3] and wide [n, 3] triples,
        const_of_pos [W] (int32: -1 a plane, -2 a wide value, else a constant index), and W"""
        def part(which, dtype=np.uint32):
            n = self.L.sim_bit_plan(self.h, which, None, 0)
            a = np.zeros(max(n, 1), dtype=np.uint32)
            self.L.sim_bit_plan(self.h, which, a.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), n)
            return a[:n].view(dtype)
        return {"code": part(0).reshape(-1, 32, 4), "inputs": part(1).reshape(-1, 3), "wide": part(2).reshape(-1, 3),
                "const_of_pos": part(3, np.int32), "W": self.W}

    def __del__(self):
        if getattr(self, "h", None):
            self.L.sim_bit_free(self.h)
            self.h = None


class SimGraph:
    """ctypes wrapper over tests/csrc/plan_host_sim.cpp"""

    def __init__(self, data: bytes, n_regs=24, fuse=True, div_batch=0, narrow=True, pow5=True, max_terms=0):
        self.L = sim_lib()
        err = ctypes.create_string_buffer(512)
        assert 0 <= div_batch <= 0xFF and 0 <= max_terms <= 0xFF
        flags = int(bool(fuse)) | (0 if narrow else 2) | (0 if pow5 else 4) | (int(div_batch) << 8) | (int(max_terms) << 16)
        self.h = self.L.sim_load2(data, len(data), n_regs, flags, err, 512)
        if not self.h:
            raise ValueError(err.value.decode())
        info = (ctypes.c_uint64 * 19)()
        self.L.sim_info(self.h, info)
        keys = ["n_nodes", "I", "W", "n_instrs", "n_regs", "n_spill", "spill_ld", "spill_st", "max_live", "n_consts",
                "live_ops", "graph_ops", "n_dot", "n_dot_mac", "inversions", "div_nodes", "slots", "n_mul", "n_addsub"]
        self.info = dict(zip(keys, [int(x) for x in info]))
        info2 = (ctypes.c_uint64 * 4)()
        self.L.sim_info2(self.h, info2)
        self.info["narrow_instrs"], self.info["widen"], self.info["n_spill_narrow"] = int(info2[0]), int(info2[1]), int(info2[2])
        self.info["pow5"] = int(info2[3])

    def eval(self, inputs):
        """inputs: list of I ints -> (witness list, status bits)"""
        assert len(inputs) == self.info["I"]
        out = ctypes.create_string_buffer(32 * self.info["W"])
        st = self.L.sim_eval(self.h, pack_u256(inputs), out)
        assert st >= 0, "malformed plan"
        return unpack_u256(out.raw), int(st)

    def eval_latency(self, inputs, mode=0, n_warps=0, n_slow_warps=0, slow_levels=0, split_dot=True, fuse=True, packet_slots=0, chain=True,
                     dataflow=False, sbox_links=True, exclusive_warp0=False, max_slots=0, coverage=False):
        """latency-mode plan on the host simulator -> (witness list, info dict).  Level plan: mode 0 / 1 = the slow-warp
        jobs run as early / as late as the protocol allows.  dataflow=True: per-warp packet streams with wait vectors;
        mode 0 / 1 / >= 2 = the next runnable warp is the lowest / the highest / a pseudo-random one
        (tests/csrc/plan_host_sim.cpp).  max_slots = 0: the LatencyOptions default.  A plan that does not compile raises
        ValueError with the compiler's message.  coverage=True returns (witness, info, coverage) with the coverage of
        this call (latency_coverage)."""
        out = ctypes.create_string_buffer(32 * self.info["W"])
        o8 = (ctypes.c_uint64 * 10)()
        opts = (ctypes.c_uint32 * 11)(n_warps, n_slow_warps, slow_levels, int(split_dot), int(fuse), packet_slots, int(chain), int(dataflow),
                                      int(sbox_links), int(exclusive_warp0), max_slots)
        cov = (ctypes.c_uint64 * len(LAT_COV_KEYS))()
        rc = self.L.sim_eval_latency3(self.h, pack_u256(inputs), out, o8, mode, opts, cov)
        if rc == -2:
            raise ValueError(self.L.sim_error(self.h).decode())
        assert rc == 0, f"latency plan failed ({rc})"
        keys = ["n_levels", "n_slots", "n_instrs", "max_width", "status", "est_cycles", "n_split", "slow_levels", "n_chained", "n_sbox_links"]
        if dataflow:
            keys[6], keys[8] = "n_rows", "n_waits"
        res = (unpack_u256(out.raw), dict(zip(keys, [int(x) for x in o8])))
        return res + (latency_coverage(list(cov)),) if coverage else res

    def code(self) -> np.ndarray:
        """the compiled program: uint32 [n_slots, 4] (isa.h: x, y, z, w of each 16-byte slot)"""
        n = self.L.sim_code(self.h, None, 0)
        out = np.zeros((n, 4), dtype=np.uint32)
        self.L.sim_code(self.h, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)), n)
        return out

    def inputs_from_json(self, js: str):
        buf = ctypes.create_string_buffer(32 * self.info["I"])
        err = ctypes.create_string_buffer(512)
        r = self.L.sim_inputs(self.h, js.encode(), buf, err, 512)
        if r:
            raise ValueError(err.value.decode())
        return unpack_u256(buf.raw)

    def reserialize(self) -> bytes:
        n = self.L.sim_reserialize(self.h, None, 0)
        buf = ctypes.create_string_buffer(n)
        self.L.sim_reserialize(self.h, buf, n)
        return buf.raw

    def __del__(self):
        if getattr(self, "h", None):
            self.L.sim_free(self.h)
            self.h = None


# ---- plan options, program coverage and corpora of the throughput interpreter ------------------------------------------
# The options the product reads when a graph is loaded (engine.cu: Engine::init_plan) or launched (GW_HOT_CONSTS,
# GW_THREADS).  "half" in GW_HOT_CONSTS stands for half of the graph's constant table.
PLAN_VARIANTS = [
    ("defaults", {}),
    ("div_batch_1", {"GW_DIV_BATCH": "1"}), ("div_batch_2", {"GW_DIV_BATCH": "2"}),
    ("div_batch_3", {"GW_DIV_BATCH": "3"}), ("div_batch_16", {"GW_DIV_BATCH": "16"}),
    ("no_dot", {"GW_FUSE_DOT": "0"}),
    ("max_terms_2", {"GW_MAX_TERMS": "2", "GW_REGS": "24"}), ("max_terms_16", {"GW_MAX_TERMS": "16", "GW_REGS": "24"}),
    ("no_narrow", {"GW_NARROW": "0"}), ("no_pow5", {"GW_FUSE_POW5": "0"}),
    ("regs_4", {"GW_REGS": "4"}), ("regs_5", {"GW_REGS": "5"}), ("regs_40", {"GW_REGS": "40"}),
    ("hot_0", {"GW_HOT_CONSTS": "0"}), ("hot_1", {"GW_HOT_CONSTS": "1"}), ("hot_half", {"GW_HOT_CONSTS": "half"}),
    ("threads_32", {"GW_THREADS": "32"}), ("threads_96", {"GW_THREADS": "96"}),
]


def sim_options(env: dict) -> dict:
    """SimGraph keyword arguments that compile the program the product compiles under `env` (PlanOptions defaults)"""
    return dict(n_regs=int(env.get("GW_REGS", 12)), fuse=env.get("GW_FUSE_DOT", "1") != "0", div_batch=int(env.get("GW_DIV_BATCH", 0)),
                narrow=env.get("GW_NARROW", "1") != "0", pow5=env.get("GW_FUSE_POW5", "1") != "0", max_terms=int(env.get("GW_MAX_TERMS", 0)))


# A constant at this table index or above is read with __ldg at every launch shape on a GPU with 227 KB of shared memory
# per block: the hot prefix is what the smallest CTA (32 threads: one 1 KB instruction ring, 4 registers of 1 KB) leaves.
COLD_CONST = (227 * 1024 - 1024 - 4 * 1024) // 32

_OP_DOT, _OP_SHRAND, _OP_SPILL_ST, _OP_SPILL_LD, _OP_INV, _OP_NZ1, _OP_POW5 = 53, 54, 49, 50, 36, 37, 55
_F_A, _F_B, _F_C, _F_NARROW = 1 << 8, 1 << 9, 1 << 10, 1 << 12


def plan_coverage(code: np.ndarray) -> dict:
    """What a compiled program (SimGraph.code()) makes eval_batch_kernel do:
    dot_cross   {(terms, header offset in its 32-slot block)} of the OP_DOTs whose slots reach the next block
    narrow_spill_st / narrow_spill_ld   narrow (8-byte) spill moves
    inv_groups  {number of OP_NZ1 in front of each OP_INV}: the sizes of the batched Div groups
    pow5        OP_POW5 instructions
    max_const_wide / max_const_narrow   the highest constant-table index read by a wide / a narrow instruction"""
    cov = dict(dot_cross=set(), narrow_spill_st=0, narrow_spill_ld=0, inv_groups=set(), pow5=0, max_const_wide=-1, max_const_narrow=-1)
    pc, nz = 0, 0
    n = len(code)
    while pc < n:
        x, y, z, w = (int(v) for v in code[pc])
        op, narrow = x & 0xFF, bool(x & _F_NARROW)
        length = 1 + (((y & 0xFF) + 1) >> 1) if op == _OP_DOT else 1
        consts = []
        if op == _OP_DOT:
            nt = y & 0xFF
            if pc % 32 + length >= 32:
                cov["dot_cross"].add((nt, pc % 32))
            for t in range(nt):
                sl = code[pc + 1 + (t >> 1)]
                lo, ci = (int(sl[2]), int(sl[3])) if t & 1 else (int(sl[0]), int(sl[1]))
                if lo & 0xF in (0, 3):
                    consts.append(ci)
        elif op == _OP_SHRAND:
            consts.append(z >> 8)
        elif op not in (_OP_POW5, _OP_SPILL_ST, _OP_SPILL_LD):
            consts += [v for f, v in ((_F_A, y), (_F_B, z), (_F_C, w)) if x & f]
        if consts:
            key = "max_const_narrow" if narrow else "max_const_wide"
            cov[key] = max(cov[key], *consts)
        if narrow and op == _OP_SPILL_ST:
            cov["narrow_spill_st"] += 1
        if narrow and op == _OP_SPILL_LD:
            cov["narrow_spill_ld"] += 1
        if op == _OP_NZ1:
            nz += 1
        if op == _OP_INV:
            cov["inv_groups"].add(nz)
            nz = 0
        cov["pow5"] += op == _OP_POW5
        pc += length
    return cov


def merge_coverage(a: dict, b: dict) -> dict:
    out = {}
    for k, v in a.items():
        out[k] = v | b[k] if isinstance(v, set) else max(v, b[k]) if k.startswith("max_") else v + b[k]
    return out


COVERAGE_FEATURES = ("dot_cross", "narrow_spill", "inv_16", "pow5", "cold_consts")


def assert_plan_coverage(cov: dict, features=COVERAGE_FEATURES):
    """the device paths the corpora below exist to reach (tests/test_gpu_plan_matrix.py), by feature:
    dot_cross    an OP_DOT of every term count 9..16 crossing a ring block from every offset it can cross from
    narrow_spill narrow spill stores and loads
    inv_16       a batched inversion of 16 Div nodes (OP_NZ1 x 16, OP_INV)
    pow5         OP_POW5
    cold_consts  wide and narrow reads of constants outside every shared-memory prefix"""
    if "dot_cross" in features:
        for nt in range(9, 17):
            length = 1 + ((nt + 1) >> 1)
            missing = set(range(32 - length, 32)) - {o for t, o in cov["dot_cross"] if t == nt}
            assert not missing, f"no OP_DOT of {nt} terms crossing a ring block from offsets {sorted(missing)}"
    if "narrow_spill" in features:
        assert cov["narrow_spill_st"] > 0 and cov["narrow_spill_ld"] > 0, "no narrow spill moves"
    if "inv_16" in features:
        assert 16 in cov["inv_groups"], f"no batched inversion of 16 Div nodes: {sorted(cov['inv_groups'])}"
    if "pow5" in features:
        assert cov["pow5"] > 0, "no OP_POW5"
    if "cold_consts" in features:
        assert min(cov["max_const_wide"], cov["max_const_narrow"]) >= COLD_CONST, "no constant outside every hot prefix"


# what each plan variant of PLAN_VARIANTS must reach on the corpus of test_plan_sim.matrix_corpus
VARIANT_FEATURES = {"defaults": ("pow5", "cold_consts"), "div_batch_16": ("inv_16",), "max_terms_16": ("dot_cross", "pow5", "cold_consts"),
                    "regs_4": ("narrow_spill", "cold_consts"), "regs_5": ("narrow_spill",), "hot_0": ("cold_consts",)}


def dot_ladder_graph(t: int, n_blocks=34):
    """Linear combinations of exactly t terms (OP_DOT under GW_MAX_TERMS >= t), each preceded by a run of cheap witness-output
    instructions.  A block (run + OP_DOT) is 33 slots mod 32, so the OP_DOT headers of consecutive blocks sit at consecutive
    offsets of the 32-slot ring blocks: every offset, crossing included.  Terms are Mul(x, c) at their worst (x = M - 1 in the
    worst-case rows, c = M - 1 or the constant whose Montgomery form is M - 1: the largest products), mixed with +-x plain
    terms and constant terms within the compiler's bound on the reduced sum."""
    r_inv = pow(1 << 256, -1, M)
    cmax = (M - 1) * r_inv % M                 # prescale(cmax) = M - 1; prescale(M - cmax, subtracted) = M - 1
    rnd = random.Random(31337 + t)
    nodes = [(po.K_INPUT, i) for i in range(7)]

    def add(node):
        nodes.append(node)
        return len(nodes) - 1
    wit = [0]
    length = 1 + ((t + 1) >> 1)
    run = (33 - length) % 32
    for k in range(n_blocks):
        for i in range(run if k else max(run, 6)):          # the first run reads every input (their loads come first)
            wit.append(add((po.K_DUO, po.DUO["Add" if i % 2 else "Sub"], 1 + i % 6, 1 + (i + 1) % 6)))
        q = k % 3 if t >= 3 else 0                          # plain terms, within the bound of plan.cpp: dot_bound
        while q and 1 + 0.18906 * (t - q) + q > 5.2:
            q -= 1
        n_const = 1 if k % 4 == 3 and t - q >= 2 else 0
        lc = None
        for j in range(t):
            sub = j % 2 == 1
            if j < t - q - n_const:
                mode = k % 4
                c = {0: M - 1, 1: (M - cmax) if sub else cmax, 2: cmax if j % 3 else M - 1}.get(mode, random_value(rnd))
                cn, x = add((po.K_CONST, c)), 1 + j % 3
                term = add((po.K_DUO, po.DUO["Mul"], x, cn) if j % 2 == 0 else (po.K_DUO, po.DUO["Mul"], cn, x))
            elif j < t - n_const:
                term = 4 + j % 3
            else:
                term = add((po.K_CONST, random_value(rnd)))
            lc = term if lc is None else add((po.K_DUO, po.DUO["Sub" if sub else "Add"], lc, term))
        wit.append(lc)
    return nodes, wit, {"x": (1, 6)}


def div_group_graph(k: int):
    """k independent Div nodes of one division level: numerators are inputs 1..k, denominators inputs k+1..2k"""
    nodes = [(po.K_INPUT, i) for i in range(2 * k + 1)]
    for j in range(k):
        nodes.append((po.K_DUO, po.DUO["Div"], 1 + j, 1 + k + j))
    return nodes, list(range(len(nodes))), {"x": (1, 2 * k)}


def div_group_rows(k: int, rnd: random.Random) -> list:
    """every pattern of zero denominators for k <= 4; first only, last only, all and none above.  A zero is 0, M or 2 M
    in turn (the raw values reduce to 0)"""
    pats = list(range(1 << k)) if k <= 4 else [1, 1 << (k - 1), (1 << k) - 1, 0]
    zeros = [0, M, 2 * M]
    rows = []
    for p in pats:
        for rep in range(2):
            num = [random_value(rnd) if rep else M - 1 for _ in range(k)]
            den = [zeros[(j + rep) % 3] if (p >> j) & 1 else (random_value(rnd) or 1) if rep else M - 1 - j for j in range(k)]
            rows.append([1] + num + den)
    return rows


def narrow_limit_graphs():
    """the shapes of test_plan_sim.test_narrow_range_limits: sums, products and negations at the +-2^62 edge of the narrow
    domain.  Returns [(bits, nodes, witness, input map)]"""
    D = po.DUO
    out = []
    for bits in (30, 31, 32, 40, 61, 62):
        mask = (1 << bits) - 1
        nodes = [(po.K_INPUT, 0), (po.K_INPUT, 1), (po.K_INPUT, 2), (po.K_CONST, mask), (po.K_CONST, 0), (po.K_CONST, 1)]
        nodes += [(po.K_DUO, D["Band"], 1, 3), (po.K_DUO, D["Band"], 2, 3)]
        a, b = 6, 7
        nodes += [(po.K_DUO, D["Mul"], a, b), (po.K_DUO, D["Sub"], 4, a), (po.K_DUO, D["Sub"], b, a), (po.K_DUO, D["Mul"], 9, b),
                  (po.K_DUO, D["Add"], a, b), (po.K_DUO, D["Add"], 12, 12), (po.K_DUO, D["Mul"], 10, 10), (po.K_UNO, 0, 8),
                  (po.K_DUO, D["Lt"], 9, 10), (po.K_DUO, D["Geq"], 10, 4), (po.K_TRES, 0, 10, 9, 13), (po.K_DUO, D["Sub"], 18, 5)]
        out.append((bits, nodes, list(range(len(nodes))), {"x": (1, 2)}))
    return out


def narrow_limit_values(bits: int) -> list:
    mask = (1 << bits) - 1
    return [mask, mask + 1, (1 << 62) - 1, 1 << 62, M - (1 << 62), M - 1, (1 << 256) - 1, 0, 1]


def const_heavy_graph(rnd: random.Random, n_wide=6400, n_narrow=1600, chain=64):
    """Several thousand distinct constants, each read once, so that the constant table is longer than any shared-memory
    prefix (COLD_CONST): long sums of Mul(x, c) (wide OP_DOT terms, or OP_MUL with a constant operand without fusion) and
    narrow chains over 16-bit slices of the inputs with constant addends, factors and comparisons (8-byte reads)."""
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(7)]

    def add(node):
        nodes.append(node)
        return len(nodes) - 1
    mask = add((po.K_CONST, 0xFFFF))
    seen = set()

    def fresh(lo, hi):
        while True:
            v = rnd.randrange(lo, hi)
            if v not in seen:
                seen.add(v)
                return add((po.K_CONST, v))
    sl = [add((po.K_DUO, D["Band"], 1 + i, mask)) for i in range(6)]
    wit = [0]
    lc = acc = None
    every = max(1, n_wide // n_narrow)
    for j in range(n_wide):                              # the two kinds interleave over the whole table
        term = add((po.K_DUO, D["Mul"], 1 + j % 6, fresh(1 << 64, M)))
        lc = term if lc is None else add((po.K_DUO, D["Add" if j % 5 else "Sub"], lc, term))
        if (j + 1) % chain == 0:
            wit.append(lc)
            lc = None
        if j % every:
            continue
        i = j // every
        s = sl[i % 6]
        kind = i % 4
        if kind == 0:
            term = add((po.K_DUO, D["Add"], s, fresh(2, 1 << 40)))
        elif kind == 1:
            term = add((po.K_DUO, D["Mul"], s, fresh(2, 1 << 20)))
        elif kind == 2:
            term = add((po.K_DUO, D["Lt"], s, fresh(2, 1 << 17)))
        else:
            term = add((po.K_DUO, D["Sub"], fresh(2, 1 << 40), s))
        acc = term if acc is None else add((po.K_DUO, D["Add"], acc, term))
        if (i + 1) % chain == 0:
            wit.append(acc)
            acc = None
    return nodes, wit, {"x": (1, 6)}


def matrix_row(rnd: random.Random, n_in: int) -> list:
    """one input row of the matrix tests: field values, raw 256-bit values >= M, edge values, neighbours of +-2^62"""
    def one():
        r = rnd.random()
        if r < 0.45:
            return random_value(rnd)
        if r < 0.6:
            return rnd.randrange(M, 1 << 256)
        if r < 0.8:
            return rnd.choice(EDGE)
        return rnd.choice([(1 << 62) + d for d in (-2, -1, 0, 1)] + [M - (1 << 62) + d for d in (-1, 0, 1, 2)])
    return [1] + [one() for _ in range(n_in)]


# ---- latency mode: options, coverage and corpus of eval_latency_kernel / eval_dataflow_kernel ---------------------------
# The options Engine::calc_latency reads when a graph's latency plan is first built (engine.cu: Engine::run_latency).
# Every variant runs the generic kernels (GW_LAT_BIT=0) with all other latency options at their defaults.
LATENCY_ENV_KEYS = ("GW_LAT_MODE", "GW_LAT_WARPS", "GW_LAT_SLOW_WARPS", "GW_LAT_EXCL", "GW_LAT_D", "GW_LAT_SPLIT", "GW_LAT_FUSE", "GW_LAT_LINKS",
                    "GW_LAT_CHAIN", "GW_LAT_BIT", "GW_LAT_WATCHDOG", "GW_LAT_DBG", "GW_LAT_CLOCKS", "GW_SINGLE_MODE")
_LAT_BOTH = [("defaults", {}), ("serial", {"GW_LAT_WARPS": "1", "GW_LAT_SLOW_WARPS": "1", "GW_LAT_D": "1"}), ("d_2", {"GW_LAT_D": "2"}),
             ("no_fuse", {"GW_LAT_FUSE": "0"}), ("links_2", {"GW_LAT_LINKS": "2"})]
LATENCY_VARIANTS = (
    [("df_" + n, e) for n, e in _LAT_BOTH] + [("level_" + n, dict(e, GW_LAT_MODE="level")) for n, e in _LAT_BOTH]
    + [("df_warps_12", {"GW_LAT_WARPS": "8", "GW_LAT_SLOW_WARPS": "4"}), ("df_excl", {"GW_LAT_EXCL": "1"}),
       ("df_excl_w7s3", {"GW_LAT_EXCL": "1", "GW_LAT_WARPS": "7", "GW_LAT_SLOW_WARPS": "3"}),
       ("df_excl_w8s4", {"GW_LAT_EXCL": "1", "GW_LAT_WARPS": "8", "GW_LAT_SLOW_WARPS": "4"}),
       ("df_no_chain", {"GW_LAT_CHAIN": "0"}), ("df_no_split", {"GW_LAT_SPLIT": "0"}), ("df_links_0", {"GW_LAT_LINKS": "0"})]
    + [("level_warps_12", {"GW_LAT_MODE": "level", "GW_LAT_WARPS": "10", "GW_LAT_SLOW_WARPS": "1"}),
       ("level_d_200", {"GW_LAT_MODE": "level", "GW_LAT_D": "200"}),
       ("level_no_split_chain", {"GW_LAT_MODE": "level", "GW_LAT_SPLIT": "0", "GW_LAT_CHAIN": "0"})])
LATENCY_VARIANTS = [(n, dict(e, GW_LAT_BIT="0")) for n, e in LATENCY_VARIANTS]

B200_SMEM_OPTIN = 232448      # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200
LAT_RING_SLOTS = 128          # engine.cu: packet ring stage / dataflow chunk (16 B slots)
LAT_CTRL_BYTES, DF_CTRL_BYTES = 320, 384


def latency_sim_options(env: dict, smem_optin=B200_SMEM_OPTIN) -> dict:
    """SimGraph.eval_latency keyword arguments that compile the latency plan the product compiles under `env` on a device
    with `smem_optin` bytes of opt-in shared memory per block (engine.cu: Engine::run_latency)"""
    geti = lambda k, d: int(env[k]) if env.get(k) else d
    dataflow = env.get("GW_LAT_MODE") != "level"
    n_warps, n_slow = geti("GW_LAT_WARPS", 6 if dataflow else 7), geti("GW_LAT_SLOW_WARPS", 3 if dataflow else 4)
    excl = geti("GW_LAT_EXCL", 0) != 0
    if dataflow:                      # rings of every physical warp, the empty ones the exclusive warp 0 leaves included
        rings = min(12, n_warps + n_slow + (2 if excl else 0))
        max_slots = min((smem_optin // 16 - DF_CTRL_BYTES // 16 - rings * 3 * LAT_RING_SLOTS) // 2, 0xFFFF)
    else:                             # one ring per main warp
        max_slots = min((smem_optin // 16 - LAT_CTRL_BYTES // 16 - n_warps * 3 * LAT_RING_SLOTS) // 2, 0xFFFF)
    links = geti("GW_LAT_LINKS", 1)
    return dict(dataflow=dataflow, n_warps=n_warps, n_slow_warps=n_slow, slow_levels=geti("GW_LAT_D", 0), split_dot=geti("GW_LAT_SPLIT", 1) != 0,
                fuse=geti("GW_LAT_FUSE", 1) != 0, packet_slots=LAT_RING_SLOTS, chain=geti("GW_LAT_CHAIN", 1) != 0,
                sbox_links=2 if links == 2 else int(links != 0), exclusive_warp0=excl, max_slots=max_slots)


# tests/csrc/plan_host_sim.cpp: enum LatCov.  Masks become sets, "max_" keys are maxima, the others counts (merge_coverage)
LAT_COV_KEYS = ("dot_shapes", "max_dot_terms", "dot_kinds", "slow_widths", "slow_ops", "slow_const", "pow5", "pow4", "muladd", "shrand", "out",
                "tern_const", "muladd_const", "max_chain", "levels_mod3", "n_levels", "empty_packet", "chunk_full", "chunk_zero", "max_wait",
                "max_phys_warps", "max_n_slots", "max_slots", "dot_shapes_m1")
_LAT_COV_MASKS = ("dot_shapes", "dot_kinds", "slow_widths", "slow_ops", "levels_mod3", "n_levels", "dot_shapes_m1")


def latency_coverage(words) -> dict:
    """the coverage record of the latency simulator as a dict; at_capacity counts plans whose value file is exactly full"""
    raw = dict(zip(LAT_COV_KEYS, (int(w) for w in words)))
    cov = {k: ({b for b in range(64) if (v >> b) & 1} if k in _LAT_COV_MASKS else v) for k, v in raw.items() if k != "max_slots"}
    cov["at_capacity"] = int(raw["max_n_slots"] == raw["max_slots"])
    return cov


_OP_DIV, _OP_POW, _OP_IDIV, _OP_MOD = 1, 4, 5, 6
DOT_SHAPES = {1 | (n << 1) | (a << 3) | (c << 4) for n in (1, 2) for a in (0, 1) for c in (0, 1)}
LATENCY_FEATURES = ("dot_shapes", "dot_generic", "slow_jobs", "slow_const", "ops", "sbox", "chains", "levels", "empty_packet", "chunks", "phys_12",
                    "warps_12")


def assert_latency_coverage(cov: dict, features=LATENCY_FEATURES):
    """the kernel paths the latency corpus exists to reach (tests/test_gpu_latency_matrix.py), by feature:
    dot_shapes   every straight-line OP_DOT shape: 1-2 products x an added value or not x a constant or not, each of them
                 with a first-product constant of M - 1 in the packet (the largest product)
    dot_generic  generic-loop OP_DOTs with all four term kinds, one of 8 terms (the most a latency plan puts in one)
    slow_jobs    slow-warp jobs of 32 lanes and of fewer, running Div, Idiv, Mod and Pow
    slow_const   slow-warp instructions with a constant operand
    ops          OP_POW5, OP_SHRAND, OP_OUT and an OP_TERN with a constant operand
    sbox         OP_POW4, OP_MULADD and an OP_MULADD with a constant operand (S-box link rewrite)
    chains       level plan: a lane running two or more headers of one packet
    levels       plans of 0, 1 and 2 levels mod 3, and of 1 and of 2 levels
    empty_packet level plan: a main warp without an instruction at some level
    chunks       dataflow plan: chunks filled to their last slot and chunks ended by a zero descriptor
    phys_12      dataflow plan: 12 physical warps (a ring and a progress counter each, the empty ones included)
    warps_12     dataflow plan: 12 physical warps, and a packet that waits for 11 other warps"""
    if "dot_shapes" in features:
        missing = DOT_SHAPES - cov["dot_shapes"]
        assert not missing, f"straight-line OP_DOT shapes never executed: {sorted(missing)}"
        missing = DOT_SHAPES - cov["dot_shapes_m1"]
        assert not missing, f"straight-line OP_DOT shapes never executed with a constant of M - 1: {sorted(missing)}"
    if "dot_generic" in features:
        assert cov["dot_kinds"] >= {0, 1, 2, 3}, f"generic OP_DOT term kinds executed: {sorted(cov['dot_kinds'])}"
        assert cov["max_dot_terms"] >= 8, f"no generic OP_DOT of 8 terms: {cov['max_dot_terms']}"
    if "slow_jobs" in features:
        assert 32 in cov["slow_widths"] and min(cov["slow_widths"] or {32}) < 32, f"slow-warp job widths: {sorted(cov['slow_widths'])}"
        missing = {_OP_DIV, _OP_POW, _OP_IDIV, _OP_MOD} - cov["slow_ops"]
        assert not missing, f"opcodes never run by a slow warp: {sorted(missing)}"
    if "slow_const" in features:
        assert cov["slow_const"] > 0, "no slow-warp instruction reads a constant"
    if "ops" in features:
        for k in ("pow5", "shrand", "out", "tern_const"):
            assert cov[k] > 0, f"no {k}"
    if "sbox" in features:
        for k in ("pow4", "muladd", "muladd_const"):
            assert cov[k] > 0, f"no {k}"
    if "chains" in features:
        assert cov["max_chain"] >= 2, "no lane chain"
    if "levels" in features:
        assert cov["levels_mod3"] == {0, 1, 2}, f"level counts mod 3: {sorted(cov['levels_mod3'])}"
        assert {1, 2} <= cov["n_levels"], f"no plan of 1 or of 2 levels: {sorted(b for b in cov['n_levels'] if b < 8)}"
    if "empty_packet" in features:
        assert cov["empty_packet"] > 0, "no level at which a main warp is idle"
    if "chunks" in features:
        assert cov["chunk_full"] > 0, "no chunk filled to its last slot"
        assert cov["chunk_zero"] > 0, "no chunk ended by a zero descriptor"
    if "phys_12" in features or "warps_12" in features:
        assert cov["max_phys_warps"] == 12, f"physical warps: {cov['max_phys_warps']}"
    if "warps_12" in features:
        assert cov["max_phys_warps"] == 12, f"physical warps: {cov['max_phys_warps']}"
        assert cov["max_wait"] == 11, f"widest wait vector: {cov['max_wait']} warps"


_LAT_COMMON = ("slow_jobs", "slow_const", "levels")
_LAT_FUSED = _LAT_COMMON + ("dot_shapes", "dot_generic", "ops")
_LAT_DF = _LAT_FUSED + ("chunks",)
_LAT_LEVEL = _LAT_FUSED + ("chains", "empty_packet")
# what each variant of LATENCY_VARIANTS must reach on latency_corpus()
LATENCY_VARIANT_FEATURES = {
    "df_defaults": _LAT_DF, "df_serial": _LAT_DF, "df_d_2": _LAT_DF, "df_no_fuse": _LAT_COMMON + ("chunks",), "df_links_2": _LAT_DF + ("sbox",),
    "level_defaults": _LAT_LEVEL, "level_serial": _LAT_LEVEL, "level_d_2": _LAT_LEVEL, "level_no_fuse": _LAT_COMMON + ("chains", "empty_packet"),
    "level_links_2": _LAT_LEVEL + ("sbox",),
    "df_warps_12": _LAT_DF + ("warps_12",), "df_excl": _LAT_DF, "df_excl_w7s3": _LAT_DF + ("phys_12",), "df_excl_w8s4": _LAT_DF + ("warps_12",),
    "df_no_chain": _LAT_DF, "df_no_split": _LAT_DF, "df_links_0": _LAT_DF,
    "level_warps_12": _LAT_LEVEL, "level_d_200": _LAT_LEVEL, "level_no_split_chain": _LAT_FUSED + ("empty_packet",),
}


def slow_const_graph(k=12):
    """Idiv, Mod and Pow of the inputs with a constant divisor / exponent on either side, in groups of k per opcode and side
    (slow-warp jobs that read constants), next to k Div of inputs by inputs.  Constants: 0, 1, small, 2^64 + 1, M - 1."""
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(7)]
    consts = []
    for v in (0, 1, 3, 255, (1 << 64) + 1, M - 1, 7, M >> 3):
        nodes.append((po.K_CONST, v))
        consts.append(len(nodes) - 1)
    wit = [0]
    for op in ("Idiv", "Mod", "Pow"):
        for j in range(k):
            x, c = 1 + j % 6, consts[j % len(consts)]
            if op == "Pow":
                c = consts[2 + j % 2] if j % 3 else consts[j % 2]      # small exponents and a large base stay cheap on the oracle
            nodes.append((po.K_DUO, D[op], x, c))
            wit.append(len(nodes) - 1)
            nodes.append((po.K_DUO, D[op], c if op != "Pow" else consts[5 - j % 2], x if op != "Pow" else 1 + j % 2))
            wit.append(len(nodes) - 1)
    for j in range(k):
        nodes.append((po.K_DUO, D["Div"], 1 + j % 6, 1 + (j + 1) % 6))
        wit.append(len(nodes) - 1)
    return nodes, wit, {"x": (1, 6)}


def dot_shape_graph(n_copies=4):
    """Linear combinations of every straight-line OP_DOT shape -- c1 x1 [+ c2 x2] [+ x3] [+ k] -- with worst-case operands
    (constants M - 1 and the one whose Montgomery form is M - 1, as in dot_ladder_graph), and the same shapes with a
    subtracted value, which must take the generic loop.  Each combination is a witness value."""
    r_inv = pow(1 << 256, -1, M)
    cmax = (M - 1) * r_inv % M
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(7)]

    def add(node):
        nodes.append(node)
        return len(nodes) - 1
    wit = [0]
    for rep in range(n_copies):
        for n_mac in (1, 2):
            for plus in (0, 1, 2):                   # 0: no added value, 1: + x3, 2: - x3 (generic loop)
                for kc in (0, 1):
                    cs = [(M - 1, cmax), (cmax, M - 1)][rep % 2]
                    lc = add((po.K_DUO, D["Mul"], 1 + rep % 2, add((po.K_CONST, cs[0]))))
                    if n_mac == 2:
                        lc = add((po.K_DUO, D["Add"], lc, add((po.K_DUO, D["Mul"], add((po.K_CONST, cs[1])), 2 + rep % 3))))
                    if plus:
                        lc = add((po.K_DUO, D["Add" if plus == 1 else "Sub"], lc, 3 + rep % 4))
                    if kc:
                        lc = add((po.K_DUO, D["Add"], lc, add((po.K_CONST, [M - 1, cmax, M - cmax, 1][rep % 4]))))
                    wit.append(lc)
    return nodes, wit, {"x": (1, 6)}


def tern_muladd_graph():
    """TernCond with a constant in each operand position (and none), and Poseidon-style S-box links with constants, so that
    the forced S-box link rewrite emits OP_MULADD with a constant operand; every result is a witness value (OP_TERN and
    OP_MULADD store through a separate OP_OUT)"""
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(7)]

    def add(node):
        nodes.append(node)
        return len(nodes) - 1
    wit = [0]
    c0, c1, c5 = add((po.K_CONST, 0)), add((po.K_CONST, M - 1)), add((po.K_CONST, 5))
    for j in range(6):
        x, y, z = 1 + j % 6, 1 + (j + 1) % 6, 1 + (j + 2) % 6
        cond = add((po.K_DUO, D["Lt"], x, y)) if j % 2 else x
        for a, b, c in ((cond, y, z), (c0 if j % 3 else c1, y, z), (cond, c1, z), (cond, y, c5), (cond, c1, c5)):
            wit.append(add((po.K_TRES, 0, a, b, c)))
    # S-box links s -> s^5 -> c * s^5 [+ k] -> ^5 ...: a link without other terms leaves OP_MULADD a constant 0 to add
    s = 1
    for r in range(8):
        x2 = add((po.K_DUO, D["Mul"], s, s))
        x4 = add((po.K_DUO, D["Mul"], x2, x2))
        x5 = add((po.K_DUO, D["Mul"], x4, s))
        wit += [x2, x4, x5]
        s = add((po.K_DUO, D["Mul"], add((po.K_CONST, (r + 2) * 0x1234567 % M)), x5))
        if r % 2:
            s = add((po.K_DUO, D["Add"], s, add((po.K_CONST, M - 1 - r))))
        wit.append(s)
    return nodes, wit, {"x": (1, 6)}


def edge_graphs():
    """[(name, nodes, witness, input map)]: inputs only, constants only, one operation, and dependent chains of 1 .. 9
    operations whose every step is also a witness value (level counts of 0, 1 and 2 mod 3, 1 and 2 levels in total)"""
    D = po.DUO
    out = [("inputs_only", [(po.K_INPUT, i) for i in range(7)], [0, 3, 1, 6, 2], {"x": (1, 6)}),
           ("consts_only", [(po.K_INPUT, 0), (po.K_CONST, 7), (po.K_CONST, M - 1), (po.K_CONST, 0)], [0, 1, 2, 3, 1], {}),
           ("one_op", [(po.K_INPUT, i) for i in range(3)] + [(po.K_DUO, D["Mul"], 1, 2)], [3], {"x": (1, 2)})]
    for n in range(1, 10):
        nodes = [(po.K_INPUT, i) for i in range(3)]
        wit, v = [], 1
        for j in range(n):
            nodes.append((po.K_DUO, D["Mul"] if j % 2 else D["Add"], v, 2))
            v = len(nodes) - 1
            wit.append(v)
        out.append((f"chain_{n}", nodes, wit, {"x": (1, 2)}))
    return out


def wide_live_graph(k: int):
    """k values live at the same time: v_i = x_(i mod 6) + c_i at one level, then w_i = v_i * v_(i+1 mod k) at the next, the
    products only as witness values.  The latency plan's value file needs k slots plus a constant few."""
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(7)]
    vs = []
    for i in range(k):
        nodes.append((po.K_CONST, 1000003 * (i + 1)))
        nodes.append((po.K_DUO, D["Add"], 1 + i % 6, len(nodes) - 1))
        vs.append(len(nodes) - 1)
    wit = [0]
    for i in range(k):
        nodes.append((po.K_DUO, D["Mul"], vs[i], vs[(i + 1) % k]))
        wit.append(len(nodes) - 1)
    return nodes, wit, {"x": (1, 6)}


def latency_rows(rnd: random.Random, n_in: int, extra=()) -> list:
    """input rows of one latency-corpus graph: an opening row that none of the checked rows repeats, the edge rows (all
    M - 1, all 0, all 2^256 - 1), `extra` and matrix rows, in an order where consecutive witnesses differ"""
    edge = [[1] + [M - 1] * n_in, [1] + [0] * n_in, [1] + [(1 << 256) - 1] * n_in]
    return [matrix_row(rnd, n_in)] + [edge[0], matrix_row(rnd, n_in), edge[1], matrix_row(rnd, n_in), edge[2]] + list(extra) + [matrix_row(rnd, n_in) for _ in range(3)]


def latency_corpus():
    """The corpus of the latency matrix (tests/test_latency_plan.py on the simulator, tests/test_gpu_latency_matrix.py on the
    GPU): [(name, nodes, witness, input map, rows)].  The plan-option matrix corpus (test_plan_sim.matrix_corpus) with
    latency rows, slow-warp job widths of 31 .. 65, slow jobs with constants, every straight-line OP_DOT shape,
    TernCond / S-box links with constants, Boolean and field-bits graphs, and edge graphs."""
    from tests.test_bitplan import boolean_graph, field_bits_graph
    from tests.test_plan_sim import matrix_corpus
    rnd = random.Random(4242)
    out = []
    for name, nodes, wit, imap, rows in matrix_corpus():
        n_in = len(rows[0]) - 1
        if name.startswith("narrow_limits"):
            rows = rows[::7]
        out.append((name, nodes, wit, imap, latency_rows(rnd, n_in, rows[:24])))
    for k in (31, 32, 33, 64, 65):
        nodes, wit, imap = div_group_graph(k)
        out.append((f"div_group_{k}", nodes, wit, imap, [matrix_row(rnd, 2 * k)] + div_group_rows(k, rnd)))
    for name, (nodes, wit, imap) in (("slow_const", slow_const_graph()), ("dot_shapes", dot_shape_graph()), ("tern_muladd", tern_muladd_graph())):
        zeros = [[1] + [0, M, 2 * M] * 2, [1, 1, 2, 3, M + 1, 2, 3], [1] + [M, 2 * M, 0] * 2, [1, 3, 1, 2, 3, M + 1, 2]]   # zero and tiny divisors
        out.append((name, nodes, wit, imap, latency_rows(rnd, 6, zeros)))
    for j in range(2):
        nodes, wit, imap = boolean_graph(rnd, n_inputs=24, n_gates=300)
        out.append((f"boolean_{j}", nodes, wit, imap, [[1] + [rnd.randrange(2) for _ in range(24)] for _ in range(24)]))
        nodes, wit, imap = field_bits_graph(rnd)
        n_in = imap["x"][1] if "x" in imap else sum(ln for _, ln in imap.values())
        out.append((f"field_bits_{j}", nodes, wit, imap, [[1] + [0] * n_in] + [[1] + [random_value(rnd) if i < 3 else rnd.randrange(2) for i in range(n_in)] for _ in range(24)]))
    for name, nodes, wit, imap in edge_graphs():
        n_in = sum(ln for _, ln in imap.values())
        out.append((name, nodes, wit, imap, latency_rows(rnd, n_in)))
    return out


def assert_rows_expose_stores(name, want):
    """want: the oracle's witness rows [B, W, 32] of one graph, in call order, row 0 the opening row.  The latency entry point
    copies the witness out of a device buffer that every call of the graph reuses, so a store the kernel skips shows the
    previous call's value: every position that is not the same in all rows must change between two consecutive checked rows."""
    w = want.reshape(len(want), -1, 32)
    varies = (w != w[:1]).any(axis=2).any(axis=0)
    changes = (w[2:] != w[1:-1]).any(axis=2).any(axis=0) if len(w) > 2 else np.zeros_like(varies)
    hidden = np.nonzero(varies & ~changes)[0]
    assert len(hidden) == 0, f"{name}: witness positions {hidden[:8].tolist()} never change between consecutive checked rows"


# ---- bit-sliced path: coverage and corpus of bit_eval_kernel / bit_expand_kernel / bit_expand_wide_kernel ------------------
BIT_NO_SLOT, BIT_NO_POS, BIT_CONTRACT = 0xFFFF, 0xFFFFFFFF, 0xFFFFFFFF      # csrc/bitplan.hpp
BIT_CHUNK_SINGLE, BIT_CHUNK_BATCH = 16, 8                                   # engine.cu: steps per TMA chunk of a header ring


def bit_chunks(n_steps: int, ch: int) -> int:
    """header-ring chunks of a bit program (steps 1 .. n_steps - 1, engine.cu: bit_eval_kernel)"""
    return -(-(n_steps - 1) // ch)


def bit_plan_coverage(plan: dict) -> dict:
    """what the kernels do with one compiled bit plan (BitSimGraph.plan): sets of step residues and ring chunk counts, the
    LUTs per step, copies, slot reuse, wide planes and their plane counts, constants, unread contract inputs and the field
    input bits by limb.  Merge records with merge_coverage."""
    code, W = plan["code"], plan["W"]
    n_steps = len(code)
    cov = {"res4": {(n_steps - 1) % 4}, "res8": {(n_steps - 1) % 8}, "res16": {(n_steps - 1) % 16},
           "chunks8": {min(bit_chunks(n_steps, BIT_CHUNK_BATCH), 7)}, "chunks16": {min(bit_chunks(n_steps, BIT_CHUNK_SINGLE), 5)},
           "step_luts": set(), "copy": 0, "multi_pos": 0, "slot_reuse": 0, "wide_writes": 0}
    written = set(int(s) for s in plan["inputs"][:, 1] if s != BIT_NO_SLOT) | {0, 1}
    stored = {}                                      # slot -> its current plane is also at a witness position
    for st in range(1, n_steps):
        ops = code[st]
        x, y, z, w = (ops[:, k].astype(np.int64) for k in range(4))
        dst = z >> 16
        real = (dst != BIT_NO_SLOT) | (w != BIT_NO_POS)
        n = int(real.sum())
        cov["step_luts"].add("1" if n == 1 else "32" if n == 32 else "2-31" if n else "0")
        copy = real & (x == 0xAA) & (dst == BIT_NO_SLOT)
        cov["copy"] += int(copy.sum())
        for a in (y[copy] & 0xFFFF).tolist():
            cov["multi_pos"] += int(stored.get(a, False))
            stored[a] = True
        cov["wide_writes"] += int(((w != BIT_NO_POS) & (w >= W)).sum())
        for d, pos in zip(dst[dst != BIT_NO_SLOT].tolist(), w[dst != BIT_NO_SLOT].tolist()):
            cov["slot_reuse"] += int(d in written)
            written.add(d)
            stored[d] = pos != BIT_NO_POS and pos < W
    wide_np = [int(t[2]) for t in plan["wide"]]
    cov["wide_planes"] = {k for k in (2, 31, 32, 33, 254) if k in wide_np} | ({"225+"} if any(k >= 225 for k in wide_np) else set())
    cov["wide_m"] = {-(-k // 32) for k in wide_np}
    cov["consts"] = int((plan["const_of_pos"] >= 0).sum())
    inp = plan["inputs"]
    contract = inp[:, 2] == BIT_CONTRACT
    cov["contract_no_slot"] = int((contract & (inp[:, 1] == BIT_NO_SLOT)).sum())
    fbits = [int(b) for b in inp[~contract, 2]]
    cov["field_limbs"] = {b >> 5 for b in fbits}
    cov["field_bits"] = {b for b in fbits if b in (31, 32, 253)}
    return cov


BIT_COVERAGE = {"res4": set(range(4)), "res8": set(range(8)), "res16": set(range(16)), "chunks8": {1, 2, 3, 4, 7},
                "chunks16": {1, 2, 3, 4}, "step_luts": {"1", "2-31", "32"}, "wide_planes": {2, 31, 32, 33, 254, "225+"},
                "wide_m": set(range(1, 9)), "field_limbs": set(range(8)), "field_bits": {31, 32, 253}}
BIT_COUNTS = ("copy", "multi_pos", "slot_reuse", "wide_writes", "consts", "contract_no_slot")


def assert_bit_coverage(cov: dict):
    for k, want in BIT_COVERAGE.items():
        assert want <= cov[k], f"bit plan coverage: {k} lacks {sorted(want - cov[k], key=str)}"
    for k in BIT_COUNTS:
        assert cov[k] > 0, f"bit plan coverage: no {k}"


def wide_counts_graph():
    """Bits2Num sums of k bits for k = 31, 32, 33 and 64 .. 250 in steps (every iteration count of the wide expansion's plane
    loop), a Num2Bits input passed through as a witness (254 planes), 2 b (the narrowest wide value: a value of one plane is a
    plane position), a masked slice, constants and one bit at three witness positions"""
    D = po.DUO
    widths = (31, 32, 33, 64, 96, 128, 160, 192, 200, 225, 250)
    n_bits = 40
    nodes = [(po.K_INPUT, i) for i in range(n_bits + 2)]
    cache = {}

    def const(v):
        if v not in cache:
            nodes.append((po.K_CONST, v))
            cache[v] = len(nodes) - 1
        return cache[v]

    def duo(op, a, b):
        nodes.append((po.K_DUO, D[op], a, b))
        return len(nodes) - 1
    f = n_bits + 1                                      # a field input: taken apart, passed through
    wit = [0, f]
    fb = [duo("Band", duo("Shr", f, const(k)), const(1)) for k in range(254)]
    wit += [fb[31], fb[32], fb[253], fb[0]]
    for i, k in enumerate(widths):
        lc = const(0)
        for j in range(k):
            b = 1 + (i * 7 + j * 3) % n_bits if j % 2 == 0 else fb[(i * 11 + j) % 254]
            lc = duo("Add", lc, duo("Mul", b, const(1 << j)))
        wit.append(lc)
    x = duo("Mul", 1, 2)
    wit += [x, const(5), x, const(0), x, const(1), duo("Band", duo("Shr", f, const(100)), const((1 << 37) - 1)), duo("Mul", 3, const(2))]
    return nodes, wit, {"x": (1, n_bits + 1)}


def bit_chain_graph(k: int, n_in=64):
    """k values alive at once: v_i = x_a ^ x_b (distinct input pairs) at one level, w_i = v_i & v_(i+1 mod k) at the next, the
    w only as witness values.  The bit plan's plane file needs about k + n_in slots; its program ~2k/32 steps."""
    D = po.DUO
    nodes = [(po.K_INPUT, i) for i in range(n_in + 1)]
    nodes.append((po.K_CONST, 2))
    two = len(nodes) - 1
    vs = []
    pairs = ((a, b) for d in range(1, n_in) for a in range(1, n_in + 1 - d) for b in (a + d,))
    for _, (a, b) in zip(range(k), pairs):
        nodes.append((po.K_DUO, D["Mul"], a, b))
        nodes.append((po.K_DUO, D["Mul"], two, len(nodes) - 1))
        nodes.append((po.K_DUO, D["Add"], a, b))
        nodes.append((po.K_DUO, D["Sub"], len(nodes) - 1, len(nodes) - 2))
        vs.append(len(nodes) - 1)
    assert len(vs) == k, "not enough input pairs"
    wit = [0]
    for i in range(k):
        nodes.append((po.K_DUO, D["Mul"], vs[i], vs[(i + 1) % k]))
        wit.append(len(nodes) - 1)
    return nodes, wit, {"x": (1, n_in)}


_bit_corpus = None


def bit_corpus():
    """The corpus of the bit-sliced matrix (tests/test_gpu_bit_matrix.py): random Boolean
    and field-bits graphs picked by their simulator step counts so that util.bit_plan_coverage of the set is full (every
    residue of the step count mod 16, header rings of 1 .. 4 and >= 7 chunks), wide_counts_graph, and the golden SHA-256.
    Entries: (name, graph bytes)."""
    global _bit_corpus
    if _bit_corpus is not None:
        return _bit_corpus
    from tests.test_bitplan import boolean_graph, field_bits_graph
    out, cov = [], None
    rnd = random.Random(5150)

    def take(name, nodes, wit, imap, force=False, data=None):
        nonlocal cov
        data = data or po.serialize_graph(nodes, wit, imap)
        g = BitSimGraph(data)
        # (not eligible: a random word sum that can reach the modulus; no LUT and no field input: pure wiring, which the
        # engine leaves to the generic kernel)
        if not g.info["eligible"] or not (g.info["n_luts"] or g.info["has_field_inputs"]):
            assert not force, (name, g.reason)
            return
        c = bit_plan_coverage(g.plan())
        new = cov is None or any(not (c[k] <= cov[k]) for k in BIT_COVERAGE)
        if force or new:
            cov = c if cov is None else merge_coverage(cov, c)
            out.append((name, data))
    take("wide_counts", *wide_counts_graph(), force=True)
    take("field_bits", *field_bits_graph(rnd, n_field=2, n_bits=6, n_gates=60), force=True)
    # step counts 2 .. ~70 come from small graphs, long ones from big graphs: keep a graph when it adds a residue or a chunk count
    for t in range(400):
        if all(BIT_COVERAGE[k] <= cov[k] for k in ("res16", "chunks8", "chunks16", "step_luts")):
            break
        n_gates = (2, 4, 8, 12, 20, 30, 45, 60, 90, 140)[t % 10]
        take(f"boolean_{t}", *boolean_graph(rnd, n_inputs=rnd.choice([3, 5, 24, 70]), n_gates=n_gates))
    take("boolean_long", *boolean_graph(rnd, n_inputs=40, n_gates=700), force=True)
    take("sha256_512", None, None, None, force=True, data=golden_graph("circuit8_sha256_512"))
    assert_bit_coverage(cov)
    _bit_corpus = out
    return out
