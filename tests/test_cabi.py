"""The C-ABI shared library: loads without a GPU, exports every symbol include/graph_witness.h
declares, graph-level entry points that need no device work behave, part 1 of the header matches the
reference's declarations, and the plain-C example compiles and links against it.  No compute calls here
(no GPU in this suite)."""
import ctypes
import importlib
import os
import re
import subprocess

import pytest

from tests import util

HEADER = os.path.join(util.ROOT, "include", "graph_witness.h")


@pytest.fixture(scope="module")
def cwc():
    subprocess.check_call(["python", os.path.join(util.ROOT, "circom-witnesscalc_b200", "build.py")])
    return importlib.import_module("circom-witnesscalc_b200")


def test_exports_match_header(cwc):
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    declared = set(re.findall(r"\b(gw_[a-z_0-9]+)\s*\(", src)) - {"gw_free_status"}     # static inline in the header
    assert declared == set(cwc.EXPORTS)
    lib = ctypes.CDLL(cwc.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    out = subprocess.check_output(["nm", "-D", "--defined-only", cwc.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert declared <= exported


def test_graph_load_and_info_without_gpu(cwc):
    g = cwc.Graph(util.golden_graph("circuit9_authV2"))
    man = util.manifest()["circuit9_authV2"]
    assert g.n_inputs == man["n_inputs"] and g.n_witness == man["n_witness"] and g.info["n_nodes"] == man["n_nodes"]
    assert g.input_signals["gistMtp"][1] == 64 and g.input_signals["authClaim"][1] == 8
    assert g.info["n_div"] == man["stats"]["op_histogram"]["Div"]
    with pytest.raises(cwc.WitnessCalcError):
        cwc.Graph(b"wtns.graph.001" + b"\x00" * 3)
    assert cwc.wtns_from_witness([1, 2]) == util.po.wtns_from_witness([1, 2])


def test_null_argument_contract(cwc):
    """src/lib.rs:51-64: null inputs / graph / zero length -> return 1 with a message"""
    lib = ctypes.CDLL(cwc.LIB_PATH)
    st = cwc.gw_status_t()
    out, n = ctypes.c_void_p(), ctypes.c_size_t()
    lib.gw_calc_witness.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p),
                                    ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(cwc.gw_status_t)]
    for args, msg in (((None, b"x", 1), b"inputs is null"), ((b"{}", None, 1), b"graph_data is null"),
                      ((b"{}", b"x", 0), b"graph_data_len is 0")):
        assert lib.gw_calc_witness(*args, ctypes.byref(out), ctypes.byref(n), ctypes.byref(st)) == 1
        assert st.code == 1 and ctypes.string_at(st.error_msg) == msg
    assert lib.gw_calc_witness(None, b"x", 1, ctypes.byref(out), ctypes.byref(n), None) == 1     # status may be NULL (lib.rs:29)


def test_no_gpu_is_a_loud_error_not_a_fallback(cwc):
    if cwc.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(cwc.WitnessCalcError, match="no CUDA device|CUDA"):
        cwc.calc_witness_wtns(util.golden_inputs("circuit1"), util.golden_graph("circuit1"))


def test_product_does_not_link_or_import_the_oracle(cwc):
    out = subprocess.check_output(["ldd", cwc.LIB_PATH], text=True)
    assert "oracle" not in out
    pkg = os.path.join(util.ROOT, "circom-witnesscalc_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".h", ".hpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle/" not in txt and "import oracle" not in txt and "from oracle" not in txt, f


def test_header_part1_is_the_reference_abi(tmp_path):
    """tests/csrc/reference_abi_part1.c restates the reference header's drop-in declarations (SURVEY.md 8(b)) and compiles
    only if include/graph_witness.h matches them; a header with a changed constant or parameter type must not compile"""
    src = os.path.join(util.ROOT, "tests", "csrc", "reference_abi_part1.c")

    def compiles(root):
        r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Wextra", "-Werror", "-fsyntax-only",
                            os.path.join(root, "tests", "csrc", "reference_abi_part1.c")], capture_output=True, text=True)
        return r.returncode == 0, r.stderr
    ok, err = compiles(util.ROOT)
    assert ok, err
    hdr = open(HEADER).read()
    for k, (old, new) in enumerate((("ERROR = 1", "ERROR = 2"), ("char *error_msg;", "const char *error_msg;"),
                                    ("size_t *wtns_len,\n                const", "uint32_t *wtns_len,\n                const"),
                                    ("const gw_status_t *status);", "gw_status_t *status);"))):
        assert hdr.count(old) == 1, old
        root = tmp_path / str(k)
        (root / "include").mkdir(parents=True)
        (root / "tests" / "csrc").mkdir(parents=True)
        (root / "include" / "graph_witness.h").write_text(hdr.replace(old, new))
        (root / "tests" / "csrc" / "reference_abi_part1.c").write_text(open(src).read())
        assert not compiles(str(root))[0], new


def test_c_example_compiles_as_c99_and_links(cwc, tmp_path):
    """examples/calc_witness.c (plain C, includes "../include/graph_witness.h" like the reference's example) compiles
    without a warning as C99 and links against the library; wrong argc -> usage on stderr, exit 1"""
    exe = tmp_path / "calc_witness_example"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-o", str(exe),
                           os.path.join(util.ROOT, "examples", "calc_witness.c"), "-L" + os.path.dirname(cwc.LIB_PATH),
                           "-lcircom_witnesscalc", "-Wl,-rpath," + os.path.dirname(cwc.LIB_PATH)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 1 and "<inputs.json> <graph.bin> <witness.wtns>" in r.stderr
    assert os.path.exists(cwc.EXAMPLE_PATH)
    # CLI contract of the reference binary (calc-witness.rs:13-19): wrong argc -> usage on stderr, exit 1
    r = subprocess.run([cwc.CLI_PATH], capture_output=True, text=True)
    assert r.returncode == 1 and "Usage:" in r.stderr and "<graph.bin> <inputs.json> <witness.wtns>" in r.stderr


def test_info_struct_is_the_same_in_the_header_the_python_binding_and_the_rust_shim():
    """gw_graph_info_t is filled by the library: a binding with fewer fields would be written past its end"""
    import re
    hdr = open(os.path.join(util.ROOT, "include", "graph_witness.h")).read()
    end = hdr.index("} gw_graph_info_t;")
    body = hdr[hdr.rindex("typedef struct", 0, end):end]
    c_fields = re.findall(r"^\s*(uint64_t|uint32_t)\s+(\w+);", body, re.M)
    cwc = importlib.import_module("circom-witnesscalc_b200")
    py_fields = [(("uint64_t" if t is ctypes.c_uint64 else "uint32_t"), n) for n, t in cwc.gw_graph_info_t._fields_]
    assert c_fields == py_fields and len(c_fields) >= 24
    rs = open(os.path.join(util.ROOT, "rust-shim", "src", "ffi.rs")).read()
    rbody = rs[rs.index("pub struct gw_graph_info_t"):]
    rbody = rbody[:rbody.index("}")]
    rs_fields = [(("uint64_t" if t == "u64" else "uint32_t"), n) for n, t in re.findall(r"pub (\w+): (u64|u32),", rbody)]
    assert rs_fields == c_fields
