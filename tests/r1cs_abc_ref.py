"""Reference (pure Python) of the ABC vectors of witness rows (gw_r1cs_abc_*), over the R1CS dicts of
tests/r1cs_ref.py, and the host build of the ABC kernel's per-constraint step, for the tests and the benchmark.

  plain layout    n = m:  A[k] = <A_k,w>, B[k] = <B_k,w>, C[k] = <C_k,w> with witness values reduced mod M
  Groth16 layout  n = the smallest power of two >= m + n_pub + 1 (n_pub = n_pub_out + n_pub_in); entry m + s,
                  s = 0 .. n_pub, has A = w_s and B = C = 0; the rest of the domain is zero (snarkjs zkey_new)
"""
from tests.r1cs_ref import M, lc_value


def abc_len(r1cs, groth16=False):
    """entries per ABC vector: m, or for Groth16 the smallest power of two >= m + n_pub + 1"""
    m = len(r1cs["constraints"])
    if not groth16:
        return m
    need = m + r1cs.get("n_pub_out", 0) + r1cs.get("n_pub_in", 0) + 1
    n = 1
    while n < need:
        n *= 2
    return n


def abc_ref(r1cs, witness, groth16=False):
    """(A, B, C): lists of n values, in the layout of the module docstring"""
    w = [v % M for v in witness]
    A, B, C = ([lc_value(con[i], w) for con in r1cs["constraints"]] for i in range(3))
    n = abc_len(r1cs, groth16)
    n_pub = r1cs.get("n_pub_out", 0) + r1cs.get("n_pub_in", 0)
    for j in range(len(A), n):
        s = j - len(r1cs["constraints"])
        A.append(w[s] if s <= n_pub else 0)
        B.append(0)
        C.append(0)
    return A, B, C


_host = {}


def abc_host_lib(emulate_ptx=False):
    """tests/csrc/r1cs_abc_host_api.cpp: the ABC kernel's per-constraint step (csrc/r1cs_eval.cuh), built for the host
    (emulate_ptx=True: with the device formulations of field.cuh)"""
    import ctypes
    import os
    from tests import util
    if emulate_ptx not in _host:
        src = [os.path.join(util.ROOT, "tests", "csrc", "r1cs_abc_host_api.cpp")] + [
            os.path.join(util.CSRC, f) for f in ("r1cs.cpp", "graph.cpp", "plan.cpp")]
        L = ctypes.CDLL(util._build("libr1csabc_ptx.so" if emulate_ptx else "libr1csabc.so", src,
                                    extra=("-DGW_EMULATE_PTX",) if emulate_ptx else ()))
        L.r1cs_abc_host_load.restype = ctypes.c_void_p
        L.r1cs_abc_host_load.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
        L.r1cs_abc_host_free.argtypes = [ctypes.c_void_p]
        L.r1cs_abc_host_eval.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_char_p]
        _host[emulate_ptx] = L
    return _host[emulate_ptx]
