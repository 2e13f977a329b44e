"""Reference (pure Python) of the batched BN254 NTT (gw_fr_ntt_batch_device) and the Groth16 quotient evaluations of
witness rows (gw_r1cs_quotient_*), over the R1CS dicts of tests/r1cs_ref.py, and the host build of the NTT arithmetic.

  M - 1 = 2^28 t, w_28 = 5^t mod M, w_n = w_28^(2^(28 - k)) for n = 2^k, g = w_2n
  forward  y_j = sum_i x_i w_n^(ij)          inverse  x_i = n^-1 sum_j y_j w_n^(-ij)
  coset    y_j = sum_i x_i (g w_n^j)^i       coset inverse: its exact inverse
  quotient h_i = A_odd[i] B_odd[i] - C_odd[i], X_odd = coset(inverse(X)) of the Groth16-layout A, B, C
           (snarkjs groth16_prove joinABC, rapidsnark's vector before the H multi-scalar multiplication)
"""
from tests.r1cs_abc_ref import abc_ref
from tests.r1cs_ref import M

W28 = pow(5, (M - 1) >> 28, M)


def root(k, inverse=False):
    w = pow(W28, 1 << (28 - k), M)
    return pow(w, M - 2, M) if inverse else w


def coset_gen(k):
    return pow(W28, 1 << (27 - k), M)


def _fft(a, w):
    n = len(a)
    if n == 1:
        return list(a)
    w2 = w * w % M
    e, o = _fft(a[0::2], w2), _fft(a[1::2], w2)
    out, t = [0] * n, 1
    for i in range(n // 2):
        u = o[i] * t % M
        out[i], out[i + n // 2] = (e[i] + u) % M, (e[i] - u) % M
        t = t * w % M
    return out


def _powers(x, n):
    out, p = [], 1
    for _ in range(n):
        out.append(p)
        p = p * x % M
    return out


def ntt(x, inverse=False, coset=False):
    """the transform of the module docstring, O(n log n); inputs any non-negative integers"""
    n = len(x)
    k = n.bit_length() - 1
    assert n == 1 << k
    x = [v % M for v in x]
    g = coset_gen(k)
    if coset and not inverse:
        x = [v * p % M for v, p in zip(x, _powers(g, n))]
    y = _fft(x, root(k, inverse))
    if inverse:
        ninv = pow(n, M - 2, M)
        f = _powers(pow(g, M - 2, M), n) if coset else [1] * n
        y = [v * ninv % M * p % M for v, p in zip(y, f)]
    return y


def ntt_naive(x, inverse=False, coset=False):
    """the same by the defining sums, O(n^2)"""
    n = len(x)
    k = n.bit_length() - 1
    w, g = root(k, inverse), coset_gen(k)
    x = [v % M for v in x]
    if not inverse:
        pts = [(g if coset else 1) * pow(w, j, M) % M for j in range(n)]
        return [sum(v * pow(p, i, M) for i, v in enumerate(x)) % M for p in pts]
    ninv = pow(n, M - 2, M)
    out = [ninv * sum(v * pow(w, i * j, M) for j, v in enumerate(x)) % M for i in range(n)]
    return [v * pow(g, (M - 2) * i, M) % M for i, v in enumerate(out)] if coset else out


def quotient_ref(r1cs, witness):
    """h of one witness row by the formula of the module docstring"""
    odd = [ntt(ntt(X, inverse=True), coset=True) for X in abc_ref(r1cs, witness, groth16=True)]
    return [(a * b - c) % M for a, b, c in zip(*odd)]


def _polymul(a, b):
    out = [0] * (len(a) + len(b) - 1)
    for i, x in enumerate(a):
        for j, y in enumerate(b):
            out[i + j] = (out[i + j] + x * y) % M
    return out


def quotient_by_division(r1cs, witness):
    """h by explicit polynomials, for a satisfying row of a small system: interpolate A, B, C on <w_n>, P = A B - C,
    H = P / (x^n - 1) (the remainder must be 0), and -2 H(g w_n^i) = (g^n - 1) H(g w_n^i)"""
    A, B, C = abc_ref(r1cs, witness, groth16=True)
    n = len(A)
    k = n.bit_length() - 1
    a, b, c = (ntt_naive(X, inverse=True) for X in (A, B, C))
    P = _polymul(a, b)
    for i, v in enumerate(c):
        P[i] = (P[i] - v) % M
    H = [0] * max(1, len(P) - n)                 # P = H (x^n - 1) + R, deg R < n
    for d in range(len(P) - 1, n - 1, -1):
        q = P[d]
        H[d - n] = q
        P[d] = 0
        P[d - n] = (P[d - n] + q) % M
    assert not any(P[:n]), "the row does not satisfy the system: x^n - 1 does not divide A B - C"
    g, w = coset_gen(k), root(k)
    pts = [g * pow(w, i, M) % M for i in range(n)]
    return [(-2 * sum(h * pow(p, e, M) for e, h in enumerate(H))) % M for p in pts]


_host = {}


def ntt_host_lib(emulate_ptx=False):
    """tests/csrc/ntt_host_api.cpp: the butterflies, the twiddle multiplication and the tables of csrc/ntt.cuh, built for
    the host (emulate_ptx=True: with the device formulations of field.cuh)"""
    import ctypes
    import os
    from tests import util
    if emulate_ptx not in _host:
        src = [os.path.join(util.ROOT, "tests", "csrc", "ntt_host_api.cpp")]
        L = ctypes.CDLL(util._build("libntt_ptx.so" if emulate_ptx else "libntt.so", src,
                                    extra=("-DGW_EMULATE_PTX",) if emulate_ptx else ()))
        L.ntt_host_tables.argtypes = [ctypes.c_uint32, ctypes.c_char_p]
        L.ntt_host_bfly.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p]
        L.ntt_host_n_tables.restype = ctypes.c_uint32
        _host[emulate_ptx] = L
    return _host[emulate_ptx]
