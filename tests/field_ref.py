"""Python-integer reference of every primitive of csrc/field.cuh, csrc/inv_safegcd.cuh, csrc/alu.cuh and the butterflies
of csrc/ntt.cuh, and the operand sets they are checked on: the host builds (tests/test_field_host.py) and the device
harness (tests/test_gpu_field.py) compare against the same formulas.

Operand domains: "c" canonical field values [0, M), "w" any 256-bit value, "s" shift amounts (canonical values, mostly
small), "n" int64 values (two's complement in limbs 0..1)."""
import random

from oracle import pyoracle as po

M = po.M
R = 1 << 256
R_MOD = R % M
R_INV = pow(R, -1, M)
MASK256 = R - 1
MASK254 = (1 << 254) - 1
HALF = M >> 1


# ---- field and integer primitives ---------------------------------------------------------------------------------------
def mul(a, b):
    return a * b % M


def mul_wide(a, b):
    return a * b


def mul_lo(a, b):
    return a * b & MASK256


def mul_hi_trunc(a, b):
    """the partial products a_j b_i with i + j >= 6 that Barrett's quotient estimate keeps, as one 512-bit sum (both code
    paths of u256_mul_hi_trunc compute exactly this sum; limbs 0..5 are 0)"""
    al = [(a >> (32 * j)) & 0xFFFFFFFF for j in range(8)]
    bl = [(b >> (32 * i)) & 0xFFFFFFFF for i in range(8)]
    return sum(al[j] * bl[i] << (32 * (i + j)) for i in range(8) for j in range(8) if i + j >= 6)


def mont_mul(a, b):
    return a * b * R_INV % M


def to_mont(a):
    return a * R_MOD % M


def from_mont(a):
    return a * R_INV % M


def add(a, b):
    return (a + b) % M


def sub(a, b):
    return (a - b) % M


def neg(a):
    return (-a) % M


def reduce256(a):
    return a % M


def shift_amount(b):
    """the reference's reading of a shift operand: 0 -> no shift, >= 254 -> the result is 0"""
    return min(b, 254)


def shr(a, b):
    n = shift_amount(b)
    return 0 if n >= 254 else a >> n


def shl(a, b):
    """(result, overflow): overflow where the reference panics (the 256-bit truncated shift is >= M); the result is then
    the circom semantics ((a << b) & (2^254 - 1)) mod M"""
    n = shift_amount(b)
    full = 0 if n >= 254 else (a << n) & MASK256
    if full < M:
        return full, 0
    return ((a << n) & MASK254) % M, 1


def bitop(a, b, which):
    """which: 0 = and, 1 = or, 2 = xor -> (result, the 256-bit result equals M); one conditional subtraction of M"""
    d = (a & b, a | b, a ^ b)[which]
    return (d - M if d >= M else d), int(d == M)


def bnot(a):
    return ((~a) & MASK254) % M


def cmp(a, b, which):
    """circom signed comparison: which 0 = lt, 1 = gt, 2 = leq, 3 = geq (values above M // 2 are negative)"""
    na, nb = a > HALF, b > HALF
    if na != nb:
        return int((na, nb, na, nb)[which])
    return int((a < b, a > b, a <= b, a >= b)[which])


def divrem(a, b):
    return a // b, a % b


def fe_pow(a, e):
    return pow(a, e, M)


def inv(a):
    """a^-1 mod M, 0 -> 0 (Fermat and safegcd alike)"""
    return pow(a, -1, M) if a % M else 0


def mont_reduce(P):
    """P * 2^-256 mod M for a 512-bit P within the bound of fe_mont_reduce (mont_reduce_limit)"""
    return P * R_INV % M


def mont_reduce_limit(ncs):
    """P < limit * 2^256 keeps (P + m M) / 2^256 below 2^ncs M and 2^256"""
    return min((1 << ncs) * M, R) - M


def dot_eval(kinds, xs, cs):
    """OP_DOT (isa.h TermKind): P = sum of x c' (T_MAC), x << 256 (T_ADDHI), (M - x) << 256 (T_SUBHI), c' (T_CONST);
    the result is P 2^-256 mod M"""
    P = 0
    for k, x, c in zip(kinds, xs, cs):
        P += (x * c, x << 256, (M - x) << 256, c)[k]
    return P * R_INV % M


def dot_ncs(n_mac, n_hi):
    """the conditional subtractions the plan compiler gives a term mix (plan.cpp: dot_bound), None when it is too wide"""
    bound = 1 + 0.18906 * n_mac + n_hi
    return None if bound > 5.25 else 1 if bound <= 2 else 2 if bound <= 4 else 3


def ntt_mul(x, w):
    """x times a pre-scaled twiddle w' = w 2^256 mod M"""
    return x * w * R_INV % M


def bfly_dif(a, b, w):
    return (a + b) % M, ntt_mul((a - b) % M, w)


def bfly_dit(a, b, w):
    t = ntt_mul(b, w)
    return (a + t) % M, (a - t) % M


def from_narrow(v):
    """canonical form of an int64 (two's complement in 64 bits)"""
    return (v - (1 << 64) if v >> 63 else v) % M


# ---- alu_exec (csrc/alu.cuh): every opcode it runs, with the status bits of isa.h --------------------------------------
ST_SHL_OVERFLOW, ST_BITWISE_EQ_M, ST_POW, ST_ID, ST_LNOT_BNOT = 1, 2, 4, 8, 16
OP_INV, OP_NZ1, OP_WIDEN, OP_TERN, OP_SQR = 36, 37, 38, 40, 52
ALU_OPS = list(range(20)) + list(range(32, 39)) + [OP_TERN, OP_SQR]
_UNDEFINED_STATUS = {"Pow": ST_POW, "Shl overflow": ST_SHL_OVERFLOW, "bitwise result == M": ST_BITWISE_EQ_M, "Id": ST_ID,
                     "Lnot": ST_LNOT_BNOT, "Bnot": ST_LNOT_BNOT}


def alu(op, a, b, c):
    """(result, status) of alu_exec on canonical operands: the value the oracle gives in "circom" mode, the status bit of
    the case where it raises ReferenceUndefined in "raise" mode; the plan compiler's own opcodes (Inv, Nz1, Widen, Sqr)
    by their isa.h definitions"""
    if op == OP_INV:
        return inv(a), 0
    if op == OP_NZ1:
        return (a or 1), 0
    if op == OP_WIDEN:
        return from_narrow(a & ((1 << 64) - 1)), 0
    if op == OP_SQR:
        return a * a % M, 0
    if op < 32:
        f = lambda mode: po.eval_duo(op, a, b, mode)
    elif op < 40:
        f = lambda mode: po.eval_uno(op - 32, a, mode)
    else:
        f = lambda mode: po.eval_tres(0, a, b, c)
    r = f("circom")
    try:
        f("raise")
        st = 0
    except po.ReferenceUndefined as e:
        st = _UNDEFINED_STATUS[str(e)]
    return r, st


# ---- operand sets -------------------------------------------------------------------------------------------------------
def _uniq(xs):
    return list(dict.fromkeys(xs))


BARRETT_A = [M - 1, M - 2, HALF + 1, 1 << 253, (1 << 253) + 1]
BARRETT_B = [M - 1, M - 2, HALF, (1 << 253) - 1, 3]
# canonical edges: the limb-ripple operands (all-ones runs, powers of 2^32 and M minus them), the sign boundary of the
# signed comparisons, 2^256 mod M and its inverse (Montgomery's 1 and R^2 reductions), Barrett's worst cases
CANON_EDGES = _uniq([0, 1, 2, 3, M - 1, M - 2, HALF, HALF - 1, HALF + 1, (1 << 253) - 1, 1 << 253, (1 << 253) + 1]
                    + [(1 << (32 * k)) - 1 for k in range(1, 8)] + [1 << (32 * k) for k in range(8)]
                    + [M - (1 << (32 * k)) for k in range(8)] + [R_MOD, pow(R_MOD, -1, M)] + BARRETT_A + BARRETT_B)
# 256-bit edges of the primitives that take any 256-bit value
WIDE_EDGES = _uniq(CANON_EDGES + [MASK256, R - (1 << 32), M, M + 1, 2 * M - 1, 5 * M - 1, 5 * M, 1 << 255, MASK256 // 3])
SHIFT_EDGES = _uniq([0, 1, 2, 31, 32, 33, 63, 64, 65, 95, 96, 127, 128, 129, 191, 192, 200, 223, 224, 225, 252, 253, 254, 255,
                     256, 257, 1 << 32, (1 << 32) + 5, 1 << 64, M - 1, 1 << 253])
NARROW_EDGES = _uniq([0, 1, 2, (1 << 31) - 1, 1 << 31, (1 << 32) - 1, 1 << 32, (1 << 62) - 1, 1 << 62, (1 << 63) - 1]
                     + [(1 << 64) - v for v in (1, 2, 1 << 31, (1 << 31) + 1, 1 << 32, (1 << 32) + 1, 1 << 62, (1 << 62) + 1, 1 << 63)])
EDGES = {"c": CANON_EDGES, "w": WIDE_EDGES, "s": SHIFT_EDGES, "n": NARROW_EDGES}

LIMB_PATTERNS = (0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF)
_TOP_CANON = (0, 1, 0x0FFFFFFF, 0x1FFFFFFF, 0x30644E71, 0x30644E72)     # M's top limb is 0x30644E72


def _limb(rnd):
    i = rnd.randrange(len(LIMB_PATTERNS) + 1)
    return rnd.getrandbits(32) if i == len(LIMB_PATTERNS) else LIMB_PATTERNS[i]


def limb_pattern(rnd: random.Random, dom="c"):
    """a value whose every limb is 0, 1, 0x7FFFFFFF, 0x80000000, 0xFFFFFFFE, 0xFFFFFFFF or random; canonical values take a
    top limb at or below M's (reduced mod M when that still is not enough)"""
    if dom == "s":
        return rnd.choice(SHIFT_EDGES) if rnd.random() < 0.5 else rnd.randrange(300)
    if dom == "n":
        return sum(_limb(rnd) << (32 * i) for i in range(2))
    v = sum(_limb(rnd) << (32 * i) for i in range(7))
    top = _limb(rnd) if dom == "w" else (rnd.choice(_TOP_CANON) if rnd.random() < 0.8 else rnd.randrange(0x30644E73))
    v |= top << 224
    return v % M if dom == "c" else v


def uniform(rnd: random.Random, dom="c"):
    if dom == "s":
        return rnd.randrange(300)
    if dom == "n":
        return rnd.getrandbits(64)
    return rnd.randrange(M) if dom == "c" else rnd.getrandbits(256)


def edge_tuples(doms):
    """the cross product of the edges of the first two operands (further operands cycle through their edges)"""
    if len(doms) == 1:
        return [(x,) for x in EDGES[doms[0]]]
    out = []
    for i, x in enumerate(EDGES[doms[0]]):
        for j, y in enumerate(EDGES[doms[1]]):
            out.append((x, y) + tuple(EDGES[d][(i + j + k) % len(EDGES[d])] for k, d in enumerate(doms[2:])))
    return out


def operand_tuples(doms, n_random, seed):
    """edges (cross product), then n_random limb-pattern tuples and n_random uniform tuples"""
    rnd = random.Random(seed)
    out = edge_tuples(doms)
    out += [tuple(limb_pattern(rnd, d) for d in doms) for _ in range(n_random)]
    out += [tuple(uniform(rnd, d) for d in doms) for _ in range(n_random)]
    return out
