"""Reference (pure Python) of the iden3 .r1cs format, version 1, and of the R1CS check, for the tests.

  file    := "r1cs" u32(version = 1) u32(n_sections) section*      sections in any order; each type at most once
  section := u32(type) u64(size) byte{size}
  type 1  := u32(n8) prime{n8} u32(n_wires) u32(n_pub_out) u32(n_pub_in) u32(n_prv_in) u64(n_labels) u32(m)
  type 2  := constraint{m};  constraint := lc(A) lc(B) lc(C);  lc := u32(n) { u32(wire) coeff{n8} }{n}
  type 3  := u64{n_wires}

An R1CS is a dict {n_wires, n_pub_out, n_pub_in, n_prv_in, n_labels, constraints}; a constraint is a triple of linear
combinations, each a list of (wire, coefficient) pairs.  Coefficients are plain little-endian integers.
"""
import struct

from oracle.pyoracle import M


def serialize_r1cs(r1cs, prime=M, n8=32, version=1, with_labels=True, extra_sections=(), order=(1, 2, 3)):
    hdr = struct.pack("<I", n8) + prime.to_bytes(n8, "little") + struct.pack(
        "<IIIIQI", r1cs["n_wires"], r1cs.get("n_pub_out", 0), r1cs.get("n_pub_in", 0), r1cs.get("n_prv_in", 0),
        r1cs.get("n_labels", r1cs["n_wires"]), len(r1cs["constraints"]))
    body = bytearray()
    for con in r1cs["constraints"]:
        for lc in con:
            body += struct.pack("<I", len(lc))
            for wire, c in lc:
                body += struct.pack("<I", wire) + int(c).to_bytes(n8, "little")
    sections = {1: hdr, 2: bytes(body)}
    if with_labels:
        sections[3] = b"".join(struct.pack("<Q", i) for i in range(r1cs["n_wires"]))
    out = [(t, sections[t]) for t in order if t in sections] + list(extra_sections)
    return b"r1cs" + struct.pack("<II", version, len(out)) + b"".join(struct.pack("<IQ", t, len(d)) + d for t, d in out)


def parse_r1cs(data: bytes):
    if data[:4] != b"r1cs":
        raise ValueError("bad magic")
    version, n_sections = struct.unpack_from("<II", data, 4)
    if version != 1:
        raise ValueError("version")
    pos, secs = 12, {}
    for _ in range(n_sections):
        t, size = struct.unpack_from("<IQ", data, pos)
        pos += 12
        if pos + size > len(data):
            raise ValueError("truncated")
        if t in secs:
            raise ValueError("duplicate section")
        secs[t] = data[pos:pos + size]
        pos += size
    if pos != len(data):
        raise ValueError("trailing bytes")
    if 4 in secs or 5 in secs:
        raise ValueError("custom gates")
    h = secs[1]
    n8 = struct.unpack_from("<I", h, 0)[0]
    prime = int.from_bytes(h[4:4 + n8], "little")
    if n8 != 32 or prime != M:
        raise ValueError("not BN254")
    n_wires, n_pub_out, n_pub_in, n_prv_in, n_labels, m = struct.unpack_from("<IIIIQI", h, 4 + n8)
    if len(h) != 4 + n8 + 28:
        raise ValueError("header size")
    body, p, cons = secs[2], 0, []
    for _ in range(m):
        con = []
        for _ in range(3):
            n = struct.unpack_from("<I", body, p)[0]
            p += 4
            lc = []
            for _ in range(n):
                wire = struct.unpack_from("<I", body, p)[0]
                if wire >= n_wires:
                    raise ValueError("wire out of range")
                lc.append((wire, int.from_bytes(body[p + 4:p + 36], "little") % M))
                p += 36
            con.append(lc)
        cons.append(tuple(con))
    if p != len(body):
        raise ValueError("constraints section size")
    if 3 in secs and len(secs[3]) != 8 * n_wires:
        raise ValueError("wire2label size")
    return {"n_wires": n_wires, "n_pub_out": n_pub_out, "n_pub_in": n_pub_in, "n_prv_in": n_prv_in,
            "n_labels": n_labels, "constraints": cons}


def lc_value(lc, witness):
    return sum(c * witness[w] for w, c in lc) % M


def check_r1cs(r1cs, witness):
    """index of the lowest violated constraint, or None.  A witness value >= M fails the first constraint reading it
    (the library's rule: such a value is not a field element)."""
    for k, con in enumerate(r1cs["constraints"]):
        if any(witness[w] >= M for lc in con for w, c in lc if c % M):
            return k
        a, b, c = (lc_value(lc, witness) for lc in con)
        if (a * b - c) % M:
            return k
    return None


_host = {}


def host_lib(emulate_ptx=False):
    """tests/csrc/r1cs_host_api.cpp: the library's .r1cs reader and the check kernel's evaluation, built for the host
    (emulate_ptx=True: with the device formulations of field.cuh)"""
    import ctypes
    import os
    from tests import util
    if emulate_ptx not in _host:
        src = [os.path.join(util.ROOT, "tests", "csrc", "r1cs_host_api.cpp")] + [
            os.path.join(util.CSRC, f) for f in ("r1cs.cpp", "graph.cpp", "plan.cpp")]
        L = ctypes.CDLL(util._build("libr1cshost_ptx.so" if emulate_ptx else "libr1cshost.so", src,
                                    extra=("-DGW_EMULATE_PTX",) if emulate_ptx else ()))
        L.r1cs_host_load.restype = ctypes.c_void_p
        L.r1cs_host_load.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
        L.r1cs_host_free.argtypes = [ctypes.c_void_p]
        L.r1cs_host_info.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_uint64)]
        L.r1cs_host_eval.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_char_p, ctypes.c_char_p]
        L.r1cs_host_check.restype = ctypes.c_uint32
        L.r1cs_host_check.argtypes = [ctypes.c_void_p, ctypes.c_char_p]
        _host[emulate_ptx] = L
    return _host[emulate_ptx]
