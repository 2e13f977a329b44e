"""Groth16 quotient evaluations of witness batches on one GPU (gw_r1cs_quotient_batch_device), next to the evaluation
and ABC of the same rows, and the batched NTT alone (gw_fr_ntt_batch_device).

  python tools/r1cs_quotient_bench.py --out DIR [--sets 8192] [--hashes 196] [--reps 3] [--ntt-gb 8]

The pair is the one of tools/r1cs_bench.py: 196 chained Poseidon-shaped permutations, 48 221 wires and 48 216
constraints, so the Groth16 domain is n = 65 536.  8 192 sets keep the witness (13 GB) and the work rows (3 x n x 32
bytes each, 52 GB) resident in HBM, far above L2.  The NTT alone runs on at least --ntt-gb GB of vectors per size.

Each rep times with CUDA events, interleaved: the evaluation, ABC in the Groth16 layout, the whole quotient (ABC plus the
transforms), then for k in {10, 12, 16, 20, 24} the forward, inverse and coset-forward NTT.  Counts, computed here:
  - IMAD.WIDE: 128 per Montgomery multiplication (64 for the product, 64 for the reduction); a transform of 2^k entries
    has (n/2) k butterflies, plus the per-entry products: the inter-pass twiddle (k > 12, two multiplications when
    its exponent is >= 4096, counted as two), the coset factor, n^-1, and in the quotient the A * B product;
  - HBM bytes from the pass structure: k <= 12 one read and one write of each vector; k > 12 two passes, plus the
    bit-reversal permutation of the standalone transform (one more read and write); the quotient reads A, B, C three
    times (column, row, column pass) and writes them three times (the last pass writes A_odd, then A_odd B_odd, then
    h into the A slot, reading it back twice).
Shares: the counts over the kernel time against the integer-pipe rate of gw_microbench_imad (same run) and 7.7 TB/s
(HBM3e, data sheet); the larger names the binding bound.  Correctness in the same run: sampled rows of h against the
Python reference (tests/r1cs_quotient_ref.py), and on sampled valid rows deg H <= n - 2 (entry n - 1 of the coset
inverse NTT of h is 0).
"""
import argparse
import importlib
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tests import r1cs_quotient_ref, r1cs_ref, util  # noqa: E402
from tools import r1cs_gen  # noqa: E402

HBM_BPS = 7.7e12
MAC_PER_MUL = 128
OK = 0xFFFFFFFF


def transform_muls(k, factor):
    """Montgomery multiplications of one transform of 2^k entries, the way ntt.cu computes it; factor: "" (forward),
    "scale" (n^-1, one product per entry) or "table" (a coset factor: two products when its exponent is >= 4096)"""
    n = 1 << k
    m = (n // 2) * k
    if k > 12:                                 # inter-pass twiddle w^(i1 j2): a second product when i1 j2 >= 4096
        n1, n2 = 1 << (k - k // 2), 1 << (k // 2)
        m += n + sum(max(0, n2 - (4095 // i1 + 1)) for i1 in range(1, n1))
    if factor == "scale" or (factor == "table" and k <= 12):
        m += n
    elif factor == "table":
        m += 2 * n - 4096
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sets", type=int, default=8192)
    ap.add_argument("--hashes", type=int, default=196)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ntt-gb", type=float, default=8.0)
    ap.add_argument("--sample", type=int, default=2, help="rows compared with the Python reference")
    a = ap.parse_args()
    import torch
    cwc = importlib.import_module("circom-witnesscalc_b200")
    if cwc.device_count() < 1:
        raise SystemExit("no CUDA device: this benchmark measures the GPU")
    os.makedirs(a.out, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()

    t0 = time.time()
    g, r = r1cs_gen.poseidon_pair(random.Random(1), n_hashes=a.hashes)
    graph, rc = cwc.Graph(g), cwc.R1cs(r1cs_ref.serialize_r1cs(r))
    t_gen = time.time() - t0
    B, W, n_in = a.sets, graph.n_witness, 4
    n = rc.abc_len(groth16=True)
    k = n.bit_length() - 1
    vals = util.random_field_batch(np.random.default_rng(2), (B, n_in + 1))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    d_in = torch.from_numpy(vals.view(np.uint8).reshape(B, -1)).cuda()
    d_w = torch.empty((B, W * 32), dtype=torch.uint8, device="cuda:0")
    d_ff = torch.empty(B, dtype=torch.int32, device="cuda:0")
    d_work = torch.empty((B, 3 * n * 32), dtype=torch.uint8, device="cuda:0")

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    steps = {
        "eval": lambda nb=B: graph.calc_witness_batch_device(0, d_in.data_ptr(), nb, d_w.data_ptr()),
        "abc_groth16": lambda nb=B: rc.abc_batch_device(0, d_w.data_ptr(), nb, d_work.data_ptr(), groth16=True),
        "quotient": lambda nb=B: rc.quotient_batch_device(0, d_w.data_ptr(), nb, d_work.data_ptr()),
    }
    for fn in steps.values():
        fn(512)
    torch.cuda.synchronize()
    ms = {s: [] for s in steps}
    for _ in range(a.reps):
        for s, fn in steps.items():
            ms[s].append(timed(fn))

    # correctness: sampled rows against the reference, deg H <= n - 2 on the GPU for sampled valid rows
    steps["quotient"]()
    rc.check_batch_device(0, d_w.data_ptr(), B, d_ff.data_ptr())
    torch.cuda.synchronize()
    all_valid = bool((d_ff.cpu().numpy().view(np.uint32) == OK).all())
    rows = sorted(random.Random(3).sample(range(B), a.sample))
    sample_ok = True
    for b in rows:
        wit = util.unpack_u256(d_w[b].cpu().numpy().tobytes())
        exp = util.pack_u256(r1cs_quotient_ref.quotient_ref(r, wit))
        sample_ok &= d_work[b, :n * 32].cpu().numpy().tobytes() == exp
    deg_rows = sorted(random.Random(4).sample(range(B), 16))
    h = torch.stack([d_work[b, :n * 32] for b in deg_rows]).contiguous()
    cwc.ntt_batch_device(0, h.data_ptr(), len(deg_rows), k, flags=cwc.NTT_INVERSE | cwc.NTT_COSET)
    torch.cuda.synchronize()
    deg_ok = not bool(h[:, (n - 1) * 32:].any())
    del h

    # the NTT alone
    ntt_ms, ntt_counts = {}, {}
    del d_work
    torch.cuda.empty_cache()
    for kk in (10, 12, 16, 20, 24):
        nv = max(1, int(a.ntt_gb * 1e9) // (32 << kk))
        buf = torch.from_numpy(util.random_field_batch(np.random.default_rng(kk), (nv, 1 << kk)).view(np.uint8)
                               .reshape(nv, -1)).cuda() if kk <= 16 else torch.randint(0, 255, (nv, 32 << kk), dtype=torch.uint8,
                                                                                       device="cuda:0")
        for name, flags in (("forward", 0), ("inverse", cwc.NTT_INVERSE), ("coset", cwc.NTT_COSET)):
            cwc.ntt_batch_device(0, buf.data_ptr(), 1, kk, flags=flags)
            torch.cuda.synchronize()
            ntt_ms[f"k{kk}_{name}"] = []
        for _ in range(a.reps):
            for name, flags in (("forward", 0), ("inverse", cwc.NTT_INVERSE), ("coset", cwc.NTT_COSET)):
                ntt_ms[f"k{kk}_{name}"].append(timed(lambda: cwc.ntt_batch_device(0, buf.data_ptr(), nv, kk, flags=flags)))
        for name in ("forward", "inverse", "coset"):
            muls = transform_muls(kk, {"forward": "", "inverse": "scale", "coset": "table"}[name])
            passes = 1 if kk <= 12 else 3
            ntt_counts[f"k{kk}_{name}"] = {"vectors": nv, "muls_per_vector": muls, "bytes_per_vector": passes * 2 * (32 << kk)}
        del buf
        torch.cuda.empty_cache()

    imad = cwc.microbench_imad(0, 0)
    rooflines = {}

    def roof(key, t_ms, macs, byts):
        t = t_ms * 1e-3
        t_int, t_hbm = macs / imad, byts / HBM_BPS
        rooflines[key] = {"ms": t_ms, "imad_wide": macs, "hbm_bytes": byts, "int_pipe_share": t_int / t,
                          "hbm_share": t_hbm / t, "binding": "integer pipe" if t_int > t_hbm else "HBM",
                          "share_of_binding_roofline": max(t_int, t_hbm) / t}

    info = rc.info()
    abc_macs = 64 * info["n_mac_terms"] + 64 * info["n_chunks"]
    q_muls = 6 * transform_muls(k, "") + 3 * (2 * n - 4096 if k > 12 else n) + n      # + n^-1 g^i of A, B, C, and A * B
    q_bytes = (11 + 9) * n * 32      # reads: 3 + 3 + 3 passes over A, B, C and A twice more; writes 3 + 3 + h, A B, A
    roof("quotient_transforms", min(ms["quotient"]) - min(ms["abc_groth16"]), B * q_muls * MAC_PER_MUL,
         B * q_bytes)
    roof("quotient_total", min(ms["quotient"]), B * (q_muls * MAC_PER_MUL + abc_macs),
         B * (W * 32 + 3 * n * 32 + q_bytes))
    for key, c in ntt_counts.items():
        roof(key, min(ntt_ms[key]), c["vectors"] * c["muls_per_vector"] * MAC_PER_MUL, c["vectors"] * c["bytes_per_vector"])
    res = {
        "gpu": gpu, "sets": B, "r1cs": info, "n": n, "generation_s": round(t_gen, 1), "ms": ms, "ntt_ms": ntt_ms,
        "ntt_counts": ntt_counts, "quotient_muls_per_row": q_muls, "imad_wide_per_s": imad, "hbm_bytes_per_s_peak": HBM_BPS,
        "rooflines": rooflines, "us_per_row_quotient": min(ms["quotient"]) * 1e3 / B,
        "all_rows_valid": all_valid, "sample_rows": rows, "sample_rows_match_reference": bool(sample_ok),
        "deg_rows": deg_rows, "deg_h_le_n_minus_2": deg_ok,
    }
    with open(os.path.join(a.out, "r1cs_quotient_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    if not (all_valid and sample_ok and deg_ok):
        raise SystemExit("wrong results")


if __name__ == "__main__":
    main()
