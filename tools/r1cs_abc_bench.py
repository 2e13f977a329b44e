"""A, B and C of witness batches on one GPU (gw_r1cs_abc_batch_device), next to the check and the evaluation of the
same rows.

  python tools/r1cs_abc_bench.py --out DIR [--sets 16384] [--hashes 196] [--reps 3]

The pair is the one of tools/r1cs_bench.py: 196 chained Poseidon-shaped permutations from tools/r1cs_gen.py, 48 221
wires and 48 216 constraints (authV2's size), so the Groth16 domain is n = 65 536.  16 384 sets keep everything in HBM
at once: 25 GB of witness computed on the device, and one output buffer of 103 GB (the Groth16 layout; the plain
layout, 76 GB, is written densely into the same buffer).  Both are far larger than L2, so every pass goes to HBM.

Each rep times, with CUDA events and in this order: the evaluation, the check, ABC in the plain layout, ABC in the
Groth16 layout, ABC in the plain layout with the verdict.  Writes DIR/r1cs_abc_bench.json with the card's name and power
limit, the times and the algorithmic counts per set:
  - IMAD.WIDE: 64 per T_MAC term and 64 per Montgomery reduction (one per chunk), plus 64 + 72 per constraint for the
    product a * b and its Barrett reduction when the verdict is computed (the check always computes it);
  - bytes: the distinct witness bytes (32 per wire, each value read once from HBM) and the output bytes (3 x n x 32).
The shares of the integer-pipe rate (gw_microbench_imad) and of 7.7 TB/s (HBM3e, data sheet) are these counts over
the kernel time; the larger one names the binding bound.  Correctness in the same run: every verdict is GW_R1CS_OK, and
a seeded sample of rows in both layouts equals the Python reference (tests/r1cs_abc_ref.py).
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

from tests import r1cs_abc_ref, r1cs_ref, util  # noqa: E402
from tools import r1cs_gen  # noqa: E402

HBM_BPS = 7.7e12
MAC_PER_TERM, MAC_PER_REDUCTION, MAC_PER_PRODUCT = 64, 64, 64 + 72
OK = 0xFFFFFFFF


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sets", type=int, default=16384)
    ap.add_argument("--hashes", type=int, default=196)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sample", type=int, default=3, help="rows compared with the Python reference, per layout")
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
    info = rc.info()
    t_gen = time.time() - t0
    B, W, n_in = a.sets, graph.n_witness, 4
    assert W == info["n_wires"]
    m, n_g = rc.abc_len(), rc.abc_len(groth16=True)
    vals = util.random_field_batch(np.random.default_rng(2), (B, n_in + 1))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    d_in = torch.from_numpy(vals.view(np.uint8).reshape(B, -1)).cuda()
    d_w = torch.empty((B, W * 32), dtype=torch.uint8, device="cuda:0")
    d_ff = torch.empty(B, dtype=torch.int32, device="cuda:0")
    d_abc = torch.empty(B * 3 * n_g * 32, dtype=torch.uint8, device="cuda:0")   # Groth16 rows; plain rows packed densely

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    def abc(groth16, verdict, n_sets=B):
        return lambda: rc.abc_batch_device(0, d_w.data_ptr(), n_sets, d_abc.data_ptr(), groth16=groth16,
                                           d_first_failed_ptr=d_ff.data_ptr() if verdict else None)

    steps = {
        "eval": lambda n_sets=B: graph.calc_witness_batch_device(0, d_in.data_ptr(), n_sets, d_w.data_ptr()),
        "check": lambda n_sets=B: rc.check_batch_device(0, d_w.data_ptr(), n_sets, d_ff.data_ptr()),
        "abc_plain": lambda n_sets=B: abc(False, False, n_sets)(),
        "abc_groth16": lambda n_sets=B: abc(True, False, n_sets)(),
        "abc_plain_verdict": lambda n_sets=B: abc(False, True, n_sets)(),
    }
    for fn in steps.values():                  # warm-up on a small batch: module load, uploads
        fn(1024)
    torch.cuda.synchronize()
    ms = {k: [] for k in steps}
    verdicts_ok = True
    for _ in range(a.reps):
        for k, fn in steps.items():
            ms[k].append(timed(fn))
            if k in ("check", "abc_plain_verdict"):
                verdicts_ok &= bool((d_ff.cpu().numpy().view(np.uint32) == OK).all())

    # seeded sample of rows in both layouts against the Python reference
    rows = sorted(random.Random(3).sample(range(B), a.sample))
    sample_ok = True
    for groth16 in (False, True):
        abc(groth16, False)()
        torch.cuda.synchronize()
        n = n_g if groth16 else m
        out = d_abc[:B * 3 * n * 32].view(B, 3 * n * 32)
        for b in rows:
            wit = util.unpack_u256(d_w[b].cpu().numpy().tobytes())
            A, Bv, C = r1cs_abc_ref.abc_ref(r, wit, groth16)
            exp = np.frombuffer(util.pack_u256(A + Bv + C), np.uint8)
            sample_ok &= bool((out[b].cpu().numpy() == exp).all())

    imad = cwc.microbench_imad(0, 0)
    macs_abc = MAC_PER_TERM * info["n_mac_terms"] + MAC_PER_REDUCTION * info["n_chunks"]
    macs_check = macs_abc + MAC_PER_PRODUCT * info["n_constraints"]
    wit_b = 32 * info["n_wires"]
    rooflines = {}
    for k, macs, out_b in (("check", macs_check, 0), ("abc_plain", macs_abc, 3 * m * 32),
                           ("abc_groth16", macs_abc, 3 * n_g * 32), ("abc_plain_verdict", macs_check, 3 * m * 32)):
        t = min(ms[k]) * 1e-3
        t_int, t_hbm = macs * B / imad, (wit_b + out_b) * B / HBM_BPS
        rooflines[k] = {"ms": min(ms[k]), "sets_per_s": B / t, "wide_macs_per_set": macs, "bytes_read_per_set": wit_b,
                        "bytes_written_per_set": out_b, "int_pipe_share": t_int / t, "hbm_share": t_hbm / t,
                        "binding": "integer pipe" if t_int > t_hbm else "HBM", "share_of_binding_roofline": max(t_int, t_hbm) / t}
    res = {
        "gpu": gpu, "sets": B, "r1cs": info, "n_plain": m, "n_groth16": n_g, "generation_s": round(t_gen, 1),
        "ms": ms, "imad_wide_per_s": imad, "hbm_bytes_per_s_peak": HBM_BPS, "rooflines": rooflines,
        "abc_plain_over_check": min(ms["abc_plain"]) / min(ms["check"]),
        "abc_groth16_over_check": min(ms["abc_groth16"]) / min(ms["check"]),
        "abc_verdict_over_check": min(ms["abc_plain_verdict"]) / min(ms["check"]),
        "all_verdicts_ok": verdicts_ok, "sample_rows": rows, "sample_rows_match_reference": sample_ok,
    }
    with open(os.path.join(a.out, "r1cs_abc_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    if not (verdicts_ok and sample_ok):
        raise SystemExit("wrong results")


if __name__ == "__main__":
    main()
