"""R1CS check throughput on one GPU, next to the evaluation of the same graph.

  python tools/r1cs_bench.py --out DIR [--sets 65536] [--hashes 196] [--reps 3]

A Poseidon-shaped (graph, R1CS) pair from tools/r1cs_gen.py stands in for a real circuit (no .r1cs of authV2 here);
196 chained permutations give about 49 000 wires and constraints, authV2's size.  The witnesses are computed on the
device (gw_calc_witness_batch_device) into one buffer and checked there (gw_r1cs_check_batch_device), each timed with
CUDA events; 65 536 sets of 49 000 wires are 103 GB, larger than L2, so every pass reads HBM.  Writes DIR/r1cs_bench.json
with the card's name and power limit, the times, and the algorithmic counts:
  - integer work per set: 64 wide multiply-adds (IMAD.WIDE) per T_MAC term, 64 per Montgomery reduction (one per
    chunk of a linear combination), 64 + 72 per constraint for the product <A,w> * <B,w> and its Barrett reduction;
  - witness reads per set: 32 B per term (what the kernel requests) and 32 B per wire (the HBM floor: each value once).
The shares of the integer-pipe peak (gw_microbench_imad, IMAD.WIDE rows/s) and of HBM (7.7 TB/s, data sheet) are the
counts over the kernel time; the larger of the two is the binding roofline.
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

from tests import r1cs_ref, util  # noqa: E402
from tools import r1cs_gen  # noqa: E402

HBM_BPS = 7.7e12
MAC_PER_TERM, MAC_PER_REDUCTION, MAC_PER_PRODUCT = 64, 64, 64 + 72


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sets", type=int, default=65536)
    ap.add_argument("--hashes", type=int, default=196)
    ap.add_argument("--reps", type=int, default=3)
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
    vals = util.random_field_batch(np.random.default_rng(2), (B, n_in + 1))
    vals[:, 0, :] = 0
    vals[:, 0, 0] = 1
    d_in = torch.from_numpy(vals.view(np.uint8).reshape(B, -1)).cuda()
    d_w = torch.empty((B, W * 32), dtype=torch.uint8, device="cuda:0")
    d_ff = torch.empty(B, dtype=torch.int32, device="cuda:0")

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    evaluate = lambda: graph.calc_witness_batch_device(0, d_in.data_ptr(), B, d_w.data_ptr())
    check = lambda: rc.check_batch_device(0, d_w.data_ptr(), B, d_ff.data_ptr())
    # warm-up on a small batch: module load, uploads
    graph.calc_witness_batch_device(0, d_in.data_ptr(), 1024, d_w.data_ptr())
    rc.check_batch_device(0, d_w.data_ptr(), 1024, d_ff.data_ptr())
    torch.cuda.synchronize()
    eval_ms = [timed(evaluate) for _ in range(a.reps)]
    check_ms = [timed(check) for _ in range(a.reps)]
    ff = d_ff.cpu().numpy().view(np.uint32)
    all_ok = bool((ff == 0xFFFFFFFF).all())
    # one corrupted row: the reported index must be the reference's
    row = d_w[B // 2].cpu().numpy()
    wit = util.unpack_u256(row.tobytes())
    k = r["constraints"][len(r["constraints"]) // 2][2][-1][0]
    wit[k] = (wit[k] + 1) % util.M
    d_w[B // 2] = torch.from_numpy(np.frombuffer(util.pack_u256(wit), np.uint8).copy()).cuda()
    check()
    torch.cuda.synchronize()
    exp = r1cs_ref.check_r1cs(r, wit)
    corrupt_ok = int(d_ff[B // 2].item()) & 0xFFFFFFFF == exp

    imad = cwc.microbench_imad(0, 0)
    ms = min(check_ms)
    macs = (MAC_PER_TERM * info["n_mac_terms"] + MAC_PER_REDUCTION * info["n_chunks"] + MAC_PER_PRODUCT * info["n_constraints"]) * B
    bytes_terms, bytes_unique = 32 * info["n_terms"] * B, 32 * info["n_wires"] * B
    t_int, t_hbm = macs / imad, bytes_unique / HBM_BPS
    res = {
        "gpu": gpu, "sets": B, "r1cs": info, "generation_s": round(t_gen, 1),
        "check_ms": check_ms, "eval_ms": eval_ms, "check_sets_per_s": B / (ms * 1e-3),
        "eval_sets_per_s": B / (min(eval_ms) * 1e-3), "check_over_eval": ms / min(eval_ms),
        "all_valid_rows_pass": all_ok, "corrupted_row_index_matches_reference": bool(corrupt_ok),
        "counts_per_set": {"wide_macs": macs // B, "bytes_requested": 32 * info["n_terms"], "bytes_unique": 32 * info["n_wires"]},
        "imad_wide_per_s": imad,
        "int_pipe_share": t_int / (ms * 1e-3), "hbm_share_unique_bytes": t_hbm / (ms * 1e-3),
        "hbm_requested_bytes_per_s": bytes_terms / (ms * 1e-3),
        "binding": "integer pipe" if t_int > t_hbm else "HBM",
        "share_of_binding_roofline": max(t_int, t_hbm) / (ms * 1e-3),
    }
    with open(os.path.join(a.out, "r1cs_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))
    if not (all_ok and corrupt_ok):
        raise SystemExit("wrong verdicts")


if __name__ == "__main__":
    main()
