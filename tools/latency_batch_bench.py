#!/usr/bin/env python3
"""Small batches on the latency kernels (gw_calc_witness_latency_batch_device, one latency CTA per input set) against the
throughput kernel (gw_calc_witness_batch_device, one lane per set), on the same seeded inputs in device memory.

  python tools/latency_batch_bench.py --out DIR [--graphs circuit9_authV2,authV2_32_32,circuit7_poseidon4]
                                      [--sizes 1,16,74,148,296,592,1184,4736,9472] [--reps 5]

Per graph and batch size n: both calls once as warm-up; the two rows of outputs compared byte for byte over all n sets and
8 sampled sets against the C oracle before any time is kept; then --reps rounds, each timing one call of each path with CUDA
events on one stream, the paths alternated.  Reported: best and median ms per call and path, the spread (max / min),
witnesses/s, and the ratio throughput / latency.  Field graphs only: a Boolean graph runs the same bit-sliced launch on both
paths.  Writes DIR/latency_batch_bench.json (one JSON object per line) and DIR/smi.csv (card name, power limit, SM clocks
of the same run)."""
import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import cref  # noqa: E402
from tests import util  # noqa: E402

SIZES = (1, 16, 74, 148, 296, 592, 1184, 4736, 9472)
GRAPHS = ("circuit9_authV2", "authV2_32_32", "circuit7_poseidon4")


def smi(out_dir):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"],
                       capture_output=True, text=True)
    text = q.stdout if q.returncode == 0 else "nvidia-smi failed\n"
    with open(os.path.join(out_dir, "smi.csv"), "w") as f:
        f.write(text)
    line = (text.splitlines()[1:2] or ["?"])[0].split(", ")
    return {"gpu": line[0], "power_limit": line[1] if len(line) > 1 else "?", "max_sm_clock": line[2] if len(line) > 2 else "?"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--graphs", default=",".join(GRAPHS))
    ap.add_argument("--sizes", default=",".join(map(str, SIZES)))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: this measurement needs the GPU")
    os.makedirs(a.out, exist_ok=True)
    cwc = importlib.import_module("circom-witnesscalc_b200")
    sizes = [int(x) for x in a.sizes.split(",")]
    card = smi(a.out)
    card["sms"] = torch.cuda.get_device_properties(0).multi_processor_count
    print(json.dumps(card), flush=True)
    s = torch.cuda.Stream()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    rows_out = []
    for name in a.graphs.split(","):
        data = util.golden_graph(name)
        g = cwc.Graph(data)
        oracle = cref.CGraph(data)
        nmax = max(sizes)
        rng = np.random.default_rng(2024)
        vals = util.random_field_batch(rng, (nmax, g.n_inputs))
        vals[:, 0, :] = 0
        vals[:, 0, 0] = 1
        inp = np.ascontiguousarray(vals.view(np.uint8).reshape(nmax, g.n_inputs, 32))
        d_in = torch.from_numpy(inp.reshape(-1).copy()).cuda()
        d_lat = torch.empty((nmax, g.n_witness * 32), dtype=torch.uint8, device="cuda")
        d_thr = torch.empty_like(d_lat)
        d_fl = torch.empty((2, nmax), dtype=torch.int32, device="cuda")

        def call(path, n):
            if path == "latency":
                g.calc_witness_latency_batch_device(0, d_in.data_ptr(), n, d_lat.data_ptr(), d_fl[0].data_ptr(), s.cuda_stream)
            else:
                g.calc_witness_batch_device(0, d_in.data_ptr(), n, d_thr.data_ptr(), d_fl[1].data_ptr(), s.cuda_stream)

        def timed(path, n):
            ev[0].record(s)
            call(path, n)
            ev[1].record(s)
            ev[1].synchronize()
            return ev[0].elapsed_time(ev[1])

        for n in sizes:
            d_lat.fill_(0xA5)
            d_thr.fill_(0x5A)
            torch.cuda.synchronize()
            call("latency", n)
            call("throughput", n)
            s.synchronize()
            same = bool(torch.equal(d_lat[:n], d_thr[:n])) and bool(torch.equal(d_fl[0, :n], d_fl[1, :n]))
            pick = sorted({0, n - 1} | set(np.random.default_rng(n).integers(0, n, 6).tolist()))
            want = oracle.evaluate_batch(np.ascontiguousarray(inp[pick]), 8).reshape(len(pick), -1)
            got = d_lat[pick].cpu().numpy()
            if not same or not np.array_equal(got, want):
                sys.exit(f"{name} n={n}: latency batch rows differ from the throughput rows or the C oracle; no time is kept")
            t = {"latency": [], "throughput": []}
            for r in range(a.reps):
                for path in (("latency", "throughput") if r % 2 == 0 else ("throughput", "latency")):
                    t[path].append(timed(path, n))
            rec = {"graph": name, "n": n, "W": g.n_witness, "reps": a.reps, **card}
            for path in t:
                best, med = min(t[path]), float(np.median(t[path]))
                rec[path] = {"best_ms": round(best, 3), "median_ms": round(med, 3), "spread": round(max(t[path]) / best, 3),
                             "witnesses_per_s": round(n / best * 1e3, 1), "all_ms": [round(x, 3) for x in t[path]]}
            rec["throughput_over_latency"] = round(rec["throughput"]["best_ms"] / rec["latency"]["best_ms"], 3)
            print(json.dumps(rec), flush=True)
            rows_out.append(rec)
        del d_in, d_lat, d_thr, d_fl
        torch.cuda.empty_cache()
        g.close()
    with open(os.path.join(a.out, "latency_batch_bench.json"), "w") as f:
        for rec in rows_out:
            f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
