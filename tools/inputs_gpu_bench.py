#!/usr/bin/env python3
"""Device input parser against the host parser, on randomised authV2 records generated as tools/parse_probe.py does.

  python tools/inputs_gpu_bench.py --out DIR [--sizes 75776,262144] [--reps 3]

Per size: (1) gw_inputs_parse_batch records/s at 1 and all host threads; (2) gw_inputs_parse_batch_device records/s
and GB/s of text, from pageable and from pinned text, whole call by the host clock, the text copy alone (CUDA events) and the kernels
from a torch.profiler run of one call, with the number of records the host had to parse (GW_TRACE_HOST);
(3) text -> witness rows in HBM by both routes (host parse + packed-row upload + gw_calc_witness_batch_device, against
device parse + gw_calc_witness_batch_device), at the first size.  Every device row is checked equal to the host row.
Writes DIR/inputs_gpu_bench.json (one JSON object per line) with the card's name and power limit."""
import argparse
import ctypes
import importlib
import json
import os
import random
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests import util  # noqa: E402

NAME = "circuit9_authV2"


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout else ("?", "?")
    return {"gpu": name.strip(), "power_limit": power.strip()}


def make_text(g, n):
    base = json.loads(util.golden_inputs(NAME))
    rnd = random.Random(1)

    def rand_like(v):
        return [rand_like(x) for x in v] if isinstance(v, list) else str(rnd.randrange(util.M))
    recs = [json.dumps({k: rand_like(v) for k, v in base.items()}) for _ in range(64)]
    return ("\n".join(recs[i % 64] for i in range(n)) + "\n").encode()


def best_of(reps, fn):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts)


def traced_marks(fn):
    """runs fn with GW_TRACE_HOST=1 and returns the 'marked' count the device parser printed"""
    os.environ["GW_TRACE_HOST"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile() as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            os.environ.pop("GW_TRACE_HOST")
        f.seek(0)
        lines = [l for l in f.read().decode().splitlines() if l.startswith("[gw inputs]")]
    return int(lines[-1].rsplit("marked ", 1)[1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--sizes", default="75776,262144")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    import torch
    cwc = importlib.import_module("circom-witnesscalc_b200")
    os.makedirs(a.out, exist_ok=True)
    g = cwc.Graph(util.golden_graph(NAME))
    info = card()
    results = []
    for si, n in enumerate(int(x) for x in a.sizes.split(",")):
        text = make_text(g, n)
        row_b = g.n_inputs * 32
        r = {"bench": "inputs_gpu", "circuit": NAME, "records": n, "text_bytes": len(text), "bytes_per_record": len(text) // n,
             "packed_row_bytes": row_b, **info}
        host_rows = None
        for threads in (1, 0):
            reps = 1 if threads == 1 else a.reps
            holder = {}
            t = best_of(reps, lambda: holder.__setitem__("rows", g.parse_inputs_batch(text, threads)))
            host_rows = holder["rows"]
            r["host_threads_%s" % ("1" if threads == 1 else "all")] = {"threads": threads or os.cpu_count(), "s": round(t, 4),
                                                                      "records_per_s": round(n / t)}
        d_rows = torch.empty(n * row_b, dtype=torch.uint8, device="cuda")
        want = torch.from_numpy(host_rows.reshape(-1)).cuda()
        pinned = torch.empty(len(text), dtype=torch.uint8).pin_memory()
        pinned.numpy()[:] = np.frombuffer(text, np.uint8)
        fp = ctypes.CDLL(cwc.LIB_PATH).gw_inputs_parse_batch_device      # the text as a raw pointer: pageable or pinned
        fp.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_size_t,
                       ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p, ctypes.POINTER(cwc.gw_status_t)]

        def dev_parse(kind):
            cnt, st = ctypes.c_size_t(0), cwc.gw_status_t()
            src = pinned.data_ptr() if kind == "pinned" else ctypes.cast(ctypes.c_char_p(text), ctypes.c_void_p).value
            rc = fp(g._h, 0, src, len(text), d_rows.data_ptr(), n, ctypes.byref(cnt), None, ctypes.byref(st))
            cwc._check(rc, st)
            assert cnt.value == n
        for kind in ("pageable", "pinned"):
            dev_parse(kind)                                  # warm-up: key table, scratch
            d_rows.fill_(0)
            marks = traced_marks(lambda: dev_parse(kind))
            torch.cuda.synchronize()
            assert torch.equal(d_rows, want), "device rows differ from the host rows"
            t = best_of(a.reps, lambda: dev_parse(kind))
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                dev_parse(kind)
                torch.cuda.synchronize()
            # the text copy on its own, the same bytes from the same kind of host memory, timed with CUDA events
            d_text = torch.empty(len(text), dtype=torch.uint8, device="cuda")
            src_t = pinned if kind == "pinned" else torch.from_numpy(np.frombuffer(text, np.uint8).copy())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            copy_ms = []
            for _ in range(a.reps):
                e0.record()
                d_text.copy_(src_t, non_blocking=(kind == "pinned"))
                e1.record()
                torch.cuda.synchronize()
                copy_ms.append(e0.elapsed_time(e1))
            del d_text, src_t
            kern_us = 0.0
            per_kernel = {}
            for e in prof.key_averages():
                dt = getattr(e, "device_time_total", None)
                if dt is None:
                    dt = e.cuda_time_total
                if "inputs_" in e.key and "kernel" in e.key:
                    kern_us += dt
                    short = e.key.split("inputs_", 1)[1].split("(")[0].split("<")[0]
                    per_kernel[short] = round(per_kernel.get(short, 0) + dt / 1e3, 3)
            r["device_" + kind] = {"s": round(t, 4), "records_per_s": round(n / t), "text_GB_per_s": round(len(text) / t / 1e9, 2),
                                   "text_copy_ms": round(min(copy_ms), 3), "text_copy_GB_per_s": round(len(text) / min(copy_ms) / 1e6, 1),
                                   "profiled_kernels_ms": round(kern_us / 1e3, 3),
                                   "kernels_ms": per_kernel, "marked_records": marks,
                                   "kernel_text_GB_per_s": round(len(text) / (kern_us * 1e-6) / 1e9, 1) if kern_us else None}
        if si == 0:
            # text -> witness rows in HBM by both routes
            d_w = torch.empty((n, g.n_witness * 32), dtype=torch.uint8, device="cuda")

            def host_route():
                rows = g.parse_inputs_batch(text, 0)
                d_in = torch.from_numpy(rows.reshape(-1)).cuda()
                g.calc_witness_batch_device(0, d_in.data_ptr(), n, d_w.data_ptr(), None, None)
                torch.cuda.synchronize()

            def device_route():
                dev_parse("pinned")
                g.calc_witness_batch_device(0, d_rows.data_ptr(), n, d_w.data_ptr(), None, None)
                torch.cuda.synchronize()
            host_route()
            device_route()
            t_w = best_of(a.reps, lambda: (g.calc_witness_batch_device(0, d_rows.data_ptr(), n, d_w.data_ptr(), None, None),
                                           torch.cuda.synchronize()))
            t_h, t_d = best_of(a.reps, host_route), best_of(a.reps, device_route)
            r["text_to_witness"] = {"witness_launch_s": round(t_w, 4), "host_route_s": round(t_h, 4), "device_route_s": round(t_d, 4),
                                    "host_route_witness_per_s": round(n / t_h), "device_route_witness_per_s": round(n / t_d)}
            del d_w
            torch.cuda.empty_cache()
        print(json.dumps(r), flush=True)
        results.append(r)
        del d_rows, want, pinned
        torch.cuda.empty_cache()
    with open(os.path.join(a.out, "inputs_gpu_bench.json"), "w") as fo:
        for r in results:
            fo.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
