#!/usr/bin/env python3
"""Headline benchmark: batched witness generation for circuit9_authV2 (BASELINE.json config 4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path (graph::evaluate for every input set) over the batch: --batch input sets
(default 262 144, BASELINE config 4).  With N > 1 ranks the batch is SHARDED over the ranks (contiguous shards, "scaling":
"strong": 262 144 sets over 1/2/4/8 GPUs as config 4 states; --scaling weak gives every rank its own --batch sets
instead).  There is no collective on the data path (witnesses are independent); torch.distributed (gloo) is used only for
the timing barrier and the max over ranks.  A rank evaluates its shard launch by launch because the witnesses of a
whole shard do not fit HBM; every launch writes its witnesses to HBM in full.

Printed JSON line (rank 0): metric witnesses/s (+ node-ops/s in `extra`);
  value        kernel-only, inputs resident in HBM, CUDA events on the launching stream, max over ranks
  e2e          the same batch through the C ABI's streaming entry point gw_calc_witness_batch_stream with pinned HOST
               inputs: H2D + kernels + D2H into the library's pinned ring + a consumer callback per chunk, all inside
               the timed region, at the FULL batch size
  roofline     integer pipe (the binding roof for authV2) with the algorithmic and the executed-work fraction,
  roofline_hbm the HBM cross-check
  cpu_baseline C restatement of the reference algorithm on the host cores (bounded sample of the same inputs)
  configs      N = 1 only: BASELINE configs 1, 2, 3, 5 at their stated sizes (kernel-only rate, binding roofline, parity bit,
               GPU vs one CPU thread latency)
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CIRCUIT_DEFAULT = "circuit9_authV2"
M = 21888242871839275222246405745257275088548364400416034343698204186575808495617
UNIT = "witnesses/s"
DUMP_BUDGET_BYTES = 60 << 20         # witness.npy of --dump-outputs (float64 limbs); the index array and headers fit beside it
DUMP_SEED = 20241


def shard_range(n_units: int, rank: int, world: int):
    """contiguous shard [lo, hi) of n_units for `rank`"""
    return n_units * rank // world, n_units * (rank + 1) // world


def launch_plan(n_sets: int, max_chunk: int, sms: int):
    """[lo, hi) per launch.  The kernel runs one persistent CTA per SM and its time steps with ceil(warps per CTA / 4)
    (four schedulers per SM), so a launch should fill whole quads of warps on every SM: chunks are multiples of
    sms x 128 input sets (sms x 32 when less fits), as large as `max_chunk` allows; the last launch takes the rest."""
    if n_sets <= 0:
        return []
    quad, wave = sms * 128, sms * 32
    chunk = max_chunk // quad * quad if max_chunk >= quad else max(max_chunk // wave * wave, wave)
    return [(lo, min(lo + chunk, n_sets)) for lo in range(0, n_sets, chunk)]


def synth_inputs(name: str, lo: int, hi: int, n_inputs: int, input_map: dict, seed: int, first_row_fixture=True) -> np.ndarray:
    """Rows [lo, hi) of the synthetic batch, uint8 [hi - lo, I, 32] (SURVEY.md 8d): set 0 = the reference's own fixture
    (a valid proof request for authV2), the others uniform in [0, M) (bits for SHA-256 and for the *NoAux flags of
    authV2).  A row is a function of (seed, row index) only -- blocks of 8192 rows have their own generator -- so every
    rank, the CPU arm and the tests see the same batch whatever slice they take."""
    from tests import util
    block = 8192
    parts = []
    for b0 in range(lo // block * block, hi, block):
        rng = np.random.default_rng([seed, b0 // block])
        vals = util.random_field_batch(rng, (block, n_inputs))
        if "sha256" in name:
            vals[:] = 0
            vals[:, :, 0] = rng.integers(0, 2, size=(block, n_inputs), dtype=np.uint64)
        for key in ("authClaimNonRevMtpNoAux", "gistMtpNoAux"):
            if key in input_map:
                off, ln = input_map[key]
                vals[:, off:off + ln, :] = 0
                vals[:, off:off + ln, 0] = rng.integers(0, 2, size=(block, ln), dtype=np.uint64)
        parts.append(vals[max(lo - b0, 0):min(hi - b0, block)])
    out = np.concatenate(parts) if parts else np.empty((0, n_inputs, 4), dtype=np.uint64)
    out[:, 0, :] = 0
    out[:, 0, 0] = 1
    if first_row_fixture and lo == 0 and hi > 0:
        try:
            from oracle import pyoracle as po
            fixture = po.deserialize_inputs(util.golden_inputs(name))
            row = [1] + [0] * (n_inputs - 1)
            for k, v in fixture.items():
                off, ln = input_map[k]
                row[off:off + ln] = v
            out[0] = np.frombuffer(util.pack_u256(row), dtype=np.uint64).reshape(n_inputs, 4)
        except FileNotFoundError:
            pass
    return np.ascontiguousarray(out).view(np.uint8).reshape(hi - lo, n_inputs, 32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for nm, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def cpu_reference_run(graph_bytes, inp, steps, warmup):
    """C restatement of the reference algorithm (oracle/ref_eval.c), all host threads, on the given input sets"""
    from oracle import cref
    cg = cref.CGraph(graph_bytes)
    cores = os.cpu_count() or 1
    for _ in range(warmup):
        cg.evaluate_batch(inp[:max(cores, 1)], cores)
    t0 = time.perf_counter()
    for _ in range(steps):
        cg.evaluate_batch(inp, cores)
    dt = (time.perf_counter() - t0) / steps
    return inp.shape[0] / dt, dt, cores, cg.n_ops


def imad_per_witness(info, executed=False):
    """SURVEY 8d cost model: 264 IMAD per field multiplication on 8x32-bit limbs; a Div = one multiplication + one
    safegcd inversion (20 rounds x 92 signed 32x32->64 multiply-adds = 3680 IMAD-equivalents).  executed=True counts
    the inversions the plan actually runs after Div batching and the 3 extra multiplications per batched division."""
    inv = 20 * 92 * 2
    if not executed:
        return 264.0 * (info["n_mul"] + info["n_div"]) + inv * info["n_div"]
    extra_mul = 3 * max(info["n_div"] - info["n_inversions"], 0) + info["n_inversions"]
    return 264.0 * (info["n_mul"] + extra_mul) + inv * info["n_inversions"]


# ---- BASELINE configs 1, 2, 3, 5 (N = 1 only) --------------------------------------------------------------------
def config_batch(cwc, torch, tag, name, B, seed, peaks, imad_peak, reps=5, warmup=3):
    """kernel-only rate of one batch config at its stated size, binding roofline, parity of sampled rows"""
    from oracle import cref
    from tests import util
    dev = torch.device("cuda", 0)
    data = util.golden_graph(name)
    g = cwc.Graph(data)
    info = g.info
    I, W = g.n_inputs, g.n_witness
    host = synth_inputs(name, 0, B, I, g.input_signals, seed, first_row_fixture=False)
    d_in = torch.from_numpy(host.reshape(B, -1)).to(dev)
    free_b, _ = torch.cuda.mem_get_info()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    launches = launch_plan(B, max(int((free_b - (6 << 30)) // max(W * 32, 1)), sms * 32), sms)
    chunk = max(hi - lo for lo, hi in launches)
    d_out = torch.empty((chunk, W * 32), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    def step():
        for lo, hi in launches:
            g.calc_witness_batch_device(0, d_in[lo:hi].data_ptr(), hi - lo, d_out.data_ptr(), None, stream.cuda_stream)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    lo, hi = launches[-1]
    rows = sorted({0, (hi - lo) // 3, (hi - lo) // 2, hi - lo - 1})
    got = d_out[rows].cpu().numpy().reshape(len(rows), W, 32)
    want = cref.CGraph(data).evaluate_batch(host[[lo + r for r in rows]], min(len(rows), os.cpu_count() or 1))
    rate = B / (ms * 1e-3)
    alg_bytes = 32.0 * (I - 1 + W)
    gbs = alg_bytes * B / (ms * 1e-3) / 1e9
    timad = imad_per_witness(info) * B / (ms * 1e-3) / 1e12
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    t_hbm, t_imad = alg_bytes / (hbm_peak * 1e9), imad_per_witness(info) / imad_peak       # seconds per witness at each roof
    # a graph that runs bit-sliced executes LUT instructions on 32 input sets per word, no field multiplications: what
    # bounds it is reading the inputs and writing 32 bytes per witness value
    bound = "hbm" if (t_hbm >= t_imad or info.get("bit_eligible")) else "imad"
    roof = ({"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak} if bound == "hbm" else
            {"bound": "imad", "achieved": timad, "peak": imad_peak / 1e12, "unit": "TIMAD/s", "frac": timad * 1e12 / imad_peak})
    res = {"config": tag, "circuit": name, "batch": B, "launches_per_step": len(launches), "ms_per_step": ms, "witnesses_per_s": rate,
           "node_ops_per_s": rate * info["n_ops"], "roofline": roof, "hbm_algorithmic_GBps": gbs, "imad_algorithmic_T": timad,
           "parity_rows_bit_exact": bool((got == want).all()), "rows_checked": len(rows), "witness_len": W, "inputs_len": I,
           "n_instrs": info["n_instrs"], "n_spill": info["n_spill"],
           "bit_sliced": bool(info.get("bit_eligible")), "bit_luts": info.get("bit_luts"), "bit_steps": info.get("bit_steps"),
           "l2": f"{chunk * W * 32 / 1e6:.0f} MB of witness written per launch (L2 is 126 MB)"}
    del d_in, d_out, g
    torch.cuda.empty_cache()
    return res


def config_single(cwc, tag, name, reps=20):
    """one witness, JSON + graph -> .wtns: the latency-mode kernel against ONE thread of the CPU restatement"""
    from oracle import cref, pyoracle as po
    from tests import util
    data = util.golden_graph(name)
    nodes, wit, imap = po.deserialize_graph(data)
    g = cwc.Graph(data)
    buf = po.build_input_buffer(nodes, imap, po.deserialize_inputs(util.golden_inputs(name)))
    row = np.frombuffer(util.pack_u256(buf), dtype=np.uint8).reshape(g.n_inputs, 32)
    ok = cwc.calc_witness_wtns(util.golden_inputs(name), data) == util.golden_wtns(name)      # gw_calc_witness, the drop-in call
    kern, wall, e2e = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter(); _, ms = g.calc_witness_latency(row); wall.append((time.perf_counter() - t0) * 1e3); kern.append(ms)
        t0 = time.perf_counter(); g.calc_witness_wtns(util.golden_inputs(name)); e2e.append((time.perf_counter() - t0) * 1e3)
    cg = cref.CGraph(data)
    cpu = []
    for _ in range(10):
        t0 = time.perf_counter(); cg.evaluate_batch(row.reshape(1, g.n_inputs, 32), 1); cpu.append((time.perf_counter() - t0) * 1e3)
    return {"config": tag, "circuit": name, "wtns_bit_exact": bool(ok), "gpu_kernel_ms": statistics.median(kern),
            "gpu_call_ms": statistics.median(wall), "gpu_json_to_wtns_ms": statistics.median(e2e),
            "cpu_port_1thread_ms": statistics.median(cpu), "gpu_over_cpu": statistics.median(cpu) / statistics.median(kern), "reps": reps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--circuit", default=CIRCUIT_DEFAULT)
    ap.add_argument("--batch", type=int, default=262144, help="input sets per step (whole job when --scaling strong, per GPU when weak)")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--chunk", type=int, default=0, help="input sets per kernel launch (0 = auto)")
    ap.add_argument("--e2e-sets", type=int, default=0, help="input sets per rank of the end-to-end leg (0 = the rank's whole shard)")
    ap.add_argument("--e2e-chunk", type=int, default=0, help="input sets per streamed chunk (0 = auto)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="input sets for the cpu_baseline leg (0 = 96 x cores)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write a fixed, seeded sample of the witnesses the last timed step computed (rank 0's shard) to DIR: "
                         "witness.npy float64 [R, W, 8] = the 32-bit little-endian limbs of each canonical witness value, "
                         "input_set.npy float64 [R] = the index of each sampled input set in the batch; at most 64 MB.  "
                         "The row copies run in the last timed step; their event-measured time is left out of the timing "
                         "(extra.dump_copy_ms_excluded)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from tests import util
    graph_bytes = util.golden_graph(a.circuit)
    metric = f"{a.circuit} witnesses/sec (batched witness generation, graph::evaluate)"
    scaling = a.scaling if world > 1 else "strong"
    B_total = a.batch if scaling == "strong" else a.batch * world

    if a.impl == "reference":
        # the reference's own CPU implementation of the path; the Rust binary cannot be built in this image
        # (no cargo/rustc), so this is its C restatement with the same cost structure, on all host threads.
        if rank != 0:
            return
        from oracle import cref
        cg = cref.CGraph(graph_bytes)
        from oracle import pyoracle as po
        _, _, imap = po.deserialize_graph(graph_bytes)
        cores = os.cpu_count() or 1
        n_sets = a.cpu_sample or 32 * cores
        inp = synth_inputs(a.circuit, 0, n_sets, cg.n_inputs, imap, 9)        # the first rows of the b200 arm's batch
        val, dt, cores, n_ops = cpu_reference_run(graph_bytes, inp, a.steps, min(a.warmup, 1))
        print(json.dumps({
            "impl": "reference", "metric": metric, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "u256 (4x64-bit Montgomery limbs)", "data": "synthetic",
            "config": {"workload": f"{a.circuit}: {n_sets} input sets per step = the first rows of the {B_total}-set batch the b200 arm evaluates (bounded sample)",
                       "graph_nodes": cg.n_nodes, "witness_len": cg.n_witness},
            "extra": {"node_ops_per_s": val * n_ops},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{n_sets} input sets x {a.steps} steps, oracle/ref_eval.c (C restatement of the reference "
                                       "algorithm: the Rust crate cannot be built in this image), one witness per thread"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    # native libraries may write to fd 1: keep stdout clean for the ONE JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(obj), flush=True)

    import torch
    import torch.distributed as dist
    cwc = importlib.import_module("circom-witnesscalc_b200")
    if not torch.cuda.is_available() or cwc.device_count() < 1:
        raise SystemExit("bench.py --impl b200 needs a CUDA device: the witness evaluator has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # plumbing only (barrier + max of the step time): gloo, the data path has no collective and the library no NCCL
        dist.init_process_group("gloo")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    g = cwc.Graph(graph_bytes)
    info = g.info
    I, W = g.n_inputs, g.n_witness
    lo_set, hi_set = shard_range(B_total, rank, world) if scaling == "strong" else (rank * a.batch, (rank + 1) * a.batch)
    B = hi_set - lo_set                                       # this rank's input sets
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    t_gen = time.perf_counter()
    host_in = synth_inputs(a.circuit, lo_set, hi_set, I, g.input_signals, seed=9)      # this rank's rows of the job's batch
    t_gen = time.perf_counter() - t_gen
    h_in = torch.from_numpy(host_in.reshape(B, I * 32)).pin_memory()
    d_in = h_in.to(dev)
    free_b, _ = torch.cuda.mem_get_info()
    # HBM budget of one launch: its witnesses (W x 32 B each) beside the spill area (allocated on first use:
    # n_spill x 32 B for each of the sms x 512 threads a launch can have) and some slack
    reserve = info["n_spill"] * 32 * sms * 512 + (3 << 30)
    max_chunk = a.chunk or min(int(max(sms * 32, (free_b - reserve) // (W * 32))), sms * 512)
    launches = launch_plan(B, max_chunk, sms)
    chunk = max(hi - lo for lo, hi in launches)
    d_out = torch.empty((chunk, W * 32), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    # --dump-outputs: the sampled rows are chosen by their index in the shard, not by launch, so that two builds whose
    # launch plans differ still dump the same input sets.  d_out only holds the current launch, so in the last timed step
    # the sampled rows are copied into d_dump after each launch, on the same stream (one cudaMemcpyAsync per row, no
    # kernel).  CUDA events bracket each group of copies, and their time is taken out of the timed total.
    d_dump, dump_rows, dump_at, dump_events = None, None, [[] for _ in launches], []
    if a.dump_outputs and rank == 0:
        n_dump = min(B, DUMP_BUDGET_BYTES // (W * 8 * 8))
        if n_dump < 1:
            raise SystemExit(f"--dump-outputs: one witness of {W} values exceeds {DUMP_BUDGET_BYTES} bytes as float64 limbs")
        dump_rows = np.sort(np.random.default_rng(DUMP_SEED).choice(B, n_dump, replace=False))
        d_dump = torch.empty((n_dump, W * 32), dtype=torch.uint8, device=dev)
        for k, r in enumerate(dump_rows):
            i = next(i for i, (lo, hi) in enumerate(launches) if lo <= r < hi)
            dump_at[i].append((k, int(r) - launches[i][0]))

    def step(dump=False):
        for (lo, hi), dumps in zip(launches, dump_at):
            g.calc_witness_batch_device(local_rank, d_in[lo:hi].data_ptr(), hi - lo, d_out.data_ptr(), None, stream.cuda_stream)
            if dump and dumps:
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(stream)
                for k, r in dumps:
                    d_dump[k].copy_(d_out[r])
                c1.record(stream)
                dump_events.append((c0, c1))

    for _ in range(a.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s in range(a.steps):
        step(dump=d_dump is not None and s == a.steps - 1)
    e1.record(stream)
    barrier()
    dump_copy_ms = sum(c0.elapsed_time(c1) for c0, c1 in dump_events)
    ms_total = e0.elapsed_time(e1) - dump_copy_ms
    clocks = sampler.stop() if sampler else None
    ms_step = max_over_ranks(ms_total) / a.steps
    value = B_total / (ms_step * 1e-3)
    n_launches = a.steps * len(launches)
    kernel_ms = ms_total / max(n_launches, 1)            # launches are back to back on one stream

    # parity of what the timed region produced (last launch) against the C oracle: 64 rows spread over the launch
    verified = None
    if rank == 0:
        from oracle import cref
        cg = cref.CGraph(graph_bytes)
        lo, hi = launches[-1]
        rows = sorted({int(x) for x in np.linspace(0, hi - lo - 1, 64)})
        got = d_out[rows].cpu().numpy().reshape(len(rows), W, 32)
        verified = bool((cg.evaluate_batch(host_in[[lo + r for r in rows]], min(len(rows), os.cpu_count() or 1)) == got).all())
    if d_dump is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        limbs = d_dump.cpu().numpy().reshape(len(dump_rows), W, 32).view("<u4")
        np.save(os.path.join(a.dump_outputs, "witness.npy"), limbs.astype(np.float64))
        np.save(os.path.join(a.dump_outputs, "input_set.npy"), (lo_set + dump_rows).astype(np.float64))
        del d_dump
    del d_out
    torch.cuda.empty_cache()

    # end to end through the C ABI: pinned HOST inputs -> gw_calc_witness_batch_stream -> consumer callback per chunk of
    # witnesses in the library's pinned ring (H2D + kernels + D2H + callback inside the timed region), whole shard
    e2e = None
    if not a.no_e2e:
        n_e = min(a.e2e_sets or B, B)
        # ring slot: at most 8 GiB, and the three slots of all ranks together at most a quarter of the free host memory
        slot_b = 8 << 30
        try:
            avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable:")][0]
            slot_b = min(slot_b, avail // (12 * world))
        except (OSError, IndexError, ValueError):
            pass
        e_chunk = a.e2e_chunk or max(32, min(slot_b // (W * 32), sms * 512) // 32 * 32)
        keep = {}

        def consumer(device, first, rows, flags):
            # the consumer touches every chunk: first row kept for verification (up to 24 chunks), flags must be clear
            if len(keep) < 24:
                keep[first] = rows[0].copy()
            return int(flags[0] != 0)
        g.calc_witness_batch_stream(h_in.data_ptr(), min(n_e, 2 * e_chunk), consumer, first_device=local_rank, chunk_sets=e_chunk)   # warm-up: pins the ring
        keep.clear()
        barrier()
        t0 = time.perf_counter()
        g.calc_witness_batch_stream(h_in.data_ptr(), n_e, consumer, first_device=local_rank, chunk_sets=e_chunk)
        dt = max_over_ranks(time.perf_counter() - t0)
        n_e_total = n_e * world if n_e != B else B_total
        e2e = {"value": n_e_total / dt, "unit": UNIT, "h2d_bytes_per_step": n_e_total * I * 32, "d2h_bytes_per_step": n_e_total * W * 32,
               "sets_per_step": n_e_total, "seconds": dt, "chunk_sets": e_chunk, "d2h_GBps": n_e_total * W * 32 / dt / 1e9,
               "api": "gw_calc_witness_batch_stream: pinned host inputs, per GPU a ring of 3 pinned chunks, consumer callback per chunk"}
        if rank == 0:
            firsts = sorted(keep)[:24]
            want = cg.evaluate_batch(host_in[firsts], min(len(firsts), os.cpu_count() or 1))
            e2e["verified_rows"] = len(firsts)
            e2e["verified_against_oracle"] = bool(all((want[i].reshape(W, 32) == keep[f]).all() for i, f in enumerate(firsts)))
        # the in-library multi-GPU path once (one process, one worker thread per GPU): rank 0 drives all N GPUs
        if world > 1:
            barrier()
            if rank == 0:
                n_lib = min(B_total, B * world)
                lib_in = synth_inputs(a.circuit, 0, min(n_lib, 32768), I, g.input_signals, seed=9)
                h_lib = torch.from_numpy(np.resize(lib_in.reshape(-1, I * 32), (n_lib, I * 32))).pin_memory()
                cnt = [0]
                lk = threading.Lock()

                def consumer2(device, first, rows, flags):
                    with lk:
                        cnt[0] += rows.shape[0]
                    return 0
                g.calc_witness_batch_stream(h_lib.data_ptr(), min(n_lib, 2 * e_chunk * world), consumer2, n_gpus=world, first_device=0, chunk_sets=e_chunk)
                cnt[0] = 0
                t0 = time.perf_counter()
                g.calc_witness_batch_stream(h_lib.data_ptr(), n_lib, consumer2, n_gpus=world, first_device=0, chunk_sets=e_chunk)
                dt2 = time.perf_counter() - t0
                e2e["in_library_n_gpus"] = {"value": n_lib / dt2, "unit": UNIT, "sets": n_lib, "delivered": cnt[0], "seconds": dt2,
                                            "api": f"one process, gw_calc_witness_batch_stream(n_gpus={world}): one worker thread per GPU"}
                del h_lib
            barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # rooflines.  Integer pipe: algorithmic IMADs against the IMAD rate measured on this GPU by the library's microbenchmark.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    imad_lo = cwc.microbench_imad(local_rank, 1)
    imad_wide = cwc.microbench_imad(local_rank, 0)
    per_launch_sets = B / max(len(launches), 1)
    alg_imad, exe_imad = imad_per_witness(info), imad_per_witness(info, executed=True)
    achieved_imad = alg_imad * per_launch_sets / (kernel_ms * 1e-3)
    bytes_per_witness = 32.0 * (I - 1 + W)
    achieved_gbs = bytes_per_witness * per_launch_sets / (kernel_ms * 1e-3) / 1e9
    # DRAM traffic of the dominant kernel from the committed one-pass ncu capture (bytes per input set x sets per launch)
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(a.circuit)
        if tj and tj.get("witness_len", W) == W:
            traffic, traffic_src = tj["dram_bytes_per_set"] * per_launch_sets, tj["source"]
    except Exception:
        pass
    roofline = {"bound": "imad", "achieved": achieved_imad / 1e12, "peak": imad_lo / 1e12, "unit": "TIMAD/s",
                "frac": achieved_imad / imad_lo, "frac_executed_work": exe_imad * per_launch_sets / (kernel_ms * 1e-3) / imad_lo,
                "traffic": traffic, "traffic_unit": "bytes per launch (dram read + write)",
                "traffic_source": traffic_src, "algorithmic_bytes_per_launch": bytes_per_witness * per_launch_sets,
                "imad_per_witness": alg_imad, "imad_per_witness_executed": exe_imad,
                "note": "algorithmic: 264 IMAD per field mul x (n_mul + n_div) + 3680 per Div (one safegcd inversion each); "
                        "executed work: the inversions left after Div batching + its 3 extra multiplications per division; peak = "
                        "mad.lo.u32 rate measured live by gw_microbench_imad (MEASURED_PEAKS.json has no integer peak)",
                "imad_wide_peak_Tops": imad_wide / 1e12}
    roofline_hbm = {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                    "traffic": traffic, "peak_source": hbm_src,
                    "note": "algorithmic bytes = 32*(I-1+W) per witness (inputs read + witness written)"}

    cpu = None
    if not a.no_cpu and world == 1:
        cores = os.cpu_count() or 1
        n_sets = min(a.cpu_sample or 96 * cores, B)
        v, dt, cores, _ = cpu_reference_run(graph_bytes, host_in[:n_sets], 1, 1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"the first {n_sets} input sets of the batch the GPU arm evaluated, oracle/ref_eval.c (C restatement of the "
                         f"reference algorithm, graph parsed once), one witness per thread, {dt:.2f} s"}

    configs = None
    if world == 1 and not a.no_configs and a.circuit == CIRCUIT_DEFAULT:
        del d_in
        torch.cuda.empty_cache()
        configs = []
        for fn in (lambda: config_single(cwc, "1: circuit5_poseidon, single witness, gw_calc_witness vs reference fixture", "circuit5_poseidon"),
                   lambda: config_batch(cwc, torch, "2a: circuit6_num2bits x 65536", "circuit6_num2bits", 65536, 6, peaks, imad_lo),
                   lambda: config_batch(cwc, torch, "2b: circuit7_poseidon4 x 65536", "circuit7_poseidon4", 65536, 7, peaks, imad_lo),
                   lambda: config_batch(cwc, torch, "3: circuit8_sha256_512 x 16384", "circuit8_sha256_512", 16384, 8, peaks, imad_lo),
                   lambda: config_single(cwc, "5: circuit9_authV2, single witness, latency mode vs one CPU thread", "circuit9_authV2"),
                   lambda: config_single(cwc, "5 (same mode, a graph with wide levels): circuit8_sha256_512, single witness vs one CPU thread", "circuit8_sha256_512")):
            try:
                configs.append(fn())
            except Exception as e:      # a failing side config must not take the headline line with it
                configs.append({"error": repr(e)})
        configs.insert(3, {"config": "4: circuit9_authV2 x 262144 over 1/2/4/8 GPUs", "see": "this line (value, e2e, roofline)"})

    line = {
        "metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": "u256 (8x32-bit limbs, canonical BN254 scalars)", "data": "synthetic",
        "config": {"workload": f"{a.circuit} (iden3 authV2(40,64)): {B_total} random input sets per step"
                               + (f" sharded over {world} GPUs ({B} per GPU)" if world > 1 and scaling == "strong" else
                                  f" ({a.batch} per GPU)" if world > 1 else "")
                               + f", {len(launches)} launches of <= {chunk} sets per GPU and step",
                   "graph_nodes": info["n_nodes"], "node_ops": info["n_ops"], "inputs_len": I,
                   "witness_len": W, "unique_input_sets": B_total, "input_gen_s": round(t_gen, 1),
                   "l2": f"every launch writes {chunk * W * 32 / 1e9:.1f} GB of witness (>> 126 MB L2), no flush needed",
                   "regs_per_witness": info["n_regs"], "spill_slots": info["n_spill"]},
        "extra": {"node_ops_per_s": value * info["n_ops"], "field_mul_per_s": value * info["n_mul"],
                  "kernel_ms_per_launch": kernel_ms, "verified_against_oracle": verified, "verified_rows": 64},
        "roofline": roofline, "roofline_hbm": roofline_hbm, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": n_launches, "clocks": clocks, "configs": configs,
    }
    if a.dump_outputs:
        line["extra"]["dump_copy_ms_excluded"] = dump_copy_ms
    if world > 1:
        dist.destroy_process_group()
    emit(line)


if __name__ == "__main__":
    main()
