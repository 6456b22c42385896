#!/usr/bin/env python
"""bench.py -- per-round query throughput of the acquisition-scoring engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--no-extras] [--dump-outputs DIR]

Headline (BASELINE.json configs[1]): MarginSampler query tail on an ImageNet-shaped pool of
80 000 x 1000 fp32 logits per GPU, budget 10 000.  A "step" is one full tail: K1 (softmax margin)
-> K1b (stable top-B) -> the B selected positions on the host.  `value` counts rows scored per
second with the logits already resident in HBM; `e2e` is the same tail through the host-buffer
C-ABI entry point (pinned host logits, H2D and D2H inside the timed region).

N > 1 (weak scaling): every rank owns its own 80 000-row shard, scores it, selects its local
top-B, and one all-gather + device merge yields the global top-B (the only exchange).

The same JSON line carries `roofline` (K1, the dominant kernel), `cpu_baseline` (the oracle port
of the reference's CPU tail on this box's host cores) and, at N = 1, `workloads`: the CoreSet
(K3+K4) and BADGE (K2+K3+K5) tails at 80 000 candidates / 50 000 labeled / B = 10 000 with their own
roofline objects -- the BADGE k-means++ streaming kernel is the north star's 90 % target.

`--impl reference` times the reference's CPU implementation of the same tail (oracle port: the
reference is Python and cannot travel to the GPU box) on all host threads.

`--dump-outputs DIR` writes what the last timed step of the headline tail returned to its caller (rank 0's caller
at N > 1): `scores.npy` (float32, this rank's 80 000 margins; not with --impl reference, whose tail returns only the
positions) and `picks.npy` (the B selected positions, as float64).  The inputs are seeded, so two builds run with the
same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROWS, N_CLASSES, BUDGET = 80000, 1000, 10000
EMB_DIM, N_LABELED = 2048, 50000
METRIC = "unlabeled samples scored/sec per AL round (ImageNet 80k pool, B=10k)"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


_TF32 = {}


def tf32_peak():
    """Dense TF32 tensor peak, MEASURED here (SURVEY.md section 8d: it is not in MEASURED_PEAKS.json): cuBLAS TF32 GEMM
    8192^3 through torch.matmul with allow_tf32, best of 10, CUDA events -- the same recipe as the driver's bf16 figure.
    Only a denominator: nothing on the product path calls it.  Falls back to bf16 / 2 without a GPU."""
    if "v" in _TF32:
        return _TF32["v"]
    val, src = None, None
    try:
        if torch.cuda.is_available():
            old = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True
            n = 8192
            a = torch.randn(n, n, device="cuda")
            b = torch.randn(n, n, device="cuda")
            best = float("inf")
            for i in range(13):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                c = a @ b
                e1.record()
                torch.cuda.synchronize()
                if i >= 3:
                    best = min(best, e0.elapsed_time(e1))
            del a, b, c
            torch.backends.cuda.matmul.allow_tf32 = old
            val, src = 2.0 * n ** 3 / (best * 1e-3) / 1e12, "measured in this run: cuBLAS TF32 GEMM 8192^3 (torch.matmul, allow_tf32), best of 10"
    except Exception:
        val = None
    if val is None:
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                val = float(json.load(fh)["bf16_tflops"]) / 2.0
        except Exception:
            val = 1590.0 / 2.0
        src = "MEASURED_PEAKS.json bf16_tflops / 2 (no live TF32 measurement possible)"
    _TF32["v"], _TF32["src"] = val, src
    return val


def ncu_traffic(kernel):
    """DRAM bytes per launch from the committed ncu --set full capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(kernel)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t_rows = []

    def __enter__(self):
        if self.index < 0:
            return self
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])
            self.t_rows.append(time.perf_counter())

    def wait_first(self, timeout=8.0):
        t0 = time.perf_counter()
        while not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, window=None):
        """window = (t0, t1) perf_counter bounds of the timed region; samples inside it are preferred, else
        every sample taken while this process kept the GPU busy (warm-up .. e2e) is used and said so."""
        sm, mx, reasons = [], [], set()
        rows = self.rows
        note = "samples span warm-up..e2e (the timed region is shorter than the 100 ms sampling period)"
        if window is not None:
            inside = [r for r, t in zip(self.rows, self.t_rows) if window[0] <= t <= window[1]]
            if inside:
                rows, note = inside, "samples inside the timed region"
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "window": note}


# ----------------------------------------------------------------------------------------------
# reference arm: the reference's CPU tail (oracle port), all host threads
# ----------------------------------------------------------------------------------------------
def cpu_margin_tail(logits, budget):
    """margin_sampler.py:33-42 on CPU, batches of 128 like the reference's loader."""
    from oracle import al_oracle as O
    scores = O.softmax_scores(logits, O.MODE_MARGIN, batch_size=128)
    return O.select_smallest(scores, budget)


def cpu_greedy_baseline(steps=20):
    """SURVEY.md section 8d: the reference's own CoreSet / k-means++ selection on the host cores -- the oracle port of
    coreset_sampler.py:59-105 on ONE partition of the paper's configuration (gen_jobs.py:11-13: 13 000 rows = 5 000
    labeled + 8 000 unlabeled), `steps` steps of each mode, extrapolated linearly to 10 partitions x 1 000 picks (the
    per-step cost grows with the labeled set, so the extrapolation favours the CPU).  The non-partitioned 130 000-row
    query the GPU workloads run needs a 67.6 GB distance matrix and cannot be run by the reference at all."""
    from oracle import al_oracle as O
    threads = host_cpu_budget()
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(5)
    rows, lab, parts, picks = 13000, 5000, 10, 1000
    ind = np.zeros(rows, dtype=bool)
    ind[:lab] = True
    out = {"unit": "samples/s", "kind": "port", "cores": threads, "extrapolated": True,
           "sample": f"one partition of {rows} rows ({lab} labeled), pairwise matrix + {steps} steps per mode of the oracle port "
                     f"of coreset_sampler.py:59-105, scaled to {parts} partitions x {picks} picks; {cpu_model()}"}
    for kind, dim, randomize in (("coreset", EMB_DIM, False), ("badge", 512, True)):
        feat = torch.relu(torch.randn(rows, dim, generator=g))
        t0 = time.perf_counter()
        dist = O.pairwise_l2_dist(feat)
        t_pair = time.perf_counter() - t0
        np.random.seed(0)
        t0 = time.perf_counter()
        O.coreset(dist, ind, steps, randomize=randomize)
        t_step = (time.perf_counter() - t0) / steps
        del dist
        round_s = parts * (t_pair + picks * t_step)
        out[kind] = {"value": N_ROWS / round_s, "seconds_per_round": round_s, "pairwise_s": t_pair, "step_ms": t_step * 1e3,
                     "dim": dim}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.manual_seed(0)
    logits = torch.randn(N_ROWS, N_CLASSES) * 3.0
    threads, cpu_budget = tune_cpu_threads(logits)
    for _ in range(args.warmup):
        cpu_margin_tail(logits, BUDGET)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        picks = cpu_margin_tail(logits, BUDGET)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, picks=picks)
    val = N_ROWS / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{N_ROWS} x {N_CLASSES} logits per step (one GPU's shard), softmax->top2->sort "
                                   f"in loader batches of 128, torch-CPU, {threads} threads (best of a probe; "
                                   f"{cpu_budget} usable CPUs); {cpu_model()}"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def dump_outputs(out_dir, **arrays):
    """DIR/<name>.npy per array: floating arrays keep float32 / float64, integer ones (positions) become float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        np.save(os.path.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def host_cpu_budget():
    """CPUs this process may really use: affinity mask and cgroup quota, not os.cpu_count()."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            with open(path) as fh:
                parts = fh.read().split()
            if path.endswith("cpu.max"):
                if parts[0] != "max":
                    n = min(n, max(1, int(float(parts[0]) / float(parts[1]) + 0.5)))
            else:
                q = int(parts[0])
                if q > 0:
                    with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as fh2:
                        n = min(n, max(1, int(q / int(fh2.read()) + 0.5)))
        except Exception:
            pass
    return max(1, n)


def tune_cpu_threads(logits):
    """The reference's loader batches are only 128 x 1000: with one OpenMP thread per hardware thread
    the tail is dominated by fork/join overhead (measured: 1.0 k samples/s at 128 threads on the GPU
    box).  Give the CPU arm its best case: probe a few thread counts on a 4096-row sample and keep the
    fastest.  `cores` in the JSON is the count actually used."""
    budget = host_cpu_budget()
    cands = sorted({c for c in (budget, budget // 2, 32, 16, 8, 4) if 1 <= c <= budget}, reverse=True)
    sample = logits[:4096]
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        cpu_margin_tail(sample[:512], 64)
        t0 = time.perf_counter()
        cpu_margin_tail(sample, 512)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
        if dt > 5.0:
            continue
    torch.set_num_threads(best)
    return best, budget


def cpu_model():
    try:
        with open("/proc/cpuinfo") as fh:
            for ln in fh:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown CPU"


def workload_config(gpus):
    return {"workload": "MarginSampler query tail (configs[1]): softmax margin + stable top-B",
            "pool_rows_per_gpu": N_ROWS, "pool_rows_total": N_ROWS * gpus, "classes": N_CLASSES,
            "budget": BUDGET, "parallelism": f"row-sharded x{gpus}",
            "l2": "inputs (320 MB logits per GPU) are larger than the 126 MB L2; no flush needed"}


# ----------------------------------------------------------------------------------------------
# extra workloads (N = 1): CoreSet and BADGE tails at the north-star shapes
# ----------------------------------------------------------------------------------------------
def run_greedy_workload(eng, kind, peak, steps, warmup, world=1, rank=0, check_picks=400):
    """CoreSet / BADGE tail at the north-star shape.  world > 1: STRONG scaling -- the same 80 000 candidates; every
    rank holds a replica of the rows (the engine's multi-GPU contract: a centre is announced as a row id), the distance
    pass (K3) and the selection loop (K4 / K5) are sharded by candidate row, and the per-step agreement on the centre
    runs inside ONE persistent kernel per rank over peer-memory windows (no NCCL call and no launch in the loop).
    The first `check_picks` picks are compared with a single-GPU run of the same loop on the same data."""
    import torch.distributed as dist
    from active_learning_b200.sharding import plan_shards
    dev = eng.device
    factored = kind == "badge"
    g = torch.Generator(device=dev).manual_seed(1000)         # candidates and labeled rows: identical on every rank
    X = torch.relu(torch.randn(N_ROWS, EMB_DIM, device=dev, generator=g))
    gy = torch.Generator(device=dev).manual_seed(1)
    Y = torch.relu(torch.randn(N_LABELED, EMB_DIM, device=dev, generator=gy))
    if factored:
        lx = torch.randn(N_ROWS, N_CLASSES, device=dev, generator=g) * 3
        ly = torch.randn(N_LABELED, N_CLASSES, device=dev, generator=gy) * 3
    rng = np.random.default_rng(0)
    us = rng.random(BUDGET)
    cand_pos = np.arange(N_LABELED, N_LABELED + N_ROWS, dtype=np.int32)
    vpos = torch.as_tensor(cand_pos, device=dev)
    full_n = N_ROWS + N_LABELED
    shard_off = shard_pos = None
    s0, s1 = 0, N_ROWS
    if world > 1:
        shard_off, shard_pos = plan_shards(cand_pos, full_n, world, leaf_aligned=factored)
        s0, s1 = int(shard_off[rank]), int(shard_off[rank + 1])
    n_loc = s1 - s0
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    out = {}
    cpad = (N_CLASSES + 3) & ~3
    XA_all = torch.empty((N_ROWS, cpad), device=dev) if factored else None
    xan_all = torch.empty(N_ROWS, device=dev) if factored else None

    def one(timed, budget=BUDGET, sharded=True):
        so, sp, a0, a1 = (shard_off, shard_pos, s0, s1) if sharded else (None, None, 0, N_ROWS)
        if world > 1:
            dist.barrier()
        if timed:
            ev[0].record()
        xn, yn = eng.row_norm2(X), eng.row_norm2(Y)
        XA = YA = xan = yan = None
        if factored:                                            # K2 over this rank's rows, then one all-gather
            XA, xan = XA_all, xan_all
            if sharded and world > 1:
                sizes = [int(shard_off[q + 1] - shard_off[q]) for q in range(world)]
                a_loc, an_loc = eng.badge_factors(lx[a0:a1], 128, row0=N_LABELED + a0, n_total=full_n)
                if len(set(sizes)) == 1:
                    dist.all_gather_into_tensor(XA_all, a_loc)
                    dist.all_gather_into_tensor(xan_all, an_loc)
                else:
                    dist.all_gather([XA_all[int(shard_off[q]):int(shard_off[q + 1])] for q in range(world)], a_loc)
                    dist.all_gather([xan_all[int(shard_off[q]):int(shard_off[q + 1])] for q in range(world)], an_loc)
            else:
                a_loc, an_loc = eng.badge_factors(lx, 128, row0=N_LABELED, n_total=full_n)
                XA_all.copy_(a_loc)
                xan_all.copy_(an_loc)
            YA, yan = eng.badge_factors(ly, 128, row0=0, n_total=full_n)
        if timed:
            ev[1].record()
        mind = torch.full((N_ROWS,), float("inf"), device=dev)
        sl = slice(a0, a1)
        eng.min_dist(X[sl], xn[sl], Y, yn, XA[sl] if factored else None, xan[sl] if factored else None, YA, yan,
                     out=mind[sl])                              # K3 over this rank's candidates
        if timed:
            ev[2].record()
        picks, stream_ms = eng.greedy_select(X, xn, mind, [0, N_ROWS], [budget], a=XA, an=xan,
                                             uniforms=us[:budget] if factored else None, vpos=vpos if factored else None,
                                             full_n=[full_n] if factored else None, time_steps=True,
                                             shard_off=so, shard_pos=sp)
        if timed:
            ev[3].record()
            torch.cuda.synchronize()
            out["prep_ms"] = ev[0].elapsed_time(ev[1])
            out["k3_ms"] = ev[1].elapsed_time(ev[2])
            out["loop_ms"] = ev[2].elapsed_time(ev[3])
            out["stream_ms"] = stream_ms
            out["select_ms"] = eng.last_greedy_timing["select_ms"]
            out["variant"] = eng.last_greedy_timing["variant"]
            out["unique"] = len(set(picks.tolist())) == budget
        return picks

    picks = None
    for _ in range(warmup):
        picks = one(False)
    tot, acc = 0.0, {}
    for _ in range(steps):
        picks = one(True)
        for k in ("prep_ms", "k3_ms", "loop_ms", "stream_ms", "select_ms"):
            acc[k] = acc.get(k, 0.0) + out[k]
        tot += out["prep_ms"] + out["k3_ms"] + out["loop_ms"]
    for k in acc:
        acc[k] /= steps
    ms = tot / steps
    match = None
    if world > 1 and check_picks > 0:                           # every rank: the same loop, unsharded, on its own GPU
        ref = one(False, budget=check_picks, sharded=False)
        same = torch.tensor([int(np.array_equal(ref, picks[:check_picks]))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        match = bool(same.item())
    if world > 1:       # device time of the slowest rank
        t = torch.tensor([ms, acc["prep_ms"], acc["k3_ms"], acc["loop_ms"], acc["stream_ms"], acc["select_ms"]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, acc["prep_ms"], acc["k3_ms"], acc["loop_ms"], acc["stream_ms"], acc["select_ms"] = [float(v) for v in t]
    row_bytes = 4 * EMB_DIM + 12 + (4 * N_CLASSES if factored else 0)
    step_ms = acc["loop_ms"] / max(BUDGET - 1, 1)               # whole loop (setup, every barrier / exchange) per step
    achieved = n_loc * row_bytes / (step_ms * 1e-3) / 1e9
    achieved_stream = n_loc * row_bytes / (max(acc["stream_ms"], 1e-9) * 1e-3) / 1e9
    flops = 2.0 * n_loc * N_LABELED * (EMB_DIM + (N_CLASSES if factored else 0))
    name = ("greedy_persist_kernel<factored,sample> (K5: TMA bulk-copy ring + LL-word agreement on the centre, one launch)"
            if factored else "greedy_persist_kernel<dense,argmax> (K4, one persistent launch)")
    return {
        "workload": (f"BADGESampler tail (configs[3] shape, global k-means++ on rank-1 factors, {world} GPU)" if factored
                     else f"CoresetSampler tail (configs[2] shape, global greedy k-center, {world} GPU)"),
        "scaling": "strong" if world > 1 else None, "rows_per_gpu": n_loc,
        "exchange": ("8-byte {tag,value} words over peer-memory windows (CUDA IPC / NVLink), inside the persistent kernel; "
                     "rows replicated, a centre is a row id") if world > 1 else None,
        "candidates": N_ROWS, "labeled": N_LABELED, "budget": BUDGET, "dim": EMB_DIM,
        "classes": N_CLASSES if factored else None,
        "value": N_ROWS / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "picks_unique": out["unique"],
        "picks_match_single_gpu": match, "picks_checked": check_picks if match is not None else None,
        "breakdown_ms": acc, "us_per_selection_step": step_ms * 1e3, "loop_variant": out.get("variant"),
        "roofline": {"kernel": name, "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "bytes_per_row_per_step": row_bytes,
                     "timing": "loop time / (B - 1): CUDA events around the whole selection loop (one launch), so every "
                               "barrier and exchange is inside",
                     "streaming_phase": {"achieved": achieved_stream, "frac": achieved_stream / peak,
                                         "us": acc["stream_ms"] * 1e3, "select_us": acc["select_ms"] * 1e3,
                                         "timing": "%globaltimer stamps of CTA 0 inside the kernel"},
                     "traffic": ncu_traffic("persist_factored_sample" if factored else "persist_dense_argmax")},
        "k3": {"kernel": "min_dist_tc_kernel (tcgen05 3xTF32 contraction, TMEM accumulators, fused min epilogue; "
                         "time includes the hi/lo operand split)",
               "bound": "tensor", "effective_fp32_tflops": flops / (acc["k3_ms"] * 1e-3) / 1e12,
               "achieved": 3 * flops / (acc["k3_ms"] * 1e-3) / 1e12, "unit": "TFLOP/s",
               "peak": tf32_peak(), "frac": 3 * flops / (acc["k3_ms"] * 1e-3) / 1e12 / tf32_peak(),
               "peak_source": _TF32.get("src"), "note": "3 tf32 MMAs per fp32 product; ncu sm__pipe_tensor_cycles_active of the same "
                                                         "kernel is in profiles/README.md"},
    }


PART_P, PART_LAB, PART_UNL, PART_BUDGET = 10, 5000, 8000, 1000     # gen_jobs.py:11-13,19: --partitions 10, 50k + 80k rows


def run_partitioned_workload(eng, kind, peak, steps, warmup, world=1, rank=0):
    """The reference's own ImageNet configuration (gen_jobs.py:11-19, partitioned_coreset_sampler.py:52-84): 130 000
    rows = 50 000 labeled + 80 000 unlabeled dealt into P = 10 partitions of 13 000 rows, 1 000 picks per partition.
    PartitionedCoreset: 2048-d embeddings, arg-max.  PartitionedBADGE: pooled 512-d gradient embeddings (K2p), D^2 draw.
    Partitions are independent: partition i runs on rank i % G (no collective inside the loop; the picks are gathered
    once), each rank runs its partitions as ONE batched persistent launch.  Like-for-like with `cpu_baseline`."""
    import torch.distributed as dist
    dev = eng.device
    badge = kind == "partitioned_badge"
    dim = 512 if badge else EMB_DIM
    mine = [i for i in range(PART_P) if i % world == rank]
    rows = PART_LAB + PART_UNL

    def data_for(i):
        g = torch.Generator(device=dev).manual_seed(7000 + i)
        f = torch.relu(torch.randn(rows, EMB_DIM, device=dev, generator=g))
        return (f, torch.randn(rows, N_CLASSES, device=dev, generator=g) * 3 if badge else None, i)

    local = [data_for(i) for i in mine]
    rng = np.random.default_rng(11)
    us_all = [rng.random(PART_BUDGET) for _ in range(PART_P)]
    nloc = len(mine)
    part_off = np.arange(nloc + 1, dtype=np.int32) * PART_UNL
    vpos = torch.as_tensor(np.tile(np.arange(PART_LAB, rows, dtype=np.int32), max(nloc, 1)), device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    out = {}

    def one(timed, budget=PART_BUDGET, which=None):
        sel = local if which is None else which
        if world > 1 and which is None:
            dist.barrier()
        if timed:
            ev[0].record()
        F = [eng.badge_pooled_embedding(lg, f, 128) for f, lg, _ in sel] if badge else [f for f, _, _ in sel]   # K2p
        if timed:
            ev[1].record()
        picks = np.zeros(0, dtype=np.int32)
        stream_ms = 0.0
        if sel:
            X = torch.cat([f[PART_LAB:] for f in F], dim=0)
            xn = eng.row_norm2(X)
            mind = torch.empty(X.shape[0], device=dev)
            for j, f in enumerate(F):                            # K3 per partition
                Y = f[:PART_LAB]
                eng.min_dist(X[j * PART_UNL:(j + 1) * PART_UNL], xn[j * PART_UNL:(j + 1) * PART_UNL], Y, eng.row_norm2(Y),
                             out=mind[j * PART_UNL:(j + 1) * PART_UNL])
            if timed:
                ev[2].record()
            po = np.arange(len(sel) + 1, dtype=np.int32) * PART_UNL
            picks, stream_ms = eng.greedy_select(
                X, xn, mind, po, [budget] * len(sel),
                uniforms=np.concatenate([us_all[pid][:budget] for _, _, pid in sel]) if badge else None,
                vpos=vpos[:len(sel) * PART_UNL] if badge else None, full_n=[rows] * len(sel) if badge else None, time_steps=True)
        elif timed:
            ev[2].record()
        if timed:
            ev[3].record()
            torch.cuda.synchronize()
            out["prep_ms"], out["k3_ms"], out["loop_ms"] = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])
            out["variant"] = eng.last_greedy_timing["variant"] if sel else None
        return picks

    picks = None
    for _ in range(warmup):
        picks = one(False)
    acc = {}
    for _ in range(steps):
        picks = one(True)
        for k in ("prep_ms", "k3_ms", "loop_ms"):
            acc[k] = acc.get(k, 0.0) + out[k] / steps
    ms = acc["prep_ms"] + acc["k3_ms"] + acc["loop_ms"]
    per_part = [picks[j * PART_BUDGET:(j + 1) * PART_BUDGET] - j * PART_UNL for j in range(nloc)]
    unique = all(len(set(p.tolist())) == PART_BUDGET for p in per_part)
    match = None
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, {mine[j]: per_part[j].tolist() for j in range(nloc)})
        allp = {k: v for d in gathered for k, v in d.items()}
        # a partition's picks do not depend on the rank that runs it: every rank recomputes the first 150 picks of a
        # partition that ANOTHER rank ran and compares
        other = [i for i in range(PART_P) if i % world == (rank + 1) % world]
        ok = 1
        if other:
            chk = one(False, budget=150, which=[data_for(other[0])])
            ok = int(np.array_equal(chk, np.asarray(allp[other[0]][:150])))
        same = torch.tensor([ok * int(len(allp) == PART_P)], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        match = bool(same.item())
        t = torch.tensor([ms, acc["prep_ms"], acc["k3_ms"], acc["loop_ms"]], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, acc["prep_ms"], acc["k3_ms"], acc["loop_ms"] = [float(v) for v in t]
    nmax = max(len([i for i in range(PART_P) if i % world == r]) for r in range(world))
    row_bytes = 4 * dim + 12
    step_ms = acc["loop_ms"] / max(PART_BUDGET - 1, 1)
    achieved = nmax * PART_UNL * row_bytes / (step_ms * 1e-3) / 1e9
    return {
        "workload": (f"{'PartitionedBADGESampler' if badge else 'PartitionedCoresetSampler'} tail, the reference's ImageNet job "
                     f"(gen_jobs.py: {PART_P} partitions x ({PART_LAB} labeled + {PART_UNL} unlabeled), {PART_BUDGET} picks each), {world} GPU"),
        "scaling": "strong" if world > 1 else None, "partitions": PART_P, "partitions_on_busiest_rank": nmax,
        "exchange": "none inside the loop: partition i runs on rank i % G, one gather of the picks" if world > 1 else None,
        "dim": dim, "candidates": PART_P * PART_UNL, "labeled": PART_P * PART_LAB, "budget": PART_P * PART_BUDGET,
        "value": PART_P * PART_UNL / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "picks_unique": unique,
        "picks_match_single_gpu": match, "breakdown_ms": acc, "us_per_selection_step": step_ms * 1e3, "loop_variant": out.get("variant"),
        "roofline": {"kernel": "greedy_persist_kernel, partitions as CTA groups of one launch", "bound": "hbm (L2 when a rank's rows fit the 126 MB L2)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "bytes_per_row_per_step": row_bytes,
                     "rows_streamed_per_step_on_busiest_rank": nmax * PART_UNL,
                     "note": "a fraction above 1 means the busiest rank's rows (8 000 x 8 KB per partition) are served from L2"},
    }


def run_mase_workload(eng, peak, steps, warmup, rank=0):
    """MASE / BASE tails (SURVEY.md section 8f rank 2) at the configs[1] shape: 80 000 x 1000 logits, a
    1000 x 2048 linear head, B = 10 000.  Per GPU (rows are independent; at N > 1 every rank times its own shard)."""
    dev = eng.device
    g = torch.Generator(device=dev).manual_seed(2000 + rank)
    logits = torch.randn(N_ROWS, N_CLASSES, device=dev, generator=g) * 3
    weight = torch.randn(N_CLASSES, EMB_DIM, device=dev, generator=g) * 0.05
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    acc = {}
    uniq = True
    for it in range(warmup + steps):
        ev[0].record()
        ginv = eng.class_gap_inv(weight)
        ev[1].record()
        mm, pred, _ = eng.mase_margins(logits, ginv, want_per_class=False)
        ev[2].record()
        pos = eng.select_smallest(mm, BUDGET)
        ev[3].record()
        mm2, pred2, radius = eng.mase_margins(logits, ginv, want_per_class=True)
        ev[4].record()
        bpos = eng.base_select(mm2, radius, pred2, BUDGET)
        ev[5].record()
        torch.cuda.synchronize()
        if it >= warmup:
            for k, (a, b) in {"gap_table_ms": (0, 1), "k6_min_ms": (1, 2), "mase_select_ms": (2, 3),
                              "k6_per_class_ms": (3, 4), "base_class_loop_ms": (4, 5)}.items():
                acc[k] = acc.get(k, 0.0) + ev[a].elapsed_time(ev[b]) / steps
            uniq = uniq and len(set(bpos.tolist())) == BUDGET and len(set(pos.tolist())) == BUDGET
        del radius
    mase_ms = acc["gap_table_ms"] + acc["k6_min_ms"] + acc["mase_select_ms"]
    base_ms = acc["gap_table_ms"] + acc["k6_per_class_ms"] + acc["base_class_loop_ms"]
    b_min, b_pc = 4 * N_CLASSES + 8, 8 * N_CLASSES + 8
    return {
        "workload": "MASESampler / BASESampler tails (logit-gap / head-geometry margins + stable selection), per GPU",
        "rows": N_ROWS, "classes": N_CLASSES, "head_dim": EMB_DIM, "budget": BUDGET, "picks_unique": uniq,
        "mase": {"value": N_ROWS / (mase_ms * 1e-3), "unit": "samples/s", "ms_per_step": mase_ms},
        "base": {"value": N_ROWS / (base_ms * 1e-3), "unit": "samples/s", "ms_per_step": base_ms,
                 "classes_with_picks": min(N_CLASSES, BUDGET)},
        "breakdown_ms": acc,
        "roofline": {"kernel": "rows_pipe_kernel<8,mase-min> (K6: minimum boundary distance, verified table pruning)", "bound": "hbm", "unit": "GB/s", "peak": peak,
                     "achieved": N_ROWS * b_min / (acc["k6_min_ms"] * 1e-3) / 1e9,
                     "frac": N_ROWS * b_min / (acc["k6_min_ms"] * 1e-3) / 1e9 / peak, "bytes_per_row": b_min,
                     "note": "the 4 MB gap table is read through L2 and not counted"},
        "roofline_per_class": {"kernel": "rows_pipe_kernel<8,mase-full> (K6: all C radii written, BASE)", "bound": "hbm", "unit": "GB/s",
                               "peak": peak, "achieved": N_ROWS * b_pc / (acc["k6_per_class_ms"] * 1e-3) / 1e9,
                               "frac": N_ROWS * b_pc / (acc["k6_per_class_ms"] * 1e-3) / 1e9 / peak, "bytes_per_row": b_pc},
    }


def run_pool_forward_workload(eng, images=2048, batch=128):
    """SURVEY.md section 8d / 8f rank 3: the query END TO END through the public sampler API -- DataLoader over host
    images -> H2D -> ResNet-50 in the reference's layout (torchvision encoder + linear head, resnet_simclr.py:6-41,
    random init, torch defaults) -> logits slab -> K1 + K1b -> indices on the host.  Then the same under
    --freeze_feature: the second query reuses the cached pool embeddings (section 8f rank 1)."""
    import torch.nn as nn
    import torchvision
    from active_learning_b200.query_strategies.get_strategy import get_strategy

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.encoder = torchvision.models.resnet50(weights=None, num_classes=N_CLASSES)
            dim = self.encoder.fc.in_features
            self.encoder.fc = nn.Identity()
            self.linear = nn.Linear(dim, N_CLASSES)

        def forward(self, x, return_features=False, specify_input_layer=None):
            if specify_input_layer:
                return self.linear(x)
            h = self.encoder(x)
            out = self.linear(h)
            return (out, h) if return_features else out

    class Pool(torch.utils.data.Dataset):
        num_classes = N_CLASSES

        def __init__(self, n):
            g = torch.Generator().manual_seed(3)
            self.x = torch.randn(n, 3, 224, 224, generator=g)

        def __len__(self):
            return self.x.shape[0]

        def __getitem__(self, i):
            return self.x[i], 0, i

    class Exp:
        url = "."

        def get_key(self):
            return "bench"

        def __getattr__(self, name):
            return lambda *a, **k: None

    torch.manual_seed(0)
    ds, net = Pool(images), Net()
    budget = images // 8
    out = {"workload": "MarginSampler.query end to end (synthetic 3x224x224 pool -> ResNet-50 fp32 forward -> K1 + K1b)",
           "images": images, "batch_size": batch, "budget": budget,
           "precision": "torch defaults: fp32 weights/activations, cuDNN conv TF32 allowed, matmul fp32",
           "data_path": "pinned double-buffered H2D on a side stream, channels-last network and batches (EngineMixin._device_batches)"}
    # loader arguments: the reference's ImageNet arg pool (arg_pools/ssp_linear_evaluation.py:12-16: 8 workers, prefetch 2) and,
    # for comparison with round 1, a single-process loader
    loaders = {"": {"batch_size": batch, "num_workers": 8, "prefetch_factor": 2},
               "_single_process_loader": {"batch_size": batch, "num_workers": 0}}
    for suffix, largs in loaders.items():
        for tag, freeze in (("uncached", False), ("freeze_feature_cached", True)):
            if suffix and freeze:
                continue
            kw = dict(early_stop_patience=0, n_epoch=1, world_size=1, model="SSLResNet50", freeze_feature=freeze,
                      ckpt_path=tempfile.mkdtemp(prefix="alq_bench_"), exp_name="b")
            s = get_strategy("MarginSampler")(ds, ds, net, {"loader_te_args": dict(largs)}, np.array([], dtype=np.int64), Exp(), None, **kw)
            s.init_network_weights()
            s.set_engine(eng)
            times = []
            sync = torch.cuda.synchronize if torch.cuda.is_available() else (lambda: None)
            for _ in range(3):                       # query 0 warms cuDNN / fills the cache; 1-2 are timed
                sync()
                t0 = time.perf_counter()
                idx, cost = s.query(float(budget))
                sync()
                times.append(time.perf_counter() - t0)
            assert cost == budget and len(set(idx)) == budget
            dt = min(times[1:])
            out[tag + suffix] = {"value": images / dt, "unit": "samples/s", "ms_per_query": dt * 1e3, "first_query_ms": times[0] * 1e3,
                                 "loader": largs}
    net.cpu()
    return out


# ----------------------------------------------------------------------------------------------
# own arm
# ----------------------------------------------------------------------------------------------
def run_own(args):
    import torch.distributed as dist
    from active_learning_b200.engine import Engine
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    group = None
    # stdout carries exactly ONE JSON line: libraries that print banners there (NCCL prints its version on the
    # first communicator) are pointed at stderr for the duration of the run
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        from active_learning_b200.sharding import ShardGroup
        group = ShardGroup()
    eng = Engine(local)
    dev = eng.device
    comm_error = None
    if world > 1:
        try:
            eng.comm_init()          # peer-memory windows: top-B exchange and the global selection loops use them
        except Exception as exc:     # e.g. CUDA IPC unavailable: fall back to the NCCL all-gather for the top-B merge
            comm_error = repr(exc)
    peak, peak_src = measured_peaks()
    MODE_MARGIN = 0

    g = torch.Generator(device=dev).manual_seed(rank)
    logits = torch.randn(N_ROWS, N_CLASSES, device=dev, generator=g) * 3.0   # this rank's shard
    scores = torch.empty(N_ROWS, dtype=torch.float32, device=dev)
    row_lo = rank * N_ROWS

    # A step = the fused K1 + K1b (+ exchange at N > 1) launch -> async D2H of the B winners into a pinned host
    # buffer (on a copy stream behind an event); steps are enqueued back to back and the host waits once after
    # the K-th (the contract's closing synchronize, which also covers the copy stream).  The headline region
    # runs the steps in order on one stream, for every N, so the per-N values are comparable and the CUDA-event
    # pair around the fused kernel times that kernel alone.  At N = 1 a second region reports the throughput with two independent
    # queries in flight (even/odd steps on two streams / engine contexts: the 148-SM scoring kernel of query
    # i+1 overlaps the 8-SM top-B cluster kernel of query i; K1 claims its tiles dynamically so CTAs that start
    # late behind the cluster kernel are not stragglers).
    host_out = [torch.empty(BUDGET, dtype=torch.int32).pin_memory() for _ in range(2)]

    def sync_all():
        if group is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run_region(depth, steps, warm):
        engines = [eng] + [Engine(local) for _ in range(depth - 1)]
        streams = [torch.cuda.Stream(device=dev) for _ in range(depth)]
        score_bufs = [scores] + [torch.empty_like(scores) for _ in range(depth - 1)]
        # the B winners leave on a copy stream behind an event, so the next step's kernel does not queue behind the
        # 40 KB D2H of this one (the region's closing wait covers the copy stream too)
        copy_stream = torch.cuda.Stream(device=dev)
        done = [torch.cuda.Event() for _ in range(4)]

        def to_host(i, k, pos):
            ev = done[i & 3]
            ev.record(streams[k])
            copy_stream.wait_event(ev)
            with torch.cuda.stream(copy_stream):
                host_out[i & 1].copy_(pos, non_blocking=True)
            pos.record_stream(copy_stream)

        def step(i, pair=None):
            k = i % depth
            e, sc = engines[k], score_bufs[k]
            with torch.cuda.stream(streams[k]):
                if pair is not None:
                    pair[0].record()
                if group is None:
                    _, pos = e.uncertainty_tail(logits, MODE_MARGIN, BUDGET, scores_out=sc)   # K1 + K1b: ONE launch
                    if pair is not None:
                        pair[1].record()
                    to_host(i, k, pos)
                elif getattr(e, "comm_ready", False):
                    # K1 + K1b + the cross-GPU exchange: ONE launch per rank (histograms summed and candidates
                    # gathered through the peer-memory windows from inside the kernel)
                    _, gp = e.uncertainty_tail_sharded(logits, MODE_MARGIN, BUDGET, row_lo, N_ROWS, N_ROWS, scores_out=sc)
                    if pair is not None:
                        pair[1].record()
                    to_host(i, k, gp)
                else:
                    _, pos = e.uncertainty_tail(logits, MODE_MARGIN, BUDGET, scores_out=sc)
                    if pair is not None:
                        pair[1].record()
                    gp = group.merge_smallest(sc, pos, row_lo, BUDGET, e, to_host=False)   # all-gather + device merge
                    to_host(i, k, gp)

        for i in range(warm * depth):
            step(i)
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        sync_all()
        l0 = sum(e.launches for e in engines)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sync_all()
        tw0 = time.perf_counter()
        ev0.record()
        for st in streams:
            st.wait_event(ev0)
        for i in range(steps):
            step(i, pairs[i])
        for st in streams + [copy_stream]:
            torch.cuda.current_stream().wait_stream(st)
        ev1.record()
        tenq = time.perf_counter()
        sync_all()
        tw1 = time.perf_counter()
        per_step = [a.elapsed_time(b) for a, b in pairs]
        return {"ms_total": ev0.elapsed_time(ev1), "k1_ms": float(np.mean(per_step)), "k1_ms_per_step": per_step,
                "launches": sum(e.launches for e in engines) - l0, "t": (tw0, tenq, tw1),
                "res": host_out[(steps - 1) & 1].clone()}

    # one nvidia-smi poller (rank 0's GPU): eight of them next to eight busy-waiting ranks oversubscribe the host cores
    clocks = ClockSampler(local if rank == 0 else -1)
    clocks.__enter__()
    clocks.wait_first(8.0 if rank == 0 else 0.0)
    R = run_region(1, args.steps, max(args.warmup, 3))
    # the region ran on `scores`, so it holds the last timed step's margins until the next region overwrites it
    dumped = {"scores": scores.cpu().numpy(), "picks": R["res"].numpy()} if args.dump_outputs else None
    t_w0, t_enq, t_w1 = R["t"]
    res, launches, ms_total, k1_ms = R["res"], R["launches"], R["ms_total"], R["k1_ms"]
    launches0 = eng.launches - launches
    pipelined = None
    if group is None:
        P2 = run_region(2, args.steps, max(args.warmup, 3))
        pipelined = {"queries_in_flight": 2, "ms_per_step": P2["ms_total"] / args.steps,
                     "value": N_ROWS / (P2["ms_total"] / args.steps * 1e-3), "unit": "samples/s",
                     "k1_event_ms_while_overlapped": P2["k1_ms"]}
    streams = [torch.cuda.current_stream()]
    with torch.cuda.stream(streams[0]):            # single query, no pipelining: latency
        lat = []
        for _ in range(5):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, pos = eng.uncertainty_tail(logits, MODE_MARGIN, BUDGET, scores_out=scores)
            host_out[0].copy_(pos, non_blocking=True)
            torch.cuda.synchronize()
            lat.append(time.perf_counter() - t0)
    latency_ms = float(np.median(lat)) * 1e3
    if group is not None:
        t = torch.tensor([ms_total, k1_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total, k1_ms = float(t[0]), float(t[1])
    ms_step = ms_total / args.steps
    value = N_ROWS * world / (ms_step * 1e-3)
    assert len(res) == BUDGET
    try:
        stream_ms, kern_ms = eng.uncertainty_tail_timing()       # in-kernel stamps of the last fused launch
    except Exception:
        stream_ms = kern_ms = None
    headline_match = None
    step_kernel_ms = {"median": float(np.median(R["k1_ms_per_step"])), "max": float(np.max(R["k1_ms_per_step"])),
                      "note": "CUDA events around the fused kernel of every timed step on this rank; a max far above the median is a "
                              "stall of one step (every rank's kernel waits for the slowest rank's launch), not kernel time"}
    if group is not None:
        allsteps = [None] * world
        dist.all_gather_object(allsteps, [round(v, 4) for v in R["k1_ms_per_step"]])
        step_kernel_ms["per_rank_max"] = [float(np.max(v)) for v in allsteps]
        step_kernel_ms["per_rank_argmax_step"] = [int(np.argmax(v)) for v in allsteps]
        step_kernel_ms["rank0_steps"] = allsteps[0]
        # the exchanged global top-B against ONE GPU selecting from the concatenated scores of all ranks
        all_scores = torch.empty(N_ROWS * world, dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(all_scores, scores)
        ref_pos = eng.select_smallest(all_scores, BUDGET).cpu()
        same = torch.tensor([int(torch.equal(ref_pos, res.cpu()))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        headline_match = bool(same.item())
        del all_scores

    # ---- e2e: host buffers through the C-ABI entry point (H2D + K1 + K1b + D2H) ----------------------
    host_logits = torch.empty((N_ROWS, N_CLASSES), dtype=torch.float32).pin_memory()
    host_logits.copy_(logits)
    for _ in range(2):
        eng.uncertainty_query_host(host_logits, MODE_MARGIN, BUDGET)
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        hp = eng.uncertainty_query_host(host_logits, MODE_MARGIN, BUDGET)
        if group is not None:
            group.merge_smallest(scores, torch.from_numpy(hp).to(dev), row_lo, BUDGET, eng)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if group is not None:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    assert np.array_equal(np.sort(hp), np.sort(eng.select_smallest(scores, BUDGET).cpu().numpy()))
    clocks.__exit__(None, None, None)

    line = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world),
        "clocks": clocks.summary((t_w0, t_w1)),
        "e2e": {"value": N_ROWS * world / e2e_s, "unit": "samples/s",
                "h2d_bytes_per_step": N_ROWS * N_CLASSES * 4, "d2h_bytes_per_step": BUDGET * 4,
                "ms_per_step": e2e_s * 1e3, "api": "alq_uncertainty_query_host (pinned host logits)"},
        "gpu_launches": int(launches),
        "picks_match_single_gpu": headline_match,
        "step_kernel_ms": step_kernel_ms,
        "host_enqueue_ms_per_step": (t_enq - t_w0) * 1e3 / args.steps,
        "latency_ms_single_query": latency_ms,
        "pipelined": pipelined,
        "roofline": {"kernel": "rows_pipe_kernel<8,margin> with the fused selection epilogue (K1 + K1b in one launch: TMA bulk-copy "
                               "pipelined softmax-margin score, then two histogram levels and the score-bucket ordering of the winners behind three grid barriers); "
                               "the CUDA events bracket the WHOLE kernel, selection included", "bound": "hbm",
                     "achieved": N_ROWS * (4 * N_CLASSES + 4) / (k1_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                     "frac": N_ROWS * (4 * N_CLASSES + 4) / (k1_ms * 1e-3) / 1e9 / peak,
                     "traffic": ncu_traffic("fused_tail_margin"), "kernel_ms": k1_ms, "peak_source": peak_src,
                     "streaming_phase": (None if not stream_ms else {
                         "us": stream_ms * 1e3, "achieved": N_ROWS * (4 * N_CLASSES + 4) / (stream_ms * 1e-3) / 1e9,
                         "frac": N_ROWS * (4 * N_CLASSES + 4) / (stream_ms * 1e-3) / 1e9 / peak, "kernel_us_in_kernel_clock": kern_ms * 1e3,
                         "timing": "%globaltimer stamps of CTA 0 inside the fused kernel: start -> every CTA has finished its rows (first "
                                   "grid barrier); the rest of the kernel is the selection epilogue (and, at N > 1, the exchange)"}),
                     "bytes_per_row": 4 * N_CLASSES + 4},
    }
    if rank == 0:
        cpu_logits = host_logits.clone()
        threads, cpu_budget = tune_cpu_threads(cpu_logits)
        t0 = time.perf_counter()
        reps = 0
        while reps < 3 and time.perf_counter() - t0 < 20:
            cp = cpu_margin_tail(cpu_logits, BUDGET)
            reps += 1
        dt = (time.perf_counter() - t0) / reps
        line["cpu_baseline"] = {
            "value": N_ROWS / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"full {N_ROWS} x {N_CLASSES} shard x{reps}, oracle port of margin_sampler.py:33-42 "
                      f"(torch-CPU softmax/topk in batches of 128 + sort), {threads} threads = best of a probe "
                      f"over {cpu_budget} usable CPUs; {cpu_model()}",
            "selection_overlap_with_gpu": (float(len(np.intersect1d(cp, res.numpy())) / BUDGET) if world == 1 else None)}
    if not args.no_extras:
        extras = {}
        for kind in ("coreset", "badge"):
            if comm_error:
                extras[kind] = {"error": comm_error}
                continue
            try:
                extras[kind] = run_greedy_workload(eng, kind, peak, steps=args.extra_steps, warmup=1, world=world, rank=rank)
            except Exception as exc:  # report, never hide
                extras[kind] = {"error": repr(exc)}
            torch.cuda.empty_cache()
        for kind in ("partitioned_coreset", "partitioned_badge"):
            try:
                extras[kind] = run_partitioned_workload(eng, kind, peak, steps=args.extra_steps, warmup=1, world=world, rank=rank)
            except Exception as exc:  # report, never hide
                extras[kind] = {"error": repr(exc)}
            torch.cuda.empty_cache()
        try:
            extras["mase_base"] = run_mase_workload(eng, peak, steps=args.extra_steps, warmup=1, rank=rank)
        except Exception as exc:  # report, never hide
            extras["mase_base"] = {"error": repr(exc)}
        torch.cuda.empty_cache()
        if world == 1:
            try:
                cpu = cpu_greedy_baseline()
                for kind, key in (("partitioned_coreset", "coreset"), ("partitioned_badge", "badge")):     # like for like
                    if "error" not in extras.get(kind, {"error": 1}):
                        extras[kind]["cpu_baseline"] = dict({k: v for k, v in cpu.items() if k not in ("coreset", "badge")}, **cpu[key])
                for kind in ("coreset", "badge"):
                    if "error" not in extras.get(kind, {"error": 1}):
                        extras[kind]["cpu_baseline"] = {"value": None, "note": "the reference cannot run the non-partitioned 130 000-row query "
                                                        "(67.6 GB distance matrix); its like-for-like configuration is workloads.partitioned_*"}
            except Exception as exc:  # report, never hide
                extras["cpu_greedy_baseline_error"] = repr(exc)
            try:
                extras["pool_forward_e2e"] = run_pool_forward_workload(eng)
            except Exception as exc:  # report, never hide
                extras["pool_forward_e2e"] = {"error": repr(exc)}
            torch.cuda.empty_cache()
        line["workloads"] = extras
        line["gpu_launches_total"] = int(eng.launches - launches0)
    if dumped is not None and rank == 0:
        dump_outputs(args.dump_outputs, **dumped)
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if group is not None:
        os.dup2(2, 1)
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the CoreSet/BADGE workloads (N=1)")
    ap.add_argument("--extra-steps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
