#!/usr/bin/env python3
"""bench.py — index-build throughput (+ QPS@recall) of arroy's distance / split / re-rank hot path on B200.

One "step" = one complete forest build (Writer::build of the reference, src/writer.rs:487-629)
over one synthetic item matrix. Contract: `python bench.py --gpus N --steps K --warmup W`
prints ONE JSON line (rank 0). `--impl reference` times the reference's CPU path instead (the
Rust crate cannot be compiled in this image, so it is the C++ restatement in oracle/, kind
"port": same AVX+FMA kernels, one task per tree on all host cores — see BASELINE.md §3).

Workloads (BASELINE.json configs; SURVEY.md §8d synthetic data: element (i,j) = gen::<f32>()
number i*d+j of StdRng::from_seed([42;32]) minus 0.5; build rng = fresh StdRng([42;32])):
  c2 (default)  1 000 000 x 768  Cosine      n_trees = 50    <- BASELINE.json configs[1]; `value`, `e2e` and the
                                                               reference arm are quoted on it (the CPU arm cannot
                                                               finish 10M rows inside the driver's steps)
  c3            10 000 000 x 768 DotProduct  n_trees = 100
  c4            10 000 000 x 1536 Cosine     n_trees = 100   (meant for 8 GPUs)
  c1            10 000 x 64      Euclidean   n_trees = 10    (raw [0,1) data)
  small         100 000 x 768    Cosine      n_trees = 16    (quick check)
  c5            4096 queries x 100 000 shared candidates, d = 768, Cosine, top-100 (own metric: queries/s)

The default (c2) line also carries, as sub-records measured in the same process:
  headline_10m  BASELINE.json's metric configuration itself: 10M x 768 Cosine, n_trees = 100 — value, roofline,
                e2e (host leaf values -> stage_items -> build_trees -> arena sink) and clocks, 2 timed steps
  query         QPS@recall100 on the c2 index: batched and one-at-a-time (p50 latency) through Reader, recall vs exact
                brute force, the oracle's nns_by_item timed on the same queries (ids compared) as `cpu_baseline`;
                `query_gmm`: the same on a Gaussian-mixture dataset drawn from the same ChaCha stream (i.i.d. uniform
                768-d data has no neighbourhood structure: recall@100 there says nothing about the index)
  c5            BASELINE configs[4] (batched 4096 x 100k re-rank) with its tensor roofline
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = bytes([42] * 32)
WORKLOADS = {
    "c2": dict(n=1_000_000, d=768, metric="cosine", n_trees=50, centre=0.5, name="C2 1Mx768 Cosine n_trees=50"),
    "c3": dict(n=10_000_000, d=768, metric="dot-product", n_trees=100, centre=0.5, name="C3 10Mx768 DotProduct n_trees=100"),
    "c4": dict(n=10_000_000, d=1536, metric="cosine", n_trees=100, centre=0.5, name="C4 10Mx1536 Cosine n_trees=100"),
    "c1": dict(n=10_000, d=64, metric="euclidean", n_trees=10, centre=0.0, name="C1 10kx64 Euclidean n_trees=10"),
    "small": dict(n=100_000, d=768, metric="cosine", n_trees=16, centre=0.5, name="small 100kx768 Cosine n_trees=16"),
    "c5": dict(n=100_000, d=768, metric="cosine", n_trees=0, centre=0.5, nq=4096, k=100, name="C5 4096 queries x 100k candidates re-rank, d=768 Cosine top-100"),
    "h10m": dict(n=10_000_000, d=768, metric="cosine", n_trees=100, centre=0.5, name="headline 10Mx768 Cosine n_trees=100"),
}
GMM_CLUSTERS, GMM_SCALE, GMM_ROW0 = 256, 0.25, 1 << 40   # mixture centres = rows GMM_ROW0.. of the same ChaCha stream


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return None


def peaks():
    d = load_peaks()
    if d:
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def tensor_peak(burst=False):
    """TF32 dense peak: half the measured dense bf16 rate (tcgen05 kind::tf32 runs at half the kind::f16 rate)."""
    d = load_peaks()
    if d and "bf16_tflops_sustained" in d:
        if burst and "bf16_tflops" in d:
            return d["bf16_tflops"] / 2.0, "measured bf16 burst %.1f TFLOP/s / 2 (TF32 rate, kernel timed alone; MEASURED_PEAKS.json)" % d["bf16_tflops"]
        return d["bf16_tflops_sustained"] / 2.0, "measured bf16 sustained %.1f TFLOP/s / 2 (TF32 rate; MEASURED_PEAKS.json)" % d["bf16_tflops_sustained"]
    return 1100.0, "fallback: nominal dense TF32 (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def derive_seeds(ab, n_trees):
    """seed chain of Writer::build (src/writer.rs:575, :795) with the product's own StdRng."""
    import numpy as np
    user = ab.StdRng.from_seed(SEED)
    s1 = bytes(np.array([user.next_u32() & 0xff for _ in range(32)], dtype=np.uint8))
    r1 = ab.StdRng.from_seed(s1)
    return [bytes(np.array([r1.next_u32() & 0xff for _ in range(32)], dtype=np.uint8)) for _ in range(n_trees)]


def base_config(wl):
    """The keys both arms print (the driver compares them)."""
    return {"workload": wl["name"], "n": wl["n"], "d": wl["d"], "distance": wl["metric"], "n_trees": wl["n_trees"]}


def run_reference(args, wl):
    """The reference's CPU path (oracle port) on all host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    import oracle
    oracle.build_lib()
    cores = os.cpu_count() or 1
    n, d, T = wl["n"], wl["d"], wl["n_trees"]
    # bounded sample: the same item matrix, as many trees as keep one step within ~tens of seconds
    t_sample = T if args.ref_trees is None else args.ref_trees
    if args.ref_trees is None and n * d >= 5e8:
        t_sample = min(T, max(8, cores // 2))
    data = oracle.synth_rows(SEED, d, 0, n, wl["centre"], threads=min(cores, 64))
    ids = np.arange(n, dtype=np.uint32)
    times = []
    scanned = 0
    for step in range(args.warmup + args.steps):
        db = oracle.Db(wl["metric"], d)
        db.set_items(ids, data)
        rng = oracle.StdRng(SEED)
        t0 = time.perf_counter()
        ref_threads = 1 if args.workload == "c1" else min(cores, t_sample)   # configs[0]: single-thread CPU reference
        db.build(rng, n_trees=t_sample, threads=ref_threads)
        dt = time.perf_counter() - t0
        scanned = db.scanned_rows
        if step >= args.warmup:
            times.append(dt)
        del db
    sec = sum(times) / len(times)
    # vectors/s of the FULL forest, extrapolated linearly in the number of trees (trees are independent)
    value = n / (sec * T / t_sample)
    line = {
        "impl": "reference", "metric": "index-build vectors/sec", "value": value, "unit": "vectors/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": base_config(wl),
        "cpu_baseline": {"value": value, "unit": "vectors/s", "cores": ref_threads, "nproc": cores, "kind": "port",
                         "sample": "%d of %d trees over the full %dx%d matrix, %d thread(s) of %d host cores (one tree per thread), extrapolated x%.2f" % (t_sample, T, n, d, ref_threads, cores, T / t_sample),
                         "scan_GBps": scanned * d * 4 / sec / 1e9},
        "e2e": {"value": value, "unit": "vectors/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def c5_cpu(wl, data_host, qh, n_queries, threads):
    """The reference's re-rank loop (oracle port) for a few queries, one query per thread."""
    import numpy as np
    import oracle
    from concurrent.futures import ThreadPoolExecutor
    n, k = wl["n"], wl["k"]
    rows = np.arange(n, dtype=np.uint32)
    m = oracle.METRICS[wl["metric"]]

    def one(i):
        return oracle.rerank(m, data_host[n + i], (float(qh[n + i]), 0.0), data_host, qh, None, rows, k)
    one(0)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        res = list(ex.map(one, range(n_queries)))
    return n_queries / (time.perf_counter() - t0), res


def c5_measure(ctx, torch, dev, wl, steps, warmup, cpu_sample=True, dump_dir=None):
    """BASELINE configs[4] on one context: returns the record (value, breakdown, tensor roofline, e2e, cpu sample).
    With dump_dir, the results of the last timed call are written there."""
    import numpy as np
    n, d, nq, k, metric = wl["n"], wl["d"], wl["nq"], wl["k"], wl["metric"]
    cores = os.cpu_count() or 1
    items = torch.empty((n + nq, d), dtype=torch.float32, device=dev)
    ctx.synth_device(SEED, d, 0, n + nq, wl["centre"], items.data_ptr())
    ctx.stage_items_device(metric, np.arange(n + nq, dtype=np.uint32), d, items.data_ptr())
    h0, _ = ctx.item_headers()
    q_host = items[n:].cpu().numpy()          # queries = the rows that continue the stream after the candidates (SURVEY.md §8d)
    qh = np.ascontiguousarray(h0[n:])
    rows = np.arange(n, dtype=np.uint32)
    out = None
    for _ in range(max(warmup, 1)):
        out = ctx.rerank_shared(q_host, qh, rows, k)
    c0 = ctx.counters()
    torch.cuda.synchronize()
    ctx.timer_start()
    t0 = time.perf_counter()
    gemm_ms = []
    for _ in range(steps):
        out = ctx.rerank_shared(q_host, qh, rows, k)
        gemm_ms.append(ctx.rerank_breakdown())
    dev_ms = ctx.timer_stop()
    wall = time.perf_counter() - t0
    c1 = ctx.counters()
    if dump_dir:
        write_outputs(dump_dir, rerank_outputs(out))
    bd = {kk: sum(b[kk] for b in gemm_ms) / len(gemm_ms) for kk in gemm_ms[0]}
    stats = ctx.rerank_stats()
    peak, peak_src = tensor_peak(burst=True)
    flop = 2.0 * nq * n * d
    ms_per_step = dev_ms / steps
    rec = {
        "metric": "batched re-rank queries/sec", "value": nq / (ms_per_step * 1e-3), "unit": "queries/s", "ms_per_step": ms_per_step, "steps": steps,
        "dtype": "f32 (tf32 tensor-core pre-filter, exact f32 re-score)",
        "config": {"workload": wl["name"], "n_candidates": n, "n_queries": nq, "d": d, "distance": metric, "k": k},
        "gpu_launches": int(c1["launches"] - c0["launches"]),
        "rerank": {"breakdown_ms": bd, "survivors_per_query": stats["survivors"] / max(stats["queries"], 1), "fallback_chunks": stats["fallback_chunks"],
                   "exact_pairs_per_s": nq * n / (ms_per_step * 1e-3)},
        "roofline": {"bound": "tensor", "kernel": "tcgemm_tf32_kernel (tcgen05.mma kind::tf32 + TMA + TMEM, fused distance-estimate epilogue)",
                     "achieved": flop / (bd["score_gemm_ms"] * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": flop / (bd["score_gemm_ms"] * 1e-3) / 1e12 / peak,
                     "peak_source": peak_src, "traffic": None,
                     "timing": "CUDA events on the library stream around the kernel inside the timed arroy_b200_rerank_shared calls"},
        "e2e": {"value": nq / (wall / steps), "unit": "queries/s", "h2d_bytes_per_step": int((c1["h2d_bytes"] - c0["h2d_bytes"]) / steps),
                "d2h_bytes_per_step": int((c1["d2h_bytes"] - c0["d2h_bytes"]) / steps), "note": "wall clock around arroy_b200_rerank_shared with pageable host buffers"},
    }
    if cpu_sample:
        import oracle
        oracle.build_lib()
        data_host = items.cpu().numpy()
        sample = min(nq, max(cores, 32))
        v, res = c5_cpu(wl, data_host, h0, sample, cores)
        same = all(out[0][i, :out[2][i]].tolist() == res[i][0].tolist() and out[1][i, :out[2][i]].tobytes() == res[i][1].tobytes() for i in range(sample))
        rec["cpu_baseline"] = {"value": v, "unit": "queries/s", "cores": cores, "nproc": cores, "kind": "port", "sample": "%d of %d queries, one query per thread" % (sample, nq),
                               "results_identical_on_sample": bool(same)}
    del items
    return rec


def run_c5(args, wl):
    """`--workload c5`: BASELINE.json configs[4] as its own bench line (replicas for N > 1)."""
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    n, d, nq, k, metric = wl["n"], wl["d"], wl["nq"], wl["k"], wl["metric"]
    cores = os.cpu_count() or 1
    if args.impl == "reference":
        if rank != 0:
            return
        import oracle
        oracle.build_lib()
        data = oracle.synth_rows(SEED, d, 0, n + nq, wl["centre"], threads=min(cores, 64))
        hdr = np.sqrt((data.astype(np.float64) ** 2).sum(1)).astype(np.float32)   # only the timing matters here
        sample = min(nq, max(2 * cores, 64))
        qps = []
        for step in range(args.warmup + args.steps):
            v, _ = c5_cpu(wl, data, hdr, sample, cores)
            if step >= args.warmup:
                qps.append(v)
        value = sum(qps) / len(qps)
        print(json.dumps({"impl": "reference", "metric": "batched re-rank queries/sec", "value": value, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": sample / value * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": {"workload": wl["name"], "n_candidates": n, "n_queries": nq, "d": d, "distance": metric, "k": k},
                          "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "nproc": cores, "kind": "port", "sample": "%d of %d queries per step, one query per thread" % (sample, nq)},
                          "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
        return
    import torch
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    import arroy_b200 as ab
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctx = ab.Context(local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    rec = c5_measure(ctx, torch, dev, wl, args.steps, args.warmup, cpu_sample=(rank == 0 and not args.no_cpu_baseline),
                     dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    t_ms = torch.tensor([rec["ms_per_step"]], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(t_ms.item())
    line = {"metric": rec["metric"], "value": world * nq / (ms_per_step * 1e-3), "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": rec["dtype"], "data": "synthetic",
            "config": rec["config"], "notes": {"parallelism": "replicas only (re-rank is single-GPU)", "l2": "score matrix (1.6 GB) and candidates (307 MB) larger than L2; no flush needed",
                                               "timing": "CUDA events on the library stream around the C-ABI call (host query / result buffers, copies included), max over ranks"},
            "gpu_launches": rec["gpu_launches"], "rerank": rec["rerank"], "roofline": rec["roofline"], "e2e": rec["e2e"], "clocks": clocks}
    line["e2e"]["value"] *= world
    if "cpu_baseline" in rec:
        line["cpu_baseline"] = rec["cpu_baseline"]
    if rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# build workloads
# ---------------------------------------------------------------------------------------------------------------------

class Rig:
    """Process-wide state of the `ours` arm: device, context, torch.distributed."""

    def __init__(self):
        import torch
        import __graft_entry__ as ge
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if self.rank == 0:
            ge.build()
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            dist.barrier()
            self.dist = dist
        import arroy_b200 as ab
        self.ab = ab
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.ctx = ab.Context(self.local_rank)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())


def synth_items(rig, wl, dataset="uniform", only_rank0=True):
    """The synthetic matrix on the device. `gmm`: row i = centre[(i * 2654435761) mod C] + GMM_SCALE * (u_i - 0.5), u and the
    centres from the same counter-based ChaCha12 stream (f32 mul, then f32 add: reproducible on the host)."""
    torch, ctx = rig.torch, rig.ctx
    n, d = wl["n"], wl["d"]
    items = torch.empty((n, d), dtype=torch.float32, device=rig.dev)
    if only_rank0 and rig.rank != 0:
        return items
    ctx.synth_device(SEED, d, 0, n, wl["centre"], items.data_ptr())
    if dataset == "gmm":
        centres = torch.empty((GMM_CLUSTERS, d), dtype=torch.float32, device=rig.dev)
        ctx.synth_device(SEED, d, GMM_ROW0, GMM_CLUSTERS, 0.5, centres.data_ptr())
        items.mul_(GMM_SCALE)
        step = 1 << 18
        for a in range(0, n, step):
            b = min(n, a + step)
            idx = (torch.arange(a, b, device=rig.dev, dtype=torch.int64) * 2654435761) % GMM_CLUSTERS
            items[a:b] += centres[idx]
    torch.cuda.synchronize()
    return items


def scan_bytes(scanned_rows, sh, d):
    """Bytes the side() scans of a build have to read BY THEIR OWN ALGORITHM (DESIGN.md, "side() through a bf16 shadow"): 2 bytes per
    element for rows that go through the bf16 pre-filter, plus the f32 row of those its error bound could not decide; 4 bytes per
    element for rows on the plain f32 path; the fused root pass reads each item row once for all trees of the wave."""
    via, resc = sh["rows_via_bf16_shadow"], sh["rows_rescored_f32"]
    f32_rows = scanned_rows - via - sh["rows_in_fused_root_pass"]
    return via * 2 * d + (resc + f32_rows + sh["fused_root_rows_read"]) * 4 * d


def timed_builds(rig, wl, items, seeds, steps, warmup):
    """`steps` timed forest builds with the items resident in HBM (device time, max over ranks)."""
    from arroy_b200 import parallel
    ctx, dist = rig.ctx, rig.dist
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    import numpy as np
    ids = np.arange(n, dtype=np.uint32)
    my_trees = list(range(rig.rank, T, rig.world))  # trees are independent units: tree t -> rank t mod world

    def one_step():
        # multi-GPU: ONE NCCL broadcast of the item buffer over NVLink, then no further data exchange
        if dist is not None:
            parallel.broadcast_items(dist, items, src=0)
            rig.torch.cuda.synchronize()
        ctx.stage_items_device(metric, ids, d, items.data_ptr())
        if metric == "dot-product":
            ctx.dot_preprocess()
        counts = ctx.build_trees_begin([seeds[t] for t in my_trees])
        # tiny all-gather of node counts so every rank can number its nodes like a single-GPU build
        parallel.gather_counts(dist, counts, T, rig.rank, rig.world, device=rig.dev if dist is not None else None)
        return counts

    for _ in range(warmup):
        one_step()
    counts = None
    c0 = ctx.counters()
    sampler = ClockSampler(rig.local_rank)
    rig.barrier()
    if rig.rank == 0:
        sampler.start()
    ctx.timer_start()
    t0 = time.perf_counter()
    scanned = 0
    alg_bytes = 0
    shadow_acc = {}
    for _ in range(steps):
        counts = one_step()
        sr = ctx.build_stats()["scanned_rows"]
        sh = ctx.build_shadow_stats()
        scanned += sr
        alg_bytes += scan_bytes(sr, sh, d)
        for k, v in sh.items():
            shadow_acc[k] = shadow_acc.get(k, 0) + v
    dev_ms = ctx.timer_stop()   # CUDA events on the library's stream (the launching stream)
    rig.barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop() if rig.rank == 0 else None
    c1 = ctx.counters()
    ms_per_step = rig.max_over_ranks(max(dev_ms, 0.0)) / steps
    sc = rig.sum_over_ranks(scanned) / steps
    ab_step = rig.sum_over_ranks(alg_bytes) / steps
    st, bd = ctx.build_stats(), ctx.build_breakdown()
    return {"alg_bytes_per_step": ab_step, "shadow_rows_per_step": {k: v / steps for k, v in shadow_acc.items()}, "last_step_alg_bytes": scan_bytes(st["scanned_rows"], ctx.build_shadow_stats(), d),
            "ms_per_step": ms_per_step, "value": n / (ms_per_step * 1e-3), "wall_ms_per_step": wall * 1e3 / steps, "clocks": clocks,
            "launches": int(c1["launches"] - c0["launches"]), "scanned_rows_per_step": sc, "stats": st, "breakdown": bd, "my_trees": my_trees,
            "last_step_counts": counts}


def build_record(wl, tb, world):
    d = wl["d"]
    sc = tb["scanned_rows_per_step"]
    return {"scanned_rows_per_step": sc, "device_steps": tb["stats"]["steps"], "create_split_calls": tb["stats"]["create_split_calls"],
            "random_splits": tb["stats"]["random_splits"], "algorithmic_GB_per_step": tb["alg_bytes_per_step"] / 1e9,
            "whole_build_GBps": tb["alg_bytes_per_step"] / 1e9 / (tb["ms_per_step"] * 1e-3),
            "f32_rows_equivalent": {"GB_per_step": sc * d * 4 / 1e9, "GBps": sc * d * 4 / 1e9 / (tb["ms_per_step"] * 1e-3),
                                    "note": "scanned rows x d x 4: what the same scans read without the bf16 pre-filter and the fused root pass (round-1 accounting)"},
            "scan_rows_per_step": tb["shadow_rows_per_step"],
            "schedule": "lockstep" if os.environ.get("ARROY_B200_LOCKSTEP") else ("persistent: one cooperative launch per wave (control CTA per tree + worker CTAs)" if tb["stats"]["steps"] == 1 else "async per-tree graph branches (control / work kernel per attempt)"),
            "misspeculated_two_means": tb["stats"].get("misspeculated_splits", 0.0), "breakdown_ms_last_step": tb["breakdown"]}


# ---------------------------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed in its last step, so that two builds of the project can be compared
# output for output (the inputs are the same seeded stream in every run)
# ---------------------------------------------------------------------------------------------------------------------

DUMP_LIMIT_BYTES = 64 << 20
# seeded samples keep the dump of c4 (100 trees over 10M x 1536) under the limit; c2 fits whole but for the normals (~300 MB)
DUMP_NODES, DUMP_SPLIT_NORMALS, DUMP_ITEMS = 1 << 18, 4096, 16384


def write_outputs(out_dir, arrays):
    """{name: array} -> out_dir/<name>.npy; float32 arrays stay float32, all others become float64 (u32 ids are exact there)."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError("outputs to dump take %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def roaring_ids(b, o):
    """Item ids of the RoaringBitmap serialized at b[o:] (portable format without run containers, as NodeCodec writes it)."""
    import numpy as np
    cookie, n = np.frombuffer(b, dtype="<u4", count=2, offset=o)
    if cookie != 12346:
        raise ValueError("unexpected roaring cookie %d" % cookie)
    keys = np.frombuffer(b, dtype="<u2", count=2 * int(n), offset=o + 8).reshape(-1, 2)
    offs = np.frombuffer(b, dtype="<u4", count=int(n), offset=o + 8 + 4 * int(n))
    parts = []
    for (key, card_m1), off in zip(keys.tolist(), offs.tolist()):
        if card_m1 + 1 > 4096:   # bitmap container
            low = np.flatnonzero(np.unpackbits(np.frombuffer(b, dtype=np.uint8, count=8192, offset=o + off), bitorder="little"))
        else:                    # array container
            low = np.frombuffer(b, dtype="<u2", count=card_m1 + 1, offset=o + off)
        parts.append((key << 16) | low.astype(np.int64))
    return np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)


def forest_outputs(ctx, wl, counts):
    """The forest that the last build_trees_begin left parked on the device, emitted as a caller receives it (node ids numbered
    like a one-GPU Writer::build: roots 0..T-1, then tree by tree, last tree first) and laid out as arrays:
      node_counts            [T]              nodes per tree, root included (what build_trees_begin returns)
      split_nodes            [<=2^18, 3 + h]  node id, left child, right child, header of the normal (NaN: no normal)
      split_normal_ids       [<=4096]         seeded sample of the split nodes ...
      split_normals          [<=4096, d]      ... and their normals (f32; NaN: no normal)
      descendants            [<=2^18, 2]      node id, number of items of the Descendants nodes
      sampled_items          [<=16384]        seeded sample of the item ids ...
      leaf_of_sampled_items  [T, <=16384]     ... and the Descendants node holding each of them in every tree
    Tables with more rows than shown are a seeded sample of their rows, in node id order."""
    import struct

    import numpy as np
    import arroy_b200 as ab
    from arroy_b200 import parallel
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    counts = np.asarray(counts, dtype=np.int64)
    base = parallel.node_id_bases(counts, T)
    arena = ab.Arena()
    ctx.build_trees_emit(list(range(T)), base, arena=arena)
    n_ids = T + int((counts - 1).sum())
    tree_of = np.empty(n_ids, dtype=np.int64)
    tree_of[:T] = np.arange(T)
    for t in range(T):
        tree_of[int(base[t]):int(base[t]) + int(counts[t]) - 1] = t
    hf = 2 if metric == "dot-product" else 1

    def sample(n_rows, k, seed):
        return np.sort(np.random.default_rng(seed).choice(n_rows, min(n_rows, k), replace=False))
    items = sample(n, DUMP_ITEMS, 0)
    slot = np.full(n, -1, dtype=np.int64)   # item ids are the rows 0..n-1 here
    slot[items] = np.arange(len(items))
    leaf = np.full((T, len(items)), -1.0)
    splits, desc = [], []
    for nid in range(n_ids):
        b = arena.get(nid)
        if b is None:
            raise RuntimeError("node %d was not emitted" % nid)
        if b[0] == 1:
            ids = roaring_ids(b, 1)
            desc.append((nid, len(ids)))
            s = slot[ids]
            leaf[tree_of[nid], s[s >= 0]] = nid
        else:
            left, right = struct.unpack_from(">II", b, 1)
            hdr = np.frombuffer(b, dtype=np.float32, count=hf, offset=9).tolist() if len(b) > 9 else [float("nan")] * hf
            splits.append([nid, left, right] + hdr)
    splits = np.array(splits, dtype=np.float64).reshape(-1, 3 + hf)
    desc = np.array(desc, dtype=np.float64).reshape(-1, 2)
    normal_ids = splits[sample(len(splits), DUMP_SPLIT_NORMALS, 1), 0]
    normals = np.full((len(normal_ids), d), np.nan, dtype=np.float32)
    for r, nid in enumerate(normal_ids):
        b = arena.get(int(nid))
        if len(b) > 9:
            normals[r] = np.frombuffer(b, dtype=np.float32, count=d, offset=9 + 4 * hf)
    del arena
    return {"node_counts": counts, "split_nodes": splits[sample(len(splits), DUMP_NODES, 2)], "split_normal_ids": normal_ids,
            "split_normals": normals, "descendants": desc[sample(len(desc), DUMP_NODES, 3)], "sampled_items": items, "leaf_of_sampled_items": leaf}


def rerank_outputs(out):
    """rerank_shared results: ids and distances per query (NaN past the query's result length)."""
    import numpy as np
    rows, dist, length = out
    valid = np.arange(rows.shape[1])[None, :] < length[:, None]
    return {"rerank_ids": np.where(valid, rows.astype(np.float64), np.nan), "rerank_distances": np.where(valid, dist, np.float32(np.nan)),
            "rerank_lengths": length}


def leaf_blob(rig, wl, items):
    """The items as raw stored Leaf values [0x00][header][d x f32] at byte-aligned-only host addresses — what LMDB hands to
    ImmutableLeafs::new. Built chunk by chunk from the device matrix (no second full host copy)."""
    import numpy as np
    ctx = rig.ctx
    n, d, metric = wl["n"], wl["d"], wl["metric"]
    ids = np.arange(n, dtype=np.uint32)
    ctx.stage_items_device(metric, ids, d, items.data_ptr())
    if metric == "dot-product":
        ctx.dot_preprocess()
    h0, h1 = ctx.item_headers()          # D::new_header / preprocess result, as stored by the writer
    hf = 2 if metric == "dot-product" else 1
    stride = 1 + 4 * hf + 4 * d           # odd => every value is byte aligned only
    blob = np.zeros(n * stride, dtype=np.uint8)
    b2 = blob.reshape(n, stride)
    b2[:, 1:5] = h0.view(np.uint8).reshape(n, 4)
    if hf == 2:
        b2[:, 5:9] = h1.view(np.uint8).reshape(n, 4)
    step = 1 << 19
    for a in range(0, n, step):
        b = min(n, a + step)
        b2[a:b, 1 + 4 * hf:] = items[a:b].cpu().numpy().view(np.uint8).reshape(b - a, 4 * d)
    ptrs = (blob.ctypes.data + np.arange(n, dtype=np.uint64) * np.uint64(stride)).astype(np.uint64)
    return blob, ptrs


def e2e_single(rig, wl, items, seeds, steps, n_warm):
    """Through the C ABI with HOST buffers on one GPU: decode + H2D + device build + D2H + NodeCodec encoding, all timed."""
    import numpy as np
    ctx, ab = rig.ctx, rig.ab
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    ids = np.arange(n, dtype=np.uint32)
    blob, ptrs = leaf_blob(rig, wl, items)
    arena = ab.Arena()
    e_times, h2d, d2h, bd = [], 0, 0, None
    for step in range(n_warm + steps):
        arena.clear()
        cc0 = ctx.counters()
        t0 = time.perf_counter()
        ctx.stage_items_ptrs(metric, d, ids, ptrs)
        if metric == "dot-product":
            ctx.dot_preprocess()
        ctx.build_trees_into_arena(arena, seeds, list(range(T)), T)
        dt = time.perf_counter() - t0
        cc1 = ctx.counters()
        if step >= n_warm:
            e_times.append(dt)
            h2d, d2h = cc1["h2d_bytes"] - cc0["h2d_bytes"], cc1["d2h_bytes"] - cc0["d2h_bytes"]
            bd = ctx.build_breakdown()
    e_sec = sum(e_times) / len(e_times)
    n_nodes, node_bytes = arena.stats()
    del arena, blob, ptrs
    return {"value": n / e_sec, "unit": "vectors/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": e_sec * 1e3, "steps": steps,
            "api": "arroy_b200_stage_items(leaf value pointers) + arroy_b200_build_trees(arena sink)", "nodes": int(n_nodes), "node_bytes": int(node_bytes),
            "build_breakdown_ms": bd}


def e2e_multi(rig, wl, items, seeds, steps, n_warm):
    """N > 1: rank 0 decodes + uploads the host leaf values, ONE NCCL broadcast straight out of the library's item buffer,
    every rank builds and encodes its trees into its own host arena."""
    import numpy as np
    from arroy_b200 import parallel
    torch, ctx, ab, dist = rig.torch, rig.ctx, rig.ab, rig.dist
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    ids = np.arange(n, dtype=np.uint32)

    class _DevView:   # zero-copy torch view of the staged item matrix of this context
        def __init__(self, ptr, shape):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": "<f4", "data": (int(ptr), False), "version": 2}
    blob = ptrs = None
    if rig.rank == 0:
        blob, ptrs = leaf_blob(rig, wl, items)
    arena = ab.Arena()
    roots = list(range(T))
    e_ms, cc0 = [], None
    for step in range(n_warm + steps):
        arena.clear()
        rig.barrier()
        if step == n_warm:
            cc0 = ctx.counters()
        t0 = time.perf_counter()
        # rank 0 decodes + uploads chunk k + 1 while chunk k is being broadcast out of / into the library's item buffers
        parallel.stage_and_broadcast(ctx, dist, rig.rank, metric, d, ids, ptrs, rig.dev)
        parallel.sharded_build(ctx, dist, rig.rank, rig.world, seeds, roots, T, arena=arena, device=rig.dev)
        rig.barrier()
        if step >= n_warm:
            e_ms.append((time.perf_counter() - t0) * 1e3)
    cc1 = ctx.counters()
    e_sec = rig.max_over_ranks(sum(e_ms) / len(e_ms)) * 1e-3
    h2d = rig.sum_over_ranks(float(cc1["h2d_bytes"] - cc0["h2d_bytes"]) / steps)
    d2h = rig.sum_over_ranks(float(cc1["d2h_bytes"] - cc0["d2h_bytes"]) / steps)
    del arena, blob, ptrs
    return {"value": n / e_sec, "unit": "vectors/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "ms_per_step": e_sec * 1e3, "steps": steps,
            "api": "rank 0: arroy_b200_stage_begin / _rows / _end (leaf value pointers) pipelined chunk by chunk with the NCCL broadcast of the item buffer; every rank: arroy_b200_build_trees_begin / _emit (arena sink) for its trees",
            "timing": "wall clock between barriers, max over ranks"}


def query_section(rig, wl, items, args, label):
    """Writer e2e + QPS@recall100 on one GPU through the host mirror (Writer.build, Reader.nns / nns_batch_by_item)."""
    import numpy as np
    ctx, ab = rig.ctx, rig.ab
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    ids = np.arange(n, dtype=np.uint32)
    host = items.cpu().numpy()
    env = ab.Env(rig.local_rank)
    env._ctx = ctx
    w = ab.Writer(env, 0, d, metric)
    w_times = []
    for step in range(3):
        w.clear()                # a FIRST build every step (re-adding items to a built index would take the incremental path)
        w.add_items(ids, host)   # Writer::add_item x n: the key/value puts are the caller's side of the API, not timed
        t0 = time.perf_counter()
        w.builder(ab.StdRng.from_seed(SEED)).n_trees(T).build()
        if step >= 1:
            w_times.append(time.perf_counter() - t0)
    ws = sum(w_times) / len(w_times)
    rec = {"dataset": label, "e2e_writer": {"value": n / ws, "unit": "vectors/s", "ms_per_step": ws * 1e3, "api": "Writer.builder(rng).n_trees(T).build()", "breakdown_ms": w.build_timings()}}
    # QPS @ recall: by_item queries for items 0..Q-1 (SURVEY §8d), top-100, default search_k
    Q, k = args.queries, 100
    reader = ab.Reader.open(env, 0, metric)
    qitems = np.arange(Q, dtype=np.uint32)
    reader.nns_batch_by_item(qitems, k)  # warm-up (stages the items, uploads the forest, sizes the scratch buffers)
    q_times = []
    for _ in range(5):
        t0 = time.perf_counter()
        out_ids, out_dist, out_len, qms = reader.nns_batch_by_item(qitems, k)
        q_times.append(time.perf_counter() - t0)
    q_sec = min(q_times)
    nsingle = min(Q, 200)
    reader.nns(k).by_item(0)
    lat, single = [], []
    for i in qitems[:nsingle]:
        t0 = time.perf_counter()
        single.append(reader.nns(k).by_item(int(i)))
        lat.append(time.perf_counter() - t0)
    lat.sort()
    assert all([s[0] for s in single[i]] == out_ids[i, :out_len[i]].tolist() for i in range(nsingle)), "batched and one-at-a-time results differ"
    # exact ground truth: the same distance over ALL rows (brute force on the device)
    allrows = np.arange(n, dtype=np.uint32)
    hits = 0
    QG = min(Q, 100)
    h0q, _ = ctx.item_headers()
    offs = (np.arange(QG + 1, dtype=np.uint64) * np.uint64(n))
    g_rows, _, g_len = ctx.rerank_batch(host[:QG], h0q[:QG], np.tile(allrows, QG), offs, k)
    for i in range(QG):
        hits += len(set(g_rows[i, :g_len[i]].tolist()) & set(out_ids[i, :out_len[i]].tolist()))
    rec["query"] = {"dataset": label, "qps_batched": Q / q_sec, "queries": Q, "k": k, "search_k": k * T, "recall_at_100": hits / (QG * k), "recall_queries": QG,
                    "batch_device_ms": qms["rerank_ms"], "qps_one_at_a_time": nsingle / sum(lat), "latency_one_at_a_time_ms": {"p50": lat[len(lat) // 2] * 1e3, "p99": lat[min(len(lat) - 1, int(len(lat) * 0.99))] * 1e3},
                    "api": "Reader.nns_batch_by_item / Reader.nns(100).by_item: device tree walk (one warp per query) + fused bf16 pre-filter / exact re-score / top-k kernel on the device-resident forest"}
    del reader
    env._ctx = None
    del w, env, host
    return rec, (out_ids, out_dist, out_len)


def cpu_build_and_queries(wl, args, gpu_results):
    """The oracle (port of the reference) on the host cores: one forest build (bounded sample of trees) and — when the sample
    is the whole forest — nns_by_item on the same queries, ids and distances compared with the GPU's."""
    import numpy as np
    import oracle
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    cores = os.cpu_count() or 1
    ids = np.arange(n, dtype=np.uint32)
    t_sample = args.ref_trees or (T if n * d < 5e9 else min(T, max(8, cores // 2)))
    data = oracle.synth_rows(SEED, d, 0, n, wl["centre"], threads=min(cores, 64))
    db = oracle.Db(metric, d)
    db.set_items(ids, data)
    t0 = time.perf_counter()
    cpu_threads = 1 if args.workload == "c1" else min(cores, t_sample)   # configs[0] names the single-thread CPU reference
    db.build(oracle.StdRng(SEED), n_trees=t_sample, threads=cpu_threads)
    sec = time.perf_counter() - t0
    out = {"cpu_baseline": {"value": n / (sec * T / t_sample), "unit": "vectors/s", "cores": cpu_threads, "nproc": cores, "kind": "port",
                            "sample": "%d of %d trees over the full %dx%d matrix in %.3f s on %d thread(s) of %d host cores, extrapolated x%.2f" % (t_sample, T, n, d, sec, cpu_threads, cores, T / t_sample)}}
    if gpu_results is not None and t_sample == T:
        out_ids, out_dist, out_len = gpu_results
        Q, k = out_ids.shape[0], 100
        lat, same = [], True
        for i in range(Q):
            t0 = time.perf_counter()
            w = db.nns_by_item(i, k)
            lat.append(time.perf_counter() - t0)
            same = same and [x[0] for x in w] == out_ids[i, :out_len[i]].tolist() and np.array([x[1] for x in w], dtype=np.float32).tobytes() == out_dist[i, :out_len[i]].tobytes()
        tot = sum(lat)
        lat.sort()
        # all cores: one query per thread (the reference's readers are independent RoTxn users)
        from concurrent.futures import ThreadPoolExecutor
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as ex:
            list(ex.map(lambda i: db.nns_by_item(i, k), range(Q)))
        par = time.perf_counter() - t0
        out["query_cpu_baseline"] = {"qps_one_thread": Q / tot, "latency_ms": {"p50": lat[Q // 2] * 1e3, "p99": lat[min(Q - 1, int(Q * 0.99))] * 1e3}, "qps_all_cores": Q / par, "cores": cores, "nproc": cores, "kind": "port",
                                     "sample": "oracle.Db.nns_by_item on the same %d queries (top-100, default search_k) over the identical 50-tree forest" % Q,
                                     "results_identical_to_gpu": bool(same)}
    return out


def headline_10m(rig, args):
    """BASELINE.json's metric configuration itself: 10M x 768 Cosine, n_trees = 100 (fits one B200: 30.7 GB)."""
    wl = WORKLOADS["h10m"]
    n, d, T = wl["n"], wl["d"], wl["n_trees"]
    ctx = rig.ctx
    items = synth_items(rig, wl)
    seeds = derive_seeds(rig.ab, T)
    tb = timed_builds(rig, wl, items, seeds, steps=2, warmup=1)
    rec = {"metric": "index-build vectors/sec", "value": tb["value"], "unit": "vectors/s", "n_gpus": rig.world, "steps": 2, "warmup": 1, "ms_per_step": tb["ms_per_step"],
           "config": base_config(wl), "dtype": "f32", "data": "synthetic", "gpu_launches": tb["launches"], "build": build_record(wl, tb, rig.world), "clocks": tb["clocks"]}
    if rig.rank == 0:
        import numpy as np
        hbm, which = peaks()
        alg = tb["alg_bytes_per_step"] / rig.world   # this rank's share (trees are spread evenly)
        loop_ms = tb["breakdown"]["loop_ms"]
        r = np.random.default_rng(0)
        normal = (r.standard_normal(d) / np.sqrt(d)).astype(np.float32)
        root_ms, _ = ctx.time_scan(normal, (0.0, 0.0), n, iters=3, flush_l2=False)
        rec["roofline"] = {"bound": "hbm", "kernel": "work_kernel_shadow (side() through the bf16 shadow + exact re-score of undecided rows + id partition)", "achieved": alg / (loop_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                           "frac": alg / (loop_ms * 1e-3) / 1e9 / hbm, "peak_source": which, "traffic": None,
                           "timing": "in the timed schedule: algorithmic scan bytes of one step / the device loop time of that step (all work_kernel launches run concurrently on 100 "
                                     "streams next to the control kernels, so this is a LOWER bound of the kernel's own rate)",
                           "root_scan": {"rows": n, "ms": root_ms, "GBps": n * d * 4 / (root_ms * 1e-3) / 1e9, "frac": n * d * 4 / (root_ms * 1e-3) / 1e9 / hbm,
                                         "note": "one plain f32 work_kernel launch over all 10M rows, timed alone with CUDA events (30.7 GB: larger than L2)"}}
    if not args.no_e2e:
        e = e2e_single(rig, wl, items, seeds, steps=2, n_warm=1) if rig.world == 1 else e2e_multi(rig, wl, items, seeds, steps=2, n_warm=1)
        rec["e2e"] = e
    del items
    rig.torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("ARROY_BENCH_WORKLOAD", "c2"), choices=sorted(WORKLOADS))
    ap.add_argument("--ref-trees", type=int, default=None, help="trees built per step by --impl reference / cpu_baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-writer-e2e", action="store_true")
    ap.add_argument("--no-query", action="store_true")
    ap.add_argument("--no-headline", action="store_true", help="skip the 10M x 768 sub-record of the default workload")
    ap.add_argument("--no-c5", action="store_true", help="skip the config-5 sub-record of the default workload")
    ap.add_argument("--queries", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step to DIR/<name>.npy (f32 / f64, at most 64 MB; "
                         "seeded samples of larger outputs), for comparing two builds on identical inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.dump_outputs and args.workload != "c5" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs of a forest build needs one process (each rank holds only its own trees)")
    wl = WORKLOADS[args.workload]
    if args.workload == "c5":
        run_c5(args, wl)
        return
    if args.impl == "reference":
        run_reference(args, wl)
        return

    import numpy as np
    rig = Rig()
    ctx, torch, rank, world = rig.ctx, rig.torch, rig.rank, rig.world
    n, d, T, metric = wl["n"], wl["d"], wl["n_trees"], wl["metric"]
    ids = np.arange(n, dtype=np.uint32)
    full = args.workload == "c2"     # the default line carries the sub-records

    items = synth_items(rig, wl)     # generated on the device of rank 0 (counter-based ChaCha12 stream)
    seeds = derive_seeds(rig.ab, T)
    tb = timed_builds(rig, wl, items, seeds, args.steps, args.warmup)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, forest_outputs(ctx, wl, tb["last_step_counts"]))
    line = {
        "metric": "index-build vectors/sec", "value": tb["value"], "unit": "vectors/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tb["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": base_config(wl),
        "notes": {"parallelism": "trees sharded t mod %d; one NCCL broadcast of the item buffer per step" % world,
                  "l2": "inputs (%.1f GB) larger than L2; no flush needed" % (n * d * 4 / 1e9), "timing": "CUDA events on the library stream, max over ranks",
                  "wall_ms_per_step": tb["wall_ms_per_step"],
                  "value": "stage (device to device) + forest build; the built forest stays in HBM. `value_incl_emit` adds the D2H of the records / normals and the NodeCodec encoding "
                           "into a host arena, i.e. what the CPU arm's step produces"},
        "gpu_launches": tb["launches"],
        "build": build_record(wl, tb, world),
    }
    if rank == 0:
        line["clocks"] = tb["clocks"]
        hbm, which = peaks()
        # roofline of the dominant kernel: work_kernel (side()/margin scan)
        os.environ["ARROY_B200_PROFILE"] = "1"
        ctx.build_trees_begin([seeds[t] for t in tb["my_trees"]])   # rank-local: no collective in here
        os.environ.pop("ARROY_B200_PROFILE")
        st = ctx.build_stats()
        scan_ms, steps_dev = st["scan_ms"], st["steps"]
        alg_bytes = scan_bytes(st["scanned_rows"], ctx.build_shadow_stats(), d)
        achieved = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
        traffic, traffic_note = None, "no ncu capture of this build of the kernel committed"
        for tp_name in ("r02_shadow_kernel_traffic.json",):
            tp = os.path.join(ROOT, "profiles", tp_name)
            if os.path.exists(tp):
                tj = json.load(open(tp))
                ratio = (tj["dram_bytes_read"] + tj["dram_bytes_write"]) / tj["algorithmic_bytes"]
                traffic = ratio * alg_bytes / max(steps_dev, 1)
                traffic_note = "avg algorithmic bytes/launch x %.4f (dram/algorithmic of %s)" % (ratio, tj["source"])
                break
        r = np.random.default_rng(0)
        normal = (r.standard_normal(d) / np.sqrt(d)).astype(np.float32)
        root_ms, _ = ctx.time_scan(normal, (0.0, 0.0), n, iters=5, flush_l2=True)
        own_alg = tb["alg_bytes_per_step"] / world
        lockstep_rec = {"GBps": achieved, "frac": achieved / hbm, "launches": steps_dev, "avg_ms": scan_ms / max(steps_dev, 1), "avg_algorithmic_GB": alg_bytes / max(steps_dev, 1) / 1e9,
                        "share_of_step": scan_ms / (st["build_ms"] if st["build_ms"] else 1.0),
                        "note": "SEPARATE untimed build in the lockstep schedule (ARROY_B200_PROFILE: one control + one work_kernel launch per step, every work_kernel launch "
                                "bracketed by CUDA events on its launching stream and running alone)"}
        root_rec = {"rows": n, "ms": root_ms, "GBps": n * d * 4 / (root_ms * 1e-3) / 1e9, "frac": n * d * 4 / (root_ms * 1e-3) / 1e9 / hbm}
        if tb["stats"]["steps"] == 1 and tb["stats"]["scan_ms"] > 0:
            # persistent schedule: the dominant kernel IS the step — one launch holds every side()/margin scan and wide partition
            kms = tb["stats"]["scan_ms"]
            k_alg = tb["last_step_alg_bytes"]
            k_f32 = tb["stats"]["scanned_rows"] * d * 4
            line["roofline"] = {
                "bound": "hbm", "kernel": "control_kernel<persistent> (worker CTAs: side() through the bf16 shadow + exact re-score, fused root pass, id partition; control CTAs: two_means / create_split / DFS)",
                "achieved": k_alg / (kms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": k_alg / (kms * 1e-3) / 1e9 / hbm, "peak_source": which,
                "traffic": (traffic * max(steps_dev, 1) / alg_bytes * k_alg) if traffic else None, "traffic_note": traffic_note,
                "timing": "live, inside the timed region: CUDA events on the launching stream around the ONE kernel launch of the last timed step; achieved = the step's "
                          "algorithmic scan bytes (bench.py scan_bytes: 2 B per element of the rows that went through the bf16 pre-filter, 4 B per element of the rows scored in f32, "
                          "the fused root pass counted once) / that duration — control CTAs' serial work included, so a lower bound of the scan rate",
                "per_launch": {"launches": 1, "avg_ms": kms, "avg_algorithmic_GB": k_alg / 1e9},
                "f32_rows_equivalent_GBps": k_f32 / (kms * 1e-3) / 1e9,
                "work_kernel_alone": lockstep_rec, "root_scan": root_rec,
            }
        else:
            line["roofline"] = {
                "bound": "hbm", "kernel": "work_kernel (side()/margin scan + id partition)", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm,
                "peak_source": which, "traffic": traffic, "traffic_note": traffic_note,
                "timing": lockstep_rec["note"] + "; the timed steps use the asynchronous per-tree schedule, whose kernels overlap",
                "per_launch": {"launches": steps_dev, "avg_ms": scan_ms / max(steps_dev, 1), "avg_algorithmic_GB": alg_bytes / max(steps_dev, 1) / 1e9},
                "in_timed_schedule": {"GBps": own_alg / (tb["breakdown"]["loop_ms"] * 1e-3) / 1e9, "frac": own_alg / (tb["breakdown"]["loop_ms"] * 1e-3) / 1e9 / hbm,
                                      "note": "algorithmic scan bytes of the last timed step / its device loop time: all kernels of the step, control kernels and launch gaps included"},
                "root_scan": root_rec, "share_of_step": scan_ms / (st["build_ms"] if st["build_ms"] else 1.0),
            }
    # ---- the same step INCLUDING node emission (like-for-like with the CPU arm, which produces complete nodes) -----------------
    if rank == 0 and world == 1 and not args.no_e2e:
        arena = rig.ab.Arena()
        ts = []
        for step in range(4):
            arena.clear()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctx.stage_items_device(metric, ids, d, items.data_ptr())
            if metric == "dot-product":
                ctx.dot_preprocess()
            ctx.build_trees_into_arena(arena, seeds, list(range(T)), T)
            if step >= 1:
                ts.append(time.perf_counter() - t0)
        line["value_incl_emit"] = {"value": n / (sum(ts) / len(ts)), "unit": "vectors/s", "ms_per_step": sum(ts) / len(ts) * 1e3, "steps": len(ts),
                                   "what": "items resident in HBM -> stage + build + D2H + NodeCodec encoding into the arena sink (wall clock)"}
        del arena
    # ---- e2e: through the C ABI with HOST buffers (what a fork of the Rust crate would call) -----------------------------------
    if args.no_e2e:
        line["e2e"] = None
    elif world == 1:
        line["e2e"] = e2e_single(rig, wl, items, seeds, steps=min(args.steps, 5), n_warm=max(1, min(args.warmup, 2)))
    elif d % 32 == 0 and metric != "dot-product":
        line["e2e"] = e2e_multi(rig, wl, items, seeds, steps=min(args.steps, 5), n_warm=1)
    else:
        line["e2e"] = None
    # ---- queries (one GPU: the re-rank is single-GPU, replicas only) -------------------------------------------------------------
    gpu_results = None
    if rank == 0 and world == 1 and not args.no_writer_e2e:
        rec, gpu_results = query_section(rig, wl, items, args, "uniform (SURVEY 8d)")
        line["e2e_writer"] = rec["e2e_writer"]
        if not args.no_query:
            line["query"] = rec["query"]
            if full:
                gitems = synth_items(rig, wl, dataset="gmm")
                grec, _ = query_section(rig, wl, gitems, args, "gaussian mixture: %d centres in [-0.5,0.5)^%d, row i = centre[(i*2654435761) mod %d] + %.2f*(u-0.5)" % (GMM_CLUSTERS, d, GMM_CLUSTERS, GMM_SCALE))
                line["query_gmm"] = grec["query"]
                line["query_gmm"]["e2e_writer_ms"] = grec["e2e_writer"]["ms_per_step"]
                del gitems
        else:
            gpu_results = None
    del items
    torch.cuda.empty_cache()
    # ---- BASELINE configs[4] as a sub-record -------------------------------------------------------------------------------------
    if full and rank == 0 and world == 1 and not args.no_c5:
        line["c5"] = c5_measure(ctx, torch, rig.dev, WORKLOADS["c5"], steps=5, warmup=2, cpu_sample=not args.no_cpu_baseline)
        torch.cuda.empty_cache()
    # ---- the metric's own configuration ----------------------------------------------------------------------------------------
    if full and not args.no_headline:
        h = headline_10m(rig, args)
        if rank == 0:
            line["headline_10m"] = h
    # ---- CPU baseline (oracle port) on a bounded sample, rank 0, N=1 only ----------------------------------------------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cb = cpu_build_and_queries(wl, args, gpu_results)
        line["cpu_baseline"] = cb["cpu_baseline"]
        if "query_cpu_baseline" in cb and "query" in line:
            line["query"]["cpu_baseline"] = cb["query_cpu_baseline"]
    if rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()
    if rig.dist is not None:
        rig.dist.barrier()
        rig.dist.destroy_process_group()


if __name__ == "__main__":
    main()
