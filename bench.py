#!/usr/bin/env python
"""bench.py -- IVF_PQ index-build Mvec/s and QPS@recall@10 (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            # our arm, config C1 (the one the metric is quoted on)
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port), same config
    python bench.py --config C2|C3|C4|C5 [--rows R]          # the other BASELINE.json configs, at size
    python bench.py --steps K --warmup W --dump-outputs DIR  # C1, plus what the last timed steps returned, as .npy

C1 (default; what the driver runs): a "step" is ONE complete IVF_PQ(256,16) index build over the
1M x 128 f32 dataset: sample -> k-means (IVF) -> residuals -> 16 sub-space k-means (PQ) -> partition id +
residual + PQ code for every row -> group by partition.  `value` is measured with the dataset already
resident in HBM; `e2e` is the same build through the C ABI from a pinned HOST buffer with the results
(partition offsets, codes, row ids, centroids, codebook) copied back to the host.  The query half of the
metric (QPS at recall@10) is in "query" / "query_table".

C2..C5: one build per step of the named configuration (rows per GPU = the config's share of one GPU, see
CONFIGS), with an in-run oracle check of a row sample (partition ids + PQ codes bit-exact), the assign
kernel's roofline against the measured tensor peak, a search batch with recall, e2e and a CPU sample.

torch is used only to synthesise the dataset on the device, for the ground truth of recall, and for
torch.distributed; nothing on the measured path is a torch op.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ROWS, DIM, NUM_PARTITIONS, NUM_SUB_VECTORS = 1_000_000, 128, 256, 16
NQ, TOPK, NPROBES = 10_000, 10, 10
WORKLOAD = "C1: SIFT-1M-shaped synthetic 1M x 128 f32, IVF_PQ num_partitions=256 num_sub_vectors=16, L2"

# BASELINE.json configs[1..4].  rows = the share ONE GPU holds when the configuration runs as BASELINE.json
# states it (C3 / C5 "over 8 B200": total / 8; C4 50M x 1536 bf16 = 153.6 GB is also an 8-way shard); every
# rank of a --gpus N run holds one such shard (weak scaling), so --gpus 8 is the configuration at full size.
CONFIGS = {
    "C2": dict(desc="C2: synthetic 10M x 768 f32 (OpenAI-ada shape), IVF_PQ 4096/96, L2, single B200",
               rows=10_000_000, total=10_000_000, d=768, dtype="f32", kind="pq", K=4096, M=96, metric="l2", ncomp=4096, nprobes=20),
    "C3": dict(desc="C3: synthetic 100M x 128 f16, IVF_PQ 8192/16, cosine, build sharded over 8 B200 (12.5M rows per GPU)",
               rows=12_500_000, total=100_000_000, d=128, dtype="f16", kind="pq", K=8192, M=16, metric="cosine", ncomp=8192, nprobes=20),
    "C4": dict(desc="C4: synthetic 50M x 1536 bf16, IVF_FLAT 4096 partitions (6.25M rows per GPU of 8)",
               rows=6_250_000, total=50_000_000, d=1536, dtype="bf16", kind="flat", K=4096, M=0, metric="l2", ncomp=4096, nprobes=4),
    "C5": dict(desc="C5: BigANN-style 1B x 128 u8, IVF_PQ 65536/32, 10k-query ADC batches across 8 B200 (125M rows per GPU)",
               rows=125_000_000, total=1_000_000_000, d=128, dtype="u8", kind="pq", K=65536, M=32, metric="l2", ncomp=65536, nprobes=32),
}


def peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], 0, set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# synthetic data on the device (same law as lance_b200/synth.py:sift_like)
# ------------------------------------------------------------------------------------------------
def device_dataset(torch, n, nq, seed, device, qseed=99):
    from lance_b200 import synth
    W, cm = synth.sift_model(DIM, 24, 1024, 1234)
    W, cm = torch.from_numpy(W).to(device), torch.from_numpy(cm).to(device)
    g = torch.Generator(device=device)
    g.manual_seed(seed)

    def draw(rows):
        out = torch.empty((rows, DIM), dtype=torch.float32, device=device)
        for s in range(0, rows, 1 << 18):
            e = min(rows, s + (1 << 18))
            comp = torch.randint(0, cm.shape[0], (e - s,), device=device, generator=g)
            z = cm[comp] + torch.randn((e - s, 24), device=device, generator=g)
            x = torch.clamp(z @ W * 12.0 + 20.0, min=0.0)
            x += torch.randn((e - s, DIM), device=device, generator=g) * 3.0
            out[s:e] = torch.clamp(torch.round(x), 0.0, 255.0)
        return out

    data = draw(n)
    g.manual_seed(qseed)  # the same queries on every rank
    return data, draw(nq)


def ground_truth(torch, data, queries, k, row_base=0, cosine=False, return_dists=False):
    """exact top-k by brute force on the device, chunked over the rows (f32, TF32 off)"""
    torch.backends.cuda.matmul.allow_tf32 = False
    q = queries.float()
    if cosine:
        q = q / q.norm(dim=1, keepdim=True)
    best_d = torch.full((q.shape[0], k), float("inf"), device=q.device)
    best_i = torch.zeros((q.shape[0], k), dtype=torch.int64, device=q.device)
    step = max(1, (1 << 28) // max(data.shape[1], 1))
    for s in range(0, data.shape[0], step):
        x = data[s:s + step].float()
        if cosine:
            x = x / x.norm(dim=1, keepdim=True)
        d2 = (x * x).sum(1)[None, :] - 2.0 * (q @ x.T) + (q * q).sum(1)[:, None]
        cd = torch.cat([best_d, d2], 1)
        ci = torch.cat([best_i, torch.arange(s, s + x.shape[0], device=q.device)[None, :].expand(q.shape[0], -1) + row_base], 1)
        o = torch.topk(cd, k, dim=1, largest=False)
        best_d, best_i = o.values, torch.gather(ci, 1, o.indices)
    if return_dists:
        return best_i, best_d
    return best_i.cpu().numpy()


def wrap_tensor(lb, t, dtype):
    a = lb.DeviceArray.__new__(lb.DeviceArray)
    a.shape, a.dtype, a.ptr, a.nbytes = tuple(t.shape), np.dtype(dtype), t.data_ptr(), t.numel() * t.element_size()
    a.free = lambda: None
    return a


# ------------------------------------------------------------------------------------------------
# CPU path (the oracle port of the reference loops), used by --impl reference and cpu_baseline
# ------------------------------------------------------------------------------------------------
def cpu_build(ob, data_host, max_iters, threads, transform_rows, sample_ivf, sample_pq):
    """One IVF_PQ(256,16) build on the host: both trainings in full, then partition id + residual + PQ code
    for the first `transform_rows` rows.  Returns (t_train_s, t_transform_s, detail)."""
    t0 = time.perf_counter()
    xs = data_host[sample_ivf]
    cent, loss, it_ivf = ob.kmeans_train(xs, NUM_PARTITIONS, max_iters=max_iters,
                                         balance_factor=float(np.float32(1.0) / np.float32(len(xs))), nthreads=threads)
    t1 = time.perf_counter()
    xp = data_host[sample_pq]
    part, _, _ = ob.compute_membership(cent, xp, nthreads=threads)
    res = ob.compute_residual(cent, xp, part, nthreads=threads)
    cb, it_pq = ob.pq_train(res, NUM_SUB_VECTORS, max_iters=max_iters, nthreads=threads)
    t2 = time.perf_counter()
    rows = data_host[:transform_rows]
    p, _, _ = ob.compute_membership(cent, rows, nthreads=threads)
    r = ob.compute_residual(cent, rows, p, nthreads=threads)
    ob.pq_encode(cb, r, nthreads=threads)
    t3 = time.perf_counter()
    # grouping (stable sort by partition) is negligible on the CPU side and left out (favours the CPU)
    return t2 - t0, t3 - t2, {"ivf_train_s": t1 - t0, "pq_train_s": t2 - t1, "transform_s_measured": t3 - t2,
                              "transform_rows": int(transform_rows), "ivf_iters": int(it_ivf),
                              "pq_iters_max": int(max(it_pq)), "model": (cent, cb)}


def cpu_query_qps(ob, model, data_host, queries_host, threads, nq):
    cent, cb = model
    p, _, _ = ob.compute_membership(cent, data_host, nthreads=threads)
    res = ob.compute_residual(cent, data_host, p, nthreads=threads)
    codes = ob.pq_encode(cb, res, nthreads=threads)
    order = np.argsort(p, kind="stable")
    off = np.zeros(NUM_PARTITIONS + 1, np.uint64)
    off[1:] = np.cumsum(np.bincount(p, minlength=NUM_PARTITIONS))
    codes_s, rid = codes[order], order.astype(np.uint64)
    t0 = time.perf_counter()
    ob.ivfpq_search(cent, cb, off, codes_s, rid, queries_host[:nq], TOPK, NPROBES, nthreads=threads)
    return nq / (time.perf_counter() - t0)


def cpu_steps(ob, data, n_rows, steps, warmup, threads, budget_s):
    """(warmup + steps) CPU builds inside `budget_s`: every step trains in full; the transform covers all
    n_rows rows when that fits the budget ("timed, not scaled"), else a bounded prefix scaled linearly."""
    rng = np.random.default_rng(0)
    n = data.shape[0]
    s_ivf = np.sort(rng.choice(n, min(n, 65536), replace=False))
    s_pq = np.sort(rng.choice(n, min(n, 65536), replace=False))
    total = warmup + steps
    rows = min(n, n_rows)
    times, detail, scaled = [], None, rows < n_rows
    t_begin = time.perf_counter()
    for i in range(total):
        left = total - i
        if i >= 1:  # size the remaining steps from what the previous one cost
            t_train, t_tr = last
            per_row = t_tr / last_rows
            room = (budget_s - (time.perf_counter() - t_begin)) / left - t_train
            fit = int(max(min(n, 20000), min(rows, room / per_row if per_row > 0 else rows)))
            fit = min(fit, n)
            if fit < rows:
                rows, scaled = fit, True
        t_train, t_tr, detail = cpu_build(ob, data, 50, threads, rows, s_ivf, s_pq)
        last, last_rows = (t_train, t_tr), rows
        if i >= warmup:
            times.append(t_train + t_tr * (n_rows / float(rows)))
    model = detail.pop("model")
    how = ("every step: IVF + PQ training in full (<= 50 iterations each, 65 536-row samples) and the transform of " +
           (f"all {n_rows} rows -- timed, not scaled" if not scaled and rows >= n_rows else
            f"{rows} of {n_rows} rows scaled linearly (the full transform did not fit the {budget_s:.0f} s budget)"))
    return float(np.mean(times)), len(times), detail, model, how


def best_threads(ob):
    """The thread count that serves the CPU arm best on THIS box: hosts with a CPU quota or busy neighbours do
    not scale to nproc, and a pool that is too wide only adds wake-up latency to ~1000 short parallel regions."""
    if os.environ.get("LB2_BENCH_THREADS"):
        return int(os.environ["LB2_BENCH_THREADS"])
    hw = ob.nthreads_default()
    rng = np.random.default_rng(0)
    x = rng.standard_normal((65536, 8)).astype(np.float32)
    init = x[:256].copy()
    best, best_t = hw, None
    for nt in sorted({hw, max(1, hw // 2), max(1, hw // 4), max(1, hw // 8), min(hw, 16), min(hw, 8)}, reverse=True):
        ob.kmeans_train(x, 256, max_iters=1, init_centroids=init, nthreads=nt)
        t0 = time.perf_counter()
        ob.kmeans_train(x, 256, max_iters=4, init_centroids=init, nthreads=nt)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t * 0.95:
            best, best_t = nt, dt
    return best


def run_reference(args):
    """The reference's own CPU implementation of the path (oracle port; the Rust toolchain and
    pylance are absent, see DESIGN.md), all host threads, same config/metric as our arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from lance_b200 import synth
    from oracle import binding as ob
    threads = best_threads(ob)
    # LB2_BENCH_REF_ROWS shrinks the host dataset (tests/test_bench_contract.py runs this arm in seconds): the
    # transform then covers that prefix and is scaled to the 1M rows of the workload, and the line says so
    n_avail = int(os.environ.get("LB2_BENCH_REF_ROWS", str(N_ROWS)))
    data = synth.sift_like(max(n_avail, 20000), DIM)
    queries = synth.sift_like_queries(2000, DIM)
    sec, nsteps, detail, model, how = cpu_steps(ob, data, N_ROWS, args.steps, args.warmup, threads,
                                               float(os.environ.get("LB2_BENCH_REF_BUDGET_S", "240")))
    scale = 1.0
    value = N_ROWS / sec / 1e6
    qrows = min(data.shape[0], 200_000)
    qps = cpu_query_qps(ob, model, data[:qrows], queries, threads, min(2000, queries.shape[0]))
    line = {
        "impl": "reference", "metric": "ivf_pq_index_build_mvec_per_s", "value": value, "unit": "Mvec/s",
        "n_gpus": args.gpus, "steps": nsteps, "warmup": args.warmup, "ms_per_step": sec * scale * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "k": TOPK, "nprobes": NPROBES},
        "cpu_baseline": {"value": value, "unit": "Mvec/s", "cores": threads, "host_threads": ob.nthreads_default(),
                         "kind": "port", "sample": how, **detail},
        "e2e": {"value": value, "unit": "Mvec/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "query": {"qps": qps, "nprobes": NPROBES, "k": TOPK, "note": f"index over {qrows} rows"},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# our arm, C1
# ------------------------------------------------------------------------------------------------
KERNEL_BYTES = {
    # algorithmic bytes per launch (SURVEY 8d / DESIGN.md "kernels"): the rows' vectors read ONCE
    "ivf_train:tc_filter": lambda ns, n: ns * DIM * 4,
    "pq_train:tc_pq_filter": lambda ns, n: ns * DIM * 4,
    "transform:tc_filter": lambda ns, n: n * DIM * 4 + n * 8,
    "transform:tc_pq_filter": lambda ns, n: n * DIM * 4 + n * NUM_SUB_VECTORS,
    "ivf_train:assign_exact": lambda ns, n: ns * DIM * 4,
    "pq_train:pq_assign_exact": lambda ns, n: ns * DIM * 4,
    "transform:assign_exact": lambda ns, n: n * DIM * 4 + n * 5,
    "transform:pq_assign_exact": lambda ns, n: n * DIM * 4 + n * 4 + n * NUM_SUB_VECTORS,
}


DUMP_ROWS = 1 << 19   # storage positions of codes / row ids kept by --dump-outputs (about 40 MB in all at C1)


def dump_outputs(path, arrays):
    """--dump-outputs: DIR/<name>.npy; float32 and integers of <= 16 bits as float32, the rest as float64 (exact:
    row ids and offsets are below 2**53)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        small = a.dtype == np.float32 or (a.dtype.kind in "iu" and a.dtype.itemsize <= 2)
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32 if small else np.float64))


def build_outputs(parts):
    """What a caller of the build receives (lb2_index_export); codes and row ids at a fixed, seeded sample of
    storage positions when there are more than DUMP_ROWS rows."""
    n = len(parts["row_ids"])
    pos = np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False)) if n > DUMP_ROWS else slice(None)
    return {"centroids": parts["centroids"], "codebook": parts["codebook"], "part_offsets": parts["part_offsets"],
            "codes": parts["codes"][pos], "row_ids": parts["row_ids"][pos]}


def load_ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` summary
    of the same kernels on the same workload (profiles/ncu_traffic.json, written by profiles/summarize_ncu.py)"""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        return {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--config", default="C1", choices=["C1"] + sorted(CONFIGS))
    ap.add_argument("--rows", type=int, default=None, help="rows per GPU (default: the configuration's share)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", default="all", choices=["all", "build", "query"],
                    help="profiling aid (ncu): restrict the run to the resident build or to the query batch")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed build step and the last timed search batch returned as "
                         "DIR/<name>.npy (rank 0; the inputs are the same on every run with the same arguments)")
    args = ap.parse_args()
    if args.dump_outputs and (args.config != "C1" or args.impl != "ours"):
        ap.error("--dump-outputs is defined on our arm of config C1")
    if args.config != "C1":
        if args.steps is None:
            args.steps = 2
        if args.warmup is None:
            args.warmup = 1
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the CPU arm is defined on config C1 (the metric's configuration)"}))
            return
        import bench_configs
        bench_configs.run(args, CONFIGS[args.config], sys.modules[__name__])
        return
    if args.steps is None:
        args.steps = 5
    if args.warmup is None:
        args.warmup = 3
    if args.rows is None:
        args.rows = N_ROWS
    if args.impl == "reference":
        run_reference(args)
        return
    assert args.warmup >= 0 and args.steps >= 1
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import torch
    import torch.distributed as dist

    import lance_b200 as lb
    if lb.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (lance_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    lb.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
        from tools import dist_util
        dist_util.init_comm(dist)  # hands the NCCL unique id to lb2_comm_init on every rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        lb.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    n = args.rows
    # each rank owns an independent shard of n rows (weak scaling: no data-path collective)
    data_t, queries_t = device_dataset(torch, n, NQ, 1000 + rank, device)
    data_dev, q_dev = wrap_tensor(lb, data_t, np.float32), wrap_tensor(lb, queries_t, np.float32)
    params = lb.IvfBuildParams(num_partitions=NUM_PARTITIONS, num_sub_vectors=NUM_SUB_VECTORS, seed=7)
    row_base = rank * n  # global row id of this shard's first row
    rid_t = torch.arange(row_base, row_base + n, dtype=torch.int64, device=device)
    rid_dev = wrap_tensor(lb, rid_t, np.uint64)

    # ---- resident build: W warm-up, K timed ----------------------------------------------------
    for _ in range(args.warmup):
        lb.IvfPqIndex.build(data_dev, "l2", params, row_ids=rid_dev).close()
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    barrier()
    lb.launch_count(reset=True)
    t_wall0 = time.time()
    lb.timer_start()
    stats = last = None
    for i in range(args.steps):
        ix = lb.IvfPqIndex.build(data_dev, "l2", params, row_ids=rid_dev)
        stats = ix.stats
        if args.dump_outputs and i == args.steps - 1:
            last = ix   # exported after the timed window
        else:
            ix.close()
    ms_total = lb.timer_stop()
    barrier()
    t_wall1 = time.time()
    launches = lb.launch_count()
    dumped = {}
    if last is not None:
        dumped = build_outputs(last.export())
        last.close()
    ms_step = max_over_ranks(ms_total / args.steps)
    clocks = sampler.summary(t_wall0, t_wall1)
    value = world * n / (ms_step * 1e-3) / 1e6
    # one extra, UNTIMED step with a CUDA-event pair around every launch -> per-kernel breakdown
    lb.profile.reset()
    lb.profile.enable(True)
    lb.timer_start()
    lb.IvfPqIndex.build(data_dev, "l2", params, row_ids=rid_dev).close()
    ms_prof = lb.timer_stop()
    lb.profile.enable(False)

    # ---- strong scaling (world > 1): the SAME 1M-row workload split over the ranks ------------------
    strong = None
    if world > 1:
        ns = N_ROWS // world
        sd = wrap_tensor(lb, data_t[:ns], np.float32)
        sr = wrap_tensor(lb, rid_t[:ns], np.uint64)
        for _ in range(2):
            lb.IvfPqIndex.build(sd, "l2", params, row_ids=sr).close()
        barrier()
        lb.timer_start()
        for _ in range(args.steps):
            lb.IvfPqIndex.build(sd, "l2", params, row_ids=sr).close()
        s_ms = max_over_ranks(lb.timer_stop() / args.steps)
        strong = {"rows_total": ns * world, "rows_per_gpu": ns, "ms_per_step": s_ms,
                  "value": ns * world / (s_ms * 1e-3) / 1e6, "unit": "Mvec/s",
                  "note": "strong scaling: 1M rows in total; the 65 536-row training samples are sharded too"}

    # ---- kernel breakdown + roofline of the dominant kernel -------------------------------------
    hbm_peak, tensor_peak, peak_src = peaks()
    traffic = load_ncu_traffic()
    fams = {}
    for fam, (cnt, ms) in sorted(lb.profile.dump().items()):
        fams[fam] = {"launches_per_step": cnt, "ms_per_step": ms, "share": ms / ms_prof}
    dom = max((f for f in fams if f in KERNEL_BYTES), key=lambda f: fams[f]["ms_per_step"])
    per_launch_ms = fams[dom]["ms_per_step"] / fams[dom]["launches_per_step"]
    alg_bytes = KERNEL_BYTES[dom](65536, n)
    achieved = alg_bytes / (per_launch_ms * 1e-3) / 1e9
    roofline = {"kernel": dom, "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic.get(dom), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": per_launch_ms,
                "note": "dominant kernel of the build step by measured time (CUDA events on the library's stream); "
                        "bytes = SURVEY 8d: the rows' vectors read once (+ ids/codes written for the full pass)"}
    roofline_all = []
    for fam in sorted(f for f in fams if f in KERNEL_BYTES):
        pl = fams[fam]["ms_per_step"] / fams[fam]["launches_per_step"]
        ab = KERNEL_BYTES[fam](65536, n)
        roofline_all.append({"kernel": fam, "avg_launch_ms": pl, "algorithmic_bytes_per_launch": ab,
                             "achieved": ab / (pl * 1e-3) / 1e9, "frac": ab / (pl * 1e-3) / 1e9 / hbm_peak,
                             "traffic": traffic.get(fam)})

    if args.only == "build":
        if rank == 0:
            print(json.dumps({"only": "build", "ms_per_step": ms_step, "value": value, "kernels": fams}))
            if args.dump_outputs:
                dump_outputs(args.dump_outputs, dumped)
        return
    # ---- e2e build: pinned host -> device -> host, through the C ABI ---------------------------
    e2e = None
    pin = None
    if args.only == "all":
        pin = lb.PinnedArray((n, DIM), np.float32)
        import ctypes as C
        lb._lib.check(lb.lib().lb2_memcpy(C.c_void_p(pin.ptr), C.c_void_p(data_t.data_ptr()), C.c_size_t(n * DIM * 4)))

        # host result buffers are allocated once, like a caller's reusable (pinned) batch buffers
        pins = {"centroids": lb.PinnedArray((NUM_PARTITIONS, DIM), np.float32),
                "codebook": lb.PinnedArray((NUM_SUB_VECTORS, 256, DIM // NUM_SUB_VECTORS), np.float32),
                "part_offsets": lb.PinnedArray((NUM_PARTITIONS + 1,), np.uint64),
                "codes": lb.PinnedArray((n, NUM_SUB_VECTORS), np.uint8), "row_ids": lb.PinnedArray((n,), np.uint64)}
        host_out = {k: v.array for k, v in pins.items()}

        def e2e_step():
            ix = lb.IvfPqIndex.build(pin, "l2", params)
            parts = ix.export(out=host_out)
            ix.close()
            return parts
        for _ in range(min(args.warmup, 2) or 1):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            parts = e2e_step()
        barrier()
        e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)
        d2h = int(parts["codes"].nbytes + parts["row_ids"].nbytes + parts["part_offsets"].nbytes +
                  parts["centroids"].nbytes + parts["codebook"].nbytes)
        e2e = {"value": world * n / (e2e_ms * 1e-3) / 1e6, "unit": "Mvec/s", "ms_per_step": e2e_ms, "steps": args.steps,
               "h2d_bytes_per_step": n * DIM * 4, "d2h_bytes_per_step": d2h,
               "timing": "host wall clock around build + export (blocking calls), barrier + device sync on both sides"}

    # ---- query: QPS @ recall@10 ------------------------------------------------------------------
    ix = lb.IvfPqIndex.build(data_dev, "l2", params, row_ids=rid_dev)
    ids_t = torch.empty((NQ, TOPK), dtype=torch.int64, device=device)
    d_t = torch.empty((NQ, TOPK), dtype=torch.float32, device=device)
    ids_dev, d_dev = wrap_tensor(lb, ids_t, np.uint64), wrap_tensor(lb, d_t, np.float32)

    def search(nprobes=NPROBES):
        """row-sharded index: every rank scans its shard for all queries, the per-rank lists are exchanged and
        merged by (distance, row id) INSIDE the library (lb2_index_search_sharded)"""
        if world == 1:
            ix.search(q_dev, TOPK, nprobes, out=(ids_dev, d_dev))
        else:
            ix.search_sharded(q_dev, TOPK, nprobes, out=(ids_dev, d_dev))
    for _ in range(max(args.warmup, 1)):
        search()
    barrier()
    lb.profile.reset()
    lb.profile.enable(True)
    lb.timer_start()
    for _ in range(args.steps):
        search()
    q_ms = max_over_ranks(lb.timer_stop() / args.steps)
    barrier()
    lb.profile.enable(False)
    if args.dump_outputs:
        dumped.update(search_ids=ids_t.cpu().numpy(), search_dists=d_t.cpu().numpy())
    scan_name = "search:pq_scan_skew"                      # the conflict-free persistent scan (large batches)
    scan_cnt, scan_ms = lb.profile.get(scan_name)
    if scan_cnt == 0:
        scan_name = "search:pq_scan"
        scan_cnt, scan_ms = lb.profile.get(scan_name)
    q_host = queries_t.cpu().numpy()
    (ix.search if world == 1 else ix.search_sharded)(q_host, TOPK, NPROBES)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ids_h, d_h = (ix.search if world == 1 else ix.search_sharded)(q_host, TOPK, NPROBES)
    q_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / args.steps)
    # ground truth over ALL shards: every rank scores its shard exactly, the lists are merged the same way
    gt_local = ground_truth(torch, data_t, queries_t[:1000], TOPK, row_base=row_base)
    if world == 1:
        gt = gt_local
    else:
        gl = [torch.empty((1000, TOPK), dtype=torch.int64, device=device) for _ in range(world)]
        dist.all_gather(gl, torch.from_numpy(gt_local).to(device))
        cand = torch.cat(gl, 1)                                   # 1000 x (world * k) global row ids
        # exact distances of the candidates: each rank scores the ones it owns, max-reduce fills the rest
        own = (cand >= row_base) & (cand < row_base + n)
        loc = torch.where(own, cand - row_base, torch.zeros_like(cand))
        vec = data_t[loc.reshape(-1)].reshape(1000, -1, DIM)
        dd = ((vec - queries_t[:1000, None, :]) ** 2).sum(2)
        dd = torch.where(own, dd, torch.full_like(dd, -1.0))
        dist.all_reduce(dd, op=dist.ReduceOp.MAX)
        o = torch.topk(dd, TOPK, dim=1, largest=False).indices
        gt = torch.gather(cand, 1, o).cpu().numpy()

    def recall_of(ids):
        return float(np.mean([len(set(ids[i].tolist()) & set(gt[i].tolist())) / TOPK for i in range(1000)]))
    recall = recall_of(ids_h.astype(np.int64))
    # BASELINE.md's table: nprobes {1, 10, 50} x batch {1, 64, 10 000}, host queries in / host results out
    query_table = []
    if args.only == "all":
        for nprobes in (1, 10, 50):
            row = {"nprobes": nprobes}
            ih, _ = (ix.search if world == 1 else ix.search_sharded)(q_host, TOPK, nprobes)
            row["recall_at_10"] = recall_of(ih.astype(np.int64))
            for bsz, reps in ((1, 100), (64, 50), (NQ, max(2, args.steps))):
                fn = ix.search if world == 1 else ix.search_sharded
                for r in range(3):
                    fn(q_host[:bsz], TOPK, nprobes)
                barrier()
                t0 = time.perf_counter()
                for r in range(reps):
                    o = (r * bsz) % max(1, NQ - bsz)
                    fn(q_host[o:o + bsz], TOPK, nprobes)
                dt = max_over_ranks((time.perf_counter() - t0) / reps)
                row[f"batch_{bsz}"] = {"e2e_qps": bsz / dt, "latency_ms": dt * 1e3}
            query_table.append(row)
    # refine operating point (the reference's published curve uses refine_factor 5..10, BASELINE.md):
    # k*refine PQ candidates re-ranked with exact distances from the resident raw vectors
    query_refine = None
    if world == 1:
        REFINE = 10
        for _ in range(2):
            ix.search_refine(data_dev, q_dev, TOPK, NPROBES, REFINE, out=(ids_dev, d_dev))
        barrier()
        lb.timer_start()
        for _ in range(args.steps):
            ix.search_refine(data_dev, q_dev, TOPK, NPROBES, REFINE, out=(ids_dev, d_dev))
        r_ms = lb.timer_stop() / args.steps
        ids_r = ids_t[:1000].cpu().numpy()
        query_refine = {"qps": NQ / (r_ms * 1e-3), "recall_at_10": recall_of(ids_r), "nprobes": NPROBES, "k": TOPK,
                        "refine_factor": REFINE, "batch": NQ, "ms_per_batch": r_ms}
    # replica mode (SURVEY 8e search (i)): every GPU holds the WHOLE index and takes nq / N of the batch
    query_replica = None
    if world > 1:
        rep_t, _ = device_dataset(torch, n, 1, 1000, device)      # rank 0's shard on every rank
        ixr = lb.IvfPqIndex.build(wrap_tensor(lb, rep_t, np.float32), "l2", params)
        qs = NQ // world
        q_slice = wrap_tensor(lb, queries_t[rank * qs:(rank + 1) * qs], np.float32)
        oi = wrap_tensor(lb, ids_t[:qs], np.uint64)
        od = wrap_tensor(lb, d_t[:qs], np.float32)
        for _ in range(2):
            ixr.search(q_slice, TOPK, NPROBES, out=(oi, od))
        barrier()
        lb.timer_start()
        for _ in range(args.steps):
            ixr.search(q_slice, TOPK, NPROBES, out=(oi, od))
        rp_ms = max_over_ranks(lb.timer_stop() / args.steps)
        query_replica = {"qps": qs * world / (rp_ms * 1e-3), "queries_per_gpu": qs, "ms_per_batch": rp_ms,
                         "indexed_rows": n, "nprobes": NPROBES, "k": TOPK}
        ixr.close()
    # the scan's own ceiling is the shared-memory gather of the lookup tables (the index is L2 resident):
    # one 4-byte LUT read per (row, sub-vector), 32 banks x 4 B per SM and clock
    lookups = NQ * NPROBES * (n / NUM_PARTITIONS) * NUM_SUB_VECTORS
    smem_peak = 148 * 32 * (clocks["sm_mhz"] or 1965.0) * 1e6       # lookups / s
    scan_launch_ms = scan_ms / max(scan_cnt, 1)
    scan_bytes = NQ * NPROBES * (n / NUM_PARTITIONS) * NUM_SUB_VECTORS + NQ * DIM * 4
    query = {"qps": NQ / (q_ms * 1e-3), "e2e_qps": NQ / (q_e2e_ms * 1e-3), "recall_at_10": recall,
             "indexed_rows": world * n, "nprobes": NPROBES, "k": TOPK, "batch": NQ, "refine_factor": None,
             "ms_per_batch": q_ms,
             "roofline": {"kernel": scan_name, "bound": "shared-memory gather (LUT lookups)", "achieved": lookups / (scan_launch_ms * 1e-3) / 1e9,
                          "peak": smem_peak / 1e9, "unit": "Glookup/s", "frac": lookups / (scan_launch_ms * 1e-3) / smem_peak,
                          "hbm_equivalent_GBps": scan_bytes / (scan_launch_ms * 1e-3) / 1e9, "avg_launch_ms": scan_launch_ms,
                          "traffic": traffic.get(scan_name)}}
    sampler.stop()

    # ---- CPU baseline (rank 0, N=1 only) ----------------------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and pin is not None:
        from oracle import binding as ob
        threads = best_threads(ob)
        sec, nsteps, detail, _, how = cpu_steps(ob, pin.array, n, 1, 0, threads, 40.0)
        cpu_baseline = {"value": n / sec / 1e6, "unit": "Mvec/s", "cores": threads, "kind": "port", "sample": how, **detail}

    if rank == 0:
        line = {
            "metric": "ivf_pq_index_build_mvec_per_s", "value": value, "unit": "Mvec/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "rows_per_gpu": n, "sharding": "row shard per GPU; the k-means loops exchange their packed partial sums once per iteration (one global IVF/PQ model); transform local; search: per-rank lists exchanged + merged in the library",
                       "cache": "inputs (512 MB) larger than L2 (126 MB)", "k": TOPK, "nprobes": NPROBES},
            "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "build_phases_ms": {"ivf_train": stats.ms_ivf_train, "pq_train": stats.ms_pq_train, "transform": stats.ms_transform,
                                "group": stats.ms_group, "ivf_iters": stats.ivf_iters, "pq_iters_max": stats.pq_iters_max},
            "strong_scaling": strong,
            "kernels": fams, "roofline": roofline, "roofline_all": roofline_all, "query": query, "query_refine": query_refine,
            "query_table": query_table, "query_replica": query_replica, "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        from lance_b200 import parallel
        parallel.comm_destroy()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
