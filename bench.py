#!/usr/bin/env python
"""Benchmark of the knowledge-base RAG hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--config cfg2|cfg3|cfg4|cfg5] [--exchange fused|nccl] [--no-graph] [--no-encoder] [--no-parity]
                  [--dump-outputs DIR]

Default workload (config.workload) = BASELINE.json configs[1] ("cfg2"): a batch of 256 queries against a 1M x 768
bf16 corpus, top-32, synthetic data (seeded randn), corpus resident in HBM.  A "step" = one batch through the fused
similarity + top-k path.

  value     queries/s with the queries already in HBM, CUDA-event timed over K steps, max over ranks; the step
            (similarity kernel -> exact re-rank -> cross-shard merge) is captured once and replayed as one CUDA graph
            (--no-graph: plain stream launches)
  e2e       queries/s through the host-buffer C-ABI call (aur_search): pinned host queries -> H2D -> kernels -> D2H
  roofline  dominant kernel (simtopk_tc): algorithmic bytes / its CUDA-event duration vs MEASURED_PEAKS.json
  parity    the answer of the timed configuration checked IN THIS RUN against the oracle (streaming exact top-k over
            the very corpus that was searched): ids bit-exact, max |dscore|; the run fails if it does not hold
  cpu_baseline  a threaded fp32 flat cosine index (oracle port) on the host cores, rank 0, N=1 only

N > 1 (torchrun): the corpus is row-sharded over the ranks (strong scaling at cfg2/cfg4); each step = local search
-> cross-shard exchange -> merge.  --exchange fused (default): the exact-re-rank kernel stores its rows straight into
every rank's peer-mapped buffer over NVLink and the merge kernel waits on delivery flags (no collective call);
--exchange nccl: one NCCL all-gather of the packed (fp64 score, id) planes + device merge.

Other arms (run by hand, results under profiles/): --config cfg4 (1024 q x 10M x 1024, top-100), cfg5 (12.5M x 768 rows
per GPU, batch-512 queries with a concurrent encoder-ingest stream), cfg3 (bge-base encoder ingest, chunks/s).

--impl reference: the reference's CPU path for the same config, timed on the host cores (the Weaviate / t2v
containers cannot run here; the oracle port restates the flat cosine search, see oracle/streaming_topk.py).
"""

from __future__ import annotations

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

CHUNK = 125_000     # rows per generated corpus chunk (seed = base + global chunk index: any rank can regenerate any chunk)

CONFIGS = {
    # name: rows (total; "per_gpu" for weak scaling), dim, nq, k, metric text, workload text
    "cfg2": dict(rows=1_000_000, dim=768, nq=256, k=32, seed=1002, qseed=2002, scaling="strong",
                 metric="RAG queries/sec (batch-256, 1M x 768 bf16, top-32)",
                 workload="batch-256 queries, 1M x 768 bf16 corpus, top-32 (BASELINE.json configs[1])"),
    "cfg4": dict(rows=10_000_000, dim=1024, nq=1024, k=100, seed=1004, qseed=2004, scaling="strong",
                 metric="RAG queries/sec (batch-1024, 10M x 1024 bf16, top-100)",
                 workload="batch-1024 queries, 10M x 1024 bf16 corpus row-sharded over the GPUs, top-100 (BASELINE.json configs[3])"),
    "cfg5": dict(rows_per_gpu=12_500_000, dim=768, nq=512, k=32, seed=1005, qseed=2005, scaling="weak",
                 metric="RAG queries/sec (batch-512, 12.5M x 768 bf16 per GPU, top-32, concurrent streaming ingest)",
                 workload="100M x 768 bf16 corpus at 8 GPUs (12.5M rows per GPU), batch-512 queries, top-32, while an ingest "
                          "stream appends 512-chunk encoder batches (BASELINE.json configs[4])"),
}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(float(r[2]) for r in self.rows if len(r) >= 7)}


# ----------------------------------------------------------------------------- synthetic corpus
def gen_chunk(dev, seed: int, gchunk: int, rows: int, dim: int):
    """Chunk `gchunk` of the corpus as a bf16 device tensor; a pure function of (seed, gchunk, rows, dim)."""
    import torch

    g = torch.Generator(device=dev).manual_seed(seed + gchunk)
    return torch.randn(rows, dim, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)


def gen_queries(dev, qseed: int, nq: int, dim: int):
    import torch

    g = torch.Generator(device=dev).manual_seed(qseed)
    return torch.randn(nq, dim, generator=g, device=dev, dtype=torch.float32).to(torch.bfloat16)


def chunk_plan(n_rows: int):
    """[(global chunk index, first row, rows)] covering [0, n_rows)."""
    return [(c, lo, min(CHUNK, n_rows - lo)) for c, lo in enumerate(range(0, n_rows, CHUNK))]


def oracle_topk_of_chunks(dev, cfg, chunks, q_dev, qsel, extra_chunks=()):
    """Exact (ids, scores) top-k of the sampled queries over the given corpus chunks [(gchunk, first row, rows)] -- the
    per-rank half of a distributed check (every rank scans its own shard on the host, rank 0 merges)."""
    import torch

    from oracle.streaming_topk import StreamingTopk

    torch.set_num_threads(max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get("WORLD_SIZE", "1")))))   # (torchrun pins OMP to 1)
    Q = q_dev.float().cpu().numpy()[qsel]
    st = StreamingTopk(Q, cfg["k"])
    for gchunk, lo, m in chunks:
        rows = gen_chunk(dev, cfg["seed"], gchunk, m, cfg["dim"]).cpu().float().numpy()
        st.add_chunk(rows, np.arange(lo, lo + m, dtype=np.int64))
    for rows, ids in extra_chunks:
        st.add_chunk(rows, ids)
    oi, osc = st.finish()
    return oi, osc.astype(np.float64), st.rows


def verify_distributed(dist, world, rank, dev, cfg, my_chunks, q_dev, got_ids, got_sc, sample, extra_chunks=()):
    """Every rank computes the oracle's exact top-k over ITS shard (regenerated chunk by chunk, device -> host), the
    per-shard lists are gathered and merged by (score desc, id asc) on rank 0 -- the oracle's global answer without one
    process scanning 100M rows -- and compared with the engine's merged result."""
    nq = q_dev.shape[0]
    qsel = np.arange(nq) if sample is None or sample >= nq else np.linspace(0, nq - 1, sample).astype(np.int64)
    t0 = time.perf_counter()
    oi, osc, scanned = oracle_topk_of_chunks(dev, cfg, my_chunks, q_dev, qsel, extra_chunks)
    parts = [None] * world
    if world > 1:
        dist.all_gather_object(parts, (oi, osc, scanned))
    else:
        parts = [(oi, osc, scanned)]
    if rank != 0:
        return None
    k = cfg["k"]
    ids = np.concatenate([p[0] for p in parts], axis=1)
    sc = np.concatenate([p[1] for p in parts], axis=1)
    m_ids = np.full((len(qsel), k), -1, np.int64)
    m_sc = np.full((len(qsel), k), -np.inf, np.float32)
    for i in range(len(qsel)):
        valid = np.nonzero(ids[i] >= 0)[0]
        order = valid[np.lexsort((ids[i, valid], -sc[i, valid]))][:k]
        m_ids[i, :len(order)] = ids[i, order]
        m_sc[i, :len(order)] = sc[i, order].astype(np.float32)
    gi, gs = got_ids[qsel], got_sc[qsel]
    exact = bool(np.array_equal(gi, m_ids))
    fin = np.isfinite(m_sc)
    dmax = float(np.max(np.abs(gs[fin] - m_sc[fin]))) if fin.any() else 0.0
    out = {"ids_exact": exact, "max_dscore": dmax, "queries_checked": int(len(qsel)), "rows_scanned": int(sum(p[2] for p in parts)),
           "checker": "oracle.streaming_topk.StreamingTopk per shard on the host cores (exact re-score = oracle.cosine_topk.exact_cosine), "
                      "per-shard lists merged by (score desc, id asc)", "seconds": round(time.perf_counter() - t0, 1)}
    if not exact or dmax > 1e-3:
        out["id_mismatches"] = int((gi != m_ids).sum())
        raise SystemExit("PARITY FAILURE: " + json.dumps(out))
    return out


# ----------------------------------------------------------------------------- CPU arm
def cpu_flat_index(cfg, n_rows: int, threads: int = 0):
    """Threaded fp32 flat cosine index over the same synthetic shape (seeded on the host), normalised at import.
    Default thread count = physical cores (half the logical CPUs): sgemm on all 128 hyper-threads of the bench box
    measured 3x SLOWER than on its 64 cores, and both CPU legs must be the CPU's best."""
    import torch

    from oracle.streaming_topk import FlatIndexF32

    ix = FlatIndexF32(cfg["dim"], threads or max(1, (os.cpu_count() or 2) // 2))
    for gchunk, lo, m in chunk_plan(n_rows):
        g = torch.Generator().manual_seed(cfg["seed"] + gchunk)
        ix.add(torch.randn(m, cfg["dim"], generator=g, dtype=torch.float32))
    Q = torch.randn(cfg["nq"], cfg["dim"], generator=torch.Generator().manual_seed(cfg["qseed"]), dtype=torch.float32)
    return ix, Q


def cpu_pure_python_qps(dim: int, k: int, n_total: int, rows: int = 1500):
    """The reference's own arithmetic (pure-Python cosine, similarity.py:84-98 restated in oracle/ref_cosine.py): one
    query against `rows` rows, extrapolated to the corpus."""
    from oracle import ref_cosine as R

    rng = np.random.default_rng(7)
    C = [[float(x) for x in row] for row in rng.standard_normal((rows, dim))]
    q = [float(x) for x in rng.standard_normal(dim)]
    t0 = time.perf_counter()
    R.topk_python(q, C, k, clamp=False)
    dt = time.perf_counter() - t0
    return 1.0 / (dt * (n_total / rows))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS["cfg2" if args.config not in CONFIGS else args.config]
    n_rows = cfg.get("rows") or cfg["rows_per_gpu"] * max(1, args.gpus)
    n_rows = int(os.environ.get("AUR_BENCH_ROWS", n_rows))          # (the contract test shrinks it)
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    ix, Q = cpu_flat_index(cfg, n_rows)
    build_s = time.perf_counter() - t0
    for _ in range(args.warmup):
        ix.search(Q, cfg["k"])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ix.search(Q, cfg["k"])
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    v = cfg["nq"] / dt
    out = {
        "impl": "reference", "metric": cfg["metric"], "value": v, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt, "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "nq": cfg["nq"], "rows": n_rows, "dim": cfg["dim"], "k": cfg["k"]},
        "cpu_baseline": {"value": v, "unit": "queries/s", "cores": cores, "threads": ix.threads, "kind": "port",
                         "sample": f"every step = {cfg['nq']} queries x the full {n_rows} x {cfg['dim']} fp32 corpus (no extrapolation); "
                                   f"vectors L2-normalised once at import ({build_s:.1f} s, outside the timed region) like Weaviate; "
                                   "per step: threaded sgemm + threaded top-k per 125k-row block + merge (torch CPU)",
                         "note": "the reference's Weaviate 1.27.6 / t2v containers cannot run here; this is the oracle's threaded flat cosine index",
                         "reference_pure_python_queries_per_s": cpu_pure_python_qps(cfg["dim"], cfg["k"], n_rows)},
        "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------- GPU arms
def _dist_setup(args):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: aurora_b200 has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    return torch, dist, world, rank, local, dev


def _barrier(torch, dist, world):
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(torch, dist, world, dev, x: float) -> float:
    if world == 1:
        return x
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_search(args, name: str):
    """cfg2 / cfg4: batch search over a row-sharded corpus (strong scaling: the corpus is fixed, N splits it)."""
    torch, dist, world, rank, local, dev = _dist_setup(args)
    from aurora_b200 import _native as N
    from aurora_b200.engine import Index
    from aurora_b200.sharded import ShardedIndex, shard_bounds

    cfg = CONFIGS[name]
    n_total, dim, nq, k = cfg["rows"], cfg["dim"], cfg["nq"], cfg["k"]
    assert n_total % CHUNK == 0 and (n_total // CHUNK) % world == 0, "shards must be whole chunks"
    row_lo, row_hi = shard_bounds(n_total, world, rank)
    n_local = row_hi - row_lo
    ix = Index(dim, n_local, dtype="bf16", device=local)
    # the C ABI reads NULL as "the index's own stream"; torch's default stream is the legacy stream (handle 0x1)
    stream = torch.cuda.current_stream().cuda_stream or 1
    for gchunk, lo, m in chunk_plan(n_total):
        if row_lo <= lo < row_hi:
            rows = gen_chunk(dev, cfg["seed"], gchunk, m, dim)
            ix.add_dev(rows.data_ptr(), m, np.arange(lo, lo + m, dtype=np.int64), stream=stream)
    q_dev = gen_queries(dev, cfg["qseed"], nq, dim)
    sh = ShardedIndex(ix, dist, world, rank, local, nq_max=nq, k_max=k, exchange=args.exchange)

    def step_dev():
        return sh.search(q_dev, k, stream=stream)

    for _ in range(max(args.warmup, 3)):
        last_i, last_s = step_dev()
    _barrier(torch, dist, world)
    step_timed = step_dev
    use_graph = args.graph and args.exchange != "nccl"
    if use_graph:           # the step as one CUDA graph (one launch per step); stream launches if capture is refused
        try:
            replay, g_ids, g_sc = sh.capture(q_dev, k)
            step_timed = replay
            last_i, last_s = g_ids, g_sc
            for _ in range(3):
                replay()
        except Exception as e:      # pragma: no cover
            sys.stderr.write(f"[bench] CUDA graph capture failed ({e}); timing stream launches instead\n")
            use_graph = False
        _barrier(torch, dist, world)

    # ---- value: K steps, queries resident in HBM, CUDA events on the launching stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        _barrier(torch, dist, world)
        e0.record()
        for _ in range(args.steps):
            step_timed()
        e1.record()
        _barrier(torch, dist, world)
        # keep the sampler running a little so short runs still get a few samples under load
        # (local search only: a time-bounded loop must not contain collectives or exchanges)
        t_end = time.time() + 1.0
        tmp_s = torch.empty(nq, k, device=dev, dtype=torch.float32)
        tmp_i = torch.empty(nq, k, device=dev, dtype=torch.int64)
        while time.time() < t_end:
            ix.search_dev(q_dev.data_ptr(), nq, k, tmp_s.data_ptr(), tmp_i.data_ptr(), stream=stream)
        torch.cuda.synchronize()
    # every step writes its answer into the same two buffers and the sampler loop above writes elsewhere: they still
    # hold what the last timed step returned
    dump = {"topk_ids": last_i.cpu().numpy().astype(np.float64), "topk_scores": last_s.cpu().numpy()} if args.dump_outputs else None
    ms = _max_over_ranks(torch, dist, world, dev, e0.elapsed_time(e1) / args.steps)
    value = nq / (ms * 1e-3)

    # ---- per-phase device time of one step (library CUDA events on the same stream)
    ph = {"kernel_ms": [], "finalize_ms": [], "merge_ms": [], "total_ms": []}
    launches = 0
    for _ in range(min(args.steps, 20)):
        _barrier(torch, dist, world)
        out_i, out_s = step_dev()
        torch.cuda.synchronize()
        st = ix.stats()
        ph["kernel_ms"].append(st["last_kernel_ms"]); ph["finalize_ms"].append(st["last_finalize_ms"])
        ph["merge_ms"].append(st["last_merge_ms"]); ph["total_ms"].append(st["last_total_ms"])
        launches = st["last_launches"]
    phases = {a: float(np.median(b)) for a, b in ph.items()}
    kernel_ms = phases["kernel_ms"]
    kernel_name = N.KERNEL_NAMES[st["last_kernel"]]
    if use_graph:           # the answer that gets checked is the graph replay's
        _barrier(torch, dist, world)
        replay()
        torch.cuda.synchronize()
        out_i, out_s = g_ids, g_sc
    got_ids, got_sc = out_i.cpu().numpy(), out_s.cpu().numpy()
    if world > 1:     # every rank must hold the same merged answer
        ref = out_i.clone()
        dist.broadcast(ref, src=0)
        same = torch.tensor([int(torch.equal(ref, out_i))], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        if int(same.item()) != 1:
            raise SystemExit("PARITY FAILURE: ranks disagree on the merged top-k")

    # ---- e2e: host buffers, H2D + D2H inside the timed region
    q_host = q_dev.cpu().pin_memory()
    h_sc = torch.empty(nq, k, dtype=torch.float32).pin_memory()
    h_id = torch.empty(nq, k, dtype=torch.int64).pin_memory()
    import ctypes as C

    lib = N.load()

    def step_e2e():
        if world == 1:
            N.check(lib.aur_search(ix._h, C.c_void_p(q_host.data_ptr()), nq, k, None, None,
                                   C.c_void_p(h_sc.data_ptr()), C.c_void_p(h_id.data_ptr())))
        else:
            q_dev.copy_(q_host, non_blocking=True)
            oi, os_ = step_dev()
            h_sc.copy_(os_, non_blocking=True)
            h_id.copy_(oi, non_blocking=True)
            torch.cuda.synchronize()

    for _ in range(3):
        step_e2e()
    _barrier(torch, dist, world)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    e2e_ms = _max_over_ranks(torch, dist, world, dev, (time.perf_counter() - t0) * 1e3 / args.steps)
    e2e = nq / (e2e_ms * 1e-3)

    parity = None
    if not args.no_parity:
        my_chunks = [c for c in chunk_plan(n_total) if row_lo <= c[1] < row_hi]
        parity = verify_distributed(dist, world, rank, dev, cfg, my_chunks, q_dev, got_ids, got_sc, sample=None if name == "cfg2" else 48)
        if rank == 0 and world == 1:      # the host-buffer call's answer too
            if not (np.array_equal(h_id.numpy(), got_ids)):
                raise SystemExit("PARITY FAILURE: aur_search (host buffers) and aur_search_dev disagree")
    if rank != 0:
        sh.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    hbm_peak, tf_peak, peak_src = _peaks()
    # queries per kernel launch: 256 per CTA pair, up to four pairs side by side on the same tiles ("query super-blocks"),
    # fewer when ceil((k + 8) / tile sets) would exceed 4 (same rule as csrc/capi.cu search_enqueue)
    n_super = 4
    while n_super > 1 and -(-(k + 8) // (74 // n_super)) > 4:
        n_super -= 1
    nq_pass = min(nq, 256 * n_super)
    passes = -(-nq // nq_pass)
    shard_bytes = n_local * dim * 2 + nq_pass * dim * 2 + nq_pass * k * 8            # per kernel launch (one 256-query pass)
    flops_pass = 2.0 * nq_pass * n_local * dim
    if name == "cfg2":
        achieved = shard_bytes / (kernel_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak}
    else:   # nq >= 512: arithmetic intensity 1024 flop/B, the tensor pipe binds (SURVEY.md 8(d))
        achieved = flops_pass / (kernel_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                "hbm_gbs_per_launch": shard_bytes / (kernel_ms * 1e-3) / 1e9, "queries_per_launch": nq_pass}
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if os.path.exists(tpath) and world == 1 and name == "cfg2":
        try:
            traffic = json.load(open(tpath))["dram_bytes_per_launch"]
        except Exception:
            traffic = None
    roof.update({"traffic": traffic, "traffic_source": "profiles/dram_traffic.json (ncu --set full capture of this kernel at this shape)" if traffic else None,
                 "kernel": "simtopk_tc_kernel", "kernel_ms": kernel_ms, "launches_per_step": passes,
                 "algorithmic_bytes": shard_bytes, "algorithmic_flops": flops_pass, "peak_source": peak_src})
    exch = None if world == 1 else (
        "fused: finalize kernel stores (fp64 score, id) rows into every rank's IPC-mapped buffer over NVLink; merge kernel waits on delivery flags"
        if args.exchange == "fused" else "one NCCL all-gather of the packed (fp64 score, id) planes + device merge")
    out = {
        "metric": cfg["metric"], "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": cfg["scaling"],
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": cfg["workload"], "nq": nq, "rows": n_total, "rows_per_gpu": n_local, "dim": dim, "k": k,
                   "parallelism": f"row-shard x{world}",
                   "l2": f"shard ({n_local * dim * 2 / 1e6:.0f} MB) vs L2 (126 MB): " + ("larger, no flush needed" if n_local * dim * 2 > 2.5e8 else "NOT much larger than L2 at this N"),
                   "kernel": kernel_name, "exchange": exch,
                   "launch": "one CUDA graph per step (search + exact re-rank + exchange/merge captured once)" if use_graph else "stream launches"},
        "e2e": {"value": e2e, "unit": "queries/s", "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": nq * dim * 2, "d2h_bytes_per_step": nq * k * 12},
        "gpu_launches": launches * args.steps,
        "phases_ms": phases,
        "parity": parity,
        "roofline": roof,
        "clocks": clk.summary(),
    }
    sh.close()
    if world == 1:
        out["cpu_baseline"] = cpu_baseline_block(cfg, n_total)
        if name == "cfg2" and not args.no_encoder:
            ix.close()
            torch.cuda.empty_cache()
            out["encoder"], emb = encoder_leg(local, args.steps)
            if dump is not None:
                dump["encoder_embeddings"] = emb
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline_block(cfg, n_rows: int) -> dict:
    cores = os.cpu_count() or 1
    t0 = time.perf_counter()
    cix, cq = cpu_flat_index(cfg, min(n_rows, 1_000_000))
    build_s = time.perf_counter() - t0
    cix.search(cq, cfg["k"])
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        cix.search(cq, cfg["k"])
    dt = (time.perf_counter() - t0) / reps
    scale = n_rows / cix.rows
    return {
        "value": cfg["nq"] / (dt * scale), "unit": "queries/s", "cores": cores, "threads": cix.threads, "kind": "port",
        "sample": f"{reps} batches of {cfg['nq']} queries x {cix.rows} x {cfg['dim']} fp32 rows ({dt:.2f} s each, normalised at import in {build_s:.1f} s)"
                  + ("" if scale == 1 else f", scaled x{scale:.0f} to {n_rows} rows"),
        "reference_pure_python_queries_per_s": cpu_pure_python_qps(cfg["dim"], cfg["k"], n_rows),
        "note": "Weaviate 1.27.6 / t2v containers cannot run here; oracle port: threaded fp32 flat cosine index on all host cores",
    }


# ----------------------------------------------------------------------------- cfg5: concurrent ingest + query
def run_cfg5(args):
    torch, dist, world, rank, local, dev = _dist_setup(args)
    from aurora_b200 import _native as N
    from aurora_b200.encoder import Encoder, EncoderConfig
    from aurora_b200.engine import Index
    from aurora_b200.sharded import ShardedIndex

    cfg = CONFIGS["cfg5"]
    per_gpu = int(os.environ.get("AUR_BENCH_ROWS", cfg["rows_per_gpu"]))
    assert per_gpu % CHUNK == 0
    dim, nq, k = cfg["dim"], cfg["nq"], cfg["k"]
    n_total = per_gpu * world
    ingest_batch, ingest_room = 512, 512 * 400
    ix = Index(dim, per_gpu + ingest_room, dtype="bf16", device=local)
    stream = torch.cuda.current_stream().cuda_stream or 1
    chunks_per_gpu = per_gpu // CHUNK
    for c in range(chunks_per_gpu):
        g = rank * chunks_per_gpu + c
        rows = gen_chunk(dev, cfg["seed"], g, CHUNK, dim)
        ix.add_dev(rows.data_ptr(), CHUNK, np.arange(g * CHUNK, (g + 1) * CHUNK, dtype=np.int64), stream=stream)
        del rows
    q_dev = gen_queries(dev, cfg["qseed"], nq, dim)
    sh = ShardedIndex(ix, dist, world, rank, local, nq_max=nq, k_max=k, exchange=args.exchange)

    # ingest stream: bge-base dims encoder, 512 chunks per batch, token lengths ~N(384, 96) (cfg3's distribution)
    ecfg = EncoderConfig()
    rng = np.random.default_rng(1005 + rank)
    lens = np.clip(np.rint(rng.normal(384, 96, ingest_batch)), 16, 512).astype(np.int64)
    cu = np.zeros(ingest_batch + 1, np.int32); cu[1:] = np.cumsum(lens)
    tok = rng.integers(1000, ecfg.vocab, size=int(cu[-1])).astype(np.int32)
    tok[cu[:-1]] = 101; tok[cu[1:] - 1] = 102
    enc = Encoder(ecfg, max_tokens=int(cu[-1]) + 256, max_seqs=ingest_batch, device=local)
    enc.load_weights(random_bert_weights(ecfg, seed=7))
    id_base = 1 << 40                                         # appended ids: disjoint from the base corpus, unique per rank
    state = {"batches": 0, "stop": False, "err": None}

    def ingest_loop():
        try:
            while not state["stop"] and (state["batches"] + 1) * ingest_batch <= ingest_room:
                b = state["batches"]
                ids = id_base + (rank << 32) + np.arange(b * ingest_batch, (b + 1) * ingest_batch, dtype=np.int64)
                enc.encode_append(ix, tok, cu, ids)
                state["batches"] = b + 1
        except Exception as e:   # pragma: no cover
            state["err"] = e

    def step_dev():
        return sh.search(q_dev, k, stream=stream)

    for _ in range(max(args.warmup, 3)):
        step_dev()
    enc.encode_append(ix, tok, cu, id_base + (rank << 32) + (1 << 30) + np.arange(ingest_batch, dtype=np.int64))   # warm the encoder
    _barrier(torch, dist, world)

    # quiet rate first (no ingest), then the concurrent phase
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_dev()
    e1.record()
    _barrier(torch, dist, world)
    quiet_ms = _max_over_ranks(torch, dist, world, dev, e0.elapsed_time(e1) / args.steps)
    st_quiet = ix.stats()                                      # kernel time of an undisturbed step (roofline)

    rows_before = ix.stats()["rows"]
    th = threading.Thread(target=ingest_loop)
    with ClockSampler(local) as clk:
        _barrier(torch, dist, world)
        t_w0 = time.perf_counter()
        th.start()
        e0.record()
        for _ in range(args.steps):
            step_dev()
        e1.record()
        torch.cuda.synchronize()
        t_w1 = time.perf_counter()
        state["stop"] = True
        th.join()
        _barrier(torch, dist, world)
    if state["err"] is not None:
        raise state["err"]
    ms = _max_over_ranks(torch, dist, world, dev, e0.elapsed_time(e1) / args.steps)
    value = nq / (ms * 1e-3)
    wall = t_w1 - t_w0
    chunks_in = torch.tensor([float(state["batches"] * ingest_batch)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(chunks_in)
    ingest_rate = float(chunks_in.item()) / wall
    st = ix.stats()
    appended = st["rows"] - rows_before

    # ---- parity of a quiescent search over base corpus + everything that was appended (sampled queries)
    out_i, out_s = step_dev()
    torch.cuda.synchronize()
    parity = None
    if not args.no_parity:
        # every rank checks its own shard (base chunks + the tail its ingest thread appended, read back from HBM)
        from oracle import cosine_topk as O

        tail_rows, tail_ids = ix.read_rows(per_gpu, st["rows"] - per_gpu)
        extra = [(O.bf16_bits_to_f32(tail_rows), tail_ids)] if len(tail_ids) else []
        my_chunks = [(rank * chunks_per_gpu + c, (rank * chunks_per_gpu + c) * CHUNK, CHUNK) for c in range(chunks_per_gpu)]
        parity = verify_distributed(dist, world, rank, dev, cfg, my_chunks, q_dev, out_i.cpu().numpy(), out_s.cpu().numpy(), sample=16,
                                    extra_chunks=extra)
        if parity is not None:
            parity["appended_rows_rank0"] = int(len(tail_ids))
    if rank != 0:
        sh.close()
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    hbm_peak, tf_peak, peak_src = _peaks()
    n_local = st_quiet["rows"]
    flops_pass = 2.0 * nq * n_local * dim                      # one launch: 512 queries = two CTA-pair super-blocks
    kernel_ms = st_quiet["last_kernel_ms"]
    out = {
        "metric": cfg["metric"], "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": cfg["workload"], "nq": nq, "rows": n_total, "rows_per_gpu": per_gpu, "dim": dim, "k": k,
                   "parallelism": f"row-shard x{world}", "l2": "shard (19.2 GB) is larger than L2: no flush needed",
                   "ingest": f"one host thread per rank: aur_encode_append of {ingest_batch} chunks ({int(cu[-1])} tokens, bge-base dims) in a loop "
                             "on the encoder's stream while the query steps run; rows become visible when a batch has landed (published row count)"},
        "concurrent": {"queries_per_s_with_ingest": value, "queries_per_s_quiet": nq / (quiet_ms * 1e-3),
                       "ingest_chunks_per_s_all_ranks": ingest_rate, "rows_appended_rank0": int(appended),
                       "wall_s": wall},
        "e2e": {"value": value, "unit": "queries/s", "note": "device-resident queries (not a host-buffer call): see the cfg2 line for the H2D/D2H path",
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": st["last_launches"] * args.steps,
        "parity": parity,
        "roofline": {"bound": "tensor", "achieved": flops_pass / (kernel_ms * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                     "frac": flops_pass / (kernel_ms * 1e-3) / 1e12 / tf_peak, "kernel": "simtopk_tc_kernel (no ingest running, one launch = all 512 queries)",
                     "kernel_ms": kernel_ms, "hbm_gbs_per_launch": n_local * dim * 2 / (kernel_ms * 1e-3) / 1e9, "peak_source": peak_src, "traffic": None},
        "clocks": clk.summary(),
    }
    sh.close()
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- cfg3: encoder ingest
def random_bert_weights(cfg, seed: int = 7):
    h, i = cfg.hidden, cfg.inter
    shapes = {"word_emb": (cfg.vocab, h), "pos_emb": (cfg.max_pos, h), "type_emb": (cfg.type_vocab, h),
              "emb_ln_g": (h,), "emb_ln_b": (h,)}
    for l in range(cfg.layers):
        for kname, shp in {"wqkv": (3 * h, h), "bqkv": (3 * h,), "wo": (h, h), "bo": (h,), "ln1_g": (h,), "ln1_b": (h,),
                           "wi": (i, h), "bi": (i,), "wo2": (h, i), "bo2": (h,), "ln2_g": (h,), "ln2_b": (h,)}.items():
            shapes[f"l{l}.{kname}"] = shp
    wrng = np.random.default_rng(seed)
    return {name: ((1.0 + 0.1 * wrng.standard_normal(shp)) if name.endswith("_g") else 0.02 * wrng.standard_normal(shp)).astype(np.float32)
            for name, shp in shapes.items()}


def synth_chunks(cfg, n_seq: int, seed: int):
    rng = np.random.default_rng(seed)
    lens = np.clip(np.rint(rng.normal(384, 96, n_seq)), 16, 512).astype(np.int64)
    cu = np.zeros(n_seq + 1, np.int32)
    cu[1:] = np.cumsum(lens)
    tok = rng.integers(1000, cfg.vocab, size=int(cu[-1])).astype(np.int32)
    tok[cu[:-1]] = 101
    tok[cu[1:] - 1] = 102
    return tok, cu, lens


def run_cfg3(args):
    """Ingest: every rank encodes its own chunk batches (bge-base dims) and appends the pooled vectors to its shard
    (aur_encode_append); no collective on the data path; chunks/s summed over the ranks.  BASELINE.json configs[2]
    names 10M chunks; the timed region is K batches of 192 chunks per rank (stated in config)."""
    torch, dist, world, rank, local, dev = _dist_setup(args)
    from aurora_b200.encoder import Encoder, EncoderConfig
    from aurora_b200.engine import Index

    cfg = EncoderConfig()
    n_seq = 192
    tok, cu, lens = synth_chunks(cfg, n_seq, 1003 + rank)
    ix = Index(cfg.hidden, n_seq * (args.steps + args.warmup + 8), dtype="bf16", device=local)
    enc = Encoder(cfg, max_tokens=int(cu[-1]) + 256, max_seqs=n_seq, device=local)
    enc.load_weights(random_bert_weights(cfg, 7))
    nxt = [0]

    def step():
        ids = (rank << 40) + np.arange(nxt[0], nxt[0] + n_seq, dtype=np.int64)
        nxt[0] += n_seq
        enc.encode_append(ix, tok, cu, ids)

    for _ in range(max(args.warmup, 3)):
        step()
    _barrier(torch, dist, world)
    dev_ms = []
    with ClockSampler(local) as clk:
        _barrier(torch, dist, world)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step()
            dev_ms.append(enc.stats()["total_ms"])
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        _barrier(torch, dist, world)
    ms_dev = _max_over_ranks(torch, dist, world, dev, float(np.mean(dev_ms)))
    ms_wall = _max_over_ranks(torch, dist, world, dev, wall_ms)
    st = enc.stats()
    flops = st["gemm_flops"] + st["attn_flops"]
    from_text = text_ingest_leg(torch, dist, world, rank, dev, enc, ix, cfg, n_seq, lens, nxt)
    # parity: the vectors that landed in the shard vs the numpy BERT oracle on two chunks
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle import bert_encoder as B
        from oracle import cosine_topk as O

        w = random_bert_weights(cfg, 7)
        ocfg = B.BertConfig(hidden=cfg.hidden, layers=cfg.layers, heads=cfg.heads, inter=cfg.inter, vocab=cfg.vocab, max_pos=cfg.max_pos, pool="cls")
        wb = {kk: (O.round_to_bf16(v) if v.ndim == 2 else v) for kk, v in w.items()}
        short = np.argsort(lens)[:2]
        rows_bits, _ = ix.read_rows(0, n_seq)
        got = O.bf16_bits_to_f32(rows_bits)
        worst = 1.0
        for sidx in short:
            t = tok[cu[sidx]:cu[sidx + 1]]
            ref = B.encode(ocfg, wb, t, np.array([0, len(t)], np.int32))[0]
            g = got[sidx]
            worst = min(worst, float(np.dot(g, ref) / (np.linalg.norm(g) * np.linalg.norm(ref))))
        parity = {"min_cosine_vs_oracle_bert": worst, "chunks_checked": 2, "tolerance": "cosine >= 0.999 (bf16 activations + bf16 stored row)"}
        if worst < 0.999:
            raise SystemExit("PARITY FAILURE: " + json.dumps(parity))
    if rank != 0:
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    _, tf_peak, peak_src = _peaks()
    out = {
        "metric": "ingest chunks/sec through the bge-base-en encoder (bf16), sharded over the GPUs", "value": world * n_seq / (ms_dev * 1e-3),
        "unit": "chunks/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[2] shape: bge-base-en dims (H768 L12 A12 I3072), random-init bf16, token ids uniform in [1000, 30522), "
                               f"lengths ~N(384,96) in [16,512]; timed region = {args.steps} batches of {n_seq} chunks per rank "
                               f"({args.steps * n_seq * world} chunks, not the full 10M), each batch encoded and appended to the rank's shard",
                   "chunks_per_batch": n_seq, "tokens_per_batch": int(st["tokens"]), "parallelism": f"dp{world} (independent shards, no collective)"},
        "e2e": {"value": world * n_seq / (ms_wall * 1e-3), "unit": "chunks/s", "ms_per_step": ms_wall,
                "h2d_bytes_per_step": int(tok.nbytes + cu.nbytes + n_seq * 16), "d2h_bytes_per_step": 0,
                "note": "wall clock of aur_encode_append from host token ids (H2D inside), vectors stay in HBM (shard append)"},
        "gpu_launches": int(st["launches"] + 2) * args.steps,
        "from_text": from_text,
        "parity": parity,
        "roofline": {"bound": "tensor", "achieved": flops / (ms_dev * 1e-3) / 1e12, "peak": tf_peak, "unit": "TFLOP/s",
                     "frac": flops / (ms_dev * 1e-3) / 1e12 / tf_peak, "peak_source": peak_src, "traffic": None,
                     "note": "whole forward over real (unpadded) tokens, per GPU"},
        "clocks": clk.summary(),
    }
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def synth_vocab_and_texts(vocab_size: int, lens, seed: int):
    """A synthetic uncased vocabulary of `vocab_size` pieces (no vocab.txt ships offline) and one text per target token
    count: words drawn from the vocabulary, every ~9th word a two-piece word, some punctuation -- runbook-like."""
    rng = np.random.default_rng(seed)
    letters = np.array(list("abcdefghijklmnopqrstuvwxyz"))
    words = set()
    while len(words) < (vocab_size - 5) * 3 // 4:
        words.add("".join(rng.choice(letters, size=int(rng.integers(2, 9)))))
    words = sorted(words)
    tails = set()
    while len(tails) < vocab_size - 5 - len(words):
        tails.add("##" + "".join(rng.choice(letters, size=int(rng.integers(1, 5)))))
    pieces = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"] + words + sorted(tails)
    tails = sorted(tails)
    texts = []
    for n in lens:
        out, toks = [], 2
        while toks < n:
            w = words[int(rng.integers(len(words)))]
            if rng.random() < 0.11 and toks + 2 <= n:
                w += tails[int(rng.integers(len(tails)))][2:]; toks += 1      # (may tokenise differently; lengths are approximate)
            out.append(w); toks += 1
            if rng.random() < 0.08 and toks < n:
                out.append(","); toks += 1
        texts.append(" ".join(out))
    return pieces, texts


def text_ingest_leg(torch, dist, world, rank, dev, enc, ix, cfg, n_seq, lens, nxt) -> dict:
    """cfg3 FROM TEXT: the same batch shape as raw text -> C++ WordPiece (all host cores) -> encoder -> shard, one
    aur_encode_text_append call per batch; and the tokenizer alone (host-side chunks/s)."""
    from aurora_b200.encoder import TextEncoder
    from aurora_b200.wordpiece import NativeTokenizer

    pieces, texts = synth_vocab_and_texts(cfg.vocab, lens, 4242 + rank)
    tok = NativeTokenizer(pieces)
    te = TextEncoder(enc, tok)
    for i in np.nonzero(tok.lengths(texts) > 512)[0]:          # the generator's counts are approximate: like the token-id leg,
        w = texts[i].split(" ")                                # no chunk is longer than the position table
        while tok.lengths([" ".join(w)])[0] > 512:
            w.pop()
        texts[i] = " ".join(w)
    tk, cu_t = tok.encode_packed(texts, 512)
    big = texts * 8                                            # 1536 chunks: enough work for all cores
    tok.encode_packed(big, 512)
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        tok.encode_packed(big, 512)
    tok_rate = reps * len(big) / (time.perf_counter() - t0)
    t1 = time.perf_counter()
    tok.encode_packed(big, 512, threads=1)
    tok_rate_1 = len(big) / (time.perf_counter() - t1)

    def step():
        ids = (rank << 40) + np.arange(nxt[0], nxt[0] + n_seq, dtype=np.int64)
        nxt[0] += n_seq
        te.encode_append(ix, texts, ids)

    for _ in range(2):
        step()
    _barrier(torch, dist, world)
    t0 = time.perf_counter()
    k = 5
    for _ in range(k):
        step()
    torch.cuda.synchronize()
    ms = _max_over_ranks(torch, dist, world, dev, (time.perf_counter() - t0) * 1e3 / k)
    return {"chunks_per_s": world * n_seq / (ms * 1e-3), "ms_per_batch": ms, "tokens_per_batch": int(cu_t[-1]),
            "call": "aur_encode_text_append (C++ WordPiece on the host cores -> encoder forward -> shard append), text bytes in",
            "tokenizer_only_chunks_per_s": tok_rate, "tokenizer_only_chunks_per_s_1_thread": tok_rate_1,
            "host_cores": os.cpu_count() or 1, "vocab": "synthetic 30522-piece uncased vocabulary (no vocab.txt offline)",
            "text_bytes_per_batch": int(sum(len(t) for t in texts))}


def encoder_leg(device: int, steps: int):
    """Second hot-path row (SURVEY.md 8 a6/a11, BASELINE.json configs[2] shape): bge-base-en
    dimensions, random-init bf16 weights, cfg3 chunk lengths ~N(384, 96) clipped to [16, 512].
    Device time of the forward (CUDA events inside the library) over `steps` batches, the same call end to end with
    host token ids in / host vectors out, and transformers' BertModel on the host cores beside it.
    Returns (result, the vectors of the last timed batch)."""
    from aurora_b200.encoder import Encoder, EncoderConfig

    cfg = EncoderConfig()
    n_seq = 192
    tok, cu, lens = synth_chunks(cfg, n_seq, 1003)
    h, i = cfg.hidden, cfg.inter
    with Encoder(cfg, max_tokens=int(cu[-1]) + 256, max_seqs=n_seq, device=device) as enc:
        enc.load_weights(random_bert_weights(cfg, 7))
        for _ in range(3):
            enc.encode_packed(tok, cu)
        dev_ms, e2e_ms = [], []
        for _ in range(steps):
            t0 = time.perf_counter()
            emb = enc.encode_packed(tok, cu)
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
            dev_ms.append(enc.stats()["total_ms"])
        st = enc.stats()
    ms, ems = float(np.median(dev_ms)), float(np.median(e2e_ms))
    flops = st["gemm_flops"] + st["attn_flops"]
    _, peak_tf, peak_src = _peaks()
    out = {
        "workload": "bge-base-en dims (H768 L12 A12 I3072), random-init bf16, 192 chunks, lengths ~N(384,96) in [16,512]",
        "chunks": n_seq, "tokens": int(st["tokens"]), "ms_per_batch": ms, "chunks_per_s": n_seq / (ms * 1e-3),
        "tokens_per_s": st["tokens"] / (ms * 1e-3), "gpu_launches_per_batch": int(st["launches"]),
        "flops_per_batch": flops, "roofline": {"bound": "tensor", "achieved": flops / (ms * 1e-3) / 1e12, "peak": peak_tf,
                                               "unit": "TFLOP/s", "frac": flops / (ms * 1e-3) / 1e12 / peak_tf,
                                               "peak_source": peak_src,
                                               "note": "whole forward (GEMMs + attention + LayerNorm + pooling) over real (unpadded) tokens"},
        "e2e": {"chunks_per_s": n_seq / (ems * 1e-3), "ms_per_batch": ems, "h2d_bytes_per_batch": int(tok.nbytes + cu.nbytes),
                "d2h_bytes_per_batch": n_seq * h * 4},
    }
    try:   # host baseline: the class the reference's t2v sidecar runs, fp32, all host cores
        import torch
        from transformers import BertConfig as HFConfig, BertModel

        n_cpu = 16
        hf = BertModel(HFConfig(vocab_size=cfg.vocab, hidden_size=h, num_hidden_layers=cfg.layers, num_attention_heads=cfg.heads,
                                intermediate_size=i, max_position_embeddings=cfg.max_pos), add_pooling_layer=False).eval()
        smax = int(lens[:n_cpu].max())
        ids = np.zeros((n_cpu, smax), np.int64)
        mask = np.zeros((n_cpu, smax), np.int64)
        for s_ in range(n_cpu):
            ids[s_, :lens[s_]] = tok[cu[s_]:cu[s_ + 1]]
            mask[s_, :lens[s_]] = 1
        with torch.no_grad():
            hf(input_ids=torch.from_numpy(ids[:2]), attention_mask=torch.from_numpy(mask[:2]))
            t0 = time.perf_counter()
            hf(input_ids=torch.from_numpy(ids), attention_mask=torch.from_numpy(mask))
            dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n_cpu / dt, "unit": "chunks/s", "cores": os.cpu_count() or 1, "kind": "reference-stack",
                               "sample": f"{n_cpu} chunks, transformers.BertModel fp32 (torch {torch.get_num_threads()} threads), one padded batch ({dt:.2f} s)"}
    except Exception as e:   # transformers missing: report, do not fail the search line
        out["cpu_baseline"] = {"unavailable": str(e)[:120]}
    return out, emb


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path: str, arrays: dict) -> None:
    """--dump-outputs: one DIR/<name>.npy per array the timed path returned in its last timed step (ids as float64,
    exact below 2**53).  The inputs are seeded, so two builds run with the same arguments can be compared output for
    output."""
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES} byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--exchange", default="fused", choices=["fused", "nccl"], help="cross-shard step at N > 1")
    ap.add_argument("--graph", dest="graph", action="store_true", default=True,
                    help="replay the step as one captured CUDA graph (default; cfg2 / cfg4, not with --exchange nccl)")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="time plain stream launches instead")
    ap.add_argument("--no-encoder", action="store_true", help="skip the encoder leg of the N=1 cfg2 run")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle check (timing experiments only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy "
                    "(cfg2 / cfg4: topk_ids, topk_scores, and encoder_embeddings when the encoder leg runs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config not in ("cfg2", "cfg4")):
        ap.error("--dump-outputs covers the GPU search arms (cfg2, cfg4)")
    if args.impl == "reference":
        run_reference(args)
    elif args.config in ("cfg2", "cfg4"):
        run_search(args, args.config)
    elif args.config == "cfg5":
        run_cfg5(args)
    else:
        run_cfg3(args)


if __name__ == "__main__":
    main()
