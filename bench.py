#!/usr/bin/env python
"""bench.py -- headline benchmark: queries/sec of brute-force top-K retrieval (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm: the reference's op sequence on host cores)

A "step" = one BruteForce.call: 4096 queries x (1M x 64) corpus -> top-100 (BASELINE configs[1]).  At N>1
the same corpus is row-sharded over the ranks (strong scaling): every rank scans its shard, ONE all-gather
of the per-shard (score, index) top-K (issued by libtfrs_b200.so's own NCCL communicator), merge on every rank.
Prints ONE JSON line (rank 0): value / e2e / roofline / cpu_baseline, plus `gather_gbs` and `adagrad_us` (the second
half of the BASELINE metric) at N = 1.  `--dump-outputs DIR` also writes the last timed step's scores and identifiers
to DIR/scores.npy and DIR/identifiers.npy.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N, d, Q, k)
    "cfg2": (1_000_000, 64, 4096, 100),    # BASELINE configs[1]: the config the metric is quoted on
    "cfg4": (8_000_000, 128, 4096, 100),   # BASELINE configs[3]: the 8-GPU sharded corpus
    "small": (131072, 64, 1024, 100),
}
METRIC = "queries/sec brute-force top-K (1Mx64 candidates)"


class ClockSampler(threading.Thread):
  """Samples nvidia-smi clocks / throttle reasons during the timed region."""

  def __init__(self, index: int):
    super().__init__(daemon=True)
    self.index = index
    self.rows = []
    self._stop = threading.Event()
    self.proc = None

  def run(self):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
      self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                    "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      for line in self.proc.stdout:
        if self._stop.is_set():
          break
        self.rows.append([x.strip() for x in line.split(",")])
    except Exception:
      pass

  def stop(self):
    self._stop.set()
    if self.proc is not None:
      try:
        self.proc.terminate()
      except Exception:
        pass

  def summary(self):
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      try:
        sm.append(float(r[0])); mx.append(float(r[1]))
        for n, v in zip(names, r[3:7]):
          if v.lower().startswith("active"):
            reasons.add(n)
      except Exception:
        continue
    if not sm:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
    sm_sorted = sorted(sm)
    busy = [x for x in sm_sorted if x > 0.5 * max(sm_sorted)] or sm_sorted
    return {"sm_mhz": busy[len(busy) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_arm_step(orc, q, c, k):
  """The reference's CPU op sequence (matmul -> top_k -> gather ids, factorized_top_k.py:603-607) under SURVEY 8d's
  protocol: torch CPU sgemm on all host threads + torch.topk(sorted=True), queries chunked by 512."""
  return orc.brute_force_torch(q, c, k, chunk=512)


def gen_corpus_block(torch, dev, b0, rows, d):
  """The synthetic corpus is defined block-wise (1M-row blocks, seed 1 + first row): every rank and the oracle leg
  regenerate exactly the same rows."""
  g = torch.Generator(device=dev)
  g.manual_seed(1 + b0)
  return torch.randn((rows, d), generator=g, device=dev)


def workload_string(name, N, d, Q, k, world):
  return (f"{name}: BruteForce top-{k}, {Q} queries x {N}x{d} corpus (N(0,1), seeds 1/2), "
          f"row-sharded over {world} GPU(s)")


def tune_cpu_threads(torch, orc, q512, c, k):
  """The CPU arm gets its best shot: MKL sgemm + torch.topk do not scale monotonically with threads on big hosts
  (128 threads were 2.5x SLOWER than 8 on this pool's box), so a few thread counts are tried on one 512-query
  chunk each and the fastest is used -- and reported."""
  n = os.cpu_count() or 1
  cands = sorted({t for t in (n, n // 2, n // 4, 32, 16, 8) if 1 <= t <= n}, reverse=True)
  best, best_rate, tried = cands[0], 0.0, {}
  for t in cands:
    torch.set_num_threads(t)
    cpu_arm_step(orc, q512[:128], c, k)   # warm the pools
    t0 = time.perf_counter()
    cpu_arm_step(orc, q512, c, k)
    rate = q512.shape[0] / (time.perf_counter() - t0)
    tried[t] = round(rate, 1)
    if rate > best_rate:
      best, best_rate = t, rate
  torch.set_num_threads(best)
  return best, best_rate, tried


def dump_outputs(dirname, scores, identifiers):
  """What a BruteForce caller receives from one step: scores [Q, k] as float32 and identifiers [Q, k] as float64 (exact for
  every integer id below 2**53).  4.9 MB in all at Q = 4096, k = 100."""
  import numpy as np
  os.makedirs(dirname, exist_ok=True)
  np.save(os.path.join(dirname, "scores.npy"), np.asarray(scores, np.float32))
  np.save(os.path.join(dirname, "identifiers.npy"), np.asarray(identifiers, np.float64))


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return 0
  import numpy as np
  import torch
  from oracle import oracle as orc
  N, d, Q, k = WORKLOADS[args.workload]
  # the same synthetic corpus / queries as the GPU arm (generated on the host: same distribution and seeds' role)
  c = np.random.default_rng(1).standard_normal((N, d), dtype=np.float32)
  q = np.random.default_rng(2).standard_normal((Q, d), dtype=np.float32)
  threads, rate, tried = tune_cpu_threads(torch, orc, q[:512], c, k)
  # bounded sample: the whole batch when --steps/--warmup of it fit in ~150 s, else the largest multiple of 512 that does
  if args.cpu_queries > 0:
    sample_q = min(Q, args.cpu_queries)
  else:
    fit = int(rate * 150.0 / (args.steps + min(args.warmup, 2))) // 512 * 512
    sample_q = max(512, min(Q, fit))
  qs = q[:sample_q]
  for _ in range(max(1, min(args.warmup, 2))):
    cpu_arm_step(orc, qs, c, k)
  t0 = time.perf_counter()
  for _ in range(args.steps):
    out = cpu_arm_step(orc, qs, c, k)
  dt = time.perf_counter() - t0
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, *out)
  value = sample_q * args.steps / dt
  world = int(os.environ.get("WORLD_SIZE", "1"))
  line = {
      "impl": "reference", "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps,
      "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
      "vs_baseline": None, "dtype": "f32", "data": "synthetic",
      "config": {"workload": workload_string(args.workload, N, d, Q, k, world),
                 "path": "CPU: torch sgemm (MKL/oneDNN) -> torch.topk(sorted) -> ids, 512-query chunks, best of several thread "
                         "counts (SURVEY 8d protocol; TensorFlow is not installable here, so this is the reference's op sequence "
                         "factorized_top_k.py:603-607 restated on torch CPU)",
                 "queries_per_step": sample_q, "threads_tried_qps": tried},
      "cpu_baseline": {"value": value, "unit": "queries/s", "cores": threads, "kind": "port",
                       "sample": f"{sample_q} of {Q} queries x {N} candidates x {args.steps} steps, {threads} of {os.cpu_count()} threads"},
      "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
      "gpu_launches": 0,
  }
  print(json.dumps(line))
  return 0


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=20)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
  ap.add_argument("--cpu-queries", type=int, default=0,
                  help="queries per CPU-arm step (0 = the whole batch; the in-line cpu_baseline leg uses a bounded sample)")
  ap.add_argument("--no-secondary", action="store_true", help="skip the gather / Adagrad / training-step figures")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-tensor-cores", action="store_true", help="force the exact CUDA-core path (debug)")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write the result of the last timed step to DIR/<name>.npy (inputs are seeded: two builds compare 1:1)")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  args.warmup = max(args.warmup, 3)
  if args.impl == "reference":
    return run_reference(args)

  import numpy as np
  import torch
  import torch.distributed as dist
  import recommenders_b200 as tfrs
  from recommenders_b200 import ops
  from recommenders_b200.layers.factorized_top_k import shard_bounds

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  if world > 1:
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=dev)

  N, d, Q, k = WORKLOADS[args.workload]
  lo, hi = shard_bounds(N, rank, world)
  # synthetic corpus: every rank generates the SAME full-corpus stream in 1M-row blocks and keeps its rows
  blocks = []
  for b0 in range(0, N, 1_000_000):
    s0, s1 = max(lo, b0), min(hi, b0 + min(1_000_000, N - b0))
    if s1 > s0:
      blk = gen_corpus_block(torch, dev, b0, min(1_000_000, N - b0), d)
      blocks.append(blk[s0 - b0:s1 - b0].clone())
      del blk
  corpus_local = torch.cat(blocks, 0) if len(blocks) > 1 else blocks[0]
  del blocks
  # NQ different query batches, rotated step by step (the timed steps never see the batch of the step before)
  NQ = 8
  g = torch.Generator(device=dev)
  g.manual_seed(2)
  query_batches = [torch.randn((Q, d), generator=g, device=dev) for _ in range(NQ)]
  queries = query_batches[0]

  layer = tfrs.layers.factorized_top_k.BruteForce(k=k)
  layer.use_tensor_cores = not args.no_tensor_cores
  if world > 1:
    layer.index_shard(corpus_local, lo, copy=False)
  else:
    layer.index(corpus_local)
  used_tc = layer._tc_index is not None and ops.tc_supported(Q, corpus_local.shape[0], d, k)

  def sync_all():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  sampler = ClockSampler(local_rank) if rank == 0 else None
  if sampler is not None:
    sampler.start()   # runs across all timed legs (nvidia-smi needs a few hundred ms before its first sample)

  # ---------------- device-resident throughput (`value`) ----------------
  for w in range(args.warmup):
    out = layer(query_batches[w % NQ])
  sync_all()
  launches0 = ops.launch_count()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  sync_all()
  e0.record()
  for st in range(args.steps):
    out = layer(query_batches[st % NQ])
  e1.record()
  torch.cuda.synchronize()
  last_batch = (args.steps - 1) % NQ
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, out[0].cpu().numpy(), out[1].cpu().numpy())
  launches = ops.launch_count() - launches0
  ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
  if world > 1:
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
  ms_total = float(ms)
  value = Q * args.steps / (ms_total * 1e-3)

  # ---------------- end-to-end through the public API with host buffers (`e2e`) ----------------
  # Every step copies ITS queries from pinned host memory and brings ITS [Q,k] result back to pinned host memory.  The
  # serving loop is pipelined two deep: H2D, the scan and D2H run on three streams, and the caller reads the result of
  # step i-2 (host-side wait on its D2H event) while step i is being submitted.  The scan itself stays on one stream.
  q_hosts = [qb.cpu().pin_memory() for qb in query_batches]
  DEPTH = 2
  s_host = [torch.empty((Q, k), dtype=torch.float32).pin_memory() for _ in range(DEPTH)]
  i_host = [torch.empty((Q, k), dtype=torch.int32).pin_memory() for _ in range(DEPTH)]
  q_dev = [torch.empty_like(queries) for _ in range(DEPTH)]
  main = torch.cuda.current_stream()
  h2d, d2h = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
  ev_h2d = [torch.cuda.Event() for _ in range(DEPTH)]
  ev_scan = [torch.cuda.Event() for _ in range(DEPTH)]
  ev_d2h = [torch.cuda.Event() for _ in range(DEPTH)]
  used = [False] * DEPTH

  def e2e_step(j):
    slot = j % DEPTH
    if used[slot]:
      ev_d2h[slot].synchronize()          # the caller consumes the result of step j - DEPTH here
      h2d.wait_event(ev_scan[slot])       # q_dev[slot] is free once that step's scan has read it
    with torch.cuda.stream(h2d):
      q_dev[slot].copy_(q_hosts[j % NQ], non_blocking=True)
      ev_h2d[slot].record(h2d)
    main.wait_event(ev_h2d[slot])
    s, i = layer(q_dev[slot])
    ev_scan[slot].record(main)
    d2h.wait_event(ev_scan[slot])
    with torch.cuda.stream(d2h):
      s_host[slot].copy_(s, non_blocking=True)
      i_host[slot].copy_(i, non_blocking=True)
      ev_d2h[slot].record(d2h)
    s.record_stream(d2h); i.record_stream(d2h)
    used[slot] = True

  def e2e_drain():
    for slot in range(DEPTH):
      if used[slot]:
        ev_d2h[slot].synchronize()

  for w in range(args.warmup):
    e2e_step(w)
  e2e_drain()
  sync_all()
  e0.record()
  for st in range(args.steps):
    e2e_step(st)
  main.wait_stream(d2h)
  e1.record()
  e2e_drain()
  torch.cuda.synchronize()
  ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
  if world > 1:
    dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
  e2e_value = Q * args.steps / (float(ms2) * 1e-3)

  # the same loop with no overlap (copy in, scan, copy out, host sync -- the latency of ONE request batch)
  def e2e_sync_step(j):
    q_dev[0].copy_(q_hosts[j % NQ], non_blocking=True)
    s, i = layer(q_dev[0])
    s_host[0].copy_(s, non_blocking=True)
    i_host[0].copy_(i, non_blocking=True)
    main.synchronize()
  for w in range(3):
    e2e_sync_step(w)
  sync_all()
  e0.record()
  for st in range(args.steps):
    e2e_sync_step(st)
  e1.record()
  torch.cuda.synchronize()
  ms2s = torch.tensor([e0.elapsed_time(e1)], device=dev)
  if world > 1:
    dist.all_reduce(ms2s, op=dist.ReduceOp.MAX)

  # ---------------- roofline of the dominant kernel (full filter pass), CUDA events inside the ABI ----------------
  roofline = None
  peaks = {}
  try:
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
  except Exception:
    pass
  if used_tc:
    ops.profile_enable(True)
    for st in range(args.steps):
      layer(query_batches[st % NQ])
    stage_ms, calls = ops.profile_read()
    ops.profile_enable(False)
    peak = peaks.get("bf16_tflops", 1590.0)
    which = "measured bf16_tflops (burst; the filter pass is timed alone)" if "bf16_tflops" in peaks else "fallback 1590"
    n_local = corpus_local.shape[0]
    flops = 2.0 * Q * n_local * d  # algorithmic: 2*Q*N*d per launch (SURVEY 8d: 128 MFLOP/query at N=1M,d=64)
    t_filter = stage_ms[2] / max(calls, 1) * 1e-3
    achieved = flops / t_filter / 1e12
    roofline = {"bound": "tensor", "kernel": "tc_scan_kernel<FILTER>", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                "frac": achieved / peak, "peak_source": which,
                # dram__bytes_read.sum + dram__bytes_write.sum of this kernel, per launch, from the committed ncu
                # --set full capture (profiles/, see profiles/README.md); only for the cfg2 single-GPU shape
                "traffic": TRAFFIC_CFG2_FILTER if (args.workload == "cfg2" and world == 1) else None, "traffic_unit": "bytes/launch",
                "whole_call_frac": (flops / (ms_total / args.steps * 1e-3) / 1e12) / peak,
                "stage_ms_per_call": {"qprep": stage_ms[0] / calls, "sample_pass+threshold": stage_ms[1] / calls,
                                      "filter_pass": stage_ms[2] / calls, "rescore+finalize": stage_ms[3] / calls}}

  # ---------------- parity of the timed outputs against the oracle (rank 0, a few rows, at EVERY N) ----------------
  checked = None
  if rank == 0:
    from oracle import oracle as orc
    rows = [0, Q // 2, Q - 1]
    s, i = out
    if world == 1:
      full = corpus_local.cpu().numpy()
    else:  # regenerate the whole corpus (same block-wise stream) for the oracle
      full = np.concatenate([gen_corpus_block(torch, dev, b0, min(1_000_000, N - b0), d).cpu().numpy()
                             for b0 in range(0, N, 1_000_000)], 0)
    es, ei = orc.topk_scan(query_batches[last_batch][rows].cpu().numpy(), full, k)
    checked = bool(np.array_equal(i[rows].cpu().numpy(), ei) and np.array_equal(s[rows].cpu().numpy(), es))
    del full

  # ---------------- second half of the BASELINE metric + training-step pieces (rank 0, N = 1) ----------------
  secondary = None
  if rank == 0 and world == 1 and not args.no_secondary:
    del layer, corpus_local
    torch.cuda.empty_cache()
    secondary = secondary_figures(torch, tfrs, ops, dev, peaks)
  if sampler is not None:
    sampler.stop()

  # ---------------- CPU baseline beside it (rank 0, N=1 only, bounded sample) ----------------
  cpu_baseline = None
  if rank == 0 and world == 1 and not args.no_cpu_baseline:
    from oracle import oracle as orc
    cq = 1024
    c_np = np.concatenate([gen_corpus_block(torch, dev, b0, min(1_000_000, N - b0), d).cpu().numpy() for b0 in range(0, N, 1_000_000)], 0)
    q_np = queries[:cq].cpu().numpy()
    threads, _, _ = tune_cpu_threads(torch, orc, q_np[:512], c_np, k)
    reps, t0 = 0, time.perf_counter()
    while reps < 2 or (time.perf_counter() - t0 < 12.0 and reps < 50):
      cpu_arm_step(orc, q_np, c_np, k); reps += 1
    dt = time.perf_counter() - t0
    cpu_baseline = {"value": cq * reps / dt, "unit": "queries/s", "cores": threads, "kind": "port",
                    "sample": f"{cq} queries x {N} candidates, {reps} reps (torch CPU sgemm -> topk, 512-query chunks, best thread count "
                              f"{threads} of {os.cpu_count()}: the reference's op sequence under SURVEY 8d's protocol)"}

  if rank == 0:
    line = {
        "metric": METRIC, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32 (fp16 tcgen05 screening, fp32 accumulate + exact fp32 re-scoring)" if used_tc else "f32",
        "data": "synthetic",
        "config": {"workload": workload_string(args.workload, N, d, Q, k, world),
                   "path": "tcgen05 screening + exact rescoring" if used_tc else "exact CUDA-core scan",
                   "l2": "inputs (fp16 image 128 MB + fp32 corpus 256 MB per 1M rows) exceed the 126 MB L2 between steps; "
                         f"{NQ} query batches rotate",
                   "parallelism": f"corpus-shard x{world}",
                   "collective": (None if world == 1 else
                                  ("tfrs_topk_sharded_f32: peer-memory exchange (NVLink P2P stores to the owner rank, owner merges 1/N of the "
                                   "queries, stores the result to every rank; epoch flags)" if getattr(layer._shard[1], "p2p", False) else
                                   "tfrs_topk_sharded_f32: one ncclAllGather issued by libtfrs_b200.so + replicated merge"))},
        "clocks": sampler.summary() if sampler is not None else None,
        "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": Q * d * 4, "d2h_bytes_per_step": Q * k * 8,
                "ms_per_step": float(ms2) / args.steps,
                "pipeline": "depth 2: H2D / scan / D2H on three streams; the caller reads step i-2's result while step i is submitted",
                "unpipelined_ms_per_step": float(ms2s) / args.steps},
        "gpu_launches": int(launches),
        "outputs_match_oracle": checked,
    }
    if roofline is not None:
      line["roofline"] = roofline
    if secondary is not None:
      line.update(secondary)
    if cpu_baseline is not None:
      line["cpu_baseline"] = cpu_baseline
    print(json.dumps(line))
  if world > 1:
    dist.barrier()
    dist.destroy_process_group()
  return 0


# dram__bytes_read.sum + dram__bytes_write.sum of tc_scan_kernel<FILTER> at cfg2 on one GPU, per launch
# (ncu --set full, profiles/r02_tc_scan_metrics.csv: 132.87 MB read + 31.38 MB written)
TRAFFIC_CFG2_FILTER = 164.25e6


def _time_ms(torch, fn, iters=20, warm=3):
  for _ in range(warm):
    fn()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize()
  e0.record()
  for _ in range(iters):
    fn()
  e1.record()
  torch.cuda.synchronize()
  return e0.elapsed_time(e1) / iters


def secondary_figures(torch, tfrs, ops, dev, peaks):
  """HBM GB/s of the embedding gather (the second half of BASELINE.json's metric: cfg5 and cfg3 shapes, uniform and
  Zipf ids) and the sparse-Adagrad / in-batch-softmax times of a cfg3 training step.  Algorithmic bytes per SURVEY 8d."""
  hbm = peaks.get("hbm_gbs", 6650.0)
  out = {}
  g = torch.Generator(device=dev); g.manual_seed(7)
  # cfg5: 26 tables [1M, 32], B = 65536 -> [B, 845 (ld 848)]
  tables = [torch.rand((1_000_000, 32), generator=g, device=dev) * 0.1 - 0.05 for _ in range(26)]
  act = torch.zeros((65536, 848), device=dev)
  bytes5 = 65536 * 26 * 32 * 4 * 2 + 26 * 65536 * 4

  def zipf(n_rows, n):
    u = torch.rand((n,), generator=g, device=dev, dtype=torch.float64)
    # inverse-CDF of a bounded Zipf(s = 1.05) on ranks 1..n_rows (continuous approximation), rank r -> row r - 1
    s = 1.05
    r = ((u * (n_rows ** (1 - s) - 1) + 1) ** (1 / (1 - s))).clamp(1, n_rows)
    return (r.to(torch.int64) - 1).to(torch.int32)

  def graph_ms(fn):
    """One call captured in a CUDA graph and replayed: the kernel's own time, not the Python binding's (26 tables of
    pointers per call cost more host time than the 90 us the kernel runs)."""
    fn(); torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
      fn()
    return _time_ms(torch, gr.replay)

  out["gather"] = {"hbm_peak_gbs": hbm, "peak_source": "measured hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650",
                   "timing": "CUDA-graph replays of one tfrs_gather_f32 call (device time; 4 id sets rotate for the uniform case)"}
  id_sets = [[torch.randint(0, 1_000_000, (65536,), generator=g, device=dev, dtype=torch.int32) for _ in range(26)] for _ in range(4)]
  ms5 = sum(graph_ms(lambda ids=ids: ops.gather(tables, ids, out=act)) for ids in id_sets) / len(id_sets)
  out["gather_gbs"] = bytes5 / ms5 / 1e6
  out["gather"]["cfg5_uniform"] = {"gbs": bytes5 / ms5 / 1e6, "us": ms5 * 1e3, "frac_of_hbm_peak": bytes5 / ms5 / 1e6 / hbm,
                                   "algorithmic_bytes": bytes5}
  zids = [zipf(1_000_000, 65536) for _ in range(26)]
  ms5z = graph_ms(lambda: ops.gather(tables, zids, out=act))
  out["gather"]["cfg5_zipf"] = {"gbs": bytes5 / ms5z / 1e6, "us": ms5z * 1e3, "frac_of_hbm_peak": bytes5 / ms5z / 1e6 / hbm,
                                "algorithmic_bytes": bytes5, "unique_ids_table0": int(zids[0].unique().numel()),
                                "note": "Zipf(1.05) ids, hot rows = low ids: staged in shared memory per CTA (bulk TMA) + L2 hits"}
  del id_sets, zids
  del tables, act
  torch.cuda.empty_cache()
  # cfg3: user table [10M, 64], item table [1M, 64], B = 16384; ids uniform and Zipf(1.05)
  ut = torch.rand((10_000_000, 64), generator=g, device=dev) * 0.1 - 0.05
  it = torch.rand((1_000_000, 64), generator=g, device=dev) * 0.1 - 0.05
  B = 16384
  for name, uid, iid in (("cfg3_uniform", torch.randint(0, 10_000_000, (B,), generator=g, device=dev, dtype=torch.int32),
                          torch.randint(0, 1_000_000, (B,), generator=g, device=dev, dtype=torch.int32)),
                         ("cfg3_zipf", zipf(10_000_000, B), zipf(1_000_000, B))):
    qo = torch.empty((B, 64), device=dev); co = torch.empty((B, 64), device=dev)
    ms3 = graph_ms(lambda: (ops.gather([ut], [uid], out=qo), ops.gather([it], [iid], out=co)))
    b3 = 2 * B * 64 * 4 * 2 + 2 * B * 4
    out["gather"][name] = {"gbs": b3 / ms3 / 1e6, "us": ms3 * 1e3, "frac_of_hbm_peak": b3 / ms3 / 1e6 / hbm, "algorithmic_bytes": b3,
                           "unique_ids": [int(uid.unique().numel()), int(iid.unique().numel())]}
    acc = torch.full_like(it, 0.1)
    grows = torch.randn((B, 64), generator=g, device=dev) * 1e-3
    msa = _time_ms(torch, lambda: ops.sparse_adagrad_(it, acc, iid, grows, 0.1))
    uniq = int(iid.unique().numel())
    ba = uniq * 64 * 4 * 4 + B * 64 * 4 + B * 4
    out["gather"][name]["adagrad_us"] = msa * 1e3
    out["gather"][name]["adagrad_gbs"] = ba / msa / 1e6
    if name == "cfg3_uniform":
      out["adagrad_us"] = msa * 1e3
    del acc
  q = ops.gather([ut], [uid]).requires_grad_(True); c = ops.gather([it], [iid]).requires_grad_(True)
  def step():
    q.grad = None; c.grad = None
    ops.inbatch_softmax_loss(q, c).backward()
  out["inbatch_softmax_fwd_bwd_us"] = _time_ms(torch, step, iters=10) * 1e3
  return out


if __name__ == "__main__":
  sys.exit(main())
