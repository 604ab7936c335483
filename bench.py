#!/usr/bin/env python
"""bench.py -- ICP scans/sec on BASELINE.json's headline configuration (cfg2), plus the other measured rows of SURVEY 8(d/e).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path (one process per GPU)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle port + verbatim octree)

A "step" registers SUB x B independent OS1-128 scans per GPU (default 4 x 256 = 1024; 131 072 points each, drawn from 512
distinct scans per GPU, consecutive sub-batches never repeat an input) against the 1 M-point warehouse map with up to 20 ICP
iterations each -- exactly what LidarSLAM::Localization does per scan -- and ends with ONE all-gather of the per-scan result
rows, enqueued on the compute stream from device memory (so_set_pose_sink; no host hop before the collective).
`value` = scans/s with the scans already resident in HBM (so_register_batch_device); `e2e` = the same through
so_register_batch with HOST (pinned) scan buffers, H2D of the scans and D2H of the results inside the timed region.
Ranks shard the scan list (no data-path collective): weak scaling.

Extra blocks on the same JSON line (rank 0; all measured in this run):
  roofline   k-NN kernel of the ICP step against the measured HBM peak, algorithmic bytes as SURVEY 8(d) defines them
  knn_cfg5   BASELINE configs[4]: 10 M queries, k = 5, 5 M-point map, queries split over the N GPUs: GB/s, fraction of peak
  cfg4       BASELINE configs[3] literally: 1024 distinct scans, fixed total, sharded over the N GPUs, one gather (strong scaling)
  wide_prior the same batch kernel path with +-0.5 m / +-5 deg priors (ICP iterations 4+ exercised)
  latency    single-scan so_register (host scan in -> pose out) on the shipped VLP-16 configuration and on cfg2
  live       live-SLAM loop: so_register + so_map_add_scan per scan on a growing ~1 M-point map
  cpu_baseline  the oracle (reference octree verbatim + restated fits / solver) on one host thread, bounded sample
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the tree may be read-only: numba's compiled-function cache (synth.py) goes to a temporary directory
os.environ.setdefault("NUMBA_CACHE_DIR", os.path.join(tempfile.gettempdir(), f"superodom_b200_numba_cache_{os.getuid()}"))

METRIC = "ICP scans/sec (128-beam, 1M-pt map)"
UNIT = "scans/s"
WORKLOAD = "cfg2: OS1-128 synthetic scans (131072 pts) vs 1M-pt local map, 20 ICP iters, planeRes 0.2, all points active"
CFG4_TOTAL = 1024
DISTINCT = 512                                   # distinct scans per GPU behind the weak-scaling step (two calls' worth: consecutive calls never repeat an input)
# SURVEY 8(d): algorithmic bytes of the k-NN = 16 B query read + k * 8 B result (u32 id + f32 d2) per query, + the map once.
KNN_BYTES_PER_QUERY = 16 + 5 * 8
# ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of ONE k_knn_scan launch / its queries (profiles/README.md says
# which capture; None where no capture of the current kernel is committed)
NCU_DRAM_BYTES_PER_QUERY = {"k_knn_scan": 76.8, "k_knn_fit": None}      # profiles/ncu_prof_r2t_metrics.csv: (26.78 MB read + 53.74 MB written) / 1 048 576 queries
DUMP_MAX_BYTES = 64 << 20


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with NVML while the timed region runs.  One sampler per job (rank 0) polls every
    GPU of the job: NVML is initialised BEFORE the warm-up (nvmlInit enumerates all GPUs and holds driver locks for a long
    time -- inside a timed region, in N processes at once, it stalled kernel launches), then polls at a low rate."""

    def __init__(self, indices, period: float = 0.02):
        super().__init__(daemon=True)
        self.indices, self.period, self.samples, self.reasons, self.stop_flag, self.max_mhz = list(indices), period, [], set(), False, None
        self.window = None
        self.nv, self.handles = None, []
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv = nv
            self.handles = [self._handle(nv, i) for i in self.indices]
            self.max_mhz = min(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM) for h in self.handles)
        except Exception as e:      # NVML missing: report that rather than fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    @staticmethod
    def _handle(nv, cuda_index):
        """NVML handle of CUDA device `cuda_index` (CUDA_VISIBLE_DEVICES may renumber): by UUID, else by index."""
        try:
            import torch
            u = str(torch.cuda.get_device_properties(cuda_index).uuid)
            return nv.nvmlDeviceGetHandleByUUID(u if u.startswith("GPU-") else "GPU-" + u)
        except Exception:
            return nv.nvmlDeviceGetHandleByIndex(cuda_index)

    def run(self):
        nv = self.nv
        if nv is None:
            return
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        try:
            while not self.stop_flag:
                if self.window is not None:                      # only while a timed region is open
                    mhz = min(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM) for h in self.handles)
                    self.samples.append(mhz)
                    for h in self.handles:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                        for bit, name in names.items():
                            if r & bit:
                                self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def open(self):
        self.window = time.perf_counter()

    def close(self):
        self.window = None

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples), "gpus_sampled": len(self.handles)}


def bind_to_gpu_numa(local: int) -> str:
    """Pin this rank (and therefore the first-touch placement of its pinned staging buffers) to the CPUs NVML reports as local
    to its GPU: GPUs 4-7 of the 8-GPU box hang off NUMA node 1, and an unbound rank stages through the far socket."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = ClockSampler._handle(nv, local)
        words = nv.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"{len(cpus)} cpus [{min(cpus)}..{max(cpus)}]"
    except Exception as e:
        return f"unbound ({type(e).__name__})"
    return "unbound"


def make_inputs(first_scan: int, n_scans: int):
    """Seeded synthetic cfg2 inputs (SURVEY 8d).  The generated arrays are kept under SO_BENCH_CACHE (default a /tmp
    directory) so that back-to-back runs on one box (N = 1, 2, 4, 8) do not repeat the CPU-side synthesis; the cache holds
    inputs only, never results."""
    from superodom_b200 import synth
    cache = os.environ.get("SO_BENCH_CACHE", "/tmp/superodom_b200_bench_inputs")       # "" disables
    path = os.path.join(cache, f"cfg2_{first_scan}_{n_scans}.npz") if cache else None
    if path and os.path.exists(path):
        try:
            z = np.load(path)
            nn = z["n"]
            offs = np.concatenate([[0], np.cumsum(nn)])
            flat = z["flat"]
            return z["map"], [flat[offs[i]:offs[i + 1]] for i in range(len(nn))], z["priors"], z["truths"]
        except Exception as e:                                 # unreadable / half-written cache: regenerate
            print(f"[bench] input cache {path} unusable ({type(e).__name__}), regenerating", file=sys.stderr)
    scene, map_xyzi = synth.make_map_for("cfg2")
    scans, priors, truths = [], [], []
    for i in range(first_scan, first_scan + n_scans):
        c = synth.make_case_on(scene, map_xyzi, "cfg2", i)
        scans.append(c["scan_xyzi"])
        priors.append(c["pose_prior"])
        truths.append(c["pose_true"])
    if path:
        try:
            os.makedirs(cache, exist_ok=True)
            tmp = path + f".{os.getpid()}.tmp.npz"
            np.savez(tmp, map=map_xyzi, flat=np.concatenate(scans, 0), n=np.array([len(x) for x in scans]), priors=np.stack(priors), truths=np.stack(truths))
            os.replace(tmp, path)                              # atomic: ranks / back-to-back runs may race on the same file
        except Exception as e:                                 # read-only or full /tmp: the cache is only a convenience
            print(f"[bench] input cache not written ({type(e).__name__}: {e})", file=sys.stderr)
    return map_xyzi, scans, np.stack(priors), np.stack(truths)


def cfg5_queries(map_xyzi: np.ndarray, first: int, count: int, block: int = 125_000) -> np.ndarray:
    """cfg5 queries [first, first+count) of the 10 M: query i = map point (i mod M) + N(0,(0.1 m)^2), drawn block by block
    (seed 3000 + block index) so that any rank can produce exactly its slice, float4 with w = 0."""
    M = len(map_xyzi)
    out = np.zeros((count, 4), np.float32)
    b0, b1 = first // block, (first + count - 1) // block
    for b in range(b0, b1 + 1):
        lo, hi = max(first, b * block), min(first + count, (b + 1) * block)
        rng = np.random.default_rng(3000 + b)
        noise = rng.normal(0, 0.1, size=(block, 3)).astype(np.float32)
        idx = (np.arange(lo, hi) % M)
        out[lo - first:hi - first, :3] = map_xyzi[idx, :3] + noise[lo - b * block:hi - b * block]
    return out


def dump_outputs(out_dir, results, **extra):
    """Write what the last timed step returned as out_dir/<name>.npy (float64): one row per scan, scans in call order, for every
    field of the result struct except the timings and padding, plus `extra` arrays.  Above DUMP_MAX_BYTES a fixed (seed 0) sample
    of the scans is written; scan_index.npy names the scans of the rows either way."""
    fields = [f for f, _ in type(results[0])._fields_ if not f.startswith("time_") and not f.endswith("_")]
    per_scan = {f: np.array([np.asarray(getattr(r, f), dtype=np.float64).reshape(-1) for r in results]) for f in fields}
    index = np.arange(len(results))
    budget = DUMP_MAX_BYTES - sum(np.asarray(a).nbytes for a in extra.values())
    row_bytes = sum(a.shape[1] * 8 for a in per_scan.values()) + 8
    if len(results) * row_bytes > budget:
        index = np.sort(np.random.default_rng(0).choice(len(results), max(0, budget // row_bytes), replace=False))
    arrays = {f: (a[index, 0] if a.shape[1] == 1 else a[index]) for f, a in per_scan.items()}
    arrays["scan_index"] = index
    arrays.update(extra)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ----------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's CPU implementation of the path on the host cores: oracle/_ref (reference octree.h compiled
    verbatim + restated fits/solver) when present, else the oracle port.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    sample = max(1, args.ref_scans)
    map_xyzi, scans, priors, truths = make_inputs(0, sample)
    ref = O.has_ref_octree()
    om = O.OracleMap(map_xyzi, ref_octree=ref)
    mode = 2 if ref else 0

    def step():
        res = [om.register(s, p, 0.2, 20, 0, knn_mode=mode, n_threads=cores, skip_map_checks=True) for s, p in zip(scans, priors)]
        assert all(r.status == 0 for r in res)
        return res
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    v = sample * args.steps / dt
    kind = "reference-octree+port" if ref else "port"
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": WORKLOAD, "scans_per_step": sample},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference-octree+port" if ref else "port",
                             "sample": f"{sample} cfg2 scans per step; k-NN = the reference's flann/octree.h compiled verbatim ({kind}); fits, Ceres LM and "
                                       f"covariance = the oracle's restatement; per-point loop on {cores} threads (a variant more generous than "
                                       f"the reference's serial loop)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from superodom_b200 import api, replay, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries the ONE JSON line and nothing else: libraries that print there (NCCL's version banner does, whatever
    # NCCL_DEBUG_FILE says) are sent to stderr at the file-descriptor level; the line goes out through the saved descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    t_phase = [time.perf_counter()]

    def phase(label):                                  # wall-clock of the untimed set-up phases, to stderr
        now = time.perf_counter()
        print(f"[bench rank {rank}] {label}: {now - t_phase[0]:.1f} s", file=sys.stderr, flush=True)
        t_phase[0] = now

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local)
    # input synthesis (numba ray casting) must not oversubscribe the host when several ranks generate at once
    os.environ.setdefault("NUMBA_NUM_THREADS", str(max(1, min(16, len(os.sched_getaffinity(0)) // max(1, min(world, 4))))))
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # stdout carries the one JSON line only (NCCL logs there by default)
        dist.init_process_group("nccl", device_id=dev)
    phase(f"import torch + process group (cpu affinity: {numa})")

    B, SUB = args.batch, args.sub_batches
    per_step = B * SUB                                               # scans per step per GPU
    # scan lists: this rank's shard of the 1024-scan cfg4 replay first, extra distinct scans after it when the shard is short
    c4b, c4e = replay.shard_range(CFG4_TOTAL, rank, world)
    n_shard = c4e - c4b if not args.no_cfg4 else 0
    map_xyzi, scans, priors, truths = make_inputs(c4b, n_shard) if n_shard else (None, [], np.zeros((0, 7)), np.zeros((0, 7)))
    n_distinct = max(B, min(DISTINCT, per_step))
    if n_shard < n_distinct:
        m2, s2, p2, t2 = make_inputs(CFG4_TOTAL + rank * n_distinct, n_distinct - n_shard)
        map_xyzi = m2 if map_xyzi is None else map_xyzi
        scans, priors, truths = scans + s2, np.concatenate([priors, p2]), np.concatenate([truths, t2])
    phase(f"synthetic inputs ({len(scans)} scans)")
    n_points = np.array([len(s) for s in scans], np.uint32)
    offs = np.concatenate([[0], np.cumsum(n_points.astype(np.int64))])
    flat = np.ascontiguousarray(np.concatenate(scans, 0))

    ctx = api.Context(device=local, max_map_points=len(map_xyzi) + 1024, max_scan_points=int(n_points.max()), max_batch=B, plane_res=0.2)
    stream = torch.cuda.Stream(device=dev)             # a real (non-legacy) stream shared by torch events and the library
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    ctx.map_set_points(map_xyzi)
    n_dev = int(offs[n_distinct])
    d_scans = torch.from_numpy(flat[:n_dev]).to(dev)
    h_pinned = torch.from_numpy(flat).pin_memory()     # first touch on the GPU-local NUMA node (bind_to_gpu_numa)
    h_view = h_pinned.numpy()
    sink = torch.zeros((per_step, replay.ROW), dtype=torch.float64, device=dev)
    gathered = torch.zeros((world * per_step, replay.ROW), dtype=torch.float64, device=dev)
    ctx.set_pose_sink(sink.data_ptr(), per_step, 0)

    def sub_range(k):                                  # scans of sub-batch k of a step: cycles through the distinct set
        g = (k * B) % n_distinct
        return g, g + B

    def step_device():
        ctx.set_pose_sink(sink.data_ptr(), per_step, 0)
        res = []
        for k in range(SUB):
            a, b = sub_range(k)
            res.append(ctx.register_batch_device(d_scans.data_ptr() + int(offs[a]) * 16, n_points[a:b], priors[a:b], 20, 0, skip_map_checks=True))
        replay.gather_rows(sink, out=gathered)         # ONE collective per step, enqueued behind the last optimiser step; nobody waits for it
        return res

    def step_host():
        ctx.set_pose_sink(sink.data_ptr(), per_step, 0)
        res = []
        for k in range(SUB):
            a, b = sub_range(k)
            res.append(ctx.register_batch(h_view[offs[a]:offs[b]], n_points[a:b], priors[a:b], 20, 0, skip_map_checks=True))
        replay.gather_rows(sink, out=gathered)
        return res

    def timed(step_fn, steps, readback=False):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            res = step_fn()
        if readback:
            host_rows = gathered.cpu()                 # the replay's gathered result, read once
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), res

    sampler = ClockSampler(range(world)) if rank == 0 else None      # torchrun on one node: local GPU indices 0..world-1
    if sampler:
        sampler.start()
    phase("context, map upload, pinned staging, NVML init")
    warm = max(args.warmup, 3)
    for _ in range(warm):
        res = step_device()
    torch.cuda.synchronize()
    phase("warm-up steps")
    # correctness guard: the timed thing really registers the scans (cm-level agreement with ground truth), and the gathered rows
    # carry the same poses the per-call result structs do
    for k, rk in enumerate(res):
        a, b = sub_range(k)
        err = np.linalg.norm(np.array([list(r.pose) for r in rk])[:, :3] - truths[a:b, :3], axis=1)
        assert all(r.status == 0 for r in rk) and err.max() < 0.05, (err.max(), [r.status for r in rk])
    g_pose, g_status, g_iters = replay.unpack_rows(gathered.cpu().numpy(), world * per_step, world)
    mine = g_pose[rank * per_step:(rank + 1) * per_step]
    assert np.array_equal(mine, np.array([list(r.pose_opt) for rk in res for r in rk])) and (g_status == 0).all()
    icp_mean = float(np.mean([r.n_iterations for rk in res for r in rk]))

    ctx.kernel_launches(reset=True)
    if sampler:
        sampler.open()
    ms, res = timed(step_device, args.steps)
    if sampler:
        sampler.close()
    launches = ctx.kernel_launches()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [r for rk in res for r in rk], gathered_rows=gathered.cpu().numpy())
    n_total = per_step * world
    value = n_total * args.steps / (ms * 1e-3)

    for _ in range(2):
        step_host()
    ctx.bytes_copied(reset=True)
    if sampler:
        sampler.open()
    ms_e2e, res_host = timed(step_host, args.steps, readback=True)
    # the host-buffer path (growing upload chunks, two streams) must give the very poses the device-resident path gave for the
    # same scans: a scan's result never depends on the batch or chunk it travels in (reported, not asserted)
    try:
        same_bits = bool(np.array_equal(np.array([list(r.pose_opt) + [r.n_iterations] for rk in res_host for r in rk]),
                                        np.array([list(r.pose_opt) + [r.n_iterations] for rk in res for r in rk])))
    except Exception as e:                             # evidence only: never fatal to the measurement
        same_bits = f"not compared: {type(e).__name__}"
    clocks = sampler.result() if sampler else None
    h2d, d2h = ctx.bytes_copied()
    d2h += gathered.numel() * 8
    e2e = n_total * args.steps / (ms_e2e * 1e-3)
    # what the host link gives a plain pinned copy on this box (after the timed regions): the denominator the e2e / value gap is read against
    nb_link = min(int(offs[n_distinct]) * 16, 512 << 20)
    link_dst = torch.empty(nb_link, dtype=torch.uint8, device=dev)
    link_src = h_pinned.view(-1).view(torch.uint8)[:nb_link]
    link_dst.copy_(link_src, non_blocking=True)
    torch.cuda.synchronize()
    l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0.record()
    for _ in range(3):
        link_dst.copy_(link_src, non_blocking=True)
    l1.record()
    torch.cuda.synchronize()
    h2d_gbs = 3 * nb_link / (l0.elapsed_time(l1) * 1e-3) / 1e9
    del link_dst
    phase("timed regions (device-resident + e2e)")

    # ---- cfg4 as BASELINE.json states it: 1024 distinct scans, fixed total, sharded, one gather (strong scaling) -------------------
    cfg4 = None
    if n_shard:
        cap4 = replay.shard_cap(CFG4_TOTAL, world)
        sink4 = torch.zeros((cap4, replay.ROW), dtype=torch.float64, device=dev)
        all4 = torch.zeros((world * cap4, replay.ROW), dtype=torch.float64, device=dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.set_pose_sink(sink4.data_ptr(), cap4, 0)
        for a in range(0, n_shard, B):
            b = min(a + B, n_shard)
            ctx.register_batch(h_view[offs[a]:offs[b]], n_points[a:b], priors[a:b], 20, 0, skip_map_checks=True)
        replay.gather_rows(sink4, out=all4)
        rows4 = all4.cpu()
        e1.record()
        torch.cuda.synchronize()
        t4 = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        p4, s4, i4 = replay.unpack_rows(rows4.numpy(), CFG4_TOTAL, world)
        err4 = np.linalg.norm(p4[c4b:c4e, :3] - truths[:n_shard, :3], axis=1)
        assert (s4 == 0).all() and err4.max() < 0.05, (err4.max(), s4.sum())
        cfg4 = {"workload": "cfg4: 1024 distinct OS1-128 scans vs the 1M-pt map, sharded over the GPUs, host (pinned) scans in, ONE gather of the poses",
                "scans_total": CFG4_TOTAL, "scans_this_rank": n_shard, "ms": float(t4.item()), "scans_per_s": CFG4_TOTAL / (float(t4.item()) * 1e-3),
                "scaling": "strong", "icp_iterations_mean": float(i4.mean()), "max_pos_err_vs_truth_m": float(err4.max())}
        ctx.set_pose_sink(sink.data_ptr(), per_step, 0)
        phase("cfg4 replay")

    # ---- cfg5: k-NN microbench, queries split over the ranks, map replicated ------------------------------------------------------
    knn5 = None
    if not args.no_cfg5:
        knn5 = run_cfg5(args, torch, dist, api, synth, rank, world, local, dev, stream, phase)

    line = None
    if rank == 0:
        peak, peak_src = _peaks()
        # roofline of the dominant kernel: one profiled sub-batch, CUDA events around every launch that has work
        ctx.set_pose_sink(None)
        ctx.profile_enable(True)
        for k in range(6):
            ctx.profile_get(k, reset=True)
        pres = ctx.register_batch_device(d_scans.data_ptr(), n_points[:B], priors[:B], 20, 0, skip_map_checks=True)
        ctx.profile_enable(False)
        ms_k, n_k = ctx.profile_get(0)          # k_knn_scan
        ms_f, n_f = ctx.profile_get(4)          # first evaluation of each solve (k_evaluate<PH_CORR> + k_lm_step)
        ms_q, n_q = ctx.profile_get(5)          # k_fit (split build)
        ms_e, n_e = ctx.profile_get(1)          # k_evaluate (+ k_lm_step)
        ms_p, n_p = ctx.profile_get(3)          # scan ordering (keys + radix sort + gather)
        queries = sum(int(r.n_iterations) * int(n) for r, n in zip(pres, n_points[:B]))      # point-passes of the k-NN kernel
        fused = bool(api.build_flags() & 1)
        kname = "k_knn_fit" if fused else "k_knn_scan"
        alg_bytes = queries * KNN_BYTES_PER_QUERY + n_k * len(map_xyzi) * 16
        achieved = alg_bytes / (ms_k * 1e-3) / 1e9 if ms_k > 0 else 0.0
        tot = ms_k + ms_q + ms_f + ms_e + ms_p + 1e-12
        per_q = NCU_DRAM_BYTES_PER_QUERY.get(kname)
        roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": per_q * queries / max(n_k, 1) if per_q else None,
                    "traffic_source": f"profiles/ (ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum of one {kname} launch per query, scaled to this launch size)",
                    "peak_source": peak_src, "launches_profiled": int(n_k), "avg_launch_ms": ms_k / max(n_k, 1),
                    "algorithmic_bytes_per_launch": alg_bytes / max(n_k, 1),
                    "algorithmic_bytes": "SURVEY 8(d): (16 B query + 5 x 8 B result) x queries of the launch + 16 B x map points once per launch",
                    "queries_per_launch": queries / max(n_k, 1),
                    "icp_step_figure": {"formula": "SURVEY 8(d) fused-ICP figure: 16 N + 16 M + 32 n_ok per ICP iteration",
                                        "bytes_per_scan_iteration": int(16 * 131072 + 16 * len(map_xyzi) / B + 32 * float(np.mean([r.iter_n_surf[0] for r in pres])))},
                    "note": "instruction-issue bound, L1/L2-resident gathers; see DESIGN.md section 4",
                    "first_evaluation": {"launches": int(n_f), "avg_launch_ms": ms_f / max(n_f, 1)},
                    "k_evaluate": {"launches": int(n_e), "avg_launch_ms": ms_e / max(n_e, 1)},
                    "k_fit": {"launches": int(n_q), "avg_launch_ms": ms_q / max(n_q, 1)},
                    "share_of_step": {kname: ms_k / tot, "k_fit": ms_q / tot, "first_evaluation": ms_f / tot, "k_evaluate": ms_e / tot, "scan_ordering": ms_p / tot}}
        phase("profiling pass")
        # ---- wide-prior variant: the same call with +-0.5 m / +-5 deg priors, so that ICP iterations 4+ actually run --------------
        wide = None
        try:
            wp = np.stack([synth.perturb_pose(truths[i], 7000 + i, dt=0.5, dth_deg=5.0) for i in range(B)])
            for _ in range(2):
                wres = ctx.register_batch_device(d_scans.data_ptr(), n_points[:B], wp, 20, 0, skip_map_checks=True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                wres = ctx.register_batch_device(d_scans.data_ptr(), n_points[:B], wp, 20, 0, skip_map_checks=True)
            e1.record()
            torch.cuda.synchronize()
            werr = np.linalg.norm(np.array([list(r.pose) for r in wres])[:, :3] - truths[:B, :3], axis=1)
            wide = {"prior": "+-0.5 m, +-5 deg per axis", "scans_per_s": 3 * B / (e0.elapsed_time(e1) * 1e-3),
                    "icp_iterations_mean": float(np.mean([r.n_iterations for r in wres])), "icp_iterations_max": int(max(r.n_iterations for r in wres)),
                    "converged_within_5cm": int((werr < 0.05).sum()), "scans": B}
        except Exception as e:
            wide = {"error": f"{type(e).__name__}: {e}"}
        phase("wide-prior variant")
        latency = run_latency(args, api, synth, local, torch, map_xyzi, scans, priors)
        phase("single-scan latency")
        live = run_live(args, api, synth, local, torch)
        phase("live-SLAM loop")
        # CPU baseline on the host cores: the oracle (reference octree verbatim when oracle/_ref travelled), 1 thread, bounded sample
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import oracle as O
            ref = O.has_ref_octree()
            om = O.OracleMap(map_xyzi, ref_octree=ref)
            mode = 2 if ref else 0
            t0 = time.perf_counter()
            ns = 0
            first = res[0]
            while ns < B and ns < 8 and (time.perf_counter() - t0 < 12.0 or ns < 2):
                ro = om.register(scans[ns], priors[ns], 0.2, 20, 0, knn_mode=mode, n_threads=1, skip_map_checks=True)
                dpos = np.abs(np.array(ro.pose)[:3] - np.array(first[ns].pose)[:3]).max()
                ns += 1
            dt = time.perf_counter() - t0
            cpu = {"value": ns / dt, "unit": UNIT, "cores": 1, "kind": "reference-octree+port" if ref else "port",
                   "sample": f"{ns} of the step's cfg2 scans, whole ICP, 1 thread (the reference's feature loop and Ceres solve are serial); "
                             f"k-NN = {'the reference flann/octree.h compiled verbatim (oracle/_ref); fits + Ceres LM = the restated port' if ref else 'oracle exact grid (port)'}"
                             f"; last |dpos| GPU-exact vs this path {dpos:.2e} m"}
        phase("cpu baseline")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": WORKLOAD, "scans_per_step_per_gpu": per_step, "scans_per_step": n_total, "sub_batches": SUB, "batch": B,
                           "distinct_scans_per_gpu": n_distinct, "parallelism": f"replay-shard x{world}",
                           "l2": f"inputs larger than L2 (every sub-batch reads {B * 2.1:.0f} MB of scans it did not touch in the previous sub-batch)",
                           "collective": "one all-gather of the per-scan rows per step, from device memory on the compute stream",
                           "timed_region_s": ms * 1e-3, "icp_iterations_executed_mean": icp_mean, "cpu_affinity": numa},
                "clocks": clocks,
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d // args.steps), "d2h_bytes_per_step": int(d2h // args.steps),
                        "ms_per_step": ms_e2e / args.steps, "h2d_link_GBps_measured": h2d_gbs,
                        "h2d_GBps_needed_at_value": value / world * 131072 * 16 / 1e9,
                        "poses_bitwise_equal_to_device_resident_path": same_bits},
                "gpu_launches": int(launches), "roofline": roofline, "knn_cfg5": knn5, "cfg4": cfg4, "wide_prior": wide, "latency": latency, "live": live,
                "cpu_baseline": cpu}
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def run_cfg5(args, torch, dist, api, synth, rank, world, local, dev, stream, phase):
    """BASELINE configs[4]: 10 M queries, k = 5, 5 M-point map; queries split evenly over the ranks, map replicated."""
    NQ = args.cfg5_queries
    scene = synth.make_scene(58.0, seed=77)
    raw = synth.sample_surfaces(scene, 0.1, seed=1234)             # 5.4 M raw samples; the per-block voxel filter runs on the device
    kctx = api.Context(device=local, max_map_points=len(raw) + 1024, max_scan_points=1024, plane_res=0.1)
    kctx.set_stream(stream.cuda_stream)
    kctx.map_add_surf(np.concatenate([raw, np.ones((len(raw), 1), np.float32)], 1))      # == synth.make_map(58, 0.1), bit for bit (tests)
    map5 = kctx.map_download(0)
    kctx.map_set_points(map5)                                      # ids = positions in map5
    M = len(map5)
    per = (NQ + world - 1) // world
    q_first = rank * per
    nq = max(0, min(NQ, q_first + per) - q_first)
    q4 = cfg5_queries(map5, q_first, nq)
    dq = torch.from_numpy(q4).to(dev)
    didx = torch.empty((nq, 5), dtype=torch.int32, device=dev)
    dd2 = torch.empty((nq, 5), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    peak, _ = _peaks()
    out = {"workload": "cfg5: 10M queries (map points + N(0,(0.1 m)^2)), k=5, vs the 5M-pt map (planeRes 0.1), queries split over the GPUs, map replicated",
           "map_points": M, "queries": NQ, "k": 5, "n_gpus": world, "peak_gbs_per_gpu": peak,
           "algorithmic_bytes": "SURVEY 8(d): 16 B query + 5 x 8 B result per query + the 16 B/pt map once per GPU",
           "l2": "256 MiB written between timed iterations (L2 flush)"}
    phase(f"cfg5 inputs (map {M} pts via the device voxel filter, {nq} queries)")
    for name, bound in (("bounded", float(np.float32(3 * np.float32(0.1)))), ("exact", 0.0)):
        times = []
        for it in range(7):
            flush.zero_()
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            kctx.knn_device(dq.data_ptr(), nq, 5, bound, didx.data_ptr(), dd2.data_ptr())
            e1.record()
            torch.cuda.synchronize()
            if it >= 3:
                times.append(e0.elapsed_time(e1))
        t = torch.tensor([float(np.median(times))], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        msk = float(t.item())
        alg = NQ * KNN_BYTES_PER_QUERY + world * 16 * M
        out[name] = {"ms": msk, "Mqueries_per_s": NQ / msk / 1e3, "algorithmic_GB": alg / 1e9, "achieved_GBps": alg / msk / 1e6,
                     "frac_of_peak": alg / msk / 1e6 / (peak * world), "found5_frac_rank0": float((didx[:, 4] != -1).float().mean().item()),
                     "includes": "cell-ordering of the queries (keys + radix sort) inside the timed call"}
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as O
        ns = 100_000
        q = q4[:ns, :3]
        om = O.OracleMap(map5)
        mode = 2 if O.has_ref_octree() else 0
        t0 = time.time()
        oi, od, of = om.knn(q, 5, mode)
        dt = time.time() - t0
        out["cpu_reference_octree_1thread"] = {"Mqueries_per_s": ns / dt / 1e6, "sample": ns, "verbatim_reference_header": bool(O.has_ref_octree())}
        gi = didx[:ns].cpu().numpy().astype(np.int64)           # the last GPU pass was the exact variant
        oi0, od0, _ = om.knn(q, 5, 0)
        out["gpu_exact_equals_oracle_exact"] = bool(np.array_equal(gi, oi0))
        out["octree_vs_exact_mismatch_queries"] = int((np.sort(oi, 1) != np.sort(oi0, 1)).any(1).sum())
        try:
            from scipy.spatial import cKDTree
            t0 = time.time()
            tree = cKDTree(map5[:, :3])
            tb = time.time() - t0
            nk = min(nq, 1_000_000)
            t0 = time.time()
            tree.query(q4[:nk, :3], k=5, workers=-1)
            dt = time.time() - t0
            out["cpu_scipy_ckdtree_allcores"] = {"Mqueries_per_s": nk / dt / 1e6, "build_s": tb, "cores": len(os.sched_getaffinity(0)),
                                                 "note": "exact kd-tree stand-in for pcl::KdTreeFLANN (PCL / FLANN are not installable here, SURVEY 8d)"}
        except Exception as e:
            out["cpu_scipy_ckdtree_allcores"] = {"error": type(e).__name__}
    kctx.close()
    phase("cfg5 k-NN microbench")
    return out


def run_latency(args, api, synth, local, torch, map2, scans2, priors2):
    """Single-scan so_register latency (host scan in -> pose out, wall clock, median of 20) beside the CPU path on one thread."""
    out = {}
    try:
        cases = {}
        c1 = synth.make_case("cfg1")
        cases["cfg1_vlp16_cap2000"] = (c1["map_xyzi"], c1["scan_xyzi"], c1["pose_prior"], 5, 2000)
        cases["cfg2_os1_128"] = (map2, scans2[0], priors2[0], 20, 0)
        for name, (m, s, p, iters, cap) in cases.items():
            c = api.Context(device=local, max_map_points=len(m) + 1024, max_scan_points=len(s), plane_res=0.2)
            c.map_set_points(m)
            for _ in range(3):
                r = c.register(s, p, iters, cap)
            wall, devt = [], []
            for _ in range(20):
                t = time.perf_counter()
                r = c.register(s, p, iters, cap)
                wall.append((time.perf_counter() - t) * 1e3)
                devt.append(r.time_ms)
            e = {"points": len(s), "map_points": len(m), "icp_iterations": int(r.n_iterations), "gpu_wall_ms_median": float(np.median(wall)),
                 "gpu_device_ms_median": float(np.median(devt))}
            if not args.no_cpu_baseline:
                from oracle import oracle as O
                ref = O.has_ref_octree()
                om = O.OracleMap(m, ref_octree=ref)
                ts = []
                for _ in range(5 if len(s) < 50000 else 2):         # median of a few runs: one cold run can be 2x off
                    t = time.perf_counter()
                    om.register(s, p, 0.2, iters, cap, knn_mode=2 if ref else 0, n_threads=1)
                    ts.append((time.perf_counter() - t) * 1e3)
                e["cpu_1thread_ms"] = float(np.median(ts))
                e["cpu_runs"] = len(ts)
                e["speedup_wall"] = e["cpu_1thread_ms"] / e["gpu_wall_ms_median"]
            out[name] = e
            c.close()
    except Exception as e:
        out["error"] = f"{type(e).__name__}: {e}"
    return out


def run_live(args, api, synth, local, torch):
    """Live-SLAM loop (LidarSlam.cpp:107-171): so_register + so_map_add_scan per scan, the map growing from the scans themselves."""
    if args.no_live:
        return None
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests", "tools"))
        import live_loop
        return live_loop.run(api, synth, device=local, n_scans=args.live_scans, cpu=not args.no_cpu_baseline)
    except Exception as e:
        return {"error": f"{type(e).__name__}: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="scans per registration call (sub-batch)")
    ap.add_argument("--sub-batches", type=int, default=4, help="registration calls per step per GPU")
    ap.add_argument("--ref-scans", type=int, default=2, help="scans per step for --impl reference")
    ap.add_argument("--cfg5-queries", type=int, default=10_000_000)
    ap.add_argument("--live-scans", type=int, default=60)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cfg4", action="store_true")
    ap.add_argument("--no-cfg5", action="store_true")
    ap.add_argument("--no-live", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the per-scan results of the last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
