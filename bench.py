#!/usr/bin/env python
"""bench.py -- verified pairs/s of the matching + verification hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (tcgen05 match -> ratio filter -> RANSAC-F) over one batch of synthetic input.
N = 1: BASELINE.json configs[1], the 50-image exhaustive run (1,225 pairs x 8192 SIFT-like features per image).
N > 1 (torchrun, one rank per GPU): BASELINE.json configs[2], the 200-image exhaustive run (19,900 pairs) block-partitioned
over the ranks -- strong scaling; every rank holds the broadcast bank, there is no data-path collective, and inside the
timed step the WHOLE result (per-pair summaries, packed match rows, inlier flags) is gathered on rank 0, which then
checks a sample of it against its own single-GPU recomputation.  ``--scaling weak`` keeps round 1's replicated block.
Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for every field.
``--dump-outputs DIR`` also writes what the last timed step returned to its caller as DIR/<name>.npy (see dump_outputs), so
that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "sfm-project_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

N_IMAGES, N_FEATS = 50, 8192
PAIR_BATCH = 2048
PAIR_BLOCK = 32
SHARD_PAIR_BATCH = int(os.environ.get("SFM_SHARD_PAIR_BATCH", 1024))   # sharded arm: batch k's rows cross NVLink while batch k+1 is swept
RANSAC_INSTR_PER_EVAL = 21.0                                            # fp32 instructions of is_inlier (csrc/ransac_f.cu): 12 FFMA, 3 FMUL, 1 FMNMX, ... per (hypothesis, correspondence)
RANSAC_FLOP_PER_EVAL = 34.0                                             # the same with an FFMA counted as two operations
E2E_PAIR_BATCH = int(os.environ.get("SFM_E2E_PAIR_BATCH", 512))   # end-to-end arm: batch k's D2H overlaps batch k+1's sweep
E2E_CHUNKS = int(os.environ.get("SFM_E2E_CHUNKS", 3))              # end-to-end arm: images uploaded in this many groups
RANSAC = dict(thr=3.0, confidence=0.99, max_iters=2000, solver="8pt", score="sym_epipolar", lo=False, seed=1)
RATIO = 0.75
OPS_PER_PAIR = 2.0 * N_FEATS * N_FEATS * 128            # algorithmic int8 ops (SURVEY.md §8d)
NOMINAL_INT8_TOPS = 4500.0
DUMP_BYTES = 64 * 10**6                                 # --dump-outputs writes at most this much


def dump_outputs(out_dir, arrays):
    """Writes ``arrays`` (name -> torch tensor or ndarray) as ``out_dir/<name>.npy``: float32 stays float32, every other
    type becomes float64 (exact for the int32 counts and indices).  Each array and its row index may fill an equal share of
    DUMP_BYTES; an array with more rows than its share holds keeps a fixed sample of them (seed 0, in ascending order, taken
    before the copy to the host), and the sampled row numbers go to ``<name>.rows.npy``.  Returns the paths written."""
    import torch

    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // (2 * max(len(arrays), 1)) - 256            # (npy header)
    written = []
    for name, a in sorted(arrays.items()):
        f32 = str(a.dtype).endswith("float32")
        shape = tuple(a.shape) or (1,)
        keep = share // max((4 if f32 else 8) * int(np.prod(shape[1:])), 8)
        if shape[0] > keep:
            rows = np.sort(np.random.default_rng(0).permutation(shape[0])[:keep])
            a = a[torch.as_tensor(rows, device=a.device)] if isinstance(a, torch.Tensor) else np.asarray(a)[rows]
            written.append(os.path.join(out_dir, f"{name}.rows.npy"))
            np.save(written[-1], rows.astype(np.float64))
        a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
        written.append(os.path.join(out_dir, f"{name}.npy"))
        np.save(written[-1], np.atleast_1d(a.astype(np.float32 if f32 else np.float64)))
    return written


def sharded_outputs(gathered, row_fields):
    """The gathered result of a sharded step as its caller reads it: the per-pair tensors, and every row field (names in
    ``row_fields``) in pair order -- pair p owns rows row_start[p] : row_start[p] + n_matches[p] of rank slices that have
    unwritten room after their rows, so the buffers themselves are not the result."""
    import torch

    out = {k: v for k, v in gathered.items() if isinstance(v, torch.Tensor) and k != "row_start" and k not in row_fields}
    if "row_start" in gathered:
        n = gathered["n_matches"].to(torch.int64)
        rows = torch.repeat_interleave(gathered["row_start"] - (torch.cumsum(n, 0) - n), n) + torch.arange(int(n.sum()), device=n.device)
        out.update({k: v.index_select(0, rows) for k, v in gathered.items() if k in row_fields})
    return out


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the bench's own kernels, from the committed ncu
    capture (profiles/traffic.json, written by tools/ncu_summary.py); {} when there is none."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            pk = json.load(f)
        return pk, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region, in-process through NVML (a thread polling
    every 20 ms).  NVML is initialised before the warm-up so that its start-up cost never lands in the timed steps;
    only samples taken between mark_begin() and mark_end() are reported."""

    def __init__(self, device_index=0):
        self.rows, self.t0, self.t1, self._stop, self.thread, self.h, self.nv = [], None, None, False, None, None, None
        try:
            import pynvml as nv

            nv.nvmlInit()
            try:
                import torch

                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                self.h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                self.h = nv.nvmlDeviceGetHandleByIndex(device_index)
            self.nv = nv
            self.max_sm = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        nv = self.nv
        while not self._stop:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((time.perf_counter(), sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.02)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self._stop = True
        if self.thread is not None:
            self.thread.join(1.0)
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "NVML unavailable"}
        rows = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or 1e300)] or self.rows
        bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap", 0x80: "hw_power_brake"}
        reasons = sorted({name for r in rows for b, name in bits.items() if r[3] & b})
        return {"sm_mhz": float(np.median([r[1] for r in rows])) if rows else None, "sm_max_mhz": self.max_sm,
                "power_w_max": max((r[2] for r in rows), default=None), "samples": len(rows), "reasons": reasons}


# ------------------------------------------------------------------------------------ reference arm (cv2 on the host)
def cv2_pairs_per_s(scene, pairs, n_sample):
    """The reference's arithmetic for this workload (BASELINE.json configs[0]): cv2 BFMatcher L2 knnMatch(k=2) + ratio +
    findFundamentalMat(FM_RANSAC) with all host threads cv2 uses, on a bounded sample of the pair list."""
    from oracle import cv2_ref

    t0 = time.perf_counter()
    verified = 0
    for i, j in pairs[:n_sample]:
        q, t, F, mask = cv2_ref.verified_pair(scene.desc[i], scene.xy[i], scene.desc[j], scene.xy[j], ratio=RATIO,
                                              thr=RANSAC["thr"], confidence=RANSAC["confidence"], max_iters=RANSAC["max_iters"])
        verified += 1
    dt = time.perf_counter() - t0
    return verified / dt, dt


_POOL_SCENE = None


def _pool_init(n_feats):
    import cv2

    from sfm_b200 import synth

    global _POOL_SCENE
    cv2.setNumThreads(1)
    _POOL_SCENE = synth.make_scene(8, n_feats, seed=2001)


def _pool_pair(ij):
    from oracle import cv2_ref

    i, j = ij
    sc = _POOL_SCENE
    cv2_ref.verified_pair(sc.desc[i], sc.xy[i], sc.desc[j], sc.xy[j], ratio=RATIO, thr=RANSAC["thr"], confidence=RANSAC["confidence"],
                          max_iters=RANSAC["max_iters"])
    return 1


def run_reference(args):
    """The reference's own CPU implementation of the path (cv2: BFMatcher L2 knnMatch(k=2) + ratio + findFundamentalMat
    FM_RANSAC -- BASELINE.json configs[0]) on this box's host cores, two ways, the faster one reported:
    (a) one process, cv2's internal threads (BFMatcher parallelises over query rows; RANSAC is serial);
    (b) a process pool over pairs, one single-threaded worker per core."""
    import multiprocessing as mp

    import cv2

    from sfm_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the GPU arm's workload at this N (N = 1: configs[1]; N > 1: configs[2], pair-sharded) -- a bounded sample of it: 8 images of the
    # same generator and seed, every pair the same 8192 x 8192 x 128 match + RANSAC-F as any pair of the full list
    world = int(os.environ.get("WORLD_SIZE", "1"))
    strong = world > 1 and args.scaling != "weak"
    wl = WORKLOADS["c3" if (args.workload == "c3" or (args.workload == "auto" and strong)) else "c2"]
    scene = synth.make_scene(8, N_FEATS, seed=wl["seed"])
    pairs = synth.exhaustive_pairs(8)
    ncpu = os.cpu_count() or 1
    n_sample = 8
    for _ in range(args.warmup):
        cv2_pairs_per_s(scene, pairs, 1)
    times = []
    for _ in range(args.steps):
        r, dt = cv2_pairs_per_s(scene, pairs, n_sample)
        times.append(dt)
    single = float(n_sample * len(times) / sum(times))
    cores_single = int(cv2.getNumThreads())
    pool_rate, pool_times, n_pool = 0.0, [], 2 * ncpu
    try:
        work = [tuple(pairs[k % len(pairs)]) for k in range(n_pool)]
        # spawn, not fork: the parent already runs cv2 / BLAS thread pools, and forking those deadlocks the children
        with mp.get_context("spawn").Pool(ncpu, initializer=_pool_init, initargs=(N_FEATS,)) as pool:
            pool.map_async(_pool_pair, work[:ncpu]).get(timeout=300)   # warm-up: every worker builds its scene
            for _ in range(max(1, min(args.steps, 5))):
                t0 = time.perf_counter()
                pool.map_async(_pool_pair, work, chunksize=1).get(timeout=300)
                pool_times.append(time.perf_counter() - t0)
        pool_rate = float(n_pool * len(pool_times) / sum(pool_times))
    except Exception as e:                                             # pragma: no cover - depends on the box
        print(f"process-pool baseline failed: {e}", file=sys.stderr)
    use_pool = pool_rate > single
    value = pool_rate if use_pool else single
    cores = ncpu if use_pool else cores_single
    ms_step = 1e3 * float(np.mean(pool_times if use_pool else times))
    sample = (f"{n_pool if use_pool else n_sample} pairs of 8192x8192x128 per step (knnMatch k=2 f32 + ratio {RATIO} + findFundamentalMat "
              f"FM_RANSAC 3.0/0.99/2000); single process with {cores_single} cv2 threads: {single:.2f} pairs/s; "
              f"pool of {ncpu} single-threaded workers: {pool_rate:.2f} pairs/s; the faster one is reported")
    line = {
        "impl": "reference", "metric": "verified pairs/s", "value": value, "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["label"] + "; bounded sample on the host cores of rank 0", "sample": sample,
                   "cv2": cv2.__version__, "host_cpus": ncpu},
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------ our arm
WORKLOADS = {
    # BASELINE.json configs[1]: the single-GPU headline (bank 66 MiB)
    "c2": dict(n_images=50, seed=2001, label="configs[1]: 50-image exhaustive matching (1,225 pairs) x 8192 features/image + RANSAC F verification"),
    # BASELINE.json configs[2]: the run north_star's "near-linear 1->8" is quoted on (bank 264 MiB)
    "c3": dict(n_images=200, seed=3001, label="configs[2]: 200-image exhaustive matching (19,900 pairs) x 8192 features/image + RANSAC F, pair-sharded"),
}


def measure_int8_gemm_tops(dev, n=8192, reps=10):
    """The library yardstick SURVEY.md §8d asks for: torch._int_mm (cuBLASLt int8) n^3, best of ``reps``, in the same run.
    Not on the product path."""
    import torch

    a = torch.randint(-128, 127, (n, n), dtype=torch.int8, device=dev)
    b = torch.randint(-128, 127, (n, n), dtype=torch.int8, device=dev)
    best = float("inf")
    for k in range(reps + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch._int_mm(a, b)
        e1.record()
        e1.synchronize()
        if k >= 2:
            best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def run_ours(args):
    import torch
    import torch.distributed as dist

    import sfm_b200
    from sfm_b200 import dist as sdist
    from sfm_b200 import matcher, synth
    from sfm_b200 import plan as splan

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- workload: N = 1 -> configs[1] (the single-GPU headline); N > 1 -> configs[2] pair-sharded (strong scaling), or
    #      with --scaling weak the N = 1 block replicated per rank
    scaling = args.scaling if args.scaling != "auto" else ("strong" if world > 1 else "weak")
    wl_name = args.workload if args.workload != "auto" else ("c3" if (world > 1 and scaling == "strong") else "c2")
    wl = WORKLOADS[wl_name]
    n_images = wl["n_images"]
    scene = synth.make_scene(n_images, N_FEATS, seed=wl["seed"])
    # (the 200-image bank is larger than L2: the pair list goes in 32 x 32 image squares, see pairs.blocked_exhaustive_pairs)
    pairs_one = sfm_b200.blocked_exhaustive_pairs(n_images, PAIR_BLOCK) if args.pair_order == "blocked" else synth.exhaustive_pairs(n_images)
    pairs_all = pairs_one if scaling == "strong" else np.concatenate([pairs_one] * world)
    P_total = len(pairs_all)
    lay = sdist.layout(P_total, world, "block")
    mine = lay.owned[rank]
    my_pairs = pairs_all[mine]

    # ---- bank: rank 0 packs it, the others receive it over NVLink (NCCL broadcast, once per job; timed on its own)
    bank = sfm_b200.DescriptorBank(-(-n_images // world) * world, N_FEATS, device=dev)
    if rank == 0:
        bank.put(0, scene.desc, xy=scene.xy)
    torch.cuda.synchronize()
    bcast_ms = []
    for _ in range(3 if world > 1 else 0):                              # first call carries NCCL's lazy connection set-up
        dist.barrier()
        torch.cuda.synchronize()
        tb = time.perf_counter()
        sdist.broadcast_bank(bank, src=0)
        torch.cuda.synchronize()
        bcast_ms.append(1e3 * (time.perf_counter() - tb))
    desc_pin = torch.from_numpy(scene.desc).pin_memory()
    xy_pin = torch.from_numpy(scene.xy).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    step_events = []

    def step_resident():
        # inputs resident in HBM.  One GPU: per-pair summaries stay on the device.  Sharded: every rank pushes its packed match
        # rows + inlier flags into rank 0's HBM over NVLink while it computes, per-pair summaries follow in one gather --
        # the whole result of the job is on rank 0 when the step ends (north_star (4)).
        if world == 1:
            return sfm_b200.match_and_verify(bank, my_pairs, ratio=RATIO, pair_ids=mine, pair_batch=PAIR_BATCH, **RANSAC)
        ev = {}
        out, res = sdist.match_and_verify_sharded(bank, pairs_all, mode="block", gather=args.gather, transport=args.transport,
                                                  events=ev, ratio=RATIO, pair_batch=SHARD_PAIR_BATCH, overlap=not args.no_overlap, **RANSAC)
        step_events.append(ev)
        return (out, res)

    def step_e2e():
        # the call a user makes, host buffers in and out: H2D of descriptors + keypoints from pinned memory, pack,
        # match, filter, verify, D2H of every pair's matches / inlier flags / F / counts into pinned memory
        # (upload in E2E_CHUNKS groups on a side stream: pairs inside the first groups are matched while later images travel,
        #  and batch k's results travel while batch k+1 is swept).  Sharded: every rank does this for its own pair block.
        if world > 1:
            # every rank uploads and packs 1/N of the images, the packed bank is all-gathered over NVLink, then every rank matches and
            # verifies its pair block and fetches its own results into its own pinned host arrays
            sdist.upload_bank_sharded(bank, desc_pin, xy_pin)
            return sfm_b200.match_and_verify(bank, my_pairs, ratio=RATIO, pair_batch=E2E_PAIR_BATCH, pair_ids=mine, fetch="view", **RANSAC)
        res, _order = sfm_b200.match_and_verify_host(desc_pin, xy_pin, my_pairs, bank=bank, n_chunks=E2E_CHUNKS, ratio=RATIO,
                                                     pair_batch=E2E_PAIR_BATCH, pair_ids=mine, fetch="view", **RANSAC)
        return res

    insitu_sweeps = []                                                  # (ms, pairs) of every sweep launch inside the timed steps (rank-local)

    def timed(fn, steps, warmup, sampler=None):
        for _ in range(warmup):
            fn()
            flush.zero_()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        step_events.clear()
        ms, host_ms, out = [], [], None
        l0 = sfm_b200.launch_count()
        if sampler is not None:
            sampler.mark_begin()
            splan.SWEEP_EVENTS = []                                    # the resident run: time every sweep launch of the timed steps
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            out = fn()
            e1.record()
            t_ret = time.perf_counter()
            host_ms.append(1e3 * (t_ret - t0))
            e1.synchronize()
            t_sync = time.perf_counter()
            ms.append(e0.elapsed_time(e1))
            if step_events and os.environ.get("SFM_HOST_TRACE"):       # CLOCK_MONOTONIC: comparable between the ranks of one box
                step_events[-1]["wall"] = (t0, t_ret, t_sync)
            if step_events and "compute" in step_events[-1]:
                step_events[-1]["t_compute"] = e0.elapsed_time(step_events[-1]["compute"])
                step_events[-1]["t_done"] = e0.elapsed_time(step_events[-1]["done"])
                if step_events[-1].get("kernels") is not None:
                    step_events[-1]["t_kernels"] = e0.elapsed_time(step_events[-1]["kernels"])
                if step_events[-1].get("fence") is not None:           # (start of the step -> the region fence has passed on this rank)
                    step_events[-1]["t_fence"] = e0.elapsed_time(step_events[-1]["fence"][1])
                tr = getattr(getattr(out[1], "plan", None), "host_trace", None) if isinstance(out, tuple) else None
                if tr:                                                 # SFM_HOST_TRACE=1: host time per batch, relative to the step's start
                    step_events[-1]["host_trace_ms"] = [round(1e3 * (x - t0), 2) for x in tr]
                    step_events[-1]["host_ms"] = round(host_ms[-1], 2)
            flush.zero_()                                              # L2 flush between timed iterations (untimed)
        if sampler is not None:
            sampler.mark_end()
        torch.cuda.synchronize()
        if sampler is not None:
            insitu_sweeps.extend((a.elapsed_time(b), n) for a, b, n in splan.SWEEP_EVENTS)
            splan.SWEEP_EVENTS = None
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([sum(ms)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                   # max over ranks
        return float(t.item()), out, (sfm_b200.launch_count() - l0) // max(steps, 1), float(np.mean(host_ms))

    sampler = ClockSampler(local)                                       # every rank watches its own GPU; rank 0 reports all of them
    sampler.start()
    total_ms, last, launches_per_step, host_ms = timed(step_resident, args.steps, args.warmup, sampler)
    clocks = sampler.stop()
    if world > 1:
        every = [None] * world
        dist.all_gather_object(every, clocks)
        if rank == 0:
            clocks = dict(every[0])
            clocks["reasons"] = sorted({r for c in every for r in (c.get("reasons") or [])})
            clocks["per_rank_sm_mhz"] = [c.get("sm_mhz") for c in every]
            clocks["per_rank_power_w_max"] = [c.get("power_w_max") for c in every]
    value = P_total * args.steps / (total_ms * 1e-3)
    gathered, res = (None, last) if world == 1 else last
    if args.dump_outputs and rank == 0:
        # what the caller of the timed path holds after the last step: the VerifiedPairs of one GPU, the gathered result when sharded
        dump_outputs(args.dump_outputs, {k: v for k, v in vars(res).items() if isinstance(v, torch.Tensor)} if world == 1
                     else sharded_outputs(gathered, splan.RowSink.ROW_BYTES))
    ev_rows = list(step_events)
    # per-rank compute time (own kernels + row pushes) and time to the end of the gather, max / min over ranks
    sharded_info = None
    if world > 1:
        tc = float(np.mean([e["t_compute"] for e in ev_rows]))
        td = float(np.mean([e["t_done"] for e in ev_rows]))
        stats = torch.tensor([tc, td, -tc, float(ev_rows[-1]["bytes_pushed"])], dtype=torch.float64, device=dev)
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        if os.environ.get("SFM_HOST_TRACE"):
            os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
            with open(os.path.join(ROOT, "gpurun_out", f"hosttrace_rank{rank}.json"), "w") as f:
                json.dump([{k: e.get(k) for k in ("t_compute", "t_kernels", "t_done", "t_fence", "host_ms", "host_trace_ms", "wall")} for e in ev_rows], f)
        per_rank = [None] * world
        dist.all_gather_object(per_rank, {"compute_ms": round(tc, 3), "kernels_ms": round(float(np.mean([e.get("t_kernels", float("nan")) for e in ev_rows])), 3),
                                          "compute_ms_each_step": [round(e["t_compute"], 2) for e in ev_rows],
                                          "region_fence_passed_at_ms_each_step": [round(e.get("t_fence", float("nan")), 2) for e in ev_rows]})
        sharded_info = {"per_rank": per_rank, "compute_ms_slowest_rank": float(mx[0]), "compute_ms_fastest_rank": float(-mx[2]), "compute_ms_rank0": tc,
                        "step_ms_rank0_until_everything_is_gathered": td,
                        "gather_ms_exposed_on_rank0": td - tc, "row_bytes_pushed_per_step_all_ranks": float(sm[3]),
                        "transport": ev_rows[-1].get("transport"), "gather": args.gather}

    # ---- end-to-end through the public API with host buffers (H2D + pack + match + verify + D2H every step)
    e2e_steps = max(1, min(args.steps, 10))
    e2e_ms, e2e_res, _, e2e_host_ms = timed(step_e2e, e2e_steps, max(1, min(args.warmup, 3)))
    e2e_value = P_total * e2e_steps / (e2e_ms * 1e-3)
    n_mine = n_images if world == 1 else max(0, min((rank + 1) * -(-n_images // world), n_images) - min(rank * -(-n_images // world), n_images))
    h2d = n_mine * (N_FEATS * 128 + N_FEATS * 8) + my_pairs.nbytes + 4 * len(my_pairs)
    d2h = int(e2e_res.d2h_bytes)
    if world > 1:
        io = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device=dev)
        dist.all_reduce(io, op=dist.ReduceOp.SUM)
        h2d, d2h = int(io[0]), int(io[1])

    # ---- sharded runs check themselves: a sample of pairs spread over every rank's block is recomputed on rank 0 alone and
    #      compared, element by element, with what the gather delivered (summaries, match rows, inlier flags)
    selfcheck, one_gpu = None, None
    if world > 1:
        if rank == 0:
            rng = np.random.default_rng(5)
            sample = np.unique(np.concatenate([rng.choice(o, size=min(12, len(o)), replace=False) for o in lay.owned if len(o)]))
            ref = sfm_b200.match_and_verify(bank, pairs_all[sample], ratio=RATIO, pair_ids=sample, pair_batch=PAIR_BATCH, fetch=True,
                                            **RANSAC).to_host()
            ok = True
            for k in ("n_matches", "n_inliers", "iters", "F"):
                ok &= bool(np.array_equal(gathered[k][torch.as_tensor(sample, device=dev)].cpu().numpy(), ref[k]))
            rows_checked = 0
            if args.gather == "full":
                start = gathered["row_start"][torch.as_tensor(sample, device=dev)].cpu().numpy()
                for k, p in enumerate(sample):
                    a, b = int(ref["offsets"][k]), int(ref["offsets"][k + 1])
                    s0 = int(start[k])
                    ok &= bool(np.array_equal(gathered["matches"][s0: s0 + (b - a)].cpu().numpy(), ref["matches"][a:b]))
                    ok &= bool(np.array_equal(gathered["inlier"][s0: s0 + (b - a)].cpu().numpy(), ref["inlier"][a:b]))
                    rows_checked += b - a
            selfcheck = {"pairs_recomputed_on_rank0": int(len(sample)), "match_rows_compared": int(rows_checked), "equal": bool(ok)}
            if not ok:
                raise AssertionError(f"sharded result differs from the single-GPU recomputation: {selfcheck}")
            # the same workload on ONE GPU (rank 0 alone, others idle): the denominator of the strong-scaling efficiency
            if scaling == "strong":
                for _ in range(2):
                    sfm_b200.match_and_verify(bank, pairs_all, ratio=RATIO, pair_batch=PAIR_BATCH, **RANSAC)
                    flush.zero_()
                one_ms = []
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    sfm_b200.match_and_verify(bank, pairs_all, ratio=RATIO, pair_batch=PAIR_BATCH, **RANSAC)
                    e1.record()
                    e1.synchronize()
                    one_ms.append(e0.elapsed_time(e1))
                    flush.zero_()
                one_gpu = {"ms_per_step": float(np.mean(one_ms)), "pairs_per_s": P_total / (float(np.mean(one_ms)) * 1e-3),
                           "what": "the same pair list on rank 0 alone (bank resident, summaries only), 3 steps after 2 warm-ups"}
        dist.barrier()

    line = None
    if rank == 0:
        # ---- roofline of the dominant kernel (the tcgen05 sweep, tensor bound), measured live with CUDA events on the launch stream
        # (the launch shape of the timed step: a one-batch job runs as two halves, plan.B pairs per sweep launch)
        step_plan = getattr(last[1] if isinstance(last, tuple) else last, "plan", None)
        per_launch = int(step_plan.B) if step_plan is not None else min(len(my_pairs), PAIR_BATCH)
        rp = my_pairs[: min(len(my_pairs), per_launch)]
        knn = torch.empty((len(rp), bank.feat_stride, 4), dtype=torch.int32, device=dev)
        for _ in range(2):
            sfm_b200.knn2(bank, rp, impl="tcgen05", out=knn, sweep_only=4)
        sw_ms = []
        for _ in range(5):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sfm_b200.knn2(bank, rp, impl="tcgen05", out=knn, sweep_only=4)             # the sweep kernel alone (no pre-fill)
            e1.record()
            e1.synchronize()
            sw_ms.append(e0.elapsed_time(e1))
        sweep_ms = float(np.mean(sw_ms))
        del knn
        peaks, peak_src = load_peaks()
        sweep_ms_isolated, achieved_isolated = sweep_ms, len(rp) * OPS_PER_PAIR / (sweep_ms * 1e-3) / 1e12
        if insitu_sweeps:
            # the duration that counts: the sweep launches of the timed steps themselves (CUDA events on the launching stream; in the
            # two-stream pipeline every launch but the first shares the SMs with the previous batch's refinement and RANSAC)
            sweep_ms = float(np.mean([m for m, _ in insitu_sweeps]))
            per_launch = float(np.mean([n for _, n in insitu_sweeps]))
        else:
            per_launch = float(len(rp))
        achieved = per_launch * OPS_PER_PAIR / (sweep_ms * 1e-3) / 1e12
        probe_ms, probe_rate = matcher.probe_int8_peak(local, 4096)
        int8_gemm_tops = measure_int8_gemm_tops(dev)
        peak = 2.0 * float(peaks["bf16_tflops"])
        # ---- verification stage alone, on the step's own correspondences
        nb = min(PAIR_BATCH, len(my_pairs))
        plan = sfm_b200.match_and_verify(bank, my_pairs[:nb], ratio=RATIO, pair_ids=mine[:nb], pair_batch=PAIR_BATCH, **RANSAC).plan   # its buffers
        # now hold the job's LAST batch (a one-batch job runs as two halves on two streams)
        torch.cuda.synchronize()                                        # the plan's packed buffers now hold one batch
        rs_ms = []
        for _ in range(3):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            plan.rerun_ransac()
            e1.record()
            e1.synchronize()
            rs_ms.append(e0.elapsed_time(e1))
        ransac_ms = float(np.mean(rs_ms))
        m_counts = plan.cur.counts[: plan.cur.P].cpu().numpy().astype(np.float64)
        iters = plan.cur.iters[: plan.cur.P].cpu().numpy().astype(np.float64)
        ransac_roof = ransac_roofline(plan, ransac_ms, m_counts, iters, peaks, clocks)
        ninl = res.n_inliers.cpu().numpy()
        all_counts = res.n_matches.cpu().numpy().astype(np.float64)
        all_iters = res.iters.cpu().numpy().astype(np.float64)
        traffic = load_traffic()

        # ---- CPU baseline: the reference's cv2 path on this box's host cores, bounded sample
        import cv2

        cpu_value, cpu_dt = cv2_pairs_per_s(scene, pairs_one, 128)
        line = {
            "metric": "verified pairs/s", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "int8", "data": "synthetic",
            "config": {
                "workload": wl["label"] + ("" if scaling == "strong" or world == 1 else f"; the block replicated on each of {world} ranks"),
                "pairs_per_rank": int(len(my_pairs)), "pairs_total": int(P_total), "images": n_images, "features_per_image": N_FEATS,
                "ratio": RATIO, "ransac": RANSAC, "pair_order": args.pair_order + (f" ({PAIR_BLOCK} x {PAIR_BLOCK} image squares)" if args.pair_order == "blocked" else ""),
                "l2": f"flushed between timed iterations (256 MiB write; bank {bank.storage.numel() / 2**20:.0f} MiB, L2 126 MB)",
                "parallelism": ("one GPU" if world == 1 else
                                f"pair list block-partitioned over {world} ranks; bank broadcast once over NCCL (untimed, reported); inside the "
                                f"timed step every rank pushes its packed match rows + inlier flags into rank 0's HBM (transport "
                                f"{sharded_info['transport']}) and the per-pair summaries follow in one dist.gather"),
                "bank_bytes": int(bank.storage.numel()),
                "bank_broadcast_ms": None if world == 1 else {"first_call": bcast_ms[0], "warm": float(min(bcast_ms[1:]))},
                "sharded": sharded_info, "selfcheck": selfcheck, "one_gpu_same_workload": one_gpu,
                "mean_matches_per_pair": float(all_counts.mean()), "mean_inliers_per_pair": float(ninl.mean()),
                "mean_hypotheses_per_pair": float(all_iters.mean()), "host_enqueue_ms_per_step": host_ms,
            },
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps,
                    "what": f"match_and_verify_host(pinned uint8 descriptors + float32 keypoints, n_chunks={E2E_CHUNKS}, pair_batch="
                            f"{E2E_PAIR_BATCH}, fetch='view'): H2D in {E2E_CHUNKS} groups on a side stream, pack, match, filter, RANSAC-F, D2H of "
                            "all matches / inlier flags / F / counts into pinned host arrays; batch k's rows travel while batch k+1 "
                            "is swept" if world == 1 else
                            f"per rank: upload + pack 1/{world} of the images from pinned host memory, NCCL all-gather of the packed bank sections over NVLink "
                            f"(dist.upload_bank_sharded), match_and_verify(pair_batch={E2E_PAIR_BATCH}, fetch='view') on the rank's pair block: all "
                            "matches / inlier flags / F / counts into the rank's own pinned host arrays (bytes are summed over ranks)"},
            "gpu_launches": int(launches_per_step),
            "clocks": clocks,
            "roofline": {
                "kernel": "sfm::match_tc_kernel (tcgen05 kind::i8 sweep)", "bound": "tensor", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic.get("match_tc_kernel"),
                "traffic_source": traffic.get("source", "none") + " -- a committed ncu capture of this command, not measured by this run",
                "peak_source": f"2 x bf16_tflops of MEASURED_PEAKS.json ({peak_src}; the file has no int8 entry, int8 dense = 2 x bf16 dense)",
                "launch_ms": sweep_ms, "pairs_per_launch": per_launch, "algorithmic_ops_per_launch": per_launch * OPS_PER_PAIR,
                "launches_timed": len(insitu_sweeps),
                "launch_ms_how": "mean over the sweep launches of the timed steps (CUDA events on the launching stream)" if insitu_sweeps
                                 else "the sweep kernel launched alone after the timed steps",
                "launch_ms_alone": sweep_ms_isolated, "achieved_alone": achieved_isolated, "frac_alone": achieved_isolated / peak,
                "frac_of_nominal_4500": achieved / NOMINAL_INT8_TOPS,
                "peak_int8_measured_tops": int8_gemm_tops, "frac_of_int8_gemm": achieved / int8_gemm_tops,
                "peak_int8_measured_how": "torch._int_mm 8192^3 (cuBLASLt int8), best of 10, this run, this GPU",
                "mma_only_probe_tops": probe_rate / 1e12, "frac_of_mma_only_probe": achieved / (probe_rate / 1e12),
                "matcher_pairs_per_s_sweep_only": per_launch / (sweep_ms * 1e-3),
            },
            "roofline_ransac": ransac_roof,
            "cpu_baseline": {"value": cpu_value, "unit": "pairs/s", "cores": int(cv2.getNumThreads()), "kind": "reference",
                             "sample": f"128 pairs of the same scene through cv2 {cv2.__version__} (knnMatch k=2 on f32 + ratio + findFundamentalMat FM_RANSAC), {cpu_dt:.1f} s"},
        }
    if world > 1:
        dist.barrier()
        for reg in bank.__dict__.get("_gather_regions", {}).values():
            reg.close()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))


def ransac_roofline(plan, ransac_ms, m_counts, iters, peaks, clocks):
    """Verification kernel against the bound that really limits it (VERDICT round 1, SURVEY.md §8d caveat): the
    correspondences live in shared memory, so the kernel is FP32-issue bound, not HBM bound.  ``H*M*16`` "algorithmic bytes"
    are kept as labelled context only."""
    hm = float((iters * m_counts).sum())
    sm_mhz = float((clocks or {}).get("sm_max_mhz") or 1965.0)
    issue_peak = 148 * 128 * sm_mhz * 1e6 / 1e12                          # T instructions / s: 148 SMs x 128 FP32 lanes
    ach = hm * RANSAC_INSTR_PER_EVAL / (ransac_ms * 1e-3) / 1e12
    return {
        "kernel": "sfm::ransac_f_kernel", "bound": "fp32 issue", "achieved": ach, "peak": issue_peak, "unit": "T fp32 instr/s", "frac": ach / issue_peak,
        "launch_ms": ransac_ms, "pairs_per_launch": int(len(m_counts)),
        "instr_per_hypothesis_point": RANSAC_INSTR_PER_EVAL, "flop_per_hypothesis_point": RANSAC_FLOP_PER_EVAL,
        "achieved_tflops": hm * RANSAC_FLOP_PER_EVAL / (ransac_ms * 1e-3) / 1e12, "peak_tflops_fma": 2.0 * issue_peak,
        "evaluations": hm, "note": "scoring only: evaluations = sum over pairs of hypotheses x correspondences (upper bound: the exact bail-out of "
                                   "later batches skips part of the stream); the minimal solves, the final mask pass and the launch's tail "
                                   "(1 CTA per pair, ~4 waves) are not credited; peak = 148 SMs x 128 FP32 lanes x max SM clock",
        "context_algorithmic_GBps_H_M_16": hm * 16.0 / (ransac_ms * 1e-3) / 1e9, "context_hbm_gbs": float(peaks["hbm_gbs"]),
        "context_note": "north_star frames scoring as HBM-bound with H*M*16 B per pair; the points are staged in shared memory, real DRAM "
                        "traffic is ~M*16 B per pair (profiles/), so that ratio is not a bandwidth and is NOT reported as frac",
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="auto", choices=["auto", "c2", "c3"], help="auto: configs[1] on one GPU, configs[2] sharded")
    ap.add_argument("--scaling", default="auto", choices=["auto", "strong", "weak"], help="N > 1: strong (default) or the N = 1 block per rank")
    ap.add_argument("--pair-order", default="blocked", choices=["blocked", "sorted"], help="exhaustive pair list in 32 x 32 image squares or (i, j)-sorted")
    ap.add_argument("--no-overlap", action="store_true", help="diagnostics: one stream (no two-stream pipeline)")
    ap.add_argument("--gather", default="full", choices=["full", "summaries"], help="what rank 0 receives inside the timed step (N > 1)")
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "sendrecv"], help="row gather transport (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
