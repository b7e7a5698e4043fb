"""Time incremental reconstruction (sfm_b200.reconstruct_device) on the bench's workloads, in one process on one GPU.

For each workload (c2 = BASELINE configs[1]: 50 images x 8192 features; c3 = configs[2]: 200 x 8192) the pairs are matched and
verified with the homography and two-view pose stages and the tracks built (match_and_verify(..., homography=True,
intrinsics=K, tracks=True)); then reconstruct_device runs with the default parameters:
  * the whole call on the host clock (it ends on a host read, so the clock covers the GPU work), median of --reps;
  * one call under torch.profiler: the kernel time of each stage (next images, gather + PnP, triangulation, bundle adjustment,
    filter) in all and per round, and the share of the call in which no kernel runs (the host's waits and work between
    launches);
  * rounds, registered images, the median rotation and centre errors after a similarity alignment to the scene's cameras,
    and the RMS reprojection error of the inlier observations;
  * at c2, the whole call at max_per_round 1, 4, 16 and 64.
The card's name, power limit and clocks are read in the same run.

    python tools/time_reconstruct.py [--configs c2,c3] [--reps 3] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "sfm-project_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {"c2": (50, 2001), "c3": (200, 3001)}       # bench.py's seeds
N_FEATS = 8192
RANSAC = dict(thr=3.0, confidence=0.99, max_iters=2000, solver="8pt", score="sym_epipolar", lo=False, seed=1)
STAGES = [("next images", ("next_score_kernel", "next_select_kernel")), ("gather + PnP", ("pnp_gather_kernel", "pnp_ransac_kernel")),
          ("triangulation", ("triangulate_kernel",)), ("bundle adjustment", ("ba_",)), ("filter", ("filter_kernel",))]


def umeyama(src, dst):
    ms, md = src.mean(0), dst.mean(0)
    a, b = src - ms, dst - md
    U, D, Vt = np.linalg.svd(b.T @ a / len(src))
    S = np.eye(3)
    if np.linalg.det(U) * np.linalg.det(Vt) < 0:
        S[2, 2] = -1
    Q = U @ S @ Vt
    s = np.trace(np.diag(D) @ S) / a.var(0).sum()
    return s, Q, md - s * Q @ ms


def errors(R, t, Rt, idx, depth):
    from scipy.spatial.transform import Rotation

    C_est = np.stack([-R[i].T @ t[i] for i in idx])
    C_true = np.stack([-Rt[i, :, :3].T @ Rt[i, :, 3] for i in idx])
    s, Q, c = umeyama(C_est, C_true)
    cen = np.linalg.norm((s * (Q @ C_est.T)).T + c - C_true, axis=1)
    rot = [np.degrees(Rotation.from_matrix(R[i] @ Q.T @ Rt[i, :, :3].T).magnitude()) for i in idx]
    return float(np.median(rot)), float(100 * np.median(cen) / depth)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", help="also write the report here")
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile

    import sfm_b200
    from sfm_b200 import mapper, synth

    if not torch.cuda.is_available():
        raise SystemExit("time_reconstruct.py measures on a GPU; none is visible")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    say(f"device: {torch.cuda.get_device_name(dev)}")
    say(f"nvidia-smi: {' | '.join(smi.splitlines())}")
    K = synth.K_INTR

    for name in args.configs.split(","):
        n_img, seed = WORKLOADS[name]
        say()
        sc = synth.make_scene(n_img, N_FEATS, seed=seed)
        bank = sfm_b200.DescriptorBank(n_img, N_FEATS, device=dev)
        bank.put(0, sc.desc, xy=sc.xy)
        res = sfm_b200.match_and_verify(bank, sfm_b200.blocked_exhaustive_pairs(n_img, 32), ratio=0.75, pair_batch=2048, tracks=True,
                                        homography=True, intrinsics=K, **RANSAC)
        Rt = np.einsum("ij,njk->nik", np.linalg.inv(K), sc.P)
        depth = float(np.median(sc.X @ Rt[0, 2, :3] + Rt[0, 2, 3]))
        say(f"== {name}: {n_img} images x {N_FEATS} features; {res.pairs.shape[0]:,} pairs; tracks {res.tracks.n_tracks:,}, observations "
            f"{res.tracks.n_obs:,}")

        def call(**kw):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            rec = mapper.reconstruct_device(res, bank.xy, K, **kw)
            torch.cuda.synchronize()
            return rec, (time.perf_counter() - t0) * 1e3

        rec, _ = call()                                     # warm-up
        ms = [call()[1] for _ in range(args.reps)]
        h = rec.to_host()
        reg = np.nonzero(h["registered"])[0]
        n_rounds = len(h["rounds"]) - 1
        say(f"whole call: median {np.median(ms):.1f} ms (min {min(ms):.1f}, max {max(ms):.1f}) over {args.reps}; status {h['status']}, "
            f"initial pair {h['init_pair']}, {n_rounds} rounds, {len(reg)} of {n_img} images registered")
        ok = h["point_status"] == 0
        e = h["obs_error"][h["obs_inlier"] == 1].astype(np.float64)
        rot, cen = errors(h["R"], h["t"], Rt, reg, depth) if len(reg) >= 3 else (float("nan"), float("nan"))
        say(f"points {int(ok.sum()):,}, inlier observations {len(e):,}, RMS reprojection error {np.sqrt(np.mean(e ** 2)):.4f} px; after a "
            f"similarity alignment: rotation error median {rot:.5f} deg, centre error median {cen:.5f} % of the median depth")
        for r in h["rounds"]:
            say(f"  round {r['round']:3d}: selected {len(r['selected']):3d}, registered {len(r['registered']):3d}"
                + (f", BA {r['ba_status']} after {r['ba_iterations']} iterations, cost {r['initial_cost']:.4e} -> {r['final_cost']:.4e}, "
                   f"filtered {r['filtered_obs']:,} observations, points {r['points']:,}" if "ba_status" in r else ""))

        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            t0 = time.perf_counter()
            call()
            wall = (time.perf_counter() - t0) * 1e6
        kern = [ev for ev in prof.events() if ev.device_type.name == "CUDA"]
        per = {s: 0.0 for s, _ in STAGES}
        for ev in kern:
            for s, keys in STAGES:
                if any(k in ev.name for k in keys):
                    per[s] += ev.time_range.elapsed_us()
        iv = sorted((ev.time_range.start, ev.time_range.end) for ev in kern)
        busy, cur_s, cur_e = 0.0, None, None
        for a, b in iv:
            if cur_e is None or a > cur_e:
                if cur_e is not None:
                    busy += cur_e - cur_s
                cur_s, cur_e = a, b
            else:
                cur_e = max(cur_e, b)
        if cur_e is not None:
            busy += cur_e - cur_s
        say(f"under torch.profiler: call {wall / 1e3:.1f} ms, kernels busy {busy / 1e3:.1f} ms; share of the call with no kernel running "
            f"(host waits and host work between launches): {100 * (1 - busy / wall):.1f} %")
        for s, _ in STAGES:
            say(f"  {s:20s} {per[s] / 1e3:9.2f} ms in all, {per[s] / 1e3 / max(n_rounds + 1, 1):8.2f} ms per round")
        if name == "c2":
            for m in (1, 4, 16, 64):
                call(max_per_round=m)
                t = [call(max_per_round=m) for _ in range(args.reps)]
                hh = t[0][0].to_host()
                say(f"max_per_round {m:3d}: whole call median {np.median([x[1] for x in t]):.1f} ms, {len(hh['rounds']) - 1} rounds, "
                    f"{int(hh['registered'].sum())} registered")
        del res, bank, rec
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
