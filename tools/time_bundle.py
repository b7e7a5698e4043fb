"""Time bundle adjustment (csrc/bundle.cu) on the bench's workloads, in one process on one GPU.

For each workload (c2 = BASELINE configs[1]: 50 images x 8192 features; c3 = configs[2]: 200 x 8192) the tracks are built in
the plan (match_and_verify(..., tracks=True)), the scene's true cameras are perturbed (rotations of about 0.3 degree, centres
moved about 1 % of the median depth), the tracks triangulated from the perturbed cameras, and every camera but image 0 (the
default gauge) is adjusted with the default parameters:
  * the whole call with CUDA events (median of --reps, L2 overwritten before each), and one call under torch.profiler: the
    time of each stage per working iteration (blocks, Schur build, factorisation and solve, back-substitution and trial
    cost, decision) and the cost of the idle iterations after the stop;
  * iterations, status, the final RMS error per coordinate against the 0.5 px pixel noise, the ground-truth errors after a
    similarity alignment before and after;
  * the float64 reference (tests/bundle_reference.py) once on the host at c2, for comparison.
The card's name, power limit and clocks are read in the same run.

    python tools/time_bundle.py [--configs c2,c3] [--reps 5] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "sfm-project_b200"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {"c2": (50, 2001), "c3": (200, 3001)}       # bench.py's seeds
N_FEATS = 8192
RANSAC = dict(thr=3.0, confidence=0.99, max_iters=2000, solver="8pt", score="sym_epipolar", lo=False, seed=1)
STAGES = [("ba_point_kernel", "blocks (J, V, V^-1)"), ("ba_camera_kernel", "Schur build"), ("ba_solve_kernel", "factorisation + solve"),
          ("ba_update_kernel", "back-substitution + trial cost"), ("ba_decide_kernel", "decision")]


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


def errors(R, t, Rt, depth):
    from scipy.spatial.transform import Rotation

    C_est = np.stack([-R[i].T @ t[i] for i in range(len(R))])
    C_true = np.stack([-Rt[i, :, :3].T @ Rt[i, :, 3] for i in range(len(R))])
    s, Q, c = umeyama(C_est, C_true)
    cen = np.linalg.norm((s * (Q @ C_est.T)).T + c - C_true, axis=1)
    rot = [np.degrees(Rotation.from_matrix(R[i] @ Q.T @ Rt[i, :, :3].T).magnitude()) for i in range(len(R))]
    return float(np.median(rot)), float(100 * np.median(cen) / depth)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--max-iters", type=int, default=50)
    ap.add_argument("--out", help="also write the report here")
    args = ap.parse_args()
    import torch
    from scipy.spatial.transform import Rotation

    import bundle_reference as br
    import sfm_b200
    from sfm_b200 import bundle, synth
    from sfm_b200 import triangulate as tri

    if not torch.cuda.is_available():
        raise SystemExit("time_bundle.py measures on a GPU; none is visible")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                          "--format=csv"], capture_output=True, text=True).stdout.strip()
    say(f"device: {torch.cuda.get_device_name(dev)}")
    say(f"nvidia-smi: {' | '.join(smi.splitlines())}")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    for name in args.configs.split(","):
        n_img, seed = WORKLOADS[name]
        say()
        sc = synth.make_scene(n_img, N_FEATS, seed=seed)
        bank = sfm_b200.DescriptorBank(n_img, N_FEATS, device=dev)
        bank.put(0, sc.desc, xy=sc.xy)
        res = sfm_b200.match_and_verify(bank, sfm_b200.blocked_exhaustive_pairs(n_img, 32), ratio=0.75, pair_batch=2048, tracks=True, **RANSAC)
        Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
        depth = float(np.median(sc.X @ Rt[0, 2, :3] + Rt[0, 2, 3]))
        rng = np.random.default_rng(seed)
        R0, t0 = Rt[:, :, :3].copy(), Rt[:, :, 3].copy()
        for i in range(1, n_img):
            C = -R0[i].T @ t0[i] + rng.normal(size=3) * 0.01 * depth / np.sqrt(3)
            R0[i] = Rotation.from_rotvec(rng.normal(size=3) * np.radians(0.3) / np.sqrt(3)).as_matrix() @ R0[i]
            t0[i] = -R0[i] @ C
        cams_h = tri.camera_table(synth.K_INTR, R0, t0)
        cams = torch.from_numpy(cams_h).to(dev)
        trk = res.tracks
        pts = tri.triangulate_tracks_device(trk, bank.xy, cams, S=bank.max_feats)
        ws = torch.empty(bundle.workspace_bytes(n_img, pts.X_buf.shape[0], pts.obs_inlier_buf.numel()), dtype=torch.uint8, device=dev)
        call = lambda: bundle.bundle_adjust_device(trk, pts, bank.xy, cams, S=bank.max_feats, workspace=ws, max_iters=args.max_iters)  # noqa: E731
        out = call().to_host()
        say(f"== {name}: {n_img} images x {N_FEATS} features; tracks {trk.n_tracks:,}, observations {trk.n_obs:,}, triangulated "
            f"{pts.counts['triangulated']:,}; used observations {out['used_obs']:,}, variable cameras {out['variable_cameras']}, adjusted "
            f"points {out['adjusted_points']:,}; max_iters {args.max_iters} ({bundle.bundle_launches(args.max_iters)} launches)")
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            call()
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        say(f"whole call: median {np.median(ms):.2f} ms (min {min(ms):.2f}, max {max(ms):.2f}) over {args.reps}")
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        per = {}
        for ev in sorted(prof.events(), key=lambda e: e.time_range.start):
            key = next((k for k, _ in STAGES if k in ev.name), None)
            if key is not None and ev.device_type.name == "CUDA":
                per.setdefault(key, []).append(ev.time_range.elapsed_us())
        it = out["iterations"]
        busy_total = 0.0
        for key, label in STAGES:
            t_us = np.array(per.get(key, []), np.float64)
            if len(t_us) == 0:
                continue
            work, idle = t_us[:it], t_us[it:]
            busy_total += work.sum()
            say(f"  {label:32s} {work.mean() / 1e3 if len(work) else 0:9.3f} ms per working iteration; idle {idle.mean() if len(idle) else 0:7.2f} us "
                f"x {len(idle)}")
        idle_all = sum(np.sum(np.array(per.get(k, []))[it:]) for k, _ in STAGES)
        say(f"  working iterations {it} ({out['accepted']} accepted): {busy_total / 1e3:.2f} ms of kernels; the idle iterations after the "
            f"stop: {idle_all / 1e3:.3f} ms of kernels in all")
        rms = np.sqrt(out["final_cost"] / (2 * out["used_obs"]))
        before = errors(R0, t0, Rt, depth)
        after = errors(out["R"], out["t"], Rt, depth)
        say(f"status {out['status']} after {it} iterations; cost {out['initial_cost']:.6e} -> {out['final_cost']:.6e}; RMS per coordinate "
            f"{rms:.4f} px (pixel noise 0.5 px)")
        say(f"ground truth after a similarity alignment: rotation error median {before[0]:.4f} -> {after[0]:.5f} deg, centre error median "
            f"{before[1]:.4f} -> {after[1]:.5f} % of the median depth")
        nv, T = out["variable_cameras"], out["adjusted_points"]
        say(f"arithmetic from shapes: S is {6 * nv} x {6 * nv}, Cholesky {(6 * nv) ** 3 / 3 / 1e9:.3f} GFLOP")
        if name == "c2":
            h = pts.to_host()
            th = trk.to_host()
            cam, pt, o, var, adj = br.problem(th["offsets"], th["obs"], h["status"], h["obs_inlier"], n_img)
            pxy = sc.xy[cam, th["obs"][o, 1]].astype(np.float64)
            t0c = time.perf_counter()
            ref = br.bundle_adjust(cams_h, h["X"], cam, pt, pxy, var, adj, max_iters=args.max_iters, ftol=1e-6)
            say(f"float64 reference (host CPU, sparse normal equations, once): {time.perf_counter() - t0c:.1f} s, {ref['iterations']} iterations, "
                f"cost {ref['cost']:.6e} (GPU {out['final_cost']:.6e}, relative difference {abs(ref['cost'] - out['final_cost']) / ref['cost']:.2e})")
        del res, bank, trk, pts, ws
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
