"""Time the track triangulation (csrc/triangulate.cu) on the bench's workloads, in one process on one GPU.

For each workload (c2 = BASELINE configs[1]: 50 images x 8192 features, 1,225 pairs; c3 = configs[2]: 200 x 8192, 19,900 pairs)
the tracks are built in the plan (match_and_verify(..., tracks=True)) from the verified rows, then triangulated with the scene's
true cameras:
  * the kernel: CUDA events around sfm_triangulate_tracks (memset + one launch), median of --reps after warm-up, L2 overwritten
    between launches; tracks/s and observations/s over that time;
  * the status histogram, the inlier fraction, the median reprojection error and the median 3-D error against the scene points;
  * the C oracle on the same tracks, once (host CPU), and whether the GPU result equals it bit for bit.
The card's name, power limit and clocks are read in the same run.

    python tools/time_triangulate.py [--configs c2,c3] [--reps 50] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="c2,c3")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", help="also write the report here")
    args = ap.parse_args()
    import torch

    import sfm_b200
    from oracle import triangulate_oracle as tro
    from sfm_b200 import synth
    from sfm_b200 import triangulate as tri

    if not torch.cuda.is_available():
        raise SystemExit("time_triangulate.py measures on a GPU; none is visible")
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
        say(f"== {name}: {n_img} images x {N_FEATS} features, exhaustive pairs (blocked order), tracks from the inlier rows "
            f"(min_pair_inliers=15), the scene's true cameras, default parameters (max_error 4 px, min_angle 1.5 deg, "
            f"max_iters 500, confidence 0.999)")
        sc = synth.make_scene(n_img, N_FEATS, seed=seed)
        bank = sfm_b200.DescriptorBank(n_img, N_FEATS, device=dev)
        bank.put(0, sc.desc, xy=sc.xy)
        pairs = sfm_b200.blocked_exhaustive_pairs(n_img, 32)
        res = sfm_b200.match_and_verify(bank, pairs, ratio=0.75, pair_batch=2048, tracks=True, **RANSAC)
        Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
        cams_h = tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])
        cams = torch.from_numpy(cams_h).to(dev)
        trk = res.tracks
        T, n_obs = trk.n_tracks, trk.n_obs
        say(f"tracks {T:,}, observations {n_obs:,}, mean length {n_obs / max(T, 1):.2f}")

        def run():
            return tri.triangulate_tracks_device(trk, bank.xy, cams, S=bank.max_feats)

        for _ in range(args.warmup):
            run()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run()
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        med = float(np.median(ms))
        say(f"sfm_triangulate_tracks: median {med:.3f} ms (min {min(ms):.3f}, max {max(ms):.3f}) over {args.reps}; "
            f"{T / (med * 1e-3) / 1e6:.2f} M tracks/s, {n_obs / (med * 1e-3) / 1e6:.1f} M observations/s")

        pts = run().to_host()
        say("statuses: " + ", ".join(f"{k} {pts[k]:,}" for k in tri.STATUS_NAMES))
        t = trk.to_host()
        ok = pts["status"] == 0
        seg = np.repeat(np.arange(T), np.diff(t["offsets"]))
        inl = pts["obs_inlier"] == 1
        pid = sc.point[t["obs"][t["offsets"][:-1], 0], t["obs"][t["offsets"][:-1], 1]]
        d3 = np.linalg.norm(pts["X"][ok] - sc.X[pid[ok]], axis=1)
        say(f"inlier observations {inl.mean():.4f}; median reprojection error of the inliers {np.median(pts['obs_error'][inl & ok[seg]]):.3f} px; "
            f"median 3-D error {np.median(d3):.5f} (scene units; points at depth 4-8)")

        t0 = time.perf_counter()
        ref = tro.triangulate_tracks(t["offsets"], t["obs"], sc.xy, cams_h)
        t_oracle = time.perf_counter() - t0
        same = all(np.array_equal(np.asarray(pts[k]).view(np.uint8), np.asarray(ref[k]).view(np.uint8))
                   for k in ("X", "n_inliers", "status", "obs_inlier", "obs_error"))
        same &= [pts[k] for k in tri.STATUS_NAMES] == ref["counts"].tolist()
        say(f"C oracle on the same tracks (host CPU, once): {t_oracle:.2f} s; GPU result == oracle bit for bit: {same}")
        del res, bank, trk
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
