"""Time registration (csrc/pnp.cu) on the bench's workloads, in one process on one GPU.

For each workload (c2 = BASELINE configs[1]: 50 images x 8192 features, 1,225 pairs; c3 = configs[2]: 200 x 8192, 19,900 pairs)
the tracks are built in the plan (match_and_verify(..., tracks=True)), triangulated from the scene's true cameras, and every image
is registered in one batch with the default parameters:
  * the gather (sfm_pnp_gather) and the RANSAC (memset + sfm_pnp_ransac), each timed with CUDA events, median of --reps after
    warm-up, L2 overwritten before every timed call; queries/s and correspondences/s over the RANSAC time;
  * the status histogram, the hypotheses drawn, the median rotation error and camera-centre error against the true cameras;
  * the C oracle on the same gathered correspondences, once (host CPU), and whether the GPU result equals it bit for bit.
The card's name, power limit and clocks are read in the same run.

    python tools/time_pnp.py [--configs c2,c3] [--reps 50] [--out FILE]
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
    from oracle import pnp_oracle as po
    from sfm_b200 import pnp
    from sfm_b200 import synth
    from sfm_b200 import triangulate as tri

    if not torch.cuda.is_available():
        raise SystemExit("time_pnp.py measures on a GPU; none is visible")
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

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        return float(np.median(ms)), min(ms), max(ms)

    for name in args.configs.split(","):
        n_img, seed = WORKLOADS[name]
        say()
        say(f"== {name}: {n_img} images x {N_FEATS} features, exhaustive pairs (blocked order), tracks from the inlier rows, points "
            f"triangulated from the scene's true cameras, every image registered in one batch, default parameters (max_error 12 px, "
            f"confidence 0.9999, max_iters 10000, min_inliers 30, min_inlier_ratio 0.25, refine_iters 10)")
        sc = synth.make_scene(n_img, N_FEATS, seed=seed)
        bank = sfm_b200.DescriptorBank(n_img, N_FEATS, device=dev)
        bank.put(0, sc.desc, xy=sc.xy)
        pairs = sfm_b200.blocked_exhaustive_pairs(n_img, 32)
        res = sfm_b200.match_and_verify(bank, pairs, ratio=0.75, pair_batch=2048, tracks=True, **RANSAC)
        Rt = np.einsum("ij,njk->nik", np.linalg.inv(synth.K_INTR), sc.P)
        cams_h = tri.camera_table(synth.K_INTR, Rt[:, :, :3], Rt[:, :, 3])
        cams = torch.from_numpy(cams_h).to(dev)
        trk = res.tracks
        pts = tri.triangulate_tracks_device(trk, bank.xy, cams, S=bank.max_feats)
        images = torch.arange(n_img, dtype=torch.int32, device=dev)
        g_xy, g_X, feature, count = pnp.gather_device(trk, pts, bank.xy, images)
        n_corr = int(count.sum())
        say(f"tracks {trk.n_tracks:,}, triangulated {pts.counts['triangulated']:,}; correspondences {n_corr:,} "
            f"({n_corr / n_img:,.0f} per image, max {int(count.max()):,})")

        g_med, g_min, g_max = timed(lambda: pnp.gather_device(trk, pts, bank.xy, images))
        say(f"sfm_pnp_gather: median {g_med:.3f} ms (min {g_min:.3f}, max {g_max:.3f}) over {args.reps}")
        r_med, r_min, r_max = timed(lambda: pnp.pnp_ransac_device(g_xy, g_X, count, cams, images))
        say(f"sfm_pnp_ransac: median {r_med:.3f} ms (min {r_min:.3f}, max {r_max:.3f}) over {args.reps}; "
            f"{n_img / (r_med * 1e-3) / 1e3:.1f} K queries/s, {n_corr / (r_med * 1e-3) / 1e6:.1f} M correspondences/s")

        out = pnp.pnp_ransac_device(g_xy, g_X, count, cams, images).to_host()
        say("statuses: " + ", ".join(f"{k} {out[k]:,}" for k in pnp.STATUS_NAMES))
        say(f"hypotheses drawn: min {out['iters'].min()}, median {int(np.median(out['iters']))}, max {out['iters'].max()}; "
            f"inlier fraction median {np.median(out['n_inliers'] / np.maximum(out['count'], 1)):.4f}")
        ok = out["status"] == 0
        rot = [np.degrees(np.arccos(np.clip((np.trace(out["R"][i] @ Rt[i, :, :3].T) - 1) / 2, -1, 1))) for i in np.nonzero(ok)[0]]
        cen = [np.linalg.norm(-out["R"][i].T @ out["t"][i] + Rt[i, :, :3].T @ Rt[i, :, 3]) for i in np.nonzero(ok)[0]]
        say(f"median rotation error {np.median(rot):.5f} deg, median camera-centre error {np.median(cen):.6f} (scene units; points at "
            f"depth 4-8)")

        h_xy, h_X, h_count = g_xy.cpu().numpy(), g_X.cpu().numpy(), count.cpu().numpy()
        t0 = time.perf_counter()
        ref = po.pnp_ransac(h_xy, h_X, h_count, cams_h, np.arange(n_img, dtype=np.int32))
        t_oracle = time.perf_counter() - t0
        same = all(np.array_equal(np.asarray(out[k]).view(np.uint8), np.asarray(ref[k]).view(np.uint8))
                   for k in ("pose", "n_inliers", "status", "mask", "iters"))
        same &= [out[k] for k in pnp.STATUS_NAMES] == ref["counts"].tolist()
        say(f"C oracle on the same correspondences (host CPU, once): {t_oracle:.2f} s; GPU result == oracle bit for bit: {same}")
        del res, bank, trk, pts
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
