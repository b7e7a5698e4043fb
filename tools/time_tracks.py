"""Time the feature-track builder (csrc/tracks.cu) on the bench's workloads, in one process on one GPU.

For each workload (c2 = BASELINE configs[1]: 50 images x 8192 features, 1,225 pairs; c3 = configs[2]: 200 x 8192, 19,900
pairs) the verified rows are produced on the device through the world-size-1 row sink, then:
  * what the tracks are: rows used, nodes, tracks, observations, conflicting / short candidates, the track-length histogram;
  * the standalone build (init + hook + finalize over the whole job) and each entry point alone: CUDA events, median of --reps
    after warm-up;
  * the hook's bytes over time: 13 B per row of a pair that passes the pair filter (12 B row + 1 B flag), over the hook's
    time -- a figure computed from the row count, not a measured DRAM rate;
  * the in-plan cost: the bench-shape match_and_verify step (bench.py's resident one-GPU step) with and without tracks=True,
    alternated, CUDA events, L2 overwritten between steps;
  * the numpy oracle on the same rows, once (and whether it equals the GPU result).
The card's name, power limit and clocks are read in the same run.

    python tools/time_tracks.py [--configs c2,c3] [--reps 20] [--out FILE]
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
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the report here")
    args = ap.parse_args()
    import torch

    import sfm_b200
    from oracle import track_oracle as to
    from sfm_b200 import dist as sdist
    from sfm_b200 import synth
    from sfm_b200 import tracks as tr

    if not torch.cuda.is_available():
        raise SystemExit("time_tracks.py measures on a GPU; none is visible")
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

    def events_ms(fn, reps, warmup, setup=None):
        for _ in range(warmup):
            if setup:
                setup()
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            if setup:
                setup()
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms.append(a.elapsed_time(b))
        return float(np.median(ms)), float(np.min(ms)), float(np.max(ms))

    for name in args.configs.split(","):
        n_img, seed = WORKLOADS[name]
        say()
        say(f"== {name}: {n_img} images x {N_FEATS} features, exhaustive pairs (blocked order), flags=inlier, min_pair_inliers=15")
        sc = synth.make_scene(n_img, N_FEATS, seed=seed)
        bank = sfm_b200.DescriptorBank(n_img, N_FEATS, device=dev)
        bank.put(0, sc.desc, xy=sc.xy)
        pairs = sfm_b200.blocked_exhaustive_pairs(n_img, 32)
        out, _ = sdist.match_and_verify_sharded(bank, pairs, ratio=0.75, pair_batch=2048, **RANSAC)
        torch.cuda.synchronize()
        P = len(pairs)
        rows_total = int(out["n_matches"].sum())
        passing = out["n_inliers"] >= 15
        rows_read = int(out["n_matches"][passing].sum())
        say(f"pairs {P}, rows {rows_total:,}, rows of pairs passing the pair filter {rows_read:,} ({int(passing.sum())} pairs)")

        # standalone, whole job, and per entry point
        t_build = events_ms(lambda: tr.build_tracks_from_rows(out, n_img, N_FEATS), args.reps, args.warmup)
        b = tr.TrackBuilder(n_img, N_FEATS, dev)
        pairs_d = torch.as_tensor(out["pairs"], device=dev)
        rs, nm, m, inl, ni = out["row_start"], out["n_matches"], out["matches"], out["inlier"], out["n_inliers"]
        t_init = events_ms(b.begin, args.reps, args.warmup)
        # the hook into a freshly initialised forest (re-hooking a finished one would only time the finds)
        t_hook = events_ms(lambda: b.hook(pairs_d, rs, nm, m, inl, ni), args.reps, args.warmup, setup=b.begin)
        t_fin = events_ms(b.finalize, args.reps, args.warmup)
        say(f"standalone build (init + hook + finalize, incl. workspace/output allocation): median {t_build[0]:.3f} ms "
            f"(min {t_build[1]:.3f}, max {t_build[2]:.3f})")
        say(f"  sfm_tracks_init     median {t_init[0]:.3f} ms")
        say(f"  sfm_tracks_hook     median {t_hook[0]:.3f} ms   bytes over time: 13 B x {rows_read:,} rows / hook time = "
            f"{13 * rows_read / (t_hook[0] * 1e-3) / 1e9:.1f} GB/s")
        say(f"  sfm_tracks_finalize median {t_fin[0]:.3f} ms")
        t = tr.build_tracks_from_rows(out, n_img, N_FEATS).to_host()
        lens = np.diff(t["offsets"])
        hist = np.bincount(lens) if len(lens) else np.zeros(1, int)
        say(f"tracks {t['n_tracks']:,}, observations {t['n_obs']:,}, conflicting candidates dropped {t['n_conflicting']:,}, "
            f"short candidates dropped {t['n_short']:,}, mean length {t['n_obs'] / max(t['n_tracks'], 1):.2f}, longest {int(lens.max()) if len(lens) else 0}")
        say("track-length histogram: " + ", ".join(f"{k}: {int(c):,}" for k, c in enumerate(hist) if c))

        # the numpy oracle on the same rows, once
        h = {k: out[k].cpu().numpy() for k in ("row_start", "n_matches", "matches", "inlier", "n_inliers")}
        h["pairs"] = out["pairs"]
        t0 = time.perf_counter()
        u, v, _ = to.used_edges(h["pairs"], h["row_start"], h["n_matches"], h["matches"], h["inlier"], h["n_inliers"], n_img, N_FEATS)
        ref = to.tracks_from_edges(u, v, n_img, N_FEATS)
        t_oracle = time.perf_counter() - t0
        same = all(np.array_equal(np.asarray(ref[k]), np.asarray(t[k])) for k in ref)
        say(f"rows used {len(u):,}, nodes {len(np.unique(np.concatenate([u, v]))):,}")
        say(f"numpy oracle on the same rows (host CPU, once): {t_oracle:.2f} s; GPU result == oracle: {same}")

        # in-plan cost: the bench-shape step with and without tracks=True, alternated
        ids = np.arange(P)
        steps = {False: [], True: []}

        def step(trk):
            return sfm_b200.match_and_verify(bank, pairs, ratio=0.75, pair_ids=ids, pair_batch=2048, tracks=trk, **RANSAC)

        for trk in (False, True):
            for _ in range(args.warmup):
                step(trk)
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for trk in (False, True):
                flush.zero_()
                a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                step(trk)
                e.record()
                e.synchronize()
                steps[trk].append(a.elapsed_time(e))
        m0, m1 = float(np.median(steps[False])), float(np.median(steps[True]))
        say(f"bench-shape step (match_and_verify, pair_batch 2048, resident bank), alternated, median of {args.reps}: "
            f"without tracks {m0:.3f} ms, with tracks=True {m1:.3f} ms (+{m1 - m0:.3f} ms, {100 * (m1 - m0) / m0:+.1f} %)")
        del out, bank
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
