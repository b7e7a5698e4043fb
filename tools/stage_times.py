"""Per-stage device times of the resident bench step (configs[1]: 1,225 pairs x 8192 features), each stage timed alone
with CUDA events on the launch stream after an L2 flush, next to the whole step.  Diagnostic, not a bench line."""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "sfm-project_b200")]
import sfm_b200  # noqa: E402
from sfm_b200 import _lib, synth  # noqa: E402

n_img = int(sys.argv[1]) if len(sys.argv) > 1 else 50
sc = synth.make_scene(n_img, 8192, seed=2001)
pairs = synth.exhaustive_pairs(n_img)
bank = sfm_b200.DescriptorBank(n_img, 8192)
bank.put(0, sc.desc, xy=sc.xy)
R = dict(thr=3.0, confidence=0.99, max_iters=2000, solver="8pt", score="sym_epipolar", lo=False, seed=1)
plan = sfm_b200.get_plan(bank, min(2048, len(pairs)), ratio=0.75, ratio_mode="cv2_f32", mutual=False, min_inliers=0,
                         prefilter=True, overlap=False, **R)        # stages timed one by one on one stream
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
L, dev = _lib.lib(), bank.device
P = min(len(pairs), plan.B)
pairs_d = torch.from_numpy(pairs[:P]).cuda()
ids_d = torch.arange(P, dtype=torch.int32, device="cuda")
st = lambda: _lib.current_stream_ptr(dev)  # noqa: E731


def timed(fn, reps=5, flush_l2=True):
    fn(); torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush_l2:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return round(float(np.median(ts)), 4)


def match(sweep_only):
    m = _lib.MatchParams()
    m.impl, m.sweep_only = plan.mprm.impl, int(sweep_only)
    m.prefilter_mode, m.prefilter_ratio = plan.fprm.ratio_mode, plan.fprm.ratio
    m.prefilter_num, m.prefilter_den = int(plan.fprm.ratio_num), int(plan.fprm.ratio_den)
    _lib.check(L.sfm_match_knn2(bank.handle, _lib.ptr(pairs_d), P, C.byref(m), _lib.ptr(plan.knn), st()), "knn2")


def filt():
    o = plan.cur
    _lib.check(L.sfm_filter_matches_packed(bank.handle, _lib.ptr(pairs_d), P, _lib.ptr(plan.knn), None, C.byref(plan.fprm), _lib.ptr(o.counts),
                                           _lib.ptr(o.offsets), _lib.ptr(o.matches), _lib.ptr(o.corr), st()), "filter")


out = {"pairs": P}
out["whole_step_ms"] = timed(lambda: plan.launch(pairs_d, ids_d))
out["sweep_ms"] = timed(lambda: match(True))
out["sweep_plus_refine_ms"] = timed(lambda: match(False))
match(False)
out["filter_3_launches_ms"] = timed(filt)
out["ransac_f_ms"] = timed(plan.rerun_ransac)
out["whole_step_warm_l2_ms"] = timed(lambda: plan.launch(pairs_d, ids_d), flush_l2=False)
out["sum_of_stages_ms"] = round(out["sweep_plus_refine_ms"] + out["filter_3_launches_ms"] + out["ransac_f_ms"], 4)
out["mean_hyp"] = float(plan.cur.iters[:P].float().mean())
print(json.dumps(out, indent=1))

# in-situ kernel durations of one whole step (CUPTI activity records through torch.profiler: no replay, no serialisation)
try:
    from torch.profiler import ProfilerActivity, profile

    flush.zero_(); torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            plan.launch(pairs_d, ids_d)
            flush.zero_()
        torch.cuda.synchronize()
    rows = {}
    for e in prof.events():
        if e.device_type.name == "CUDA" or "kernel" in e.name.lower():
            rows.setdefault(e.name[:60], []).append(e.device_time if hasattr(e, "device_time") else e.cuda_time)
    print(json.dumps({k: [round(x / 1e3, 4) for x in v] for k, v in rows.items()}, indent=1))
except Exception as ex:  # diagnostic only
    print("profiler unavailable:", ex)
