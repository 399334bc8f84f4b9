"""Times the camera-pose step (csrc/pnp.cu) on the GPU and writes one JSON file (default profiles/r03_pnp_rates.json).

Workload: 32 views of 368 x 512 pixels (synthetic scenes of tests/golden/pnp_synth.py, 30 % outliers), resident in HBM,
every pixel masked.  Two modes, each timed with CUDA events over >= 10 repetitions after warm-up:
  readme   the README flow: one GPU focal per view (estimate_focal: quantile + Weiszfeld) + 100 hypotheses per view
  sweep    the default 'individual' mode: 100 candidate focals x niter_PnP=10 per view
The scoring kernel's own time comes from a separate torch.profiler run.  A point test is one (hypothesis, pixel) pair;
it costs OPS_PER_TEST fp32 instructions on the FMA pipe (9 FMA for P X, 2 FMA for the residuals, 1 MUL + 1 FMA for the
squared error, 2 MUL for 25 w^2); the share of peak is the instruction rate over SMs x 128 lanes x max SM clock.
If cv2 is importable, the reference-equivalent cv2.solvePnPRansac time per view on the host cores is added.

    python tools/pnp_rates.py [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPS_PER_TEST = 15
VIEWS, H, W = 32, 368, 512


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True).stdout.strip().split(", ")
    return dict(name=q[0], power_limit_w=float(q[1]), max_sm_clock_mhz=float(q[2]),
                sms=torch.cuda.get_device_properties(0).multi_processor_count)


def timed(fn, warmup=3, reps=10):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return dict(median_ms=float(np.median(times)), min_ms=float(np.min(times)), max_ms=float(np.max(times)), reps=reps)


def kernel_ms(fn, reps=3):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "pnp_" in ev.key:
            name = ev.key.split("pnp_")[1].split("_kernel")[0]
            out[name] = out.get(name, 0.0) + ev.device_time_total / 1e3 / reps  # us -> ms per call
    return out


def cv2_per_view(pts, mask, focals, niter):
    import cv2
    idx = np.flatnonzero(mask.reshape(-1))
    pix = np.stack([idx % W, idx // W], 1).astype(np.float32)
    p3 = pts.reshape(-1, 3)[idx]
    t0 = time.perf_counter()
    for f in focals:
        K = np.float32([(f, 0, W / 2), (0, f, H / 2), (0, 0, 1)])
        cv2.solvePnPRansac(p3, pix, K, None, iterationsCount=niter, reprojectionError=5, flags=cv2.SOLVEPNP_SQPNP)
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_pnp_rates.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "pnp_rates.py measures on the GPU"
    from fast3r_b200 import ops
    from tests.golden.pnp_synth import make_scene
    info = gpu_info()
    scenes = [make_scene(300 + v, H, W, 420.0 + 5 * v, 0.3) for v in range(VIEWS)]
    pts = torch.from_numpy(np.stack([s[0] for s in scenes])).cuda()
    conf = torch.from_numpy(np.stack([s[1] for s in scenes])).cuda()
    mask = torch.ones(VIEWS, H, W, dtype=torch.uint8, device="cuda")
    n = H * W
    sweep_f = torch.from_numpy(np.tile(np.geomspace(max(H, W) / 2, 3 * max(H, W), 100).astype(np.float32),
                                       (VIEWS, 1))).cuda()

    def readme():
        thr = ops.conf_quantile(conf.reshape(VIEWS, n), 0.10)
        f = ops.focal_weiszfeld(pts, conf, thr, None, iters=100)
        return ops.pnp_ransac(pts, mask, f.reshape(VIEWS, 1).contiguous(), None, iters=100)

    def sweep():
        return ops.pnp_ransac(pts, mask, sweep_f, None, iters=10)

    res = dict(gpu=info, workload=dict(views=VIEWS, h=H, w=W, masked_pixels_per_view=n, inputs="HBM-resident"),
               ops_per_test=OPS_PER_TEST)
    fma_instr_per_s = info["sms"] * 128 * info["max_sm_clock_mhz"] * 1e6
    for name, fn, hyps in (("readme", readme, 100), ("sweep", sweep, 1000)):
        t = timed(fn)
        k = kernel_ms(fn)
        tests = VIEWS * hyps * n
        score_ms = k.get("score", float("nan"))
        res[name] = dict(call=t, kernels_ms=k, hypotheses_per_view=hyps, point_tests=tests,
                         per_view_ms=t["median_ms"] / VIEWS,
                         score_tests_per_s=tests / (score_ms / 1e3),
                         score_share_of_fma_peak=tests * OPS_PER_TEST / (score_ms / 1e3) / fma_instr_per_s)
        print(name, json.dumps(res[name]), flush=True)
    try:
        import cv2  # noqa: F401
        p0, m0 = scenes[0][0], np.ones((H, W), bool)
        known = cv2_per_view(p0, m0, [420.0], 100)
        sw = cv2_per_view(p0, m0, np.geomspace(max(H, W) / 2, 3 * max(H, W), 100), 10)
        res["cv2_reference_equivalent_s_per_view"] = dict(readme_known_focal_niter100=known, sweep_100x10=sw,
                                                          host_threads=torch.get_num_threads(), cpu=os.cpu_count())
    except ImportError:
        res["cv2_reference_equivalent_s_per_view"] = "not measured"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["gpu"]), "->", args.out)


if __name__ == "__main__":
    main()
