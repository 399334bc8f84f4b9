"""Writes tests/golden/pnp_scenes.pt: for every scene of tests/golden/pnp_synth.py, the result of the reference's own
fast_pnp (fast3r/dust3r/cloud_opt/init_im_poses.py:300-350, cv2.solvePnPRansac with SQPnP) in the known-focal mode
(niter_PnP=100) and in the focal sweep (100 focals x niter_PnP=10): focal, c2w, the inlier count cv2 returned, and cv2's
pose recounted with the kernel's inlier test (tests/pnp_oracle.py), so that scores compare like with like.  Inputs are not
stored: they are regenerated from the seed and checked against the stored sha256.

Needs the reference sources and cv2 (build container only):  python tools/make_golden_pnp.py"""
import os
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tests import pnp_oracle as O  # noqa: E402
from tests.golden import pnp_synth as S  # noqa: E402


def recount(c2w, f, pts, mask):
    H, W, _ = pts.shape
    w2c = np.linalg.inv(np.asarray(c2w, np.float64))
    P = O.projection32(w2c[:3, :3], w2c[:3, 3], float(np.float32(f)), float(np.float32(W / 2)), float(np.float32(H / 2)))
    idx = np.flatnonzero(mask.reshape(-1))
    uv = np.stack([idx % W, idx // W], 1).astype(np.float64)
    inl, _ = O.inlier_mask(P[None], pts.reshape(-1, 3)[idx], uv)
    return int(inl.sum())


def main():
    import cv2
    sys.modules.setdefault("roma", types.ModuleType("roma"))
    from oracle.ref_harness import import_reference
    import_reference()
    import fast3r.dust3r.cloud_opt.init_im_poses as ip

    calls = []
    real = cv2.solvePnPRansac

    def spy(*a, **k):
        r = real(*a, **k)
        calls.append((float(a[2][0, 0]), len(r[3]) if r[0] and r[3] is not None else 0))
        return r

    out = {}
    for name in S.SCENES:
        pts, conf, truth = S.scene(name)
        mask = conf > 1.0
        entry = dict(params=S.SCENES[name], sha256=S.digest(pts, conf), truth=truth)
        for mode, focal, niter in (("known", truth["f"], 100), ("sweep", None, 10)):
            cv2.setRNGSeed(0)
            calls.clear()
            ip.cv2.solvePnPRansac = spy
            try:
                f, c2w = ip.fast_pnp(torch.from_numpy(pts), focal, torch.from_numpy(mask), "cpu", niter_PnP=niter)
            finally:
                ip.cv2.solvePnPRansac = real
            c2w = c2w.numpy()
            returned = max(n for _, n in calls)
            entry[mode] = dict(focal=float(f), c2w=c2w, returned=returned, recount=recount(c2w, f, pts, mask))
            print(name, mode, f"focal {float(f):.1f} (true {truth['f']})", "returned", returned,
                  "recount", entry[mode]["recount"], flush=True)
        out[name] = entry
    torch.save(out, os.path.join(ROOT, "tests", "golden", "pnp_scenes.pt"))


if __name__ == "__main__":
    main()
