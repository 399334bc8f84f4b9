"""Camera poses on the B200 (csrc/pnp.cu through ops.pnp_ransac and postprocess.estimate_camera_poses / fast_pnp):
per-hypothesis inlier counts against the numpy oracle, pose and focal against the truth and the reference's cv2 results
stored in tests/golden/pnp_scenes.pt, determinism and batching, edge cases and the public API."""
import os

import numpy as np
import pytest
import torch

from tests import pnp_oracle as O
from tests.golden import pnp_synth as S
from tests.test_pnp_cpu import _check_known, _check_sweep, recount

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gold(golden_dir):
    return torch.load(os.path.join(golden_dir, "pnp_scenes.pt"), weights_only=False)


def _run(pts, mask, focals, iters, pp=None):
    from fast3r_b200 import ops
    p = torch.from_numpy(np.ascontiguousarray(pts)).cuda()
    m = torch.from_numpy(np.ascontiguousarray(mask).astype(np.uint8)).cuda()
    f = torch.from_numpy(np.ascontiguousarray(focals, np.float32)).cuda()
    s, b, c = ops.pnp_ransac(p, m, f, pp, iters=iters)
    torch.cuda.synchronize()
    return s.cpu().numpy(), b.cpu().numpy(), c.cpu().numpy()


@pytest.mark.parametrize("H,W,n_focals,iters", [(64, 96, 20, 5), (368, 512, 1, 100)])
def test_counts_match_oracle(H, W, n_focals, iters):
    pts, conf, truth = S.make_scene(21, H, W, 0.8 * max(H, W), 0.3)
    mask = conf > 1.0
    focals = np.geomspace(max(H, W) / 2, 3 * max(H, W), n_focals).astype(np.float32) if n_focals > 1 else \
        np.float32([truth["f"]])
    s, b, _ = _run(pts[None], mask[None], focals[None], iters)
    o = O.pnp_view(pts, mask, focals, None, iters)
    diff = np.abs(s[0].astype(np.int64) - o["scores"])
    assert np.all(diff <= o["band"]), (diff.max(), o["band"][diff > o["band"]])
    assert o["scores"].max() > 0.5 * mask.sum()
    assert tuple(b[0]) == o["best"] or s[0].reshape(-1)[b[0][0] * iters + b[0][1]] == s[0].max()


@pytest.mark.parametrize("mode", ["known", "sweep"])
def test_fixture_scenes(gold, mode):
    from fast3r_b200 import postprocess
    for name in S.SCENES:
        pts, conf, truth = S.scene(name)
        mask = conf > 1.0
        focal, c2w = postprocess.fast_pnp(torch.from_numpy(pts).cuda(), truth["f"] if mode == "known" else None,
                                          torch.from_numpy(mask).cuda(), niter_PnP=100 if mode == "known" else 10)
        assert c2w.dtype == torch.float32 and c2w.shape == (4, 4) and c2w.is_cuda
        c2w = c2w.cpu().numpy().astype(np.float64)
        rc = recount(c2w, focal, pts, mask)
        if mode == "known":
            assert type(focal) is float
            _check_known(name, gold[name], focal, c2w, rc)
        else:
            assert type(focal) is np.float64
            _check_sweep(name, gold[name], focal, rc)


def test_batching_and_determinism():
    views = [S.make_scene(100 + v, 96, 128, 140.0 + v, 0.3 * (v % 3)) for v in range(32)]
    pts = np.stack([v[0] for v in views])
    mask = np.stack([v[1] > 1.0 for v in views])
    focals = np.tile(np.geomspace(64, 384, 8).astype(np.float32), (32, 1))
    a = _run(pts, mask, focals, 6)
    b = _run(pts, mask, focals, 6)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    for v in range(32):
        one = _run(pts[v:v + 1], mask[v:v + 1], focals[v:v + 1], 6)
        for x, y in zip(a, one):
            assert np.array_equal(x[v:v + 1], y), v
    assert np.all(a[1][:, 0] >= 0)


def test_cpu_and_cuda_inputs_agree():
    from fast3r_b200 import postprocess
    pts, conf, truth = S.scene("outliers30")
    mask = torch.from_numpy(conf > 1.0)
    f1, c1 = postprocess.fast_pnp(torch.from_numpy(pts), None, mask, niter_PnP=10)
    f2, c2 = postprocess.fast_pnp(torch.from_numpy(pts).cuda(), None, mask.cuda(), niter_PnP=10)
    assert f1 == f2 and c1.device.type == "cpu" and torch.equal(c1, c2.cpu())


def _fails(pts, mask, niter=10):
    from fast3r_b200 import postprocess
    f, c = postprocess.fast_pnp(torch.from_numpy(pts).cuda(), 100.0, torch.from_numpy(mask).cuda(), niter_PnP=niter)
    return f is None and c is None


def test_edges():
    from fast3r_b200 import ops
    pts, conf, truth = S.scene("clean")
    H, W, _ = pts.shape
    few = np.zeros((H, W), bool)
    few[5, 5:8] = True
    assert _fails(pts, few)                                  # 3 masked pixels (host-side check)
    # the kernel path with < 4 and with 0 masked pixels, next to a good view in the same call
    m = np.stack([conf > 1.0, few, np.zeros((H, W), bool)])
    s, b, c = _run(np.stack([pts] * 3), m, np.float32([[truth["f"]]] * 3), 10)
    assert b[0, 0] == 0 and tuple(b[1]) == (-1, -1) and tuple(b[2]) == (-1, -1) and not s[1:].any()
    assert np.all(c[1:] == 0) and np.isfinite(c[0]).all()
    nan = pts.copy()
    nan[::2] = np.nan
    nan[1::2] = np.inf
    assert _fails(nan, conf > 1.0)                            # NaN / inf points everywhere
    part = pts.copy()
    part[:, ::3] = np.nan                                     # some NaN points: the rest still gives a pose
    assert not _fails(part, conf > 1.0)
    line = np.zeros_like(pts)
    line[..., 0] = np.arange(W, dtype=np.float32)[None] * 0.01
    line[..., 2] = 5.0
    assert _fails(line, conf > 1.0)                           # collinear masked set
    for z in (0.0, -1.0):                                     # points at z <= 0: no fault, a valid result either way
        flat = pts.copy()
        flat[..., 2] = z
        from fast3r_b200 import postprocess
        f, c2w = postprocess.fast_pnp(torch.from_numpy(flat).cuda(), 100.0, torch.from_numpy(conf > 1.0).cuda())
        assert (f is None and c2w is None) or (f == 100.0 and torch.isfinite(c2w).all())
    with pytest.raises(RuntimeError, match="f3r_pnp_ransac"):
        ops.pnp_ransac(torch.from_numpy(pts[None]).cuda(), torch.ones(1, H, W, dtype=torch.uint8, device="cuda"),
                       torch.ones(1, 1, device="cuda"), None, iters=0)


def test_estimate_camera_poses_api(golden_dir):
    from fast3r_b200 import postprocess
    g = torch.load(os.path.join(golden_dir, "tiny_b2_n2.pt"), weights_only=False)
    preds = [{k: v.clone() for k, v in p.items()} for p in g["preds"]]
    postprocess.align_local_pts3d_to_global(preds, None)
    for method in ("individual", "first_view_from_global_head", "first_view_from_local_head"):
        poses, focals = postprocess.estimate_camera_poses(preds, niter_PnP=10, focal_length_estimation_method=method)
        assert len(poses) == 2 and all(len(p) == 2 for p in poses)
        for i in range(2):
            for v in range(2):
                if focals[i][v] is None:
                    assert np.array_equal(poses[i][v], np.eye(4))
                else:
                    assert poses[i][v].dtype == np.float32 and np.isfinite(poses[i][v]).all()
        if method == "first_view_from_global_head":
            for i in range(2):
                want = postprocess.estimate_focal(preds[0]["pts3d_in_other_view"][i:i + 1], preds[0]["conf"][i:i + 1],
                                                  min_conf_thr_percentile=10)
                assert all(f is None or f == want for f in focals[i])
    with pytest.raises(ValueError):
        postprocess.estimate_camera_poses(preds, focal_length_estimation_method="median")
