"""The geometry tail every caller runs on the forward's outputs (SURVEY.md §8 row f2, first slice), on the GPU.

Same names, arguments and results as the reference:

* ``align_local_pts3d_to_global(preds, views, min_conf_thr_percentile=0)`` -
  MultiViewDUSt3RLitModule.align_local_pts3d_to_global (fast3r/models/multiview_dust3r_module.py:427-549): adds
  ``pts3d_local_aligned_to_global`` (B, H, W, 3) to every pred.  The reference loops over (view, batch item) pairs in a
  CPU thread pool (torch.quantile + boolean gathers + roma SVD per pair); here all pairs go through three kernels
  (exact radix-select quantile, masked moments + Umeyama solve, streaming apply).
* ``estimate_focal(pts3d_i, conf_i, pp=None, min_conf_thr_percentile=10)`` - multiview_dust3r_module.py:1081-1109
  (returns a python float), and ``estimate_focal_knowing_depth(pts3d, pp, focal_mode="weiszfeld")`` -
  fast3r/dust3r/post_process.py:19-79 (returns a (B,) tensor).

* ``estimate_camera_poses(preds, views=None, niter_PnP=10, focal_length_estimation_method='individual')`` -
  MultiViewDUSt3RLitModule.estimate_camera_poses (multiview_dust3r_module.py:806-869, :1038-1078) returning
  ``(poses_c2w_all, estimated_focals_all)``, and ``fast_pnp(pts3d, focal, msk, device=None, pp=None, niter_PnP=10,
  num_guessed_focals=100)`` - fast3r/dust3r/cloud_opt/init_im_poses.py:300-350.  The reference runs one
  cv2.solvePnPRansac (SQPnP) per view and candidate focal on the CPU; here every view of a shape goes through one
  P3P-RANSAC call (csrc/pnp.cu): the same mask (conf > 1), pixel grid, focal candidates, 5 px threshold and
  first-strictly-best focal, with a Levenberg-Marquardt refit on the inliers in place of SQPnP's.  The inlier test is
  division-free, so it differs from cv2.projectPoints only for points at depth exactly 0 (never inliers here).  Poses
  are not bit-identical to OpenCV's (its RANSAC draws from its own generator); they are deterministic.

NOT here (documented in DESIGN.md §1): the "median" focal mode.  Tensors may live on the CPU (what ``inference()`` returns) or on a CUDA device; CPU inputs are
copied to ``device`` (default cuda:0) and the results copied back, so the function is a drop-in either way.  There is
no CPU implementation: without the CUDA library this raises.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import numpy as np

import torch

from . import ops

_GROUP = 64  # (view, batch) pairs stacked per kernel call: bounds the staging copy to ~64 x 5.3 MB at 512x368


def _device_of(t: torch.Tensor, device) -> torch.device:
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise RuntimeError("fast3r_b200.postprocess needs a CUDA device (there is no CPU path)")
    return torch.device(device if device is not None else "cuda:0")


def _f32(t: torch.Tensor, dev: torch.device) -> torch.Tensor:
    return t.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()


def align_local_pts3d_to_global(preds: List[Dict], views: List[Dict], min_conf_thr_percentile: float = 0, device=None) -> None:
    for pred in preds:
        for key, what in (("pts3d_local", "Key 'pts3d_local' not found in preds."),
                          ("conf_local", "Key 'conf_local' not found in preds."),
                          ("pts3d_in_other_view", "Key 'pts3d_in_other_view' not found in preds."),
                          ("conf", "Key 'conf' (global head confidence) not found in preds.")):
            if key not in pred:
                raise ValueError(what)
    if not preds:
        return
    dev = _device_of(preds[0]["pts3d_local"], device)
    q = float(min_conf_thr_percentile) / 100.0
    for g0 in range(0, len(preds), _GROUP):
        group = preds[g0:g0 + _GROUP]
        gviews = views[g0:g0 + _GROUP] if views is not None else [{}] * len(group)
        shapes = {tuple(p["pts3d_local"].shape) for p in group}
        if len(shapes) != 1:  # mixed resolutions: one call per pred
            for p, v in zip(group, gviews):
                _align_group([p], [v], q, dev)
        else:
            _align_group(group, gviews, q, dev)


def _align_group(group: List[Dict], gviews: List[Dict], q: float, dev: torch.device) -> None:
    b, h, w, _ = group[0]["pts3d_local"].shape
    n = h * w
    x = torch.cat([_f32(p["pts3d_local"], dev).reshape(b, n, 3) for p in group])
    y = torch.cat([_f32(p["pts3d_in_other_view"], dev).reshape(b, n, 3) for p in group])
    conf = torch.cat([_f32(p["conf"], dev).reshape(b, n) for p in group])
    valid = None
    if any("valid_mask" in v for v in gviews):
        valid = torch.cat([
            (v["valid_mask"].to(dev).reshape(b, n) if "valid_mask" in v else torch.ones(b, n, dtype=torch.bool, device=dev))
            .to(torch.uint8) for v in gviews]).contiguous()
    thr = ops.conf_quantile(conf, q)
    rts = ops.similarity_fit(x, y, conf, thr, valid)
    out = ops.similarity_apply(x, rts)
    for i, p in enumerate(group):
        src = p["pts3d_local"]
        aligned = out[i * b:(i + 1) * b].reshape(b, h, w, 3)
        p["pts3d_local_aligned_to_global"] = aligned.to(device=src.device, dtype=src.dtype)  # no copy if already there


def estimate_focal(pts3d_i: torch.Tensor, conf_i: torch.Tensor, pp: Optional[torch.Tensor] = None,
                   min_conf_thr_percentile: float = 10, device=None) -> float:
    b, h, w, three = pts3d_i.shape
    assert three == 3
    assert b == 1  # the reference processes one sample at a time
    dev = _device_of(pts3d_i, device)
    pts = _f32(pts3d_i, dev)
    conf = _f32(conf_i, dev).reshape(b, h, w)
    thr = ops.conf_quantile(conf.reshape(b, h * w), float(min_conf_thr_percentile) / 100.0)
    ppt = None if pp is None else _f32(torch.as_tensor(pp), dev).reshape(b, 2)
    return float(ops.focal_weiszfeld(pts, conf, thr, ppt, iters=100)[0])


def estimate_focal_knowing_depth(pts3d: torch.Tensor, pp: torch.Tensor, focal_mode: str = "weiszfeld", device=None) -> torch.Tensor:
    if focal_mode != "weiszfeld":
        raise ValueError(f"bad {focal_mode=} (only 'weiszfeld' is implemented on the GPU)")
    b, h, w, three = pts3d.shape
    assert three == 3
    dev = _device_of(pts3d, device)
    ppt = _f32(torch.as_tensor(pp), dev).reshape(-1, 2).expand(b, 2).contiguous()
    return ops.focal_weiszfeld(_f32(pts3d, dev), None, None, ppt, iters=10).to(pts3d.device)


_FOCAL_METHODS = ("individual", "first_view_from_global_head", "first_view_from_local_head")


def _pnp_group(pts: List[torch.Tensor], confs: List[torch.Tensor], focals: List, niter_PnP: int, dev: torch.device):
    """One f3r_pnp_ransac call over same-shape views.  focals[j]: candidate list (np.float64 array or [float]) of view j.
    Returns [(pose c2w float32 (4, 4) or None, focal or None)]."""
    p = torch.stack([_f32(t, dev) for t in pts])
    m = torch.stack([(c.to(dev) > 1.0) for c in confs]).to(torch.uint8).contiguous()
    f32 = torch.tensor(np.asarray(focals, dtype=np.float64), dtype=torch.float32).to(dev)
    _, best, c2w = ops.pnp_ransac(p, m, f32, None, iters=niter_PnP)
    best, c2w = best.cpu().numpy(), c2w.cpu().numpy()
    out = []
    for j in range(len(pts)):
        k = int(best[j, 0])
        if k < 0:
            out.append((None, None))
            continue
        pose = np.eye(4, dtype=np.float32)
        pose[:3] = c2w[j]
        out.append((pose, focals[j][k]))
    return out


def _candidates(focal, h: int, w: int, num_guessed_focals: int):
    if focal is None:  # init_im_poses.py:310-312, evaluated in float64
        s = max(w, h)
        return np.geomspace(s / 2, s * 3, num=num_guessed_focals)
    return [focal]


def fast_pnp(pts3d: torch.Tensor, focal, msk: torch.Tensor, device=None, pp=None, niter_PnP: int = 10,
             num_guessed_focals: int = 100):
    """Pose of one view from its pointmap pts3d (H, W, 3) and boolean mask (H, W): ``(best_focal, c2w)`` with c2w a
    float32 (4, 4) tensor, or ``(None, None)`` when fewer than 4 pixels are masked or no hypothesis has an inlier.
    focal None sweeps ``num_guessed_focals`` candidates (np.geomspace(S/2, 3S), S = max(H, W)), otherwise focal is kept.
    The work runs on pts3d's CUDA device (CPU inputs: on ``device`` if it is a CUDA device, else cuda:0); c2w is
    returned on ``device`` if given, else on pts3d's device."""
    if int(msk.sum()) < 4:
        return None, None
    h, w, three = pts3d.shape
    assert three == 3
    out_dev = torch.device(device) if device is not None else pts3d.device
    dev = _device_of(pts3d, device if out_dev.type == "cuda" else None)
    cands = _candidates(focal, h, w, num_guessed_focals)
    p = _f32(pts3d, dev).unsqueeze(0)
    m = msk.to(dev).to(torch.uint8).reshape(1, h, w).contiguous()
    f32 = torch.tensor(np.asarray(cands, dtype=np.float64), dtype=torch.float32).reshape(1, -1).to(dev)
    ppt = None if pp is None else _f32(torch.as_tensor(pp), dev).reshape(1, 2)
    _, best, c2w = ops.pnp_ransac(p, m, f32, ppt, iters=niter_PnP)
    k = int(best[0, 0])
    if k < 0:
        return None, None
    pose = torch.eye(4, dtype=torch.float64)
    pose[:3] = c2w[0].cpu()
    return cands[k], pose.to(torch.float32).to(out_dev)


def estimate_camera_poses(preds: List[Dict], views=None, niter_PnP: int = 10,
                          focal_length_estimation_method: str = "individual", device=None):
    """Camera-to-world pose and focal of every view of every batch item: ``(poses_c2w_all, estimated_focals_all)``,
    lists over the B batch items of lists over the N views.  A pose is a float32 (4, 4) numpy array; a view whose pose
    cannot be estimated gets np.eye(4) and focal None.  'individual' sweeps 100 focals per view (niter_PnP hypotheses
    each); the 'first_view_*' methods estimate one focal per batch item from its first view (estimate_focal,
    min_conf_thr_percentile=10) and keep it."""
    batch_size = len(preds[0]["pts3d_in_other_view"])
    if focal_length_estimation_method not in _FOCAL_METHODS:
        raise ValueError(f"Unknown focal_length_estimation_method: {focal_length_estimation_method}")
    key_pts, key_conf = {"first_view_from_global_head": ("pts3d_in_other_view", "conf"),
                         "first_view_from_local_head": ("pts3d_local_aligned_to_global", "conf_local")}.get(
        focal_length_estimation_method, (None, None))
    items = []  # (batch item, view, pts (H, W, 3), conf (H, W), candidate focals)
    for i in range(batch_size):
        focal = None
        if key_pts is not None:
            focal = estimate_focal(preds[0][key_pts][i].unsqueeze(0), preds[0][key_conf][i].unsqueeze(0),
                                   min_conf_thr_percentile=10, device=device)
        for v, pred in enumerate(preds):
            pts, conf = pred["pts3d_in_other_view"][i], pred["conf"][i]
            h, w = pts.shape[0], pts.shape[1]
            items.append((i, v, pts, conf, _candidates(focal, h, w, 100)))
    results = {}
    if items:
        dev = _device_of(items[0][2], device)
        by_shape: Dict[tuple, list] = {}
        for it in items:
            by_shape.setdefault((tuple(it[2].shape), len(it[4])), []).append(it)
        for group_all in by_shape.values():
            for g0 in range(0, len(group_all), _GROUP):
                group = group_all[g0:g0 + _GROUP]
                res = _pnp_group([it[2] for it in group], [it[3] for it in group], [it[4] for it in group], niter_PnP, dev)
                for it, r in zip(group, res):
                    results[(it[0], it[1])] = r
    poses_c2w_all, estimated_focals_all = [], []
    for i in range(batch_size):
        poses, focals = [], []
        for v in range(len(preds)):
            pose, f = results[(i, v)]
            poses.append(np.eye(4) if pose is None else pose)
            focals.append(f)
        poses_c2w_all.append(poses)
        estimated_focals_all.append(focals)
    return poses_c2w_all, estimated_focals_all
