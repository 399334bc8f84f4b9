"""Seeded synthetic PnP scenes with a known answer (tests/test_pnp_*.py, tools/make_golden_pnp.py): a pinhole camera
(focal f, principal point (W/2, H/2), world-to-camera R, t) looking at a smooth depth surface; each pixel (x, y) holds the
world point seen there, with Gaussian 3-D noise, and a fraction of pixels is replaced by gross outliers.  The confidence
map puts some pixels at or below 1 (not used by the pose estimate)."""
import hashlib

import numpy as np

# name: (seed, H, W, focal, outlier fraction)
SCENES = {
    "clean": (11, 96, 128, 150.0, 0.0),
    "outliers30": (12, 96, 128, 150.0, 0.3),
    "outliers60": (13, 96, 128, 110.0, 0.6),
    "portrait": (14, 512, 368, 420.0, 0.3),
}


def rotation(rng, max_deg=20.0):
    axis = rng.standard_normal(3)
    axis /= np.linalg.norm(axis)
    th = np.deg2rad(rng.uniform(0.3, 1.0) * max_deg)
    k = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(th) * k + (1 - np.cos(th)) * k @ k


def make_scene(seed, H, W, focal, outliers, noise=0.0005):
    """Returns pts (H, W, 3) fp32, conf (H, W) fp32 and the truth dict(f, R, t, depth)."""
    rng = np.random.default_rng(seed)
    R = rotation(rng)
    t = rng.uniform(-0.5, 0.5, 3)
    y, x = np.mgrid[:H, :W].astype(np.float64)
    depth = 4.0 + 1.8 * np.sin(x / W * 5.0 + rng.uniform(0, 6)) * np.cos(y / H * 4.0 + rng.uniform(0, 6))
    xc = np.stack([(x - W / 2) / focal * depth, (y - H / 2) / focal * depth, depth], -1)
    xc += rng.standard_normal(xc.shape) * noise * depth[..., None]
    pts = (xc - t) @ R  # X = R^T (Xc - t)
    bad = rng.random((H, W)) < outliers
    pts[bad] += rng.uniform(-2.0, 2.0, (int(bad.sum()), 3))
    conf = 1.0 + rng.gamma(2.0, 1.0, (H, W))
    conf[rng.random((H, W)) < 0.1] = rng.uniform(0.5, 1.0)
    return pts.astype(np.float32), conf.astype(np.float32), dict(f=focal, R=R, t=t, depth=4.0)


def scene(name):
    seed, H, W, f, out = SCENES[name]
    return make_scene(seed, H, W, f, out)


def digest(pts, conf):
    return hashlib.sha256(np.ascontiguousarray(pts).tobytes() + np.ascontiguousarray(conf).tobytes()).hexdigest()
