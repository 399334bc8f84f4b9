"""Camera poses without a GPU: fast3r_b200/csrc/pnp_math.h compiled for the host against the numpy oracle
(tests/pnp_oracle.py), the oracle's inlier test against cv2.projectPoints, the oracle pipeline against the reference's
cv2 results stored in tests/golden/pnp_scenes.pt, the host logic of postprocess.estimate_camera_poses against the
reference's, and the C ABI's argument checks."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from tests import pnp_oracle as O
from tests.golden import pnp_synth as S

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "fast3r_b200", "csrc")


@pytest.fixture(scope="module")
def hostlib(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    so = str(tmp_path_factory.mktemp("pnp") / "libpnp_host.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", CSRC,
                           os.path.join(HERE, "pnp_math_host.cpp"), "-o", so])
    lib = C.CDLL(so)
    lib.f3r_test_pnp_sample4.argtypes = [C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]
    lib.f3r_test_p3p.argtypes = [C.c_void_p] * 4
    lib.f3r_test_hypothesis.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p]
    lib.f3r_test_chol6.argtypes = [C.c_void_p] * 3
    return lib


@pytest.fixture(scope="module")
def gold(golden_dir):
    return torch.load(os.path.join(golden_dir, "pnp_scenes.pt"), weights_only=False)


def rot(rng):
    q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
    return q * np.sign(np.linalg.det(q))


def rot_deg(a, b):
    return float(np.degrees(np.arccos(np.clip((np.trace(a[:3, :3].T @ b[:3, :3]) - 1) / 2, -1, 1))))


def true_c2w(truth):
    c = np.eye(4)
    c[:3, :3] = truth["R"].T
    c[:3, 3] = -truth["R"].T @ truth["t"]
    return c


def test_sampler_stream_matches_oracle(hostlib):
    out = np.zeros(4, np.uint32)
    for m in (0, 3, 4, 5, 7, 100, 188416, 1 << 24):
        for k in range(6):
            for i in range(25):
                ok = hostlib.f3r_test_pnp_sample4(m, k, i, out.ctypes.data)
                want = O.sample4(m, k, i)
                assert (want is not None) == bool(ok), (m, k, i)
                if want is not None:
                    assert list(out) == want and len(set(want)) == 4 and max(want) < m


def test_p3p_solution_set_matches_oracle(hostlib):
    """1000 random minimal problems: the header's solutions contain the true pose and, where the oracle (np.roots) sees
    the same number of well-separated solutions, equal the oracle's - to 1e-9 for at least 95 % of them and to 1e-4 for
    all (the rest are configurations where the pose amplifies the last bits of the quartic's root)."""
    rng = np.random.default_rng(0)
    diffs = []
    for _ in range(1000):
        R, t = rot(rng), rng.uniform(-1, 1, 3) + [0, 0, 6]
        X = rng.uniform(-2, 2, (3, 3))
        xc = X @ R.T + t
        b = np.ascontiguousarray(xc / np.linalg.norm(xc, axis=1, keepdims=True))
        Rs, ts = np.zeros(36), np.zeros(12)
        n = hostlib.f3r_test_p3p(b.ctypes.data, np.ascontiguousarray(X).ctypes.data, Rs.ctypes.data, ts.ctypes.data)
        ours = [(Rs[9 * s:9 * s + 9].reshape(3, 3), ts[3 * s:3 * s + 3]) for s in range(n)]
        assert any(np.abs(r - R).max() < 1e-7 and np.abs(tt - t).max() < 1e-7 for r, tt in ours)
        theirs = O.p3p(b, X)
        gaps = [np.abs(t1 - t2).max() for j, (_, t1, _) in enumerate(theirs) for (_, t2, _) in theirs[j + 1:]]
        if any(ill for _, _, ill in theirs) or len(theirs) != n or (gaps and min(gaps) < 1e-2):
            continue  # (near-)double root: both solvers are right only to sqrt(eps) there
        for r, tt in ours:
            diffs.append(min(max(np.abs(r - r2).max(), np.abs(tt - t2).max() / 6) for r2, t2, _ in theirs))
    diffs = np.array(diffs)
    assert len(diffs) > 1500 and diffs.max() < 1e-4 and np.mean(diffs < 1e-9) >= 0.95, (len(diffs), diffs.max())


def test_hypothesis_picks_the_true_pose(hostlib):
    rng = np.random.default_rng(1)
    f, cx, cy = 300.0, 256.0, 184.0
    for _ in range(200):
        R, t = rot(rng), rng.uniform(-1, 1, 3) + [0, 0, 8]
        X = rng.uniform(-2, 2, (4, 3))
        xc = X @ R.T + t
        uv = np.stack([f * xc[:, 0] / xc[:, 2] + cx, f * xc[:, 1] / xc[:, 2] + cy], 1)
        pose = np.zeros(12)
        assert hostlib.f3r_test_hypothesis(np.ascontiguousarray(X).ctypes.data, np.ascontiguousarray(uv).ctypes.data,
                                           f, cx, cy, pose.ctypes.data)
        assert np.abs(pose[:9].reshape(3, 3) - R).max() < 1e-6 and np.abs(pose[9:] - t).max() < 1e-5
        r2, t2 = O.hypothesis(X, uv, f, cx, cy)
        assert np.abs(r2 - R).max() < 1e-6 and np.abs(t2 - t).max() < 1e-5


def test_chol6_solve(hostlib):
    rng = np.random.default_rng(2)
    for _ in range(50):
        a = rng.standard_normal((6, 6))
        a = a @ a.T + 0.1 * np.eye(6)
        b = rng.standard_normal(6)
        up = np.concatenate([a[i, i:] for i in range(6)])
        x = np.zeros(6)
        assert hostlib.f3r_test_chol6(up.ctypes.data, b.ctypes.data, x.ctypes.data)
        assert np.allclose(x, np.linalg.solve(a, b), rtol=1e-9, atol=1e-12)
    up = np.concatenate([(-np.eye(6))[i, i:] for i in range(6)])
    assert not hostlib.f3r_test_chol6(up.ctypes.data, np.ones(6).ctypes.data, np.zeros(6).ctypes.data)


def test_inlier_test_matches_projectpoints():
    """The division-free test equals cv2.projectPoints + err^2 <= 25 on every pixel with z != 0 outside the rounding
    band."""
    cv2 = pytest.importorskip("cv2")
    pts, conf, truth = S.scene("outliers30")
    H, W, _ = pts.shape
    f, cx, cy = np.float32(truth["f"]), np.float32(W / 2), np.float32(H / 2)
    rng = np.random.default_rng(3)
    R = truth["R"] @ cv2.Rodrigues(rng.standard_normal(3) * 2e-3)[0]  # a slightly wrong pose: many borderline points
    t = truth["t"] + rng.standard_normal(3) * 0.01
    X = pts.reshape(-1, 3).astype(np.float64)
    uv = np.stack(np.meshgrid(np.arange(W), np.arange(H)), -1).reshape(-1, 2).astype(np.float64)
    K = np.array([[f, 0, cx], [0, f, cy], [0, 0, 1]], np.float64)
    proj, _ = cv2.projectPoints(X, cv2.Rodrigues(R)[0], t, K, None)
    err2 = np.sum((proj.reshape(-1, 2) - uv) ** 2, 1)
    inl, band = O.inlier_mask(O.projection32(R, t, float(f), float(cx), float(cy))[None], X, uv)
    z = X @ R[2] + t[2]
    keep = (z != 0) & ~band[0]
    assert keep.sum() > 0.9 * len(X) and 0 < inl[0][keep].sum() < keep.sum()
    # fp32 P vs cv2's fp64 projection: compare where the fp64 error is clearly away from the threshold
    clear = keep & (np.abs(err2 - 25) > 0.05)
    assert np.array_equal(inl[0][clear], err2[clear] <= 25)


def test_scene_inputs_match_fixture(gold):
    for name in S.SCENES:
        pts, conf, _ = S.scene(name)
        assert S.digest(pts, conf) == gold[name]["sha256"], name


def _check_known(name, g, focal, c2w, recount):
    truth = g["truth"]
    cv = g["known"]
    assert focal == truth["f"]
    tc = true_c2w(truth)
    assert rot_deg(c2w, tc) < 0.05, name
    # cv2's own pose carries its error to the truth: the distance to it is bounded by that plus ours
    assert rot_deg(c2w, cv["c2w"]) < 0.05 + rot_deg(cv["c2w"], tc), name
    assert np.linalg.norm(c2w[:3, 3] - tc[:3, 3]) < 2e-3 * truth["depth"], name
    assert recount >= 0.99 * cv["recount"], name


def _check_sweep(name, g, focal, recount):
    truth, cv = g["truth"], g["sweep"]
    assert recount >= 0.99 * cv["recount"], name
    if abs(cv["focal"] / truth["f"] - 1) < 0.05:
        assert abs(focal / truth["f"] - 1) < 0.10, (name, focal)


def recount(c2w, f, pts, mask):
    H, W, _ = pts.shape
    w2c = np.linalg.inv(np.asarray(c2w, np.float64))
    P = O.projection32(w2c[:3, :3], w2c[:3, 3], float(np.float32(f)), float(np.float32(W / 2)), float(np.float32(H / 2)))
    idx = np.flatnonzero(mask.reshape(-1))
    uv = np.stack([idx % W, idx // W], 1).astype(np.float64)
    inl, _ = O.inlier_mask(P[None], pts.reshape(-1, 3)[idx], uv)
    return int(inl.sum())


@pytest.mark.parametrize("mode", ["known", "sweep"])
def test_oracle_pipeline_against_cv2(gold, mode):
    for name in S.SCENES:
        pts, conf, truth = S.scene(name)
        mask = conf > 1.0
        H, W, _ = pts.shape
        cands = [truth["f"]] if mode == "known" else np.geomspace(max(H, W) / 2, 3 * max(H, W), 100)
        o = O.pnp_view(pts, mask, np.float32(cands), None, 100 if mode == "known" else 10)
        assert o["best"] is not None and o["cost"] <= o["cost0"]
        c2w = np.eye(4)
        c2w[:3] = o["c2w"]
        focal = cands[o["best"][0]]
        rc = recount(c2w, focal, pts, mask)
        if mode == "known":
            _check_known(name, gold[name], focal, c2w, rc)
        else:
            _check_sweep(name, gold[name], focal, rc)


# ------------------------------------------------------------------ host logic of estimate_camera_poses
class _OracleOps:
    """postprocess.ops with the CUDA entry points replaced: the geometry tail by tests/abi_emulator.py, pnp_ransac by
    the oracle."""

    def __init__(self):
        from tests import abi_emulator
        self._emu = abi_emulator

    def __getattr__(self, name):
        return getattr(self._emu, name)

    @staticmethod
    def pnp_ransac(pts, mask, focals, pp=None, iters=10):
        return O.pnp_ransac(pts, mask, focals, pp, iters)


@pytest.fixture()
def host_post(monkeypatch):
    from fast3r_b200 import postprocess
    monkeypatch.setattr(postprocess, "ops", _OracleOps())
    monkeypatch.setattr(postprocess, "_device_of", lambda t, device: torch.device("cpu"))
    return postprocess


def _tiny_preds(golden_dir, post):
    g = torch.load(os.path.join(golden_dir, "tiny_b2_n2.pt"), weights_only=False)
    preds = [{k: v.clone() for k, v in p.items()} for p in g["preds"]]
    post.align_local_pts3d_to_global(preds, None)
    preds[1]["conf"][1] = 0.5  # batch item 1, view 1: no pixel above 1 -> the failure values
    preds[1]["conf"][1, 0, :3] = 2.0
    return preds


def test_estimate_camera_poses_structure_and_failures(host_post, golden_dir):
    preds = _tiny_preds(golden_dir, host_post)
    for method in ("individual", "first_view_from_global_head", "first_view_from_local_head"):
        poses, focals = host_post.estimate_camera_poses(preds, niter_PnP=3, focal_length_estimation_method=method)
        assert len(poses) == len(focals) == 2 and all(len(p) == 2 for p in poses) and all(len(f) == 2 for f in focals)
        assert poses[1][1].dtype == np.float64 and np.array_equal(poses[1][1], np.eye(4)) and focals[1][1] is None
        for i, v in ((0, 0), (0, 1), (1, 0)):  # random pointmaps: a view may also fail, with the failure values
            if focals[i][v] is None:
                assert poses[i][v].dtype == np.float64 and np.array_equal(poses[i][v], np.eye(4))
                continue
            assert poses[i][v].dtype == np.float32 and poses[i][v].shape == (4, 4), (method, i, v)
            assert type(focals[i][v]) is (np.float64 if method == "individual" else float), (method, type(focals[i][v]))
        assert sum(f is not None for f in focals[0] + focals[1]) >= 1, (method, focals)
    with pytest.raises(ValueError, match="Unknown focal_length_estimation_method: median"):
        host_post.estimate_camera_poses(preds, focal_length_estimation_method="median")
    no_local = [{k: v for k, v in p.items() if k != "pts3d_local_aligned_to_global"} for p in preds]
    with pytest.raises(KeyError):
        host_post.estimate_camera_poses(no_local, focal_length_estimation_method="first_view_from_local_head")


def test_estimate_camera_poses_matches_reference(host_post, golden_dir):
    """The reference's MultiViewDUSt3RLitModule.estimate_camera_poses on the same preds: same structure, dtypes,
    first-view focals and failure values (poses differ: the reference runs OpenCV's RANSAC)."""
    pytest.importorskip("cv2")
    from oracle.ref_harness import reference_available, import_reference_lit_module
    if not reference_available():
        pytest.skip("reference sources not available")
    try:
        lit_mod = import_reference_lit_module()
    except Exception as e:  # a training-stack dependency that cannot be stubbed here
        pytest.skip(f"reference Lightning module not importable: {e!r}")
    preds = _tiny_preds(golden_dir, host_post)
    for method in ("individual", "first_view_from_global_head", "first_view_from_local_head"):
        ref_p, ref_f = lit_mod.MultiViewDUSt3RLitModule.estimate_camera_poses(
            [dict(p) for p in preds], niter_PnP=3, focal_length_estimation_method=method)
        our_p, our_f = host_post.estimate_camera_poses(preds, niter_PnP=3, focal_length_estimation_method=method)
        for i in range(2):
            for v in range(2):
                a, b = np.asarray(ref_p[i][v]), our_p[i][v]
                assert a.shape == b.shape == (4, 4), (method, i, v)
                if ref_f[i][v] is None or our_f[i][v] is None:  # random pointmaps: either side may fail on a view
                    continue
                assert a.dtype == b.dtype and type(ref_f[i][v]) is type(our_f[i][v]), (method, i, v, a.dtype, b.dtype)
                if method != "individual":
                    assert abs(ref_f[i][v] - our_f[i][v]) <= 1e-3 * abs(ref_f[i][v]), (method, i, v)
        assert np.array_equal(our_p[1][1], np.eye(4)) and our_p[1][1].dtype == np.float64 and our_f[1][1] is None
        assert np.array_equal(np.asarray(ref_p[1][1]), np.eye(4)) and ref_f[1][1] is None


# ------------------------------------------------------------------ C ABI
def test_pnp_cabi_rejects_bad_arguments_before_any_cuda_call():
    from fast3r_b200 import lib as L
    lib = L.load()
    ws = lib.f3r_pnp_workspace(2, 8, 8, 3, 5)
    assert ws > 0 and ws % 256 == 0 and lib.f3r_pnp_workspace(0, 8, 8, 3, 5) == 0
    assert lib.f3r_pnp_workspace(1, 8, 8, 0, 5) == 0 and lib.f3r_pnp_workspace(1, 8, 8, 1, 0) == 0
    a = 256
    cases = [
        ((None, a, 1, 8, 8, a, 1, None, 5, a, a, a, a, 1 << 20, None), "null operand"),
        ((a, a, 1, 8, 8, a, 1, None, 5, a, a, None, a, 1 << 20, None), "null operand"),
        ((a, a, 1, 8, 8, a, 0, None, 5, a, a, a, a, 1 << 20, None), "n_focals must be >= 1"),
        ((a, a, 1, 8, 8, a, 1, None, 0, a, a, a, a, 1 << 20, None), "iters must be >= 1"),
        ((a, a, 0, 8, 8, a, 1, None, 5, a, a, a, a, 1 << 20, None), "bad shape"),
        ((a, a, 1, 1 << 13, 1 << 12, a, 1, None, 5, a, a, a, a, 1 << 40, None), "bad shape"),
        ((a, a, 1, 8, 8, a, 1, None, 5, a, a, a, a, 16, None), "workspace too small"),
        ((a, a, 1, 8, 8, a, 1, None, 5, a, a, a, a + 8, 1 << 20, None), "not 256-byte aligned"),
    ]
    for args, msg in cases:
        assert lib.f3r_pnp_ransac(*args) != 0
        err = lib.f3r_last_error().decode()
        assert err.startswith("f3r_pnp_ransac") and msg in err, err
