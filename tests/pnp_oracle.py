"""numpy fp64 restatement of the PnP-RANSAC pipeline of fast3r_b200/csrc/pnp.cu (checker only; the product never imports
it).  Same sampler, same inlier test (evaluated in fp64 on the fp32 projection matrices, with the count of points whose
error lies in the rounding band around the 5 px threshold), same selection and refit.  The minimal solver is written
independently of csrc/pnp_math.h: the quartic's roots come from np.roots (companion-matrix eigenvalues) and the pose
from an SVD alignment of the two point triangles, so a mistake in one cannot hide in the other."""
from __future__ import annotations

import numpy as np

SEED = 0x3f3a2b1c0d0e0f10
MAX_DRAWS = 64
MIN_SINE = 1e-5
LM_STEPS = 10
BAND = 1e-4          # relative half-width of the rounding band around err^2 = 25
_M64 = (1 << 64) - 1


def splitmix64(x: int) -> int:
    z = (x + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def draw(m: int, k: int, i: int, d: int) -> int:
    h = splitmix64(splitmix64(splitmix64(SEED ^ k) ^ i) ^ d)
    return ((h >> 32) * m) >> 32


def sample4(m: int, k: int, i: int):
    """4 distinct entries of range(m) for hypothesis (k, i), or None."""
    if m < 4:
        return None
    out = []
    for d in range(MAX_DRAWS):
        e = draw(m, k, i, d)
        if e not in out:
            out.append(e)
            if len(out) == 4:
                return out
    return None


def _collinear(p):
    d1, d2 = p[1] - p[0], p[2] - p[0]
    return not np.linalg.norm(np.cross(d1, d2)) > MIN_SINE * np.linalg.norm(d1) * np.linalg.norm(d2)


def _align(pw, pc):
    """R, t with pc = R pw + t for two congruent triangles (Kabsch)."""
    mw, mc = pw.mean(0), pc.mean(0)
    u, _, vt = np.linalg.svd((pc - mc).T @ (pw - mw))
    s = np.diag([1.0, 1.0, np.sign(np.linalg.det(u @ vt))])
    r = u @ s @ vt
    return r, mc - r @ mw


def p3p(b, X):
    """Grunert's quartic (Haralick et al. 1994) solved with np.roots.  b: 3 unit bearings, X: 3 world points.
    Returns [(R, t, ill_conditioned)], ill_conditioned flagging roots with a small non-zero imaginary part."""
    b, X = np.asarray(b, np.float64), np.asarray(X, np.float64)
    ca, cb, cg = b[1] @ b[2], b[0] @ b[2], b[0] @ b[1]
    a2, b2, c2 = np.sum((X[1] - X[2]) ** 2), np.sum((X[0] - X[2]) ** 2), np.sum((X[0] - X[1]) ** 2)
    if not (a2 > 0 and b2 > 0 and c2 > 0) or _collinear(X):
        return []
    p, q = (a2 - c2) / b2, (a2 + c2) / b2
    A = [(p - 1) ** 2 - 4 * c2 / b2 * ca ** 2,
         4 * (p * (1 - p) * cb - (1 - q) * ca * cg + 2 * c2 / b2 * ca ** 2 * cb),
         2 * (p ** 2 - 1 + 2 * p ** 2 * cb ** 2 + 2 * (b2 - c2) / b2 * ca ** 2 - 4 * q * ca * cb * cg
              + 2 * (b2 - a2) / b2 * cg ** 2),
         4 * (-p * (1 + p) * cb + 2 * a2 / b2 * cg ** 2 * cb - (1 - q) * ca * cg),
         (1 + p) ** 2 - 4 * a2 / b2 * cg ** 2]
    if not A[0] != 0 or not np.all(np.isfinite(A)):
        return []
    out = []
    for root in np.roots(A):
        scale = max(1.0, abs(root))
        if abs(root.imag) > 1e-6 * scale:
            continue
        ill = abs(root.imag) > 0
        v = root.real
        for _ in range(3):  # Newton polish: eigenvalues of the companion matrix lose digits near close roots
            d = np.polyval(np.polyder(A), v)
            if d == 0:
                break
            v = v - np.polyval(A, v) / d
        den = 2 * (cg - v * ca)
        s1sq = b2 / (1 + v * v - 2 * v * cb)
        if den == 0 or not s1sq > 0:
            continue
        u = ((p - 1) * v * v - 2 * p * cb * v + 1 + p) / den
        s = np.sqrt(s1sq) * np.array([1.0, u, v])
        if not (s[1] > 0 and s[2] > 0 and np.all(np.isfinite(s))):
            continue
        pc = s[:, None] * b
        if _collinear(pc):
            continue
        r, t = _align(X, pc)
        out.append((r, t, ill))
    return out


def bearings(uv, f, cx, cy):
    x = np.stack([(uv[:, 0] - cx) / f, (uv[:, 1] - cy) / f, np.ones(len(uv))], 1)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def reproj_err2(r, t, f, cx, cy, X, uv):
    xc = X @ r.T + t
    z = xc[..., 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        e = (f * xc[..., 0] / z + cx - uv[..., 0]) ** 2 + (f * xc[..., 1] / z + cy - uv[..., 1]) ** 2
    return np.where(z > 0, e, np.inf)


def hypothesis(X4, uv4, f, cx, cy):
    """(R, t) of one hypothesis: P3P on the first three correspondences, the fourth picks; None if invalid."""
    X4, uv4 = np.asarray(X4, np.float64), np.asarray(uv4, np.float64)
    if not np.all(np.isfinite(X4)):
        return None
    best, best_e = None, np.inf
    for r, t, _ in p3p(bearings(uv4[:3], f, cx, cy), X4[:3]):
        e = float(reproj_err2(r, t, f, cx, cy, X4[3], uv4[3]))
        if e < best_e:
            best, best_e = (r, t), e
    return best


def projection32(r, t, f, cx, cy):
    K = np.array([[f, 0, cx], [0, f, cy], [0, 0, 1.0]])
    return (K @ np.concatenate([r, t[:, None]], 1)).astype(np.float32).reshape(12)


def inlier_mask(P32, X, uv):
    """fp64 evaluation of the kernel's division-free test for projection matrices P32 [h, 12] over points X [m, 3]:
    (inlier [h, m], in_band [h, m]) where in_band marks |err^2 - 25| within BAND relative (fp32 rounding may flip those)."""
    P = np.asarray(P32, np.float32).astype(np.float64).reshape(-1, 3, 4)
    Xh = np.concatenate([np.asarray(X, np.float64), np.ones((len(X), 1))], 1)
    with np.errstate(invalid="ignore", over="ignore"):
        q = np.einsum("hrc,mc->hrm", P, Xh)
        e0 = q[:, 0] - uv[None, :, 0] * q[:, 2]
        e1 = q[:, 1] - uv[None, :, 1] * q[:, 2]
        lhs, rhs = e0 * e0 + e1 * e1, 25.0 * q[:, 2] * q[:, 2]
        inl = (lhs <= rhs) & (q[:, 2] != 0)
        band = np.abs(lhs - rhs) <= BAND * rhs
    return inl, band


def lm_refit(r, t, X, uv, f, cx, cy, steps=LM_STEPS):
    """Levenberg-Marquardt on the reprojection error over X, uv (the inliers), left-multiplied so(3) increment,
    Marquardt damping, a step that does not lower the cost is rejected.  Returns (R, t, initial cost, final cost)."""
    def evaluate(r, t):
        q = X @ r.T
        xc = q + t
        z = xc[:, 2]
        if not np.all(z > 0):
            return np.inf, None, None
        res = np.stack([f * xc[:, 0] / z + cx - uv[:, 0], f * xc[:, 1] / z + cy - uv[:, 1]], 1)
        gx, gzu, gzv = f / z, -f * xc[:, 0] / z ** 2, -f * xc[:, 1] / z ** 2
        zero = np.zeros_like(z)
        ju = np.stack([gzu * q[:, 1], gx * q[:, 2] - gzu * q[:, 0], -gx * q[:, 1], gx, zero, gzu], 1)
        jv = np.stack([-gx * q[:, 2] + gzv * q[:, 1], -gzv * q[:, 0], gx * q[:, 0], zero, gx, gzv], 1)
        cost = float(np.sum(res ** 2))
        return (cost if np.isfinite(cost) else np.inf), ju.T @ ju + jv.T @ jv, ju.T @ res[:, 0] + jv.T @ res[:, 1]

    cost, jtj, jtr = evaluate(r, t)
    cost0, lam = cost, 1e-3
    for _ in range(steps):
        if jtj is None:
            break
        a = jtj + lam * np.diag(np.diag(jtj))
        try:
            np.linalg.cholesky(a)
            d = np.linalg.solve(a, -jtr)
        except np.linalg.LinAlgError:
            lam = min(lam * 10, 1e12)
            continue
        th = np.linalg.norm(d[:3])
        k = d[:3] / th if th > 0 else np.zeros(3)
        kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        e = np.eye(3) + np.sin(th) * kx + (1 - np.cos(th)) * kx @ kx
        r2, t2 = e @ r, t + d[3:]
        c2, jtj2, jtr2 = evaluate(r2, t2)
        if c2 < cost:
            r, t, cost, jtj, jtr, lam = r2, t2, c2, jtj2, jtr2, max(lam * 0.1, 1e-12)
        else:
            lam = min(lam * 10, 1e12)
    return r, t, cost0, cost


def pnp_view(pts, mask, focals, pp, iters):
    """One view: pts [H, W, 3] fp32, mask [H, W] bool, focals [F] fp32, pp (cx, cy) fp32 or None.
    Returns dict(scores [F, iters], band [F, iters], best (k, i) or None, c2w [3, 4] or None, cost0, cost, pose)."""
    H, W, _ = pts.shape
    cx, cy = (np.float32(W / 2), np.float32(H / 2)) if pp is None else (np.float32(pp[0]), np.float32(pp[1]))
    cx, cy = float(cx), float(cy)
    idx = np.flatnonzero(np.asarray(mask).reshape(-1))
    X = np.asarray(pts, np.float32).reshape(-1, 3)[idx].astype(np.float64)
    uv = np.stack([idx % W, idx // W], 1).astype(np.float64)
    nf = len(focals)
    nan = np.full(12, np.nan, np.float32)
    Ps, poses = [], []
    for k in range(nf):
        f = float(np.float32(focals[k]))
        for i in range(iters):
            e = sample4(len(idx), k, i)
            hyp = None if e is None else hypothesis(X[e], uv[e], f, cx, cy)
            poses.append(hyp)
            Ps.append(nan if hyp is None else projection32(hyp[0], hyp[1], f, cx, cy))
    Ps = np.stack(Ps)
    scores = np.zeros(len(Ps), np.int64)
    band = np.zeros(len(Ps), np.int64)
    step = max(1, int(2e7 // max(1, len(X))))
    for h0 in range(0, len(Ps), step):
        inl, bnd = inlier_mask(Ps[h0:h0 + step], X, uv)
        scores[h0:h0 + step] = inl.sum(1)
        band[h0:h0 + step] = bnd.sum(1)
    out = dict(scores=scores.reshape(nf, iters), band=band.reshape(nf, iters), best=None, c2w=None, cost0=None,
               cost=None, pose=None)
    if len(idx) < 4 or scores.max() == 0:
        return out
    h = int(np.argmax(scores))  # first maximum = lowest (k, i)
    k = h // iters
    r, t = poses[h]
    inl, _ = inlier_mask(Ps[h:h + 1], X, uv)
    f = float(np.float32(focals[k]))
    r, t, c0, c1 = lm_refit(r, t, X[inl[0]], uv[inl[0]], f, cx, cy)
    out.update(best=(k, h % iters), c2w=np.concatenate([r.T, (-r.T @ t)[:, None]], 1), cost0=c0, cost=c1, pose=(r, t))
    return out


def pnp_ransac(pts, mask, focals, pp=None, iters=10):
    """Same contract as fast3r_b200.ops.pnp_ransac, on torch tensors, computed by pnp_view (CPU, numpy)."""
    import torch
    V = pts.shape[0]
    F = focals.shape[1]
    scores = torch.zeros(V, F, iters, dtype=torch.int32)
    best = torch.full((V, 2), -1, dtype=torch.int32)
    c2w = torch.zeros(V, 3, 4, dtype=torch.float64)
    for v in range(V):
        o = pnp_view(pts[v].cpu().numpy(), mask[v].cpu().numpy() != 0, focals[v].cpu().numpy(),
                     None if pp is None else pp[v].cpu().numpy(), iters)
        scores[v] = torch.from_numpy(o["scores"].astype(np.int32))
        if o["best"] is not None:
            best[v] = torch.tensor(o["best"], dtype=torch.int32)
            c2w[v] = torch.from_numpy(o["c2w"])
    return scores, best, c2w
