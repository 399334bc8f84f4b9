"""Torch-tensor wrappers over the C ABI.  torch is plumbing here (device memory + streams); every op below
is one call into libfast3r_b200.so on ``torch.cuda.current_stream()``.  No op has a PyTorch fallback."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import lib as L

BF16, F32 = torch.bfloat16, torch.float32

# Optional per-launch CUDA-event timing of the dominant kernel (bench.py's live roofline measurement).
# When set to a list, attention() appends (batch, heads, sq, skv, start_event, end_event), recorded on the
# launching stream.
KERNEL_TIMER = None


def _stream(t: Optional[torch.Tensor] = None) -> int:
    """The current stream OF THE TENSOR'S DEVICE (callers need not have made that device current)."""
    return torch.cuda.current_stream(t.device if t is not None else None).cuda_stream


class _on_device:
    """CUDA runtime calls inside the library (cudaFuncSetAttribute, launches) act on the CURRENT device: make the
    operand's device current for the duration of the call."""

    def __init__(self, t: torch.Tensor):
        self.idx = t.device.index if t.is_cuda else None

    def __enter__(self):
        self.prev = None
        if self.idx is not None and torch.cuda.current_device() != self.idx:
            self.prev = torch.cuda.current_device()
            torch.cuda.set_device(self.idx)

    def __exit__(self, *exc):
        if self.prev is not None:
            torch.cuda.set_device(self.prev)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("fast3r_b200 ops need CUDA tensors (there is no CPU path)")
    return t.data_ptr()


def _chk(t: torch.Tensor, dtype, name: str):
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")


def gemm(a: torch.Tensor, wt: torch.Tensor, *, w: int, h: int = 1, nb: int = 1, taps: int = 1,
         bias: Optional[torch.Tensor] = None, out0: Optional[torch.Tensor] = None,
         out1: Optional[torch.Tensor] = None, res0: Optional[torch.Tensor] = None,
         res1: Optional[torch.Tensor] = None, act: int = L.ACT_NONE, epi: int = L.EPI_STORE,
         ldo: Optional[int] = None, split_col: int = 0, out0b: Optional[torch.Tensor] = None, ldo_b: int = 0,
         tok_per_img: int = 0, grid_w: int = 0, rope_cols: int = 0, rope_cos=None, rope_sin=None,
         emb_table=None, emb_ids=None, ct_k: int = 0, ct_cout: int = 0, w4=None, b4=None, pts=None, conf=None):
    """Fused GEMM / implicit conv (f3r_gemm).  a: bf16 (..., K) channels-last with nb*h*w pixels;
    wt: bf16 (N, taps, K)."""
    _chk(a, BF16, "a"); _chk(wt, BF16, "wt")
    n, k = wt.shape[0], wt.shape[-1]
    assert wt.numel() == n * taps * k
    assert a.shape[-1] == k and a.numel() == nb * h * w * k, (a.shape, nb, h, w, k)
    d = L.GemmDesc()
    d.a, d.wt = _ptr(a), _ptr(wt)
    d.n, d.k, d.taps = n, k, taps
    d.w, d.h, d.nb = w, h, nb
    d.a_ld = k
    d.epi, d.act = epi, act
    d.ldo = ldo if ldo is not None else (ct_cout if epi == L.EPI_CONVT else n)
    d.split_col, d.ldo_b = split_col, ldo_b
    d.tok_per_img, d.grid_w, d.rope_cols = tok_per_img, grid_w, rope_cols
    d.ct_k, d.ct_cout = ct_k, ct_cout
    if bias is not None:
        _chk(bias, F32, "bias")
    d.bias = _ptr(bias)
    if res0 is not None:
        assert res0.dtype in (BF16, F32) and res0.is_contiguous()
        d.res0_f32 = int(res0.dtype == F32)
    d.res0 = _ptr(res0)
    if res1 is not None:
        _chk(res1, BF16, "res1")
    d.res1 = _ptr(res1)
    if out0 is not None:
        assert out0.dtype in (BF16, F32) and out0.is_contiguous()
        d.out0_f32 = int(out0.dtype == F32)
    d.out0 = _ptr(out0)
    if out0b is not None:
        assert out0 is not None and out0b.dtype == out0.dtype
    d.out0b = _ptr(out0b)
    if out1 is not None:
        _chk(out1, BF16, "out1")
    d.out1 = _ptr(out1)
    d.rope_cos, d.rope_sin = _ptr(rope_cos), _ptr(rope_sin)
    d.emb_table, d.emb_ids = _ptr(emb_table), _ptr(emb_ids)
    d.w4, d.b4, d.pts, d.conf = _ptr(w4), _ptr(b4), _ptr(pts), _ptr(conf)
    with _on_device(a):
        L.check(L.load().f3r_gemm(C.byref(d), _stream(a)), "f3r_gemm")


def gemm_x3(a: torch.Tensor, wt3: torch.Tensor, *, a_relu: bool = False, **kw):
    """Parity-mode GEMM: a fp32 (..., K) is split into bf16 [hi | lo | hi] (optionally of relu(a)) and multiplied with
    wt3 = bf16 (N, taps, 3K) packed as [Whi | Whi | Wlo]: hi*hi + lo*hi + hi*lo accumulated in fp32."""
    _chk(a, F32, "a")
    k = a.shape[-1]
    assert wt3.shape[-1] == 3 * k, (wt3.shape, k)
    a3 = torch.empty(a.shape[:-1] + (3 * k,), dtype=BF16, device=a.device)
    split3(a, a3, relu=a_relu)
    return gemm(a3, wt3, **kw)


def split3(x: torch.Tensor, out: torch.Tensor, relu: bool = False):
    _chk(x, F32, "x"); _chk(out, BF16, "out")
    k = x.shape[-1]
    assert out.numel() == 3 * x.numel()
    with _on_device(x):
        L.check(L.load().f3r_split3(_ptr(x), _ptr(out), x.numel() // k, k, int(relu), _stream(x)), "f3r_split3")


def add_f32(dst: torch.Tensor, src: torch.Tensor):
    _chk(dst, F32, "dst"); _chk(src, F32, "src")
    assert dst.numel() == src.numel()
    with _on_device(dst):
        L.check(L.load().f3r_add_f32(_ptr(dst), _ptr(src), dst.numel(), _stream(dst)), "f3r_add_f32")


def linear(a: torch.Tensor, wt: torch.Tensor, bias=None, **kw):
    """y = a @ wt.T (+bias ...) for a bf16 (M, K), wt bf16 (N, K)."""
    return gemm(a, wt, w=a.numel() // a.shape[-1], bias=bias, **kw)


NUM_SMS = 148


def pick_kv_split(units: int, key_blocks: int, max_split: int = 8) -> int:
    """Key slices per (batch, head, 256-row query tile) unit so that units * slices CTAs fill whole waves of the 148
    SMs (one CTA per SM): minimises ceil(units*s / 148) / s; every slice keeps >= 16 key blocks (below that the extra
    prologues and the merge pass cost more than the idle SMs, measured at N=4); 1 = no slicing."""
    if units >= 3 * NUM_SMS:
        return 1
    best, best_cost = 1, None
    for s_ in range(1, max_split + 1):
        if s_ > 1 and key_blocks // s_ < 16:
            break
        cost = -(-units * s_ // NUM_SMS) / s_ * (1.0 + 0.01 * (s_ - 1))  # (+1 % per extra slice: merge + prologues)
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = s_, cost
    return best


def attention_partial(q: torch.Tensor, kv: torch.Tensor, part_o: torch.Tensor, part_lse: torch.Tensor, *, part_base: int,
                      n_split: int, batch: int, heads: int, sq: int, kv_rows_total: int, kv_row0: int, skv: int,
                      scale: float):
    """Attends q to the keys [kv_row0, kv_row0 + skv) of kv (batch*kv_rows_total, ldkv), cut into n_split slices; slice s
    fills slot part_base + s of part_o (slots, batch*sq, heads*64) fp32 / part_lse (slots, batch, heads, sq) fp32."""
    _chk(q, BF16, "q"); _chk(kv, BF16, "kv"); _chk(part_o, F32, "part_o"); _chk(part_lse, F32, "part_lse")
    ldq, ldkv = q.shape[-1], kv.shape[-1]
    assert q.numel() == batch * sq * ldq and kv.numel() == batch * kv_rows_total * ldkv
    slots = part_o.shape[0]
    assert part_base + n_split <= slots and part_o.numel() == slots * batch * sq * heads * 64
    assert part_lse.numel() == slots * batch * heads * sq
    with _on_device(q):
        L.check(L.load().f3r_attention_partial(_ptr(q), ldq, _ptr(kv), ldkv, kv_rows_total, kv_row0, skv, n_split,
                                               _ptr(part_o), _ptr(part_lse), part_base, batch, heads, sq, float(scale),
                                               _stream(q)), "f3r_attention_partial")


def attention_merge(part_o: torch.Tensor, part_lse: torch.Tensor, n_parts: int, out: torch.Tensor, *, batch: int,
                    heads: int, sq: int):
    _chk(part_o, F32, "part_o"); _chk(part_lse, F32, "part_lse"); _chk(out, BF16, "out")
    assert out.numel() == batch * sq * out.shape[-1] and n_parts <= part_o.shape[0]
    with _on_device(out):
        L.check(L.load().f3r_attention_merge(_ptr(part_o), _ptr(part_lse), n_parts, _ptr(out), out.shape[-1], batch,
                                             heads, sq, _stream(out)), "f3r_attention_merge")


def attention(q: torch.Tensor, kv: torch.Tensor, out: torch.Tensor, *, batch: int, heads: int, sq: int, skv: int,
              scale: float, lse: Optional[torch.Tensor] = None, kv_split: Optional[int] = None):
    """q (batch*sq, ldq) bf16, kv (batch*skv, ldkv) bf16 [K | V], out (batch*sq, ldo) bf16.  When the launch would
    leave SMs idle (few query tiles), the keys are cut into slices (more CTAs) and merged (pick_kv_split)."""
    _chk(q, BF16, "q"); _chk(kv, BF16, "kv"); _chk(out, BF16, "out")
    ldq, ldkv, ldo = q.shape[-1], kv.shape[-1], out.shape[-1]
    assert q.numel() == batch * sq * ldq and kv.numel() == batch * skv * ldkv and out.numel() == batch * sq * ldo
    timer = KERNEL_TIMER
    st = torch.cuda.current_stream(q.device)
    if timer is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
    ns = kv_split if kv_split is not None else (
        1 if lse is not None else pick_kv_split(batch * heads * ((sq + 255) // 256), (skv + 127) // 128))
    if ns > 1:
        part_o = torch.empty(ns, batch * sq, heads * 64, dtype=F32, device=q.device)
        part_lse = torch.empty(ns, batch, heads, sq, dtype=F32, device=q.device)
        attention_partial(q, kv, part_o, part_lse, part_base=0, n_split=ns, batch=batch, heads=heads, sq=sq,
                          kv_rows_total=skv, kv_row0=0, skv=skv, scale=scale)
        attention_merge(part_o, part_lse, ns, out, batch=batch, heads=heads, sq=sq)
    else:
        with _on_device(q):
            L.check(L.load().f3r_attention(_ptr(q), ldq, _ptr(kv), ldkv, _ptr(out), ldo, _ptr(lse), batch, heads, sq, skv,
                                           float(scale), st.cuda_stream), "f3r_attention")
    if timer is not None:
        e1.record(st)
        timer.append((batch, heads, sq, skv, e0, e1))


def attention_x3(q: torch.Tensor, kv: torch.Tensor, out: torch.Tensor, *, batch: int, heads: int, sq: int, skv: int,
                 scale: float, lse: Optional[torch.Tensor] = None):
    """Parity-mode attention: q (batch*sq, ldq), kv (batch*skv, ldkv) [K | V], out (batch*sq, ldo), all fp32."""
    _chk(q, F32, "q"); _chk(kv, F32, "kv"); _chk(out, F32, "out")
    ldq, ldkv, ldo = q.shape[-1], kv.shape[-1], out.shape[-1]
    assert q.numel() == batch * sq * ldq and kv.numel() == batch * skv * ldkv and out.numel() == batch * sq * ldo
    lib = L.load()
    nbytes = int(lib.f3r_attention_x3_workspace(batch, heads, sq, skv))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=q.device)  # caching allocator: >= 512-byte aligned
    with _on_device(q):
        L.check(lib.f3r_attention_x3(_ptr(q), ldq, _ptr(kv), ldkv, _ptr(out), ldo, _ptr(lse), _ptr(ws), nbytes, batch,
                                     heads, sq, skv, float(scale), _stream(q)), "f3r_attention_x3")


def transformer_blocks(x: torch.Tensor, blocks, *, batch: int, seq: int, heads: int, eps: float, scale: float,
                       rope=None):
    """n consecutive transformer blocks on the fp32 residual stream x (batch*seq, D), in place, in ONE library call
    (f3r_transformer_blocks).  `blocks`: objects with n1w, n1b, n2w, n2b, qkv_w, qkv_b, proj_w, proj_b, fc1_w, fc1_b,
    fc2_w, fc2_b (bf16 weights [N, 1, K], fp32 biases); rope: dict(P=tokens per image, gw=grid width, cos=, sin=) or None."""
    _chk(x, F32, "x")
    D = x.shape[-1]
    hidden = blocks[0].fc1_w.shape[0]
    arr = (L.BlockWeights * len(blocks))()
    for i, b in enumerate(blocks):
        for name, t in (("norm1_w", b.n1w), ("norm1_b", b.n1b), ("norm2_w", b.n2w), ("norm2_b", b.n2b),
                        ("qkv_w", b.qkv_w), ("qkv_b", b.qkv_b), ("proj_w", b.proj_w), ("proj_b", b.proj_b),
                        ("fc1_w", b.fc1_w), ("fc1_b", b.fc1_b), ("fc2_w", b.fc2_w), ("fc2_b", b.fc2_b)):
            setattr(arr[i], name, _ptr(t))
    lib = L.load()
    rows = batch * seq
    assert x.numel() == rows * D
    nbytes = int(lib.f3r_transformer_workspace(rows, D, hidden))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    with _on_device(x):
        L.check(lib.f3r_transformer_blocks(arr, len(blocks), _ptr(x), batch, seq, D, heads, hidden, float(eps), float(scale),
                                           rope["gw"] if rope else 0, rope["P"] if rope else 0,
                                           _ptr(rope["cos"]) if rope else None, _ptr(rope["sin"]) if rope else None,
                                           _ptr(ws), nbytes, _stream(x)), "f3r_transformer_blocks")


def layernorm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float, out: torch.Tensor):
    _chk(x, F32, "x"); _chk(w, F32, "w"); _chk(b, F32, "b")
    assert out.dtype in (BF16, F32) and out.is_contiguous() and out.numel() == x.numel()
    dim = x.shape[-1]
    with _on_device(x):
        L.check(L.load().f3r_layernorm(_ptr(x), _ptr(w), _ptr(b), _ptr(out), int(out.dtype == F32), x.numel() // dim,
                                       dim, float(eps), _stream(x)), "f3r_layernorm")


def im2col_patch(img: torch.Tensor, out: torch.Tensor):
    _chk(img, F32, "img")
    assert out.dtype in (BF16, F32) and out.is_contiguous()
    n, c, h, w = img.shape
    assert c == 3 and out.numel() == n * (h // 16) * (w // 16) * 768
    with _on_device(img):
        L.check(L.load().f3r_im2col_patch(_ptr(img), _ptr(out), int(out.dtype == F32), n, h, w, _stream(img)),
                "f3r_im2col_patch")


def im2col3x3s2(x: torch.Tensor, out: torch.Tensor, n: int, h: int, w: int, c: int, ho: int, wo: int):
    _chk(x, BF16, "x"); _chk(out, BF16, "out")
    assert x.numel() == n * h * w * c and out.numel() == n * ho * wo * 9 * c
    with _on_device(x):
        L.check(L.load().f3r_im2col3x3s2(_ptr(x), _ptr(out), n, h, w, c, ho, wo, _stream(x)), "f3r_im2col3x3s2")


def upsample2x(x: torch.Tensor, out: torch.Tensor, n: int, h: int, w: int, c: int, ho: int, wo: int):
    assert x.dtype in (BF16, F32) and x.dtype == out.dtype and x.is_contiguous() and out.is_contiguous()
    assert x.numel() == n * h * w * c and out.numel() == n * ho * wo * c
    with _on_device(x):
        L.check(L.load().f3r_upsample2x(_ptr(x), _ptr(out), int(x.dtype == F32), n, h, w, c, ho, wo, _stream(x)),
                "f3r_upsample2x")


def cast_bf16(x: torch.Tensor, out: torch.Tensor):
    _chk(x, F32, "x"); _chk(out, BF16, "out")
    assert x.numel() == out.numel()
    with _on_device(x):
        L.check(L.load().f3r_cast_bf16(_ptr(x), _ptr(out), x.numel(), _stream(x)), "f3r_cast_bf16")


# ------------------------------------------------------------------ geometry tail (csrc/geometry.cu)
def conf_quantile(conf: torch.Tensor, q: float) -> torch.Tensor:
    """conf fp32 [views, n] -> thr fp32 [views] = torch.quantile(conf[v], q) (exact, linear interpolation)."""
    _chk(conf, F32, "conf")
    assert conf.dim() == 2
    thr = torch.empty(conf.shape[0], dtype=F32, device=conf.device)
    with _on_device(conf):
        L.check(L.load().f3r_conf_quantile(_ptr(conf), conf.shape[0], conf.shape[1], float(q), _ptr(thr), _stream(conf)),
                "f3r_conf_quantile")
    return thr


def similarity_fit(x: torch.Tensor, y: torch.Tensor, conf: Optional[torch.Tensor] = None,
                   thr: Optional[torch.Tensor] = None, valid: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x, y fp32 [views, n, 3]; conf fp32 [views, n] with thr fp32 [views]; valid uint8 [views, n].  Returns rts
    fp32 [views, 13] (R row-major, t, s) with y ~ s R x + t over conf >= thr & valid (fallbacks as the reference)."""
    _chk(x, F32, "x"); _chk(y, F32, "y")
    views, n = x.shape[0], x.shape[1]
    assert x.shape == y.shape == (views, n, 3)
    if conf is not None:
        _chk(conf, F32, "conf"); _chk(thr, F32, "thr")
        assert conf.shape == (views, n) and thr.shape == (views,)
    if valid is not None:
        _chk(valid, torch.uint8, "valid")
        assert valid.shape == (views, n)
    lib = L.load()
    nbytes = lib.f3r_similarity_fit_workspace(views)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=x.device)
    rts = torch.empty(views, 13, dtype=F32, device=x.device)
    with _on_device(x):
        L.check(lib.f3r_similarity_fit(_ptr(x), _ptr(y), _ptr(conf), _ptr(thr), _ptr(valid), views, n, _ptr(rts), _ptr(ws),
                                       nbytes, _stream(x)), "f3r_similarity_fit")
    return rts


def similarity_apply(x: torch.Tensor, rts: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[v] = s_v (x[v] R_v^T) + t_v, fp32 [views, n, 3]."""
    _chk(x, F32, "x"); _chk(rts, F32, "rts")
    views, n = x.shape[0], x.shape[1]
    assert x.shape == (views, n, 3) and rts.shape == (views, 13)
    if out is None:
        out = torch.empty_like(x)
    _chk(out, F32, "out")
    assert out.shape == x.shape
    with _on_device(x):
        L.check(L.load().f3r_similarity_apply(_ptr(x), _ptr(rts), _ptr(out), views, n, _stream(x)), "f3r_similarity_apply")
    return out


def focal_weiszfeld(pts: torch.Tensor, conf: Optional[torch.Tensor] = None, thr: Optional[torch.Tensor] = None,
                    pp: Optional[torch.Tensor] = None, iters: int = 100) -> torch.Tensor:
    """pts fp32 [views, H, W, 3]; conf fp32 [views, H, W] with thr fp32 [views]; pp fp32 [views, 2] or None (image
    centre).  Returns focal fp32 [views]."""
    _chk(pts, F32, "pts")
    views, h, w = pts.shape[0], pts.shape[1], pts.shape[2]
    assert pts.shape == (views, h, w, 3)
    if conf is not None:
        _chk(conf, F32, "conf"); _chk(thr, F32, "thr")
        assert conf.shape == (views, h, w) and thr.shape == (views,)
    if pp is not None:
        _chk(pp, F32, "pp")
        assert pp.shape == (views, 2)
    lib = L.load()
    nbytes = lib.f3r_focal_workspace(views)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=pts.device)
    focal = torch.empty(views, dtype=F32, device=pts.device)
    with _on_device(pts):
        L.check(lib.f3r_focal_weiszfeld(_ptr(pts), _ptr(conf), _ptr(thr), _ptr(pp), views, h, w, int(iters), _ptr(focal),
                                        _ptr(ws), nbytes, _stream(pts)), "f3r_focal_weiszfeld")
    return focal


# ------------------------------------------------------------------ camera poses (csrc/pnp.cu)
def pnp_ransac(pts: torch.Tensor, mask: torch.Tensor, focals: torch.Tensor, pp: Optional[torch.Tensor] = None,
               iters: int = 10):
    """pts fp32 [views, H, W, 3]; mask uint8 [views, H, W]; focals fp32 [views, n_focals] (candidates per view); pp fp32
    [views, 2] or None (= (W/2, H/2)).  Per view, `iters` P3P-RANSAC hypotheses per candidate focal, the best refined by
    Levenberg-Marquardt (f3r_pnp_ransac).  Returns scores int32 [views, n_focals, iters] (inliers at <= 5 px),
    best int32 [views, 2] = (k, i) of the selected hypothesis or (-1, -1), c2w fp64 [views, 3, 4]."""
    _chk(pts, F32, "pts"); _chk(mask, torch.uint8, "mask"); _chk(focals, F32, "focals")
    views, h, w = pts.shape[0], pts.shape[1], pts.shape[2]
    assert pts.shape == (views, h, w, 3) and mask.shape == (views, h, w)
    assert focals.dim() == 2 and focals.shape[0] == views
    n_focals = focals.shape[1]
    if pp is not None:
        _chk(pp, F32, "pp")
        assert pp.shape == (views, 2)
    lib = L.load()
    nbytes = int(lib.f3r_pnp_workspace(views, h, w, n_focals, int(iters)))
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=pts.device)  # caching allocator: >= 512-byte aligned
    scores = torch.empty(views, n_focals, max(int(iters), 0), dtype=torch.int32, device=pts.device)
    best = torch.empty(views, 2, dtype=torch.int32, device=pts.device)
    c2w = torch.empty(views, 3, 4, dtype=torch.float64, device=pts.device)
    with _on_device(pts):
        L.check(lib.f3r_pnp_ransac(_ptr(pts), _ptr(mask), views, h, w, _ptr(focals), n_focals, _ptr(pp), int(iters),
                                   _ptr(scores), _ptr(best), _ptr(c2w), _ptr(ws), nbytes, _stream(pts)), "f3r_pnp_ransac")
    return scores, best, c2w
