"""Headline benchmark: views/sec of one Fast3R ViT-L/512 forward pass over N synthetic 512x368 views.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--views V] [--impl ours|reference|library] [--dump-outputs DIR]

* ours, 1 GPU: BASELINE.json configs[1] (N=32 views, 512x368, bf16 tensor-core operands) on one B200 is the
  headline `value`; `config.extra` adds configs[2] (N=320, long-sequence regime) with its own roofline, the
  per-GEMM rates of the fusion-decoder linears, and the "library bar" (the UNMODIFIED reference model on the same B200
  under bf16 autocast + SDPA-flash, from oracle/_ref).
* ours, N GPUs (torchrun, one rank per GPU): the SAME total N=32 workload, views sharded by contiguous ranges
  (sequence-parallel fusion decoder, K|V exchange per layer over NCCL) -> "scaling": "strong"; `config.extra` adds the
  sharded-vs-unsharded parity of the run and, at 8 GPUs, configs[3] (N=1000).
* --impl reference: the reference's OWN `inference(..., dtype="32")` on the host CPU cores (oracle/_ref, made by
  oracle/make_ref.py), on BASELINE configs[0] (N=4 views per step) - a bounded sample of the workload.  Falls back to
  the CPU oracle port when oracle/_ref is missing.

One JSON line on stdout (rank 0).  `value` = views/s with inputs resident in HBM; `e2e` = the same metric through
the reference-facing API `inference()` from pinned host buffers including H2D and D2H.  `--dump-outputs DIR` writes
the preds of the last timed headline step (see dump_outputs); the inputs and weights are seeded, so two builds run with
the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 368, 512
P_TOK, DMODEL, DEPTH = 736, 1024, 24


def flops_total(n):  # BASELINE.md §3, GFLOP -> FLOP
    return (1304.15 * n + 53.25 * n * n) * 1e9


def flops_decoder(n):
    return (446.07 * n + 53.25 * n * n) * 1e9


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        """Start of the timed region: samples taken before this call are dropped (nvidia-smi needs ~1 s to come up, so
        the sampler is started ahead of the region)."""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        t0 = getattr(self, "t0", 0.0)
        for ts, ln in self.lines:
            if ts < t0:
                continue
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        med = sm[len(sm) // 2] if sm else None
        return {"sm_mhz": med, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def make_views(n, device=None, pinned=False, seed0=1234, only=None):
    """SURVEY §8(d) synthetic views.  `only` = (lo, hi): materialise just that range (sequence-parallel ranks never touch
    the other views' pixels); the rest share one placeholder tensor of the right shape."""
    import numpy as np
    import torch
    views, placeholder = [], None
    for i in range(n):
        if only is not None and not (only[0] <= i < only[1]):
            if placeholder is None:
                placeholder = torch.zeros(1, 3, H, W)
            img = placeholder
        else:
            g = torch.Generator().manual_seed(seed0 + i)
            img = torch.rand(1, 3, H, W, generator=g) * 2 - 1
            if pinned:
                img = img.pin_memory()
            if device is not None:
                img = img.to(device)
        views.append(dict(img=img, true_shape=np.int32([[H, W]]), idx=i, instance=str(i), dataset="synthetic",
                          label=f"v{i}"))
    return views


DUMP_BYTES = 60 * 10 ** 6


def dump_outputs(preds, out_dir, seed=0):
    """Writes the preds of one forward - per key the views stacked, (N, B, H, W[, C]) - as float32 `out_dir/<key>.npy`.
    When they exceed DUMP_BYTES, every key keeps the same seeded sample of pixel positions, (N, B, P[, C]), so that
    two builds run with the same arguments can be compared value for value."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    out = {k: torch.stack([p[k] for p in preds]).float() for k, v in preds[0].items()
           if torch.is_tensor(v) and v.is_floating_point()}
    total = sum(v.numel() * 4 for v in out.values())
    for k, v in out.items():
        if total > DUMP_BYTES:
            hw = v.shape[2] * v.shape[3]
            idx = torch.randperm(hw, generator=torch.Generator().manual_seed(seed))[:hw * DUMP_BYTES // total]
            v = v.flatten(2, 3)[:, :, idx.sort().values.to(v.device)]
        np.save(os.path.join(out_dir, f"{k}.npy"), v.cpu().numpy())


def pick_cpu_threads():
    """The box may expose more logical CPUs than the container's quota allows: pick the torch thread count that
    actually maximises matmul throughput (a few short probes) instead of blindly using os.cpu_count()."""
    import torch
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, 128, avail) if c <= avail} | {min(avail, 8)})
    a = torch.randn(2048, 2048)
    best, best_t = cands[0], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ a
        t0 = time.time()
        for _ in range(5):
            a @ a
        dt = time.time() - t0
        if dt < best_t * 0.9:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


# ----------------------------------------------------------------------------- the reference itself (oracle/_ref)
def reference_model(device="cpu"):
    """The UNMODIFIED reference Fast3R (ViT-L dicts, random init under manual_seed(0), SURVEY §8(d)) and its
    inference().  Returns None when no reference copy is available."""
    import torch
    try:
        from oracle.ref_harness import import_reference, reference_available
        if not reference_available():
            return None
        import logging
        logging.disable(logging.WARNING)
        RefFast3R, ref_inference = import_reference()
    except Exception:
        return None
    from fast3r_b200 import vit_large_args
    enc, dec, head = vit_large_args()
    torch.manual_seed(0)
    with torch.device(device):
        model = RefFast3R(dict(enc), dict(dec), dict(head)).eval()
    model = model.to(device)  # buffers built from numpy (image_idx_emb) ignore the device context
    return model, ref_inference


def cpu_reference_sample(n_views, steps, warmup):
    """Times the reference's own inference(dtype="32") (kind "reference") - or the oracle port (kind "port") - on the
    host cores.  Returns (seconds per step, kind, cores)."""
    import torch
    cores = pick_cpu_threads()
    ref = reference_model("cpu")
    views = make_views(n_views)
    if ref is not None:
        model, ref_inference = ref

        def step():
            torch.manual_seed(7)
            ref_inference([dict(v) for v in views], model, torch.device("cpu"), dtype="32", verbose=False)
        kind = "reference"
    else:
        from oracle import fast3r_oracle as O
        from fast3r_b200 import Fast3R, vit_large_args
        enc, dec, head = vit_large_args()
        torch.manual_seed(0)
        sd = Fast3R(enc, dec, head).state_dict()
        imgs = [v["img"] for v in views]

        def step():
            torch.manual_seed(7)
            O.forward(sd, enc, dec, head, imgs)
        kind = "port"
    with torch.no_grad():
        for _ in range(warmup):
            step()
        t0 = time.time()
        for _ in range(steps):
            step()
        dt = (time.time() - t0) / steps
    return dt, kind, cores


def sample_text(n_sample, n_work, kind):
    src = ("the reference's own inference(dtype='32') (oracle/_ref, unmodified fast3r package)" if kind == "reference"
           else "the CPU oracle port (oracle/fast3r_oracle.py)")
    ratio = (flops_total(n_work) / n_work) / (flops_total(n_sample) / n_sample)
    return (f"{n_sample} views 368x512 per step (BASELINE configs[0]) through {src}, fp32, torch CPU flash-SDPA, all host "
            f"threads; global attention grows with N^2: a view costs x{ratio:.2f} more FLOPs at N={n_work} than at "
            f"N={n_sample}, so CPU views/s at N={n_work} would be ~value/{ratio:.2f}")


def run_reference(args, rank, world):
    if rank != 0:
        return
    n_sample = args.ref_views
    dt, kind, cores = cpu_reference_sample(n_sample, args.steps, 1 if args.warmup >= 1 else 0)
    v = n_sample / dt
    sample = sample_text(n_sample, args.views, kind)
    line = {"impl": "reference", "metric": "views_per_sec", "value": v, "unit": "views/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": f"Fast3R ViT-L/512 forward, N={args.views} views 512x368, random-init weights",
                       "measured_views_per_step": n_sample, "same_config": n_sample == args.views, "kind": kind,
                       "sample": sample,
                       "extrapolated_views_per_sec_at_workload_N":
                           v / ((flops_total(args.views) / args.views) / (flops_total(n_sample) / n_sample))},
            "cpu_baseline": {"value": v, "unit": "views/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "views/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- library bar (reference on the B200)
def library_bar(n_views, dev, steps=3, warmup=2):
    """The UNMODIFIED reference model on this GPU: bf16 autocast + SDPA-flash (BASELINE.md §4 item 4) - torch/cuBLAS/
    cuDNN/flash kernels, none of ours.  Returns a dict (or {"unavailable": why})."""
    import torch
    try:
        ref = reference_model(dev)
        if ref is None:
            return {"unavailable": "no reference copy (oracle/_ref missing)"}
        model, ref_inference = ref
        views = make_views(n_views, device=dev)
        for v in views:  # Fast3R.forward (unlike inference()) does not collate: it wants tensors
            v["true_shape"] = torch.from_numpy(v["true_shape"]).to(dev)

        def step():
            torch.manual_seed(7)
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                return model(views)
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        del model
        torch.cuda.empty_cache()
        return {"views": n_views, "ms_per_forward": ms, "views_per_sec": n_views / (ms * 1e-3),
                "achieved_tflops_whole_forward": flops_total(n_views) / (ms * 1e-3) / 1e12,
                "what": "reference Fast3R.forward (oracle/_ref) on this B200, torch.autocast(bfloat16), "
                        "attn_implementation=flash_attention (SDPA flash), device-resident inputs"}
    except Exception as e:  # the bar is context, never a reason to lose the headline number
        torch.cuda.empty_cache()
        return {"unavailable": repr(e)[:300]}


def run_library(args, rank, world, local_rank):
    import torch
    if rank != 0:
        return
    torch.cuda.set_device(local_rank)
    r = library_bar(args.views, torch.device("cuda", local_rank), steps=args.steps, warmup=max(1, min(args.warmup, 3)))
    print(json.dumps({"impl": "library", "metric": "views_per_sec", "value": r.get("views_per_sec"), "unit": "views/s",
                      "n_gpus": 1, "config": {"workload": f"N={args.views} views 512x368"}, **r}), flush=True)


# ----------------------------------------------------------------------------- ours
def gemm_rates(dev, peak_tf):
    """The four linears of one fusion-decoder block at N=32 (M = 23 552 tokens), each timed alone with CUDA events,
    L2 flushed by a 512 MB write between launches."""
    import torch
    from fast3r_b200 import ops, lib as L
    M = 32 * P_TOK
    bf, f32 = torch.bfloat16, torch.float32
    g = torch.Generator(device="cpu").manual_seed(1)
    mk = lambda *s: (torch.randn(*s, generator=g) * 0.05).to(bf).to(dev)  # noqa: E731
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    x = torch.zeros(M, DMODEL, dtype=f32, device=dev)
    cases = {
        "qkv": (mk(M, 1024), mk(3072, 1, 1024), dict(out0=torch.empty(M, 1024, dtype=bf, device=dev), ldo=1024,
                                                       split_col=1024, out0b=torch.empty(M, 2048, dtype=bf, device=dev),
                                                       ldo_b=2048)),
        "proj": (mk(M, 1024), mk(1024, 1, 1024), dict(out0=x, res0=x)),
        "fc1_gelu": (mk(M, 1024), mk(4096, 1, 1024), dict(out0=torch.empty(M, 4096, dtype=bf, device=dev), act=L.ACT_GELU)),
        "fc2": (mk(M, 4096), mk(1024, 1, 4096), dict(out0=x, res0=x)),
    }
    out = {}
    for name, (a, w, kw) in cases.items():
        bias = torch.zeros(w.shape[0], dtype=f32, device=dev)
        ts = []
        for it in range(7):
            flush.fill_(it)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.linear(a, w, bias, **kw)
            e1.record()
            torch.cuda.synchronize()
            if it >= 2:
                ts.append(e0.elapsed_time(e1))
        ms = sorted(ts)[len(ts) // 2]
        tf = 2.0 * M * w.shape[0] * w.shape[2] / (ms * 1e-3) / 1e12
        out[name] = {"us": ms * 1e3, "tflops": tf, "frac_of_measured_peak": tf / peak_tf}
    return out


def ingest_rates(dev, hbm_gbs):
    """SURVEY §8 f3: resize + crop + normalise of load_images() for a 12-Mpixel photo (4032x3024 -> 512x384): the GPU kernels
    (f3r_ingest_rgb8, bit-exact with Pillow) vs Pillow itself on one host core (what the reference's loop does per image)."""
    import numpy as np
    import torch
    from PIL import Image
    from fast3r_b200.ingest import ingest_rgb8
    h, w = 3024, 4032
    img = np.random.default_rng(0).integers(0, 256, (h, w, 3), dtype=np.uint8)
    u8 = torch.from_numpy(img).to(dev)
    out = torch.empty(3, 384, 512, dtype=torch.float32, device=dev)
    for _ in range(3):
        ingest_rgb8(u8, 512, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        ingest_rgb8(u8, 512, out=out)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / 20 * 1e3
    pil = Image.fromarray(img)
    t0 = time.time()
    for _ in range(3):
        pil.resize((512, 384), Image.LANCZOS)
    cpu_ms = (time.time() - t0) / 3 * 1e3
    nbytes = h * w * 3 + 2 * h * 512 * 3 + 3 * 384 * 512 * 4   # source read + 8-bit intermediate write/read + fp32 out
    return {"image": "4032x3024 RGB8 -> 3x384x512 fp32 (LANCZOS, crop, normalise)", "gpu_us_per_image": us,
            "gpu_images_per_sec": 1e6 / us, "algorithmic_bytes": nbytes, "achieved_gbs": nbytes / us / 1e3,
            "frac_of_measured_hbm": nbytes / us / 1e3 / hbm_gbs, "pillow_cpu_ms_per_image_1_core": cpu_ms,
            "note": "decode (PIL, host threads) and the H2D copy of the decoded image are outside this number"}


def geometry_rates(dev, hbm_gbs):
    """SURVEY §8 f2 (first slice): align_local_pts3d_to_global for N=32 views at 512x368 - the GPU kernels (quantile, masked
    moments + Umeyama, apply) on device-resident preds vs the oracle restatement on one host core for one view (the
    reference runs one such task per (view, batch item) in a CPU thread pool), plus the 100-iteration Weiszfeld focal."""
    import numpy as np
    import torch
    from fast3r_b200 import ops
    from oracle import geometry_oracle as go
    views, h, w = 32, 368, 512
    n = h * w
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(views, n, 3, device=dev, generator=g) + 2
    y = 1.5 * x.flip(-1).contiguous() + 0.01 * torch.randn(views, n, 3, device=dev, generator=g)
    conf = 1 + torch.exp(torch.randn(views, n, device=dev, generator=g))
    out = torch.empty_like(x)

    def align():
        thr = ops.conf_quantile(conf, 0.3)
        ops.similarity_apply(x, ops.similarity_fit(x, y, conf, thr), out)

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e3

    us = timed(align, 20)
    thr30 = ops.conf_quantile(conf, 0.3)
    rts30 = ops.similarity_fit(x, y, conf, thr30)
    parts = {"quantile": timed(lambda: ops.conf_quantile(conf, 0.3), 20),
             "fit": timed(lambda: ops.similarity_fit(x, y, conf, thr30), 20),
             "apply": timed(lambda: ops.similarity_apply(x, rts30, out), 20)}
    nbytes = views * n * (5 * 4 + 28 + 24)  # 5 quantile passes over conf; fit reads x, y, conf; apply reads x, writes out
    pts = x.reshape(views, h, w, 3)
    cmap = conf.reshape(views, h, w)
    thr10 = ops.conf_quantile(conf, 0.1)
    us_f = timed(lambda: ops.focal_weiszfeld(pts[:1], cmap[:1], thr10[:1], None, iters=100), 5)
    t0 = time.time()
    go.align_local_to_global(x[0].reshape(h, w, 3).cpu().numpy(), cmap[0].cpu().numpy(), y[0].reshape(h, w, 3).cpu().numpy(), None, 30.0)
    cpu_ms = (time.time() - t0) * 1e3
    t0 = time.time()
    go.estimate_focal(pts[0].cpu().numpy(), cmap[0].cpu().numpy())
    cpu_f_ms = (time.time() - t0) * 1e3
    return {"workload": "align_local_pts3d_to_global, 32 views 512x368, 30th-percentile confidence mask",
            "gpu_us_per_32_views": us, "gpu_views_per_sec": views / us * 1e6, "algorithmic_bytes": nbytes,
            "achieved_gbs": nbytes / us / 1e3, "frac_of_measured_hbm": nbytes / us / 1e3 / hbm_gbs,
            "gpu_us_by_kernel": parts, "apply_gbs": views * n * 24 / parts["apply"] / 1e3,
            "oracle_cpu_ms_per_view_1_core": cpu_ms, "focal_weiszfeld_100it_gpu_us_per_view": us_f,
            "focal_oracle_cpu_ms_per_view_1_core": cpu_f_ms,
            "note": "inputs resident in HBM; PnP-RANSAC (fast_pnp) is not part of this slice"}


def attention_roofline(timer, n_views, ms_step, clocks, peak_tf, peak_src):
    att = [(b, h, sq, skv, a.elapsed_time(z)) for (b, h, sq, skv, a, z) in timer if skv == n_views * P_TOK]
    if not att:
        return None, 0.0
    att_ms = sum(t[4] for t in att) / len(att)
    sq = att[0][2]
    att_flops = 4.0 * sq * (n_views * P_TOK) * DMODEL  # QK^T + PV, 2 FLOP/MAC, all heads
    ach = att_flops / (att_ms * 1e-3) / 1e12
    roof = {"kernel": "attention_kernel (fusion decoder global attention, 24 launches/step)", "bound": "tensor",
            "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "peak_source": peak_src,
            "ms_per_launch": att_ms, "flops_per_launch": att_flops,
            # not measured inside this run: the ncu --set full figure lives in profiles/ (r02_ncu_attn_*.txt)
            "traffic": None,
            "algorithmic_bytes_per_launch": 2.0 * DMODEL * (2 * sq + 2 * n_views * P_TOK),
            "share_of_step": DEPTH * att_ms / ms_step}
    try:  # the binding unit at head_dim 64 is the special-function unit (16 ex2 / clk / SM)
        clk = (clocks or {}).get("sm_mhz") or 1965.0
        exps = float(sq) * (n_views * P_TOK) * (DMODEL // 64)
        roof["sfu"] = {"exp2_per_launch": exps, "peak_exp2_per_s": 148 * 16 * clk * 1e6,
                       "frac": exps / (att_ms * 1e-3) / (148 * 16 * clk * 1e6), "sm_mhz": clk}
    except Exception:
        pass
    return roof, att_ms


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from fast3r_b200 import Fast3R, vit_large_args, inference, lib as L, ops
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    enc, dec, head = vit_large_args()
    torch.manual_seed(0)
    with torch.device(dev):  # random-init ViT-L weights created directly in HBM (no checkpoint available offline)
        model = Fast3R(enc, dec, head).eval()
    sp = None
    if world > 1:
        from fast3r_b200.parallel import enable_sequence_parallel, shard_views
        sp = enable_sequence_parallel(model, gather_preds=False)
    peak_tf, hbm, peak_src = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def timed_device(views, steps, warmup):
        """K forwards with device-resident inputs; returns (ms/step max over ranks, launches, attention timer)."""
        def step():
            torch.manual_seed(7)
            return model(views)
        for _ in range(warmup):
            step()
        barrier()
        timer = []
        ops.KERNEL_TIMER = timer
        n0 = L.launch_count()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            step()
        last = step()  # only the last step's preds are kept, so earlier steps allocate exactly as before
        e1.record()
        barrier()
        ops.KERNEL_TIMER = None
        return e0.elapsed_time(e1) / steps, L.launch_count() - n0, timer, last

    # ================= headline: N = args.views (default 32, BASELINE configs[1]) =================
    N = args.views
    rng = shard_views(N, world)[rank] if world > 1 else None
    views_dev = make_views(N, device=dev, only=rng)
    views_host = make_views(N, pinned=True, only=rng)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        torch.manual_seed(7)
        model(views_dev)
    torch.cuda.synchronize()
    sampler.mark()
    if sp is not None:
        sp.timers = []
    ms, launches, timer, last = timed_device(views_dev, args.steps, 0)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(last, args.dump_outputs)
    del last
    roof, att_ms = attention_roofline(timer, N, ms, clocks, peak_tf, peak_src)
    sp_trace = None
    if sp is not None and sp.timers:
        tr = sp.timers
        sp.timers = None
        n = len(tr)
        avg = lambda f: sum(f(e) for e in tr) / n  # noqa: E731
        sp_trace = {"calls": n,
                    "attend_total_ms": avg(lambda e: e[0].elapsed_time(e[3])),
                    "local_chunk_attention_ms": avg(lambda e: e[0].elapsed_time(e[1])),
                    "remote_chunks_attention_incl_wait_ms": avg(lambda e: e[1].elapsed_time(e[2])),
                    "merge_ms": avg(lambda e: e[2].elapsed_time(e[3])),
                    "allgather_on_comm_stream_ms": avg(lambda e: e[4].elapsed_time(e[5])),
                    "allgather_end_after_local_end_ms": avg(lambda e: e[1].elapsed_time(e[5]))}
        att_ms = sp_trace["attend_total_ms"]
        sq = (rng[1] - rng[0]) * P_TOK
        flops = 4.0 * sq * (N * P_TOK) * DMODEL
        ach = flops / (att_ms * 1e-3) / 1e12
        roof = {"kernel": "attention_kernel key-range partials + merge incl. exposed K|V exchange wait "
                          "(fusion decoder global attention, 24 per step)", "bound": "tensor", "achieved": ach,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "peak_source": peak_src,
                "ms_per_launch": att_ms, "flops_per_launch": flops, "traffic": None,
                "share_of_step": DEPTH * att_ms / ms}

    # ---- end to end through inference() (pinned host -> device -> host)
    def step_e2e():
        torch.manual_seed(7)
        vs = [dict(v) for v in views_host]  # loss_of_one_batch overwrites view["img"] with the device copy
        return inference(vs, model, dev, dtype=torch.bfloat16, verbose=False)
    for _ in range(min(args.warmup, 2) or 1):
        step_e2e()
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    g0.record()
    for _ in range(args.steps):
        res = step_e2e()
    g1.record()
    barrier()
    ms_e2e = max(g0.elapsed_time(g1), (time.time() - t0) * 1e3) / args.steps  # D2H is synchronous: wall >= events
    n_local = (rng[1] - rng[0]) if rng is not None else N
    h2d = n_local * 3 * H * W * 4                      # fp32 images of this rank's views
    d2h = sum(v.numel() * v.element_size() for p in res["preds"] for v in p.values() if hasattr(v, "numel"))
    del res
    ms, ms_e2e, att_ms_max = allmax([ms, ms_e2e, att_ms])
    if roof is not None:
        ach = roof["flops_per_launch"] / (att_ms_max * 1e-3) / 1e12
        roof.update(achieved=ach, frac=ach / peak_tf, ms_per_launch=att_ms_max, share_of_step=DEPTH * att_ms_max / ms)

    extra = {}
    if sp_trace is not None:
        extra["sp_attention_trace_rank0"] = sp_trace
        kvx = next(iter(sp._kvx.values()), None)
        extra["sp_kv_transport"] = ("copy-engine pulls from symmetric peer memory (torch symmetric memory)"
                                    if (kvx is not None and kvx.sym_state) else "NCCL all-gather on a side stream")
    # ================= sharded vs un-sharded parity of THIS run (world > 1) =================
    if world > 1:
        torch.manual_seed(7)
        out_sp = model(views_dev)
        model.sp_group, model.image_id_rank_offset = None, 0   # single-device forward with the rank-0 id stream
        full = make_views(N, device=dev)
        torch.manual_seed(7)
        out_1 = model(full)
        model.sp_group, model.image_id_rank_offset = sp, None
        worst = 0.0
        for i in range(rng[0], rng[1]):
            for k in out_1[i]:
                a, b = out_sp[i][k].float(), out_1[i][k].float()
                worst = max(worst, float((a - b).abs().max() / b.abs().max().clamp_min(1e-30)))
        extra["sp_parity_max_rel"] = allmax([worst])[0]
        del out_sp, out_1, full
    torch.cuda.empty_cache()

    # ================= further BASELINE configs (few steps each, own roofline) =================
    def extra_config(n_views, steps=2, warmup=1):
        r = shard_views(n_views, world)[rank] if world > 1 else None
        vd = make_views(n_views, device=dev, only=r)
        if sp is not None:
            sp.timers = []
        m, _l, tm = timed_device(vd, steps, warmup)[:3]
        rf, am = attention_roofline(tm, n_views, m, clocks, peak_tf, peak_src)
        if sp is not None and sp.timers:   # sharded: the attention of a layer = key-range partials + merge (+ exposed wait)
            tr, sp.timers = sp.timers[-DEPTH * steps:], None
            am = sum(e[0].elapsed_time(e[3]) for e in tr) / len(tr)
            fl = 4.0 * (r[1] - r[0]) * P_TOK * (n_views * P_TOK) * DMODEL
            rf = {"kernel": "attention_kernel key-range partials + merge incl. exposed K|V exchange wait", "bound": "tensor",
                  "peak": peak_tf, "unit": "TFLOP/s", "peak_source": peak_src, "flops_per_launch": fl, "traffic": None}
        m, am = allmax([m, am])
        if rf is not None:
            a = rf["flops_per_launch"] / (am * 1e-3) / 1e12
            rf.update(achieved=a, frac=a / peak_tf, ms_per_launch=am, share_of_step=DEPTH * am / m)
        del vd
        torch.cuda.empty_cache()
        return {"views": n_views, "tokens": n_views * P_TOK, "steps": steps, "ms_per_forward": m,
                "views_per_sec": n_views / (m * 1e-3), "achieved_tflops_whole_forward": flops_total(n_views) / (m * 1e-3) / 1e12,
                "decoder_tflops_per_gpu_upper_bound": flops_decoder(n_views) / world / (m * 1e-3) / 1e12,
                "roofline": rf}
    if not args.no_extras and N == 32:
        if world == 1:
            extra["N320_1gpu"] = extra_config(320)
        if world == 8:
            extra["N320_8gpu"] = extra_config(320)
            extra["N1000_8gpu"] = extra_config(1000)
        if world == 1:
            extra["decoder_gemms_M23552"] = gemm_rates(dev, peak_tf)
            try:
                extra["ingest_12mpix"] = ingest_rates(dev, hbm)
            except Exception as e:  # context only
                extra["ingest_12mpix"] = {"unavailable": repr(e)[:200]}
            try:
                extra["geometry_tail_N32"] = geometry_rates(dev, hbm)
            except Exception as e:  # context only
                extra["geometry_tail_N32"] = {"unavailable": repr(e)[:200]}
    if rank == 0 and world == 1 and not args.no_extras and not args.no_library_bar:
        extra["library_bar_N32"] = library_bar(32, dev)
    if rank != 0:
        return
    line = {"metric": "views_per_sec", "value": N / (ms * 1e-3), "unit": "views/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"Fast3R ViT-L/512 forward, N={N} views 512x368 (BASELINE configs[1] shape), "
                                   "random-init weights, fp32 pointmaps out",
                       "views": N, "tokens": N * P_TOK,
                       "parallelism": "single GPU" if world == 1 else f"sequence-parallel x{world} (K|V exchange/layer)",
                       "l2": "working set (1.3 GB weights + GBs of activations per step) exceeds the 126 MB L2; no explicit flush",
                       "achieved_tflops_whole_forward": flops_total(N) / (ms * 1e-3) / 1e12,
                       "extra": extra},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": N / (ms_e2e * 1e-3), "unit": "views/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "note": "bytes of rank 0 (its own views / preds); the input views are not copied back"},
            "roofline": roof}
    if world == 1 and not args.no_cpu_baseline:
        dt, kind, cores = cpu_reference_sample(args.ref_views, 1, 0)
        line["cpu_baseline"] = {"value": args.ref_views / dt, "unit": "views/s", "cores": cores, "kind": kind,
                                "sample": f"one forward, {dt:.1f} s: " + sample_text(args.ref_views, N, kind)}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--views", type=int, default=32)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "library"])
    ap.add_argument("--ref-views", type=int, default=4, help="views per CPU reference step (BASELINE configs[0])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip config.extra (N=320 / N=1000 / GEMM rates / library bar)")
    ap.add_argument("--no-library-bar", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the preds of the last timed step as DIR/<key>.npy (float32; a seeded pixel sample when "
                         "the whole output is larger than 60 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200 (no CPU fallback); use --impl reference for the CPU arm")
    if args.impl == "library":
        run_library(args, rank, world, local_rank)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
