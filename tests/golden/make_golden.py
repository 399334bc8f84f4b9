"""Generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference) on CPU fp32.

Run in the build container only:  python tests/golden/make_golden.py
(The GPU box has no /root/reference; tests there read the committed fixtures.)
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle.ref_harness import import_reference  # noqa: E402
from oracle.fast3r_oracle import tiny_args, vit_large_args  # noqa: E402
from tests.golden.synth import synth_state_dict, synth_images  # noqa: E402

Fast3R, inference = import_reference()
from fast3r.croco.models.blocks import Block  # noqa: E402
from fast3r.croco.models.pos_embed import RoPE2D  # noqa: E402


def half(t):
    return t.detach().clone()


def run_tiny(B, N, H, W, tag, dec_over=None, head_over=None, train_mode=False):
    enc, dec, head = tiny_args()
    dec.update(dec_over or {})
    head.update(head_over or {})
    torch.manual_seed(0)
    model = Fast3R(dict(enc), dict(dec), dict(head)).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    sd = synth_state_dict(shapes, seed=0)
    model.load_state_dict(sd)
    if train_mode:
        model.train()  # forward-only check of the training-mode variants (scale 1/8, per-view heads; SURVEY a13)
    taps = {}

    def hook(name):
        def f(_m, _i, o):
            taps[name] = half(o[0] if isinstance(o, tuple) else o)
        return f

    model.encoder.patch_embed.register_forward_hook(hook("patch_embed"))
    for i, b in enumerate(model.encoder.enc_blocks):
        b.register_forward_hook(hook(f"enc_block{i}"))
    model.encoder.register_forward_hook(hook("enc_out"))
    model.decoder.decoder_embed.register_forward_hook(hook("dec_embed_linear"))
    for i, b in enumerate(model.decoder.dec_blocks):
        if i in (0, 5, 11):
            b.register_forward_hook(hook(f"dec_block{i}"))
    dpt = model.downstream_head.dpt
    for i in range(4):
        dpt.scratch.layer_rn[i].register_forward_hook(hook(f"layer_rn{i}"))
    for i in (3, 4):
        getattr(dpt.scratch, f"refinenet{i}").register_forward_hook(hook(f"path{i}_uncropped"))
    dpt.head.register_forward_hook(hook("head_out"))

    imgs = synth_images(N, B, H, W)
    views = [dict(img=imgs[i], true_shape=torch.tensor([[H, W]] * B, dtype=torch.int32), idx=i, instance=str(i),
                  dataset="synthetic", label=f"v{i}") for i in range(N)]
    # record the ids the reference will draw (same RNG stream, replayed)
    torch.manual_seed(7)
    seed = torch.randint(0, 2 ** 32, (1,)).item()
    g = torch.Generator(); g.manual_seed(seed)
    ids = torch.zeros(B, N, dtype=torch.long)
    for b in range(B):
        ids[b, 1:] = torch.randperm(999, generator=g)[: N - 1] + 1
    torch.manual_seed(7)
    with torch.no_grad():
        preds = model(views)
    keep = None if (B == 1 and not dec_over and not head_over and not train_mode) else ()
    snap = {k: v for k, v in taps.items() if keep is None or k in keep}  # snapshot (later runs re-fire the hooks)
    out = dict(shapes=shapes, taps=snap, image_ids=ids, B=B, N=N, H=H, W=W, weight_seed=0, rng_seed=7,
               dec_over=dec_over or {}, head_over=head_over or {}, train_mode=train_mode,
               preds=[{k: half(v) for k, v in p.items()} for p in preds])
    if B == 1 and not dec_over and not head_over and not train_mode:
        # the public API on the same inputs (inference(): collate, dtype="32", to_cpu)
        views1 = [dict(img=imgs[i], true_shape=np.int32([[H, W]]), idx=i, instance=str(i),
                       dataset="synthetic", label=f"v{i}") for i in range(N)]
        torch.manual_seed(7)
        res = inference(views1, model, torch.device("cpu"), dtype="32", verbose=False)
        for a, b in zip(res["preds"], preds):
            for k in a:
                assert torch.equal(a[k], b[k]), k
        out["inference_keys"] = sorted(res.keys())
        out["inference_view_keys"] = sorted(res["views"][0].keys())
        # calibration: the reference's own bf16-autocast path vs its fp32 path
        torch.manual_seed(7)
        res16 = inference(views1, model, torch.device("cpu"), dtype=torch.bfloat16, verbose=False)
        gap = {}
        for k in preds[0]:
            a = torch.cat([p[k].float().flatten() for p in res16["preds"]])
            b = torch.cat([p[k].float().flatten() for p in preds])
            gap[k] = ((a - b).norm() / b.norm()).item()
        out["ref_bf16_vs_fp32_relL2"] = gap
        print(tag, "ref bf16 vs fp32 gap", gap)
    torch.save(out, os.path.join(HERE, f"{tag}.pt"))
    sz = os.path.getsize(os.path.join(HERE, f"{tag}.pt"))
    print(tag, "saved", sz / 1e6, "MB; pts abs mean", preds[0]["pts3d_in_other_view"].abs().mean().item(),
          "conf mean", preds[0]["conf"].mean().item())


def run_tiny_mixed(tag="tiny_mixed_res"):
    """Views of different resolutions in one forward (reference per-view path, fast3r/models/fast3r.py:276-294, 407-428)."""
    enc, dec, head = tiny_args()
    torch.manual_seed(0)
    model = Fast3R(dict(enc), dict(dec), dict(head)).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth_state_dict(shapes, seed=0))
    sizes = [(64, 96), (48, 64), (64, 96), (32, 48)]
    B = 1
    imgs = [synth_images(1, B, h, w, seed0=1234 + i)[0] for i, (h, w) in enumerate(sizes)]
    views = [dict(img=imgs[i], true_shape=torch.tensor([[h, w]] * B, dtype=torch.int32), idx=i, instance=str(i),
                  dataset="synthetic", label=f"v{i}") for i, (h, w) in enumerate(sizes)]
    torch.manual_seed(7)
    with torch.no_grad():
        preds = model(views)
    out = dict(shapes=shapes, sizes=sizes, B=B, weight_seed=0, rng_seed=7,
               preds=[{k: half(v) for k, v in p.items()} for p in preds])
    torch.save(out, os.path.join(HERE, f"{tag}.pt"))
    print(tag, "saved", os.path.getsize(os.path.join(HERE, f"{tag}.pt")) / 1e6, "MB")


def run_blocks():
    """ViT-L-width single transformer blocks (D=1024, 16 heads): encoder flavour (RoPE100, LN 1e-6,
    scale 1/8) and decoder flavour (no RoPE, LN 1e-5, eval scale 0.16019 / train 0.125)."""
    from functools import partial
    import torch.nn as nn
    out = {}
    gh, gw, n = 5, 8, 2
    x = torch.randn(n, gh * gw, 1024, generator=torch.Generator().manual_seed(11))
    yy, xx = torch.meshgrid(torch.arange(gh), torch.arange(gw), indexing="ij")
    pos = torch.stack((yy.reshape(-1), xx.reshape(-1)), -1)[None].expand(n, -1, -1).contiguous()
    enc_blk = Block(dim=1024, num_heads=16, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                    rope=RoPE2D(freq=100.0), attn_implementation="pytorch_naive").eval()
    shapes = {k: tuple(v.shape) for k, v in enc_blk.state_dict().items()}
    sd = synth_state_dict(shapes, seed=3)
    enc_blk.load_state_dict(sd)
    dec_blk = Block(dim=1024, num_heads=16, mlp_ratio=4.0, qkv_bias=True, norm_layer=nn.LayerNorm,
                    attn_implementation="pytorch_naive", attn_bias_for_inference_enabled=True).eval()
    dec_blk.load_state_dict(sd)
    with torch.no_grad():
        out["enc_block"] = enc_blk(x, pos)
        out["dec_block_eval"] = dec_blk(x.reshape(1, -1, 1024), None)
        dec_blk.train()
        out["dec_block_train"] = dec_blk(x.reshape(1, -1, 1024), None)
        q = torch.randn(2, 16, gh * gw, 64, generator=torch.Generator().manual_seed(12))
        out["rope_q"] = q
        out["rope_out"] = RoPE2D(freq=100.0)(q, pos)
    out.update(shapes=shapes, x=x, pos=pos, weight_seed=3)
    torch.save(out, os.path.join(HERE, "vitl_blocks.pt"))
    print("vitl_blocks saved", os.path.getsize(os.path.join(HERE, "vitl_blocks.pt")) / 1e6, "MB")


def run_tiny_portrait(tag="tiny_portrait"):
    """Training-style configuration: ManyAR_PatchEmbed + landscape_only=True heads; view 1 is a PORTRAIT image stored
    transposed in the landscape buffer (true_shape = (W, H)) - fast3r/dust3r/patch_embed.py:59-105,
    fast3r/dust3r/utils/misc.py:74-104."""
    enc, dec, head = tiny_args()
    enc.update(patch_embed_cls="ManyAR_PatchEmbed")
    head.update(landscape_only=True)
    torch.manual_seed(0)
    model = Fast3R(dict(enc), dict(dec), dict(head)).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth_state_dict(shapes, seed=0))
    B, N, H, W = 1, 3, 64, 96
    imgs = synth_images(N, B, H, W)
    true_shapes = [(H, W), (W, H), (H, W)]
    views = [dict(img=imgs[i], true_shape=torch.tensor([true_shapes[i]] * B, dtype=torch.int32), idx=i, instance=str(i),
                  dataset="synthetic", label=f"v{i}") for i in range(N)]
    torch.manual_seed(7)
    with torch.no_grad():
        preds = model(views)
    out = dict(shapes=shapes, B=B, N=N, H=H, W=W, true_shapes=true_shapes, weight_seed=0, rng_seed=7,
               enc_over=dict(patch_embed_cls="ManyAR_PatchEmbed"), head_over=dict(landscape_only=True),
               preds=[{k: half(v) for k, v in p.items()} for p in preds])
    torch.save(out, os.path.join(HERE, f"{tag}.pt"))
    print(tag, "saved", os.path.getsize(os.path.join(HERE, f"{tag}.pt")) / 1e6, "MB", {k: tuple(v.shape) for k, v in preds[1].items()})


def run_vitl_n4(tag="vitl_n4_368x512", stride=4):
    """BASELINE.json configs[0]: full ViT-L/512 (24+24 layers, 2 DPT heads), N=4 views 512x368, fp32 on CPU through the
    reference's own inference(..., dtype="32").  The full-resolution preds are 24 MB, so the fixture keeps every
    `stride`-th pixel in y and x (each pixel depends on the whole network) plus per-view full-resolution moments."""
    import time
    enc, dec, head = vit_large_args()
    torch.manual_seed(0)
    model = Fast3R(dict(enc), dict(dec), dict(head)).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth_state_dict(shapes, seed=5))
    N, B, H, W = 4, 1, 368, 512
    imgs = synth_images(N, B, H, W)
    views = [dict(img=imgs[i], true_shape=np.int32([[H, W]]), idx=i, instance=str(i), dataset="synthetic",
                  label=f"v{i}") for i in range(N)]
    torch.manual_seed(7)
    t0 = time.time()
    res = inference(views, model, torch.device("cpu"), dtype="32", verbose=False)
    dt = time.time() - t0
    preds = res["preds"]
    sub = [{k: v[:, ::stride, ::stride].contiguous().clone() for k, v in p.items()} for p in preds]
    mom = [{k: (float(v.double().mean()), float(v.double().std()), float(v.double().abs().max())) for k, v in p.items()}
           for p in preds]
    # calibration on this config: the reference's own bf16-autocast path vs its fp32 path
    torch.manual_seed(7)
    res16 = inference(views, model, torch.device("cpu"), dtype=torch.bfloat16, verbose=False)
    gap = {}
    for k in preds[0]:
        a = torch.cat([p[k].float().flatten() for p in res16["preds"]])
        b = torch.cat([p[k].float().flatten() for p in preds])
        gap[k] = ((a - b).norm() / b.norm()).item()
    out = dict(N=N, B=B, H=H, W=W, stride=stride, weight_seed=5, rng_seed=7, preds_sub=sub, moments=mom,
               ref_bf16_vs_fp32_relL2=gap, ref_cpu_seconds=dt, ref_cpu_threads=torch.get_num_threads())
    torch.save(out, os.path.join(HERE, f"{tag}.pt"))
    print(tag, "saved", os.path.getsize(os.path.join(HERE, f"{tag}.pt")) / 1e6, "MB;", f"{dt:.1f} s on",
          torch.get_num_threads(), "threads; ref bf16 vs fp32 gap", gap)


def run_inference_call(tag="tiny_b1_n3_inference_call"):
    """The call the reference's own inference(..., dtype="32") makes on the model for the tiny_b1_n3 views: the collated
    views, the keyword arguments, and the grad / autocast state around it (inference_multiview.py:22-95)."""
    enc, dec, head = tiny_args()
    torch.manual_seed(0)
    model = Fast3R(dict(enc), dict(dec), dict(head)).eval()
    shapes = {k: tuple(v.shape) for k, v in model.state_dict().items()}
    model.load_state_dict(synth_state_dict(shapes, seed=0))
    N, B, H, W = 3, 1, 64, 96
    imgs = synth_images(N, B, H, W)
    views = [dict(img=imgs[i], true_shape=np.int32([[H, W]]), idx=i, instance=str(i), dataset="synthetic",
                  label=f"v{i}") for i in range(N)]
    calls = []

    def recording_model(vs, **kw):
        calls.append(dict(views=[{k: v.clone() if torch.is_tensor(v) else v for k, v in x.items()} for x in vs],
                          kwargs=kw, grad_enabled=torch.is_grad_enabled(),
                          autocast_enabled=torch.is_autocast_enabled("cpu")))
        return model(vs, **kw)

    torch.manual_seed(7)
    inference(views, recording_model, torch.device("cpu"), dtype="32", verbose=False)
    assert len(calls) == 1
    torch.save(calls[0], os.path.join(HERE, f"{tag}.pt"))
    print(tag, "saved", os.path.getsize(os.path.join(HERE, f"{tag}.pt")) / 1e6, "MB", calls[0]["kwargs"])


def run_load_images(tag="load_images", n_sample=4096):
    """The reference's own load_images(dir, size=512) on PNG files (lossless) of seeded random images.  The full fp32
    outputs are 8 MB, so the fixture keeps per image the true_shape, the sha256 of the full array and a seeded sample
    of its values."""
    import hashlib
    import tempfile
    from PIL import Image
    from fast3r.dust3r.utils.image import load_images
    sizes = [(800, 600), (600, 800), (1024, 1024), (321, 123)]
    with tempfile.TemporaryDirectory() as d:
        for i, (w, h) in enumerate(sizes):
            a = np.random.default_rng(100 + i).integers(0, 256, (h, w, 3), dtype=np.uint8)
            Image.fromarray(a).save(os.path.join(d, f"im{i}.png"))
        views = load_images(d, size=512, verbose=False)
    rng = np.random.default_rng(0)
    out = []
    for v in views:
        img = np.ascontiguousarray(v["img"][0].numpy(), np.float32)
        idx = np.sort(rng.choice(img.size, n_sample, replace=False))
        out.append(dict(true_shape=torch.from_numpy(np.asarray(v["true_shape"][0])), shape=tuple(img.shape),
                        sha256=hashlib.sha256(img.tobytes()).hexdigest(), index=torch.from_numpy(idx),
                        values=torch.from_numpy(img.reshape(-1)[idx].copy())))
    torch.save(dict(sizes=sizes, seeds=[100 + i for i in range(len(sizes))], size=512, views=out),
               os.path.join(HERE, f"{tag}.pt"))
    print(tag, "saved", os.path.getsize(os.path.join(HERE, f"{tag}.pt")) / 1e6, "MB")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "consumers":
        run_inference_call()
        run_load_images()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "vitl_n4":
        run_vitl_n4()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "portrait":
        run_tiny_portrait()
        sys.exit(0)
    run_tiny(1, 3, 64, 96, "tiny_b1_n3")
    run_tiny(2, 2, 48, 64, "tiny_b2_n2")
    # configuration quirks the replacement must honour (SURVEY.md Q3 / Q14 / Q16)
    run_tiny(1, 3, 64, 96, "tiny_noattnbias", dec_over=dict(attn_bias_for_inference_enabled=False))
    run_tiny(1, 3, 64, 96, "tiny_fixedidx", dec_over=dict(random_image_idx_embedding=False))
    run_tiny(1, 2, 32, 48, "tiny_nolocal_n2", head_over=dict(with_local_head=False))
    run_tiny(1, 1, 48, 48, "tiny_single_view")
    run_tiny_mixed()
    run_tiny(1, 3, 32, 48, "tiny_trainmode", train_mode=True)
    run_blocks()
    run_tiny_portrait()
    run_vitl_n4()
