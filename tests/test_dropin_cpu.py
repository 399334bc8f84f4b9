"""Drop-in boundary beyond forward(): hub mixin, config containers, DUSt3R checkpoint loading, portrait views, and the
reference's own consumers (its inference(), MultiViewDUSt3RLitModule, estimate_camera_poses) running on this model.
CPU only: the kernels are replaced by tests/abi_emulator.py.  The Lightning-module test needs the reference fast3r
package importable and skips without it; the others read fixtures recorded from the reference under tests/golden/."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from tests.conftest import rel_l2
from tests.golden.synth import synth_state_dict, synth_images


@pytest.fixture()
def emulated(monkeypatch):
    import fast3r_b200.model as M
    from tests import abi_emulator
    monkeypatch.setattr(M, "ops", abi_emulator)
    monkeypatch.setattr(M, "_require_cuda", lambda device: None)
    return M


def test_hub_mixin_roundtrip(tmp_path):
    """Fast3R.from_pretrained(local_dir) / save_pretrained like the reference (fast3r/models/fast3r.py:45-49, README.md:84)."""
    from fast3r_b200 import Fast3R, tiny_args
    m = Fast3R(*tiny_args())
    m.save_pretrained(str(tmp_path))
    assert {"config.json", "model.safetensors"} <= set(os.listdir(tmp_path))
    m2 = Fast3R.from_pretrained(str(tmp_path))
    assert m2.encoder_args == m.encoder_args and m2.decoder_args == m.decoder_args and m2.head_args == m.head_args
    for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert torch.equal(a, b), k


def test_mapping_configs_are_accepted():
    """omegaconf DictConfig / ListConfig look like Mapping / Sequence: the ctor must turn them into plain containers
    (reference: OmegaConf.to_container, fast3r.py:59-66)."""
    from collections.abc import Mapping, Sequence
    from fast3r_b200 import Fast3R, tiny_args

    class DictCfg(Mapping):
        def __init__(self, d): self._d = {k: wrap(v) for k, v in d.items()}
        def __getitem__(self, k): return self._d[k]
        def __iter__(self): return iter(self._d)
        def __len__(self): return len(self._d)

    class ListCfg(Sequence):
        def __init__(self, v): self._v = [wrap(x) for x in v]
        def __getitem__(self, i): return self._v[i]
        def __len__(self): return len(self._v)

    def wrap(v):
        return DictCfg(v) if isinstance(v, dict) else ListCfg(v) if isinstance(v, (list, tuple)) else v

    enc, dec, head = tiny_args()
    m = Fast3R(DictCfg(enc), DictCfg(dec), DictCfg(head))
    assert type(m.head_args) is dict and type(m.head_args["depth_mode"]) is list and m.head_args == head


def test_unsupported_head_modes_are_refused():
    from fast3r_b200 import Fast3R, tiny_args
    enc, dec, head = tiny_args()
    for bad in (dict(conf_mode=["exp", 1, 100.0]), dict(depth_mode=["exp", -10.0, 10.0]), dict(depth_mode=["linear", float("-inf"), float("inf")])):
        with pytest.raises(NotImplementedError):
            Fast3R(enc, dec, dict(head, **bad))


def test_load_from_dust3r_checkpoint(tmp_path):
    """Encoder + downstream_head1 of a DUSt3R checkpoint are taken over, everything else is left (fast3r.py:162-239)."""
    from fast3r_b200 import Fast3R, tiny_args
    m = Fast3R(*tiny_args())
    sd = m.state_dict()
    g = torch.Generator().manual_seed(1)
    ck = {}
    for k, v in sd.items():
        if k.startswith("encoder."):
            ck[k[len("encoder."):]] = torch.randn(v.shape, generator=g)
        elif k.startswith("downstream_head."):
            ck[k.replace("downstream_head.", "downstream_head1.", 1)] = torch.randn(v.shape, generator=g)
    for k in list(ck):  # scratch.layer_rn.{i} aliases scratch.layer{i+1}_rn (one tensor in the module)
        if ".scratch.layer_rn." in k:
            i = int(k.split(".scratch.layer_rn.")[1].split(".")[0])
            ck[k] = ck[k.replace(f".scratch.layer_rn.{i}.", f".scratch.layer{i + 1}_rn.")]
    ck["dec_blocks.0.attn.qkv.weight"] = torch.zeros(3)   # DUSt3R decoder weights are ignored
    path = str(tmp_path / "DUSt3R_ViTLarge_BaseDecoder_512_dpt.pth")
    torch.save({"model": ck}, path)
    before = {k: v.clone() for k, v in sd.items()}
    loaded, not_loaded = m.load_from_dust3r_checkpoint(path)
    after = m.state_dict()
    assert "dec_blocks.0.attn.qkv.weight" in not_loaded
    for k in after:
        if k.startswith("encoder."):
            assert torch.equal(after[k], ck[k[len("encoder."):]]), k
        elif k.startswith("downstream_head."):
            assert torch.equal(after[k], ck[k.replace("downstream_head.", "downstream_head1.", 1)]), k
        else:
            assert torch.equal(after[k], before[k]), k


def _portrait_model_views(M, g):
    from fast3r_b200 import tiny_args
    enc, dec, head = tiny_args()
    enc.update(g["enc_over"]); head.update(g["head_over"])
    model = M.Fast3R(enc, dec, head).eval()
    model.load_state_dict(synth_state_dict(g["shapes"], seed=g["weight_seed"]))
    imgs = synth_images(g["N"], g["B"], g["H"], g["W"])
    views = [dict(img=im, true_shape=torch.tensor([g["true_shapes"][i]] * g["B"], dtype=torch.int32), idx=i,
                  instance=str(i)) for i, im in enumerate(imgs)]
    return model, views


@pytest.mark.parametrize("precision,tol", [("bf16", 2e-2), ("fp32", 1e-3)])
def test_portrait_view_against_reference_fixture(emulated, golden_dir, precision, tol):
    """ManyAR_PatchEmbed + landscape_only heads with one portrait view (stored transposed): reference outputs."""
    g = torch.load(os.path.join(golden_dir, "tiny_portrait.pt"))
    model, views = _portrait_model_views(emulated, g)
    model.set_precision(precision)
    torch.manual_seed(g["rng_seed"])
    preds = model(views)
    for p, q in zip(preds, g["preds"]):
        for k in q:
            assert p[k].shape == q[k].shape
    for k in g["preds"][0]:
        e = rel_l2(torch.cat([p[k].flatten() for p in preds]), torch.cat([q[k].flatten() for q in g["preds"]]))
        assert e < tol, (k, e)


def test_portrait_needs_manyar_configuration(emulated, golden_dir):
    from fast3r_b200 import tiny_args
    g = torch.load(os.path.join(golden_dir, "tiny_portrait.pt"))
    model = emulated.Fast3R(*tiny_args()).eval()   # PatchEmbedDust3R / landscape_only=False (inference configuration)
    imgs = synth_images(2, 1, g["H"], g["W"])
    views = [dict(img=imgs[0], true_shape=torch.tensor([[g["H"], g["W"]]])),
             dict(img=imgs[1], true_shape=torch.tensor([[g["W"], g["H"]]]))]
    with pytest.raises(ValueError):
        model(views)


# ------------------------------------------------------------------ the reference's own consumers on this model
def _reference_or_skip():
    from oracle.ref_harness import reference_available, import_reference
    if not reference_available():
        pytest.skip("reference sources not available")
    return import_reference()


def _tiny(M, golden_dir, tag="tiny_b1_n3"):
    from fast3r_b200 import tiny_args
    g = torch.load(os.path.join(golden_dir, f"{tag}.pt"))
    model = M.Fast3R(*tiny_args()).eval()
    model.load_state_dict(synth_state_dict(g["shapes"], seed=g["weight_seed"]))
    imgs = synth_images(g["N"], g["B"], g["H"], g["W"])
    views = [dict(img=im, true_shape=np.int32([[g["H"], g["W"]]]), idx=i, instance=str(i), dataset="synthetic",
                  label=f"v{i}") for i, im in enumerate(imgs)]
    return g, model, views


def test_reference_inference_function_drives_this_model(emulated, golden_dir):
    """The call fast3r.dust3r.inference_multiview.inference (the reference's code, unmodified) makes on the model -
    collated views, keyword arguments, grad and autocast state, recorded by tests/golden/make_golden.py - replayed on
    the B200 model object."""
    g, model, views = _tiny(emulated, golden_dir)
    call = torch.load(os.path.join(golden_dir, "tiny_b1_n3_inference_call.pt"))
    assert len(call["views"]) == len(views)
    for v, r in zip(views, call["views"]):
        assert torch.equal(v["img"], r["img"])
    model.set_precision("fp32")
    torch.manual_seed(g["rng_seed"])
    with torch.set_grad_enabled(call["grad_enabled"]), torch.autocast("cpu", enabled=call["autocast_enabled"]):
        preds = model(call["views"], **call["kwargs"])
    assert len(preds) == len(g["preds"])
    for p, q in zip(preds, g["preds"]):
        for k in q:
            assert rel_l2(p[k], q[k]) < 1e-3, k


def _stub_lightning_stack():
    """Import stubs for the packages multiview_dust3r_module.py pulls in at module level and this image lacks
    (multiview_dust3r_module.py:1-24).  Nothing of the reference is modified."""
    import torch.nn as nn

    def mod(name, **attrs):
        m = sys.modules.get(name) or types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    class LightningModule(nn.Module):
        def save_hyperparameters(self, *a, **k): pass
        @property
        def device(self): return torch.device("cpu")

    class _Metric(nn.Module):
        def __init__(self, *a, **k): super().__init__()
        def update(self, *a, **k): pass
        def compute(self): return torch.tensor(0.0)

    class BaseAggregator(_Metric):
        def __init__(self, fn=None, default_value=None, nan_strategy=None, state_name="value", **k):
            super().__init__()
            setattr(self, state_name, default_value)

    for name in ("roma", "open3d", "pl_bolts", "pl_bolts.optimizers", "lightning.pytorch", "lightning.pytorch.loggers"):
        mod(name)
    mod("lightning", LightningModule=LightningModule)
    mod("lightning.pytorch.loggers.wandb", WandbLogger=type("WandbLogger", (), {}))
    mod("torchmetrics", MaxMetric=_Metric, MeanMetric=_Metric, MinMetric=_Metric, SumMetric=_Metric, Metric=_Metric)
    mod("torchmetrics.aggregation", BaseAggregator=BaseAggregator)
    mod("pl_bolts.optimizers.lr_scheduler", LinearWarmupCosineAnnealingLR=type("LinearWarmupCosineAnnealingLR", (), {}))


def test_lightning_module_and_pose_estimation_on_this_model(emulated, golden_dir, tmp_path):
    """MultiViewDUSt3RLitModule.load_for_inference(net) + forward, the isinstance(self.net, Fast3R) branch of
    _load_pretrained_weights (multiview_dust3r_module.py:998-1017) and estimate_camera_poses (:811-869) with the B200
    model installed under the reference's class name (fast3r_b200.compat.install)."""
    _reference_or_skip()
    _stub_lightning_stack()
    from fast3r_b200 import compat
    try:
        compat.install()
        try:
            import fast3r.models.multiview_dust3r_module as lit_mod
        except Exception as e:  # a dependency of the training stack that cannot be stubbed here
            pytest.skip(f"reference Lightning module not importable in this image: {e!r}")
        assert lit_mod.Fast3R is emulated.Fast3R
        g, model, views = _tiny(emulated, golden_dir)
        lit = lit_mod.MultiViewDUSt3RLitModule.load_for_inference(model)
        assert lit.net is model and not lit.training
        tviews = [dict(v, true_shape=torch.from_numpy(v["true_shape"])) for v in views]
        torch.manual_seed(g["rng_seed"])
        preds = lit(tviews)
        for p, q in zip(preds, g["preds"]):
            for k in q:
                assert rel_l2(p[k], q[k]) < 2e-2, k
        # pretrained Fast3R checkpoint ('net.' prefix) goes through the isinstance(self.net, Fast3R) branch
        sd2 = synth_state_dict(g["shapes"], seed=3)
        ck = str(tmp_path / "fast3r.ckpt")
        torch.save({"state_dict": {"net." + k: v for k, v in sd2.items()}}, ck)
        lit.pretrained = ck
        lit._load_pretrained_weights()
        assert torch.equal(model.state_dict()["decoder.decoder_embed.weight"], sd2["decoder.decoder_embed.weight"])
        # the step every caller runs right after the forward: focal + PnP pose per view from pts3d_local / conf
        poses, focals = lit_mod.MultiViewDUSt3RLitModule.estimate_camera_poses([dict(p) for p in g["preds"]], niter_PnP=10)
        ours = [{k: v.clone() for k, v in p.items()} for p in preds]
        poses2, focals2 = lit_mod.MultiViewDUSt3RLitModule.estimate_camera_poses(ours, niter_PnP=10)
        assert len(poses2[0]) == len(views) and len(focals2[0]) == len(views)
        assert all(np.isfinite(np.asarray(p)).all() for p in poses2[0])
    finally:
        compat.uninstall()
