"""Image ingest (SURVEY §8 f3), CPU side: the C oracle (oracle/ingest_oracle.c, a restatement of Pillow's 8-bit resampler +
the crop / normalise of load_images) is pinned bit-exactly against Pillow / torchvision themselves - the third-party
dependencies the reference calls (fast3r/dust3r/utils/image.py:32, 68-159) - and against what the reference's own
load_images() returned on image files (a recorded fixture); the library's HOST tap-table function is checked against
the oracle."""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import ingest_oracle as O

SIZES = [(640, 480), (4032, 3024), (3024, 4032), (300, 200), (1000, 1000), (97, 131), (512, 384), (513, 384), (2000, 350),
         (1920, 1080)]


def _img(w, h, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


@pytest.mark.parametrize("w,h", SIZES)
def test_resize_matches_pillow_bit_exact(w, h):
    from PIL import Image
    img = _img(w, h, w * 7 + h)
    for size in (512, 224):
        nw, nh, filt = O.resize_plan(w, h, size)
        ref = np.asarray(Image.fromarray(img).resize((nw, nh), Image.LANCZOS if filt == O.LANCZOS else Image.BICUBIC))
        assert np.array_equal(O.resize_rgb8(img, nw, nh, filt), ref), (w, h, size)


@pytest.mark.parametrize("w,h", SIZES)
def test_full_ingest_matches_pil_torchvision_pipeline(w, h):
    """resize + center crop + ToTensor + Normalize exactly as load_images() composes them (image.py:118-146)."""
    import torchvision.transforms as tvf
    from PIL import Image
    norm = tvf.Compose([tvf.ToTensor(), tvf.Normalize((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))])
    img = _img(w, h, 3 * w + h)
    for size, square_ok in ((512, False), (512, True), (224, False)):
        pil = Image.fromarray(img)
        W1, H1 = pil.size
        S = max(pil.size)
        le = round(size * max(W1 / H1, H1 / W1)) if size == 224 else size
        interp = Image.LANCZOS if S > le else Image.BICUBIC
        pil = pil.resize(tuple(int(round(x * le / S)) for x in pil.size), interp)
        W, H = pil.size
        cx, cy = W // 2, H // 2
        if size == 224:
            half = min(cx, cy)
            pil = pil.crop((cx - half, cy - half, cx + half, cy + half))
        else:
            halfw, halfh = ((2 * cx) // 16) * 8, ((2 * cy) // 16) * 8
            if not square_ok and W == H:
                halfh = 3 * halfw / 4
            pil = pil.crop((cx - halfw, cy - halfh, cx + halfw, cy + halfh))
        ref = norm(pil).numpy()
        out, (H2, W2) = O.ingest(img, size, square_ok)
        assert (H2, W2) == ref.shape[1:], (w, h, size)
        assert np.array_equal(out, ref), (w, h, size, float(np.abs(out - ref).max()))


def test_reference_load_images_on_files(golden_dir):
    """The reference's own load_images() (PNG files, lossless) against the oracle pipeline.  The fixture, recorded by
    tests/golden/make_golden.py, holds per image the reference's true_shape, the sha256 of its full fp32 output and a
    seeded sample of the values."""
    g = torch.load(os.path.join(golden_dir, "load_images.pt"))
    assert len(g["views"]) == len(g["sizes"])
    for (w, h), seed, v in zip(g["sizes"], g["seeds"], g["views"]):
        out, shape = O.ingest(_img(w, h, seed), g["size"])
        assert tuple(v["true_shape"].tolist()) == tuple(shape)
        assert out.shape == v["shape"], (w, h)
        assert np.array_equal(out.reshape(-1)[v["index"].numpy()], v["values"].numpy()), (w, h)
        assert hashlib.sha256(np.ascontiguousarray(out, np.float32).tobytes()).hexdigest() == v["sha256"], (w, h)


def test_library_tap_tables_match_oracle():
    """f3r_resample_coeffs (host function of libfast3r_b200.so, no CUDA needed) vs the oracle's tables."""
    from fast3r_b200 import lib as L
    lib = L.load()
    for (n_in, n_out, filt) in [(4032, 512, 1), (3024, 384, 1), (300, 512, 0), (1000, 512, 1), (97, 64, 1), (513, 512, 1)]:
        ks = lib.f3r_resample_ksize(n_in, n_out, filt)
        assert ks == O.lib().f3r_oracle_ksize(n_in, n_out, filt)
        b1, k1 = np.empty((n_out, 2), np.int32), np.empty((n_out, ks), np.int32)
        b2, k2 = np.empty((n_out, 2), np.int32), np.empty((n_out, ks), np.int32)
        span = lib.f3r_resample_coeffs(n_in, n_out, filt, b1.ctypes.data_as(C.c_void_p), k1.ctypes.data_as(C.c_void_p))
        O.lib().f3r_oracle_coeffs(n_in, n_out, filt, b2.ctypes.data_as(C.c_void_p), k2.ctypes.data_as(C.c_void_p))
        assert np.array_equal(b1, b2) and np.array_equal(k1, k2)
        assert span >= int((b1[:, 0] + b1[:, 1]).max() - b1[:, 0].min()) // max(1, (n_out + 63) // 64) - 1 and span > 0
