"""Pins the preprocess oracle (oracle/preprocess_ref.py): against Pillow + torchvision running here,
and against the reference's test_tensors fixtures (their sha256 in the committed golden), both from the
stored decoded pixels and from the reference's own test images (tests/golden/reference_images)."""
import hashlib
import os

import numpy as np
import pytest

from oracle import preprocess_ref as P

GOLD = os.path.join(os.path.dirname(__file__), "golden", "preprocess_ref.npz")
REF_IMAGES = os.path.join(os.path.dirname(__file__), "golden", "reference_images")


def _torchvision_transform(n_px):
    from torchvision import transforms as T
    from torchvision.transforms import InterpolationMode
    return T.Compose([T.Resize(n_px, interpolation=InterpolationMode.BICUBIC), T.CenterCrop(n_px),
                      lambda im: im.convert("RGB"), T.ToTensor(), T.Normalize(P.OPENAI_MEAN, P.OPENAI_STD)])


@pytest.mark.parametrize("shape", [(224, 224), (300, 224), (224, 301), (375, 500), (500, 375), (225, 226), (97, 64),
                                   (1, 1), (3, 700), (1333, 800), (449, 448)])
def test_oracle_matches_pillow_torchvision(shape):
    from PIL import Image
    rng = np.random.default_rng(shape[0] * 7919 + shape[1])
    px = rng.integers(0, 256, (*shape, 3), dtype=np.uint8)
    ref = _torchvision_transform(224)(Image.fromarray(px)).numpy()
    got = P.preprocess(px)
    assert got.dtype == np.float32 and got.shape == (3, 224, 224)
    assert np.array_equal(got, ref)


def test_oracle_other_size():
    from PIL import Image
    px = np.random.default_rng(5).integers(0, 256, (400, 640, 3), dtype=np.uint8)
    ref = _torchvision_transform(336)(Image.fromarray(px)).numpy()
    assert np.array_equal(P.preprocess(px, 336), ref)


def test_oracle_matches_committed_reference_golden():
    g = np.load(GOLD)
    n = 0
    for name in g["names"]:
        key = f"pixels_{name}"
        if key not in g.files:
            continue
        got = P.preprocess(g[key])
        assert hashlib.sha256(got.tobytes()).digest() == g[f"sha256_{name}"].tobytes(), name
        n += 1
    assert n == 4


def test_oracle_matches_reference_fixtures():
    """The reference's 7 test images, decoded with Pillow, against the sha256 of the float32 tensors its
    preprocess produced for them (test_tensors/*.pkl; tests/golden/make_preprocess_golden.py)."""
    from PIL import Image
    g = np.load(GOLD)
    seen = 0
    for name in g["names"]:
        px = np.asarray(Image.open(os.path.join(REF_IMAGES, f"{name}.jpg")).convert("RGB"))
        got = P.preprocess(px)
        assert hashlib.sha256(got.tobytes()).digest() == g[f"sha256_{name}"].tobytes(), name
        seen += 1
    assert seen == 7


def test_pack_images_layout_and_mode_conversion():
    """Host side of the GPU transform: the packed batch layout of b200_preproc_run and the RGB conversion
    (no CUDA involved)."""
    from PIL import Image
    from clip_retrieval_b200.preprocess import pack_images, to_rgb8

    rng = np.random.default_rng(0)
    a = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    g = rng.integers(0, 256, (4, 3), dtype=np.uint8)
    buf, off, hh, ww = pack_images([a, Image.fromarray(g, mode="L"), Image.fromarray(a).convert("RGBA")])
    assert hh.tolist() == [5, 4, 5] and ww.tolist() == [7, 3, 7]
    assert off.tolist() == [0, 105, 141] and buf.size == 105 + 36 + 105 and buf.dtype == np.uint8
    assert np.array_equal(buf[:105].reshape(5, 7, 3), a)
    assert np.array_equal(buf[105:141].reshape(4, 3, 3), np.repeat(g[:, :, None], 3, axis=2))
    assert np.array_equal(buf[141:].reshape(5, 7, 3), a)
    assert np.array_equal(to_rgb8(g), np.repeat(g[:, :, None], 3, axis=2))
    with pytest.raises(ValueError):
        to_rgb8(np.zeros((4, 4, 3), np.float32))
    e = pack_images([])
    assert e[0].size == 0 and e[1].size == 0
