"""Image preprocessing of the predict API against vectors produced by the reference's own
transform (tests/golden/make_golden.py::preprocess_case): PIL decode -> Resize((224,224)) ->
ToTensor -> Normalize (data/preprocess.py:117-121, api/inference.py:140-170)."""
import io
import os

import numpy as np
import pytest
import torch
from PIL import Image

from conftest import GOLDEN
from vqa_b200.inference import VQAInference


@pytest.fixture(scope="module")
def g():
    return np.load(os.path.join(GOLDEN, "preprocess.npz"))


def test_identity_at_224_matches_reference_transform(g):
    inf = VQAInference()
    img = Image.fromarray(g["id224.u8"], "RGB")
    out = inf.preprocess_image(img)
    assert tuple(out.shape) == (1, 3, 224, 224) and out.dtype == torch.float32
    np.testing.assert_allclose(out[0].numpy(), g["id224.out"], rtol=0, atol=1e-6)
    assert np.array_equal(inf.preprocess_image_u8(img).numpy(), g["id224.u8"])


@pytest.mark.parametrize("name", ["down", "up", "odd"])
def test_resize_is_bit_exact_with_reference(g, name):
    """uint8 result of the PIL antialiased bilinear resize is bit-exact; the float output's moments match."""
    inf = VQAInference()
    img = Image.fromarray(g[f"{name}.u8"], "RGB")
    u8 = inf.preprocess_image_u8(img)          # a CUDA tensor where a GPU resizes it, else PIL's result on the host
    assert np.array_equal(u8.cpu().numpy(), g[f"{name}.resized_u8"])
    t64 = inf.preprocess_image(img).double()
    np.testing.assert_allclose([float(t64.sum()), float(t64.abs().sum())], g[f"{name}.out_moments"], rtol=1e-6)


def test_accepts_bytes_paths_and_non_rgb(g, tmp_path):
    inf = VQAInference()
    img = Image.fromarray(g["id224.u8"], "RGB")
    buf = io.BytesIO()
    img.save(buf, format="PNG")
    path = str(tmp_path / "x.png")
    img.save(path)
    a = inf.preprocess_image_u8(img)
    assert torch.equal(a, inf.preprocess_image_u8(buf.getvalue())) and torch.equal(a, inf.preprocess_image_u8(path))
    gray = inf.preprocess_image_u8(img.convert("L"))
    assert tuple(gray.shape) == (224, 224, 3) and torch.equal(gray[..., 0], gray[..., 1])


def test_no_cpu_path():
    with pytest.raises(RuntimeError):
        VQAInference(device="cpu").load()


# (300, 3) .. (2000, 5) and (70000, 5) straddle Pillow's vertical-first rule (height > 100 * width); (1, 300) and
# (300, 1) are one-pixel strips; (3000, 4000) is a photo-sized downscale.
RESIZE_SHAPES = [(300, 400), (100, 160), (333, 211), (224, 500), (640, 224), (17, 23), (225, 223), (1, 1),
                 (300, 3), (301, 3), (1000, 3), (205, 2), (225, 2), (2000, 5), (70000, 5), (1, 300), (300, 1), (3000, 4000)]


@pytest.mark.parametrize("hw", RESIZE_SHAPES)
def test_resize_restatement_is_bit_exact_with_pil(hw):
    """vqa_b200/resize.py (windows + 22-bit weights handed to the CUDA kernels, pass order) and the numpy two-pass
    restatement in oracle/resize_oracle.py against PIL.Image.resize(BILINEAR) itself."""
    from oracle.resize_oracle import numpy_resize
    from vqa_b200.resize import coeffs
    rng = np.random.default_rng(hw[0] * 7919 + hw[1])
    img = rng.integers(0, 256, (hw[0], hw[1], 3), dtype=np.uint8)
    want = np.asarray(Image.fromarray(img, "RGB").resize((224, 224), Image.BILINEAR))
    assert np.array_equal(numpy_resize(img, 224, 224), want)
    b, kk = coeffs(hw[1], 224)
    assert b.shape == (224, 2) and kk.shape[0] == 224 and (b[:, 0] + b[:, 1] <= hw[1]).all()
    assert (kk.sum(axis=1) - (1 << 22)).__abs__().max() <= kk.shape[1]      # weights sum to 1.0 in fixed point


def test_resize_restatement_matches_golden(g):
    from oracle.resize_oracle import numpy_resize
    for name in ("down", "up", "odd"):
        assert np.array_equal(numpy_resize(g[f"{name}.u8"], 224, 224), g[f"{name}.resized_u8"])
