"""CPU oracle for the PIL-exact antialiased bilinear resize (SURVEY 8(f) row f1).

TEST INFRASTRUCTURE ONLY: nothing in the product package imports this module.  It restates in numpy the two integer
passes that ``csrc/resize.cu`` runs on the GPU (horizontal first except for very tall images, intermediate rounded to
uint8, then the other pass; each output = clip8((2^21 + sum(pixel * weight)) >> 22)), i.e. Pillow's
``Image.resize(..., BILINEAR)`` on 8-bit images (``src/libImaging/Resample.c``; reached by the reference through ``transforms.Resize((224, 224))``,
data/preprocess.py:117-121, api/inference.py:153-167).  The windows and 22-bit fixed-point weights come from the same
host function the product uses (``vqa_b200.resize.coeffs``).

Parity status: PINNED -- ``tests/test_preprocess.py`` checks it against ``PIL.Image.resize`` itself on eighteen geometries
and against the committed golden vectors (``tests/golden/preprocess.npz``, made by ``tests/golden/make_golden.py`` through
the reference's own transform).
"""
import numpy as np

from vqa_b200.resize import PRECISION_BITS, coeffs, vertical_first


def _h_pass(x: np.ndarray, out_w: int) -> np.ndarray:
    b, kk = coeffs(x.shape[1], out_w)
    out = np.empty((x.shape[0], out_w, x.shape[2]), dtype=np.int64)
    for xx in range(out_w):
        x0, n = int(b[xx, 0]), int(b[xx, 1])
        acc = (x[:, x0:x0 + n, :] * kk[xx, :n].astype(np.int64)[None, :, None]).sum(axis=1) + (1 << (PRECISION_BITS - 1))
        out[:, xx, :] = np.clip(acc >> PRECISION_BITS, 0, 255)
    return out


def _v_pass(x: np.ndarray, out_h: int) -> np.ndarray:
    b, kk = coeffs(x.shape[0], out_h)
    out = np.empty((out_h, x.shape[1], x.shape[2]), dtype=np.int64)
    for yy in range(out_h):
        y0, n = int(b[yy, 0]), int(b[yy, 1])
        acc = (x[y0:y0 + n, :, :] * kk[yy, :n].astype(np.int64)[:, None, None]).sum(axis=0) + (1 << (PRECISION_BITS - 1))
        out[yy, :, :] = np.clip(acc >> PRECISION_BITS, 0, 255)
    return out


def numpy_resize(img: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """CPU restatement of the two integer passes (uint8 [H, W, C] -> [out_h, out_w, C]) in Pillow's pass order
    (``vqa_b200.resize.vertical_first``); test infrastructure."""
    h, w, _ = img.shape
    x = img.astype(np.int64)
    passes = [(w != out_w, lambda t: _h_pass(t, out_w)), (h != out_h, lambda t: _v_pass(t, out_h))]
    if vertical_first(h, w, out_h):
        passes.reverse()
    for needed, run in passes:
        if needed:
            x = run(x)
    return x.astype(np.uint8)
