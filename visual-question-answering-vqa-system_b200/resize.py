"""PIL-exact antialiased bilinear resize, coefficient side (host) -- SURVEY 8(f) row f1.

The reference resizes through ``torchvision.transforms.Resize((224, 224))`` on PIL images
(data/preprocess.py:117-121, api/inference.py:153-167), i.e. Pillow's ``Image.resize(..., BILINEAR)``.
Pillow is a third-party dependency of the reference (``Pillow>=9.5.0`` in requirements.txt; 12.2.0 in this
image; C source ``src/libImaging/Resample.c`` is not vendored), so its published algorithm is restated here:

* separable, horizontal pass first, then vertical; the intermediate image is rounded to uint8.  An image more than
  100 times taller than wide that shrinks vertically goes vertical pass first (``vertical_first``): the installed
  Pillow (12.2.0) does so in ``Image.resize``, earlier releases always ran horizontal first, and this module follows
  the installed one;
* triangle filter with support ``max(scale, 1)``; per output pixel a window ``[xmin, xmin + n)`` with
  ``xmin = int(center - support + 0.5)``, weights normalised to sum 1 in double precision;
* 8-bit path: weights become 22-bit fixed point (round half away from zero), each output is
  ``clip8((2^21 + sum(pixel * weight)) >> 22)``.

The windows / fixed-point weights are computed here in double precision exactly as the C code does and handed
to the CUDA kernels (``csrc/resize.cu``), which do the two integer passes.  Bit-exactness against PIL itself is
tested on the CPU (``oracle/resize_oracle.py`` restates the two integer passes in numpy) and on the GPU.
"""
from __future__ import annotations

import math
from functools import lru_cache
from typing import Tuple

import numpy as np

PRECISION_BITS = 32 - 8 - 2


def vertical_first(in_h: int, in_w: int, out_h: int) -> bool:
    """Pass order of ``Image.resize``: True when Pillow resizes rows before columns (``in_h > 100 * in_w`` and the
    height shrinks).  The two orders round the intermediate image differently, so they give different bytes."""
    return in_h > in_w * 100 and out_h < in_h


@lru_cache(maxsize=256)
def coeffs(in_size: int, out_size: int) -> Tuple[np.ndarray, np.ndarray]:
    """(bounds int32 [out, 2] = (xmin, count), weights int32 [out, ksize]) of one pass (precompute_coeffs +
    normalize_coeffs_8bpc of Pillow's Resample.c for the bilinear filter, whole-image box)."""
    scale = filterscale = in_size / out_size
    if filterscale < 1.0:
        filterscale = 1.0
    support = 1.0 * filterscale                   # bilinear filter support is 1.0
    ksize = int(math.ceil(support)) * 2 + 1
    bounds = np.zeros((out_size, 2), dtype=np.int32)
    kk = np.zeros((out_size, ksize), dtype=np.int32)
    ss = 1.0 / filterscale
    for xx in range(out_size):
        center = (xx + 0.5) * scale
        xmin = int(center - support + 0.5)        # C (int) cast: truncation toward zero
        if xmin < 0:
            xmin = 0
        xmax = int(center + support + 0.5)
        if xmax > in_size:
            xmax = in_size
        xmax -= xmin
        k = [0.0] * ksize
        ww = 0.0
        for x in range(xmax):
            t = (x + xmin - center + 0.5) * ss
            if t < 0.0:
                t = -t
            w = 1.0 - t if t < 1.0 else 0.0
            k[x] = w
            ww += w
        for x in range(xmax):
            if ww != 0.0:
                k[x] /= ww
        for x in range(ksize):
            v = k[x] * (1 << PRECISION_BITS)
            kk[xx, x] = int(v - 0.5) if k[x] < 0 else int(v + 0.5)
        bounds[xx, 0], bounds[xx, 1] = xmin, xmax
    return bounds, kk
