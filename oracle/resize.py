"""Oracle for ``skimage.transform.resize(img, (64, 64), anti_aliasing=True)``.

Serves improved_detection.py:99 (CAE_improved_modeltrain.py:93).  The arithmetic is
the REAL scipy.ndimage ``gaussian_filter`` + ``zoom`` that skimage itself calls
(pinned); the wrapper logic (sigma, mode mapping, clipping) is restated per
SURVEY.md A.3.  ``resize_formula`` is the closed-form restatement the CUDA kernel
implements, checked against scipy in tests/test_oracle.py.  Test infrastructure only.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage as ndi

OUT = 64


def resize(img: np.ndarray, out_shape=(OUT, OUT)) -> np.ndarray:
    img = np.asarray(img, dtype=np.float64)
    factors = np.array(img.shape, dtype=np.float64) / np.array(out_shape, dtype=np.float64)
    sigma = np.maximum(0, (factors - 1) / 2)
    filtered = ndi.gaussian_filter(img, sigma, cval=0, mode="mirror")
    zoom = [1 / f for f in factors]
    out = ndi.zoom(filtered, zoom, order=1, mode="mirror", cval=0, grid_mode=True)
    return np.clip(out, img.min(), img.max())


def _mirror(i: np.ndarray, n: int) -> np.ndarray:
    if n == 1:
        return np.zeros_like(i)
    p = 2 * n - 2
    i = np.abs(i) % p
    return np.where(i >= n, p - i, i)


def gaussian_weights(sigma: float):
    radius = int(4.0 * sigma + 0.5)
    x = np.arange(-radius, radius + 1, dtype=np.float64)
    w = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return w / w.sum(), radius


def resize_formula(img: np.ndarray, out: int = OUT) -> np.ndarray:
    """Closed-form restatement (A.3): separable mirror Gaussian then separable
    pixel-centre bilinear with mirror indexing, then clip to the input range."""
    a = np.asarray(img, dtype=np.float64)
    for ax in (0, 1):
        n = a.shape[ax]
        sigma = max(0.0, (n / out - 1) / 2)
        if sigma > 1e-15:
            w, r = gaussian_weights(sigma)
            idx = _mirror(np.arange(n)[:, None] + np.arange(-r, r + 1)[None, :], n)
            # tap by tap: a 1024-px side has 61 taps, too many to gather all at once
            acc = np.zeros_like(a)
            for j in range(2 * r + 1):
                acc += w[j] * (a[idx[:, j]] if ax == 0 else a[:, idx[:, j]])
            a = acc
    h, w_ = a.shape

    def taps(n):
        cc = (np.arange(out) + 0.5) * (n / out) - 0.5
        i0 = np.floor(cc)
        t = cc - i0
        i0 = i0.astype(np.int64)
        return _mirror(i0, n), _mirror(i0 + 1, n), t

    r0, r1, tr = taps(h)
    c0, c1, tc = taps(w_)
    rows = (1 - tr)[:, None] * a[r0] + tr[:, None] * a[r1]
    res = rows[:, c0] * (1 - tc)[None, :] + rows[:, c1] * tc[None, :]
    return np.clip(res, float(np.min(img)), float(np.max(img)))
