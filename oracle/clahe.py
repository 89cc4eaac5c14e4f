"""Oracle for ``exposure.equalize_adapthist(cell, clip_limit=0.02)``.

Serves improved_detection.py:98 (CAE_improved_modeltrain.py:92).  scikit-image is
not installable here, so this is a NumPy restatement of the published algorithm
(skimage/exposure/_adapthist.py, 0.19-0.25 line of releases) following SURVEY.md
A.2 step by step -- PARITY UNPINNED against the real library.  Test
infrastructure only.
"""
from __future__ import annotations

import numpy as np

NR_OF_GRAY = 1 << 14
NBINS = 256
BIN_SIZE = 1 + NR_OF_GRAY // NBINS       # 65 -> bins 0..252


def quantise(cell: np.ndarray) -> np.ndarray:
    """A.2 steps 1-2: img_as_float then rescale to 0..16383 and round half even."""
    if cell.dtype == np.uint16:
        v = cell.astype(np.float64) * (1.0 / 65535.0)
    elif cell.dtype == np.uint8:                # img_as_float: multiply by 1 / imax_in
        v = cell.astype(np.float64) * (1.0 / 255.0)
    else:
        v = cell.astype(np.float64)
    vmin, vmax = float(v.min()), float(v.max())
    if vmin != vmax:
        v = (v - vmin) / (vmax - vmin)
        v = v * float(NR_OF_GRAY - 1) + 0.0
    else:                                   # rescale_intensity's degenerate branch
        v = np.clip(v, 0.0, float(NR_OF_GRAY - 1))
    return np.round(v).astype(np.uint16)


def kernel_size(shape):
    return tuple(max(s // 8, 1) for s in shape)


def padding(shape, k):
    before = [kk // 2 for kk in k]
    after = [(kk - s % kk) % kk + int(np.ceil(kk / 2.0)) for kk, s in zip(k, shape)]
    return before, after


def clip_histogram(hist: np.ndarray, clim: int) -> np.ndarray:
    """A.2 step 8 on one 256-bin histogram (modified in place, exact integers)."""
    over = hist > clim
    excess = int(hist[over].sum()) - int(over.sum()) * clim
    hist[over] = clim

    incr = excess // hist.size
    upper = clim - incr
    low = hist < upper
    excess -= int(low.sum()) * incr
    hist[low] += incr

    mid = (hist >= upper) & (hist < clim)
    excess += int(hist[mid].sum()) - int(mid.sum()) * clim
    hist[mid] = clim

    while excess > 0:
        prev = excess
        for index in range(hist.size):
            under = hist < clim
            step = max(1, int(np.count_nonzero(under)) // excess)
            sel = under[index::step]
            hist[index::step][sel] += 1
            excess -= int(np.count_nonzero(sel))
            if excess <= 0:
                break
        if prev == excess:
            break
    return hist


def tile_maps(bins: np.ndarray, k, clim: int) -> np.ndarray:
    """A.2 steps 6-9: per-tile clipped histograms -> integer mapping tables
    [ns_hist_r, ns_hist_c, 256] (int64)."""
    kh, kw = k
    nh = [bins.shape[0] // kh - 1, bins.shape[1] // kw - 1]
    maps = np.empty((nh[0], nh[1], NBINS), np.int64)
    npx = kh * kw
    for i in range(nh[0]):
        for j in range(nh[1]):
            t = bins[kh // 2 + i * kh: kh // 2 + (i + 1) * kh,
                     kw // 2 + j * kw: kw // 2 + (j + 1) * kw]
            h = np.bincount(t.ravel(), minlength=NBINS).astype(np.int64)
            h = clip_histogram(h, clim)
            out = np.cumsum(h).astype(np.float64)
            out *= float(NR_OF_GRAY - 1) / npx
            out += 0.0
            np.clip(out, None, float(NR_OF_GRAY - 1), out=out)
            maps[i, j] = out.astype(np.int64)
    return maps


def interpolate(bins: np.ndarray, maps: np.ndarray, k) -> np.ndarray:
    """A.2 steps 10-11: bilinear blend of the 4 neighbouring tile mappings,
    accumulated in float32 in edge order (0,0),(0,1),(1,0),(1,1), truncated to uint16."""
    kh, kw = k
    npr, npc = bins.shape[0] // kh, bins.shape[1] // kw
    mp = np.pad(maps, [(1, 1), (1, 1), (0, 0)], mode="edge")
    cr = np.arange(kh) / kh
    cc = np.arange(kw) / kw
    Y = np.arange(bins.shape[0])
    X = np.arange(bins.shape[1])
    I, a = Y // kh, Y % kh
    J, b = X // kw, X % kw
    res = np.zeros(bins.shape, np.float32)
    b64 = bins.astype(np.int64)
    for er in (0, 1):
        wr = cr[a] if er else 1 - cr[a]
        for ec in (0, 1):
            wc = cc[b] if ec else 1 - cc[b]
            mapped = mp[(I + er)[:, None], (J + ec)[None, :], b64]
            coef = wc[None, :] * wr[:, None]
            res += (mapped * coef).astype(np.float32)
    assert npr * kh == bins.shape[0] and npc * kw == bins.shape[1]
    return res.astype(np.uint16)


def clip_count(clip_limit: float, k) -> int:
    """A.2 step 5: the per-bin count limit of a tile of ``k[0] x k[1]`` pixels; clip_limit 0 is plain
    AHE (no clipping)."""
    npx = k[0] * k[1]
    return int(np.clip(clip_limit * npx, 1, None)) if clip_limit > 0 else NR_OF_GRAY


def clahe_levels(cell: np.ndarray, clip_limit: float = 0.02) -> np.ndarray:
    """The uint16 levels before the final [0,1] rescale (the bit-exact integer core)."""
    q = quantise(cell)
    k = kernel_size(cell.shape)
    before, after = padding(cell.shape, k)
    qp = np.pad(q, [(before[0], after[0]), (before[1], after[1])], mode="reflect")
    bins = (qp // BIN_SIZE).astype(np.uint16)
    res = interpolate(bins, tile_maps(bins, k, clip_count(clip_limit, k)), k)
    return res[before[0]: res.shape[0] - after[0], before[1]: res.shape[1] - after[1]]


def equalize_adapthist(cell: np.ndarray, clip_limit: float = 0.02) -> np.ndarray:
    """det:98.  uint16 [h, w] -> float64 [h, w] in [0, 1]."""
    r = clahe_levels(cell, clip_limit).astype(np.float64)
    rmin, rmax = float(r.min()), float(r.max())
    if rmin != rmax:
        r = (r - rmin) / (rmax - rmin)
        return r * 1.0 + 0.0
    return np.clip(r, 0.0, 1.0)
