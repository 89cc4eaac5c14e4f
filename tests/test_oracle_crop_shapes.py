"""The crop-stage oracle (CLAHE levels, resize) at the bbox shapes the GPU crop sweep
(tests/test_gpu_crop_sweep.py) holds the kernels to: 1-pixel sides, sides below the 8-px
tile split, oblong boxes and 1024-px sides.  Before the oracle is the reference there, the
closed-form resize is checked against the real scipy.ndimage path and the CLAHE invariants
of tests/test_oracle.py are checked at each shape.  CPU only."""
import numpy as np
import pytest

from oracle import clahe, resize

# (h, w) of the bboxes the GPU sweep runs at clip limit 0.02 (sides > 1024 are refused by the
# kernel and have no oracle counterpart)
SWEEP_SHAPES = [
    (1, 1), (1, 2), (1, 7), (1, 50), (1, 96), (1, 97), (1, 300),
    (2, 1), (7, 1), (50, 1), (96, 1), (97, 1), (300, 1),
    (2, 2), (2, 7), (2, 50), (2, 97), (7, 2), (97, 2),
    # kh = max(h // 8, 1) changes; ntr = ceil(h / kh) reaches 15
    (7, 7), (8, 8), (9, 9), (15, 15), (16, 16), (17, 17), (23, 23), (7, 23), (23, 7), (8, 15), (16, 9),
    # no blur / identity zoom / first blur
    (63, 63), (64, 64), (65, 65), (64, 65), (63, 65),
    # the fast path's side limit
    (95, 95), (96, 96), (97, 97), (96, 97), (97, 96),
    # gaussian radius 1 -> 2
    (111, 111), (112, 112), (111, 40),
    (127, 127), (128, 128), (129, 129),
    (12, 90), (90, 12), (40, 700), (700, 40),
    # at and just above the shared-memory byte limits of the classes (26 KB, 92 KB, 206 KB)
    (57, 93), (88, 59), (91, 120), (167, 93), (104, 256), (161, 212),
    # kernel size 29 x 50: 0.02 * 29 * 50 and 0.02 * 1450 round to different clip counts
    (232, 400),
    (1023, 1023), (1024, 1024),
]


def _noise(shape, seed=0):
    return np.random.default_rng(seed).integers(0, 65536, shape).astype(np.uint16)


@pytest.mark.parametrize("shape", SWEEP_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_resize_formula_matches_scipy_at_sweep_shapes(shape):
    a = np.random.default_rng(shape[0] * 7919 + shape[1]).random(shape)
    ref = resize.resize(a)
    assert ref.shape == (64, 64)
    assert np.abs(ref - resize.resize_formula(a)).max() < 1e-14
    assert ref.min() >= a.min() and ref.max() <= a.max()


@pytest.mark.parametrize("shape", SWEEP_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_clahe_invariants_at_sweep_shapes(shape):
    cell = _noise(shape, seed=shape[0] + 3 * shape[1])
    k = clahe.kernel_size(shape)
    before, after = clahe.padding(shape, k)
    for s, kk, b, a in zip(shape, k, before, after):
        assert (s + b + a) % kk == 0 and (s + b + a) // kk == -(-s // kk) + 1
    q = clahe.quantise(cell)
    qp = np.pad(q, [(before[0], after[0]), (before[1], after[1])], mode="reflect")
    bins = (qp // clahe.BIN_SIZE).astype(np.uint16)
    maps = clahe.tile_maps(bins, k, clahe.clip_count(0.02, k))
    # every tile's map is monotone and inside the 14-bit range
    assert (np.diff(maps, axis=-1) >= 0).all()
    assert maps.min() >= 0 and maps.max() <= 16383
    lv = clahe.clahe_levels(cell)
    assert lv.shape == shape and lv.dtype == np.uint16 and lv.max() <= 16383
    out = clahe.equalize_adapthist(cell)
    assert out.shape == shape and out.dtype == np.float64
    if lv.min() != lv.max():
        assert out.min() == 0.0 and out.max() == 1.0
    else:
        assert out.min() >= 0.0 and out.max() <= 1.0


def test_clip_count_rule():
    """clip_limit * the tile's pixel count (one product, as skimage and the kernel compute it), at
    least 1; clip_limit 0 is plain AHE.  Both oracle entry points use this one rule."""
    assert clahe.clip_count(0.0, (12, 12)) == clahe.NR_OF_GRAY
    assert clahe.clip_count(0.02, (1, 1)) == 1
    assert clahe.clip_count(0.02, (29, 50)) == int(0.02 * 1450) == 29     # 0.02 * 29 * 50 rounds to 28.999...
    cell = _noise((100, 130), seed=4)
    for clip_limit in (0.0, 0.005, 0.02, 0.05):
        lv = clahe.clahe_levels(cell, clip_limit).astype(np.float64)
        np.testing.assert_array_equal(clahe.equalize_adapthist(cell, clip_limit),
                                      (lv - lv.min()) / (lv.max() - lv.min()))
    # AHE really does not clip: its levels differ from the clipped ones on noise
    assert not np.array_equal(clahe.clahe_levels(cell, 0.0), clahe.clahe_levels(cell, 0.02))
