"""The crop stage (csrc/crop.cu: bbox crop, equalize_adapthist, resize(..., anti_aliasing=True),
float32 cast) against the oracle in every one of its five work classes:

  fast 0 / fast 1 ........ crop_fast_kernel, clip count 1, sides <= 96, fast_layout <= 26 / 42 KB
  general 0 / general 1 .. crop_clahe_resize_kernel, cell_bytes <= 92 / 206 KB of shared memory
  general 2 .............. crop_clahe_resize_kernel on global scratch; a side > 1024 is refused

Cell records are built directly (no cia_filter gates), so the sweep reaches 1-pixel sides,
oblong boxes, boxes on field and buffer edges and cells at each class's byte limit.  Which
class took a cell is read back from the device work lists and checked against a Python
mirror of the classification.  Each cell is held to:
  * CLAHE levels (uint16) equal to oracle.clahe.clahe_levels, bit for bit;
  * the fp64 crop within 1e-12 of resize(equalize_adapthist(cell)) -- the levels are exact
    integers, so all that is left is fp64 rounding in the resize;
  * the float32 crop equal to the float32 rounding of the fp64 crop.
The image buffer is a view inside a larger tensor whose margins hold 65535, so a read
outside the fields changes min / max and shows as a wrong level.
"""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from oracle import clahe as oclahe
from oracle import resize as oresize
from test_oracle_crop_shapes import SWEEP_SHAPES

pytestmark = pytest.mark.gpu

CLASS_NAMES = ("fast 0", "fast 1", "general 0", "general 1", "general 2")
FAST_LIMITS = (26 * 1024, 42 * 1024)
GENERAL_LIMITS = (92 * 1024, 206 * 1024)
WS_CROP_SCRATCH = 2
CROP64_ATOL = 1e-12
CIA_E_UNSUPPORTED = -6


# ---- Python mirror of crop_classify_all_kernel (csrc/crop.cu) ------------------------------
def _a16(x):
    return (x + 15) & ~15


def _geom(h, w):
    kh, kw = max(h // 8, 1), max(w // 8, 1)
    return kh, kw, -(-h // kh), -(-w // kw)


def fast_layout_total(h, w):
    """fast_layout(h, w, ntiles, npix).total: the fast kernel's dynamic shared memory."""
    kh, kw, ntr, ntc = _geom(h, w)
    pitch = ((w + 14) >> 3) << 3
    u0 = _a16(h * pitch * 2)
    o = u0 + _a16(h * w) + _a16(ntr * ntc * 18 * 4) + kh * kw * 32 + _a16(257 * 2) + _a16(h * 4) + _a16(w * 4)
    return max(o, u0 + 4 * 176 * 8)


def cell_bytes(h, w):
    kh, kw, ntr, ntc = _geom(h, w)
    return _a16(h * w) + _a16(2 * h * w) + _a16(max(ntr * ntc * 256 * 2, 64 * w * 8))


def fast_eligible(h, w, clip_limit):
    if not (1 <= h <= 96 and 1 <= w <= 96) or not clip_limit > 0:
        return False
    kh, kw, _, _ = _geom(h, w)
    cl = clip_limit * (kh * kw)
    if not cl >= 1.0:
        cl = 1.0
    return int(cl) == 1 and kh * kw <= 256


def expected_class(h, w, clip_limit):
    if fast_eligible(h, w, clip_limit):
        need = fast_layout_total(h, w)
        for c, lim in enumerate(FAST_LIMITS):
            if need <= lim:
                return c
    if h > 1024 or w > 1024:
        return 4
    need = cell_bytes(h, w)
    return 2 if need <= GENERAL_LIMITS[0] else (3 if need <= GENERAL_LIMITS[1] else 4)


# ---- cell contents -------------------------------------------------------------------------
def _blob(h, w):
    yy, xx = np.mgrid[0:h, 0:w]
    return np.exp(-(((yy - h / 2) / max(h / 3, 1)) ** 2 + ((xx - w / 2) / max(w / 3, 1)) ** 2))


def make_content(kind, h, w, rng):
    if kind == "noise":                       # uniform over the full uint16 range
        return rng.integers(0, 65536, (h, w)).astype(np.uint16)
    if kind == "poisson":
        return np.minimum(rng.poisson(300 + 2500 * _blob(h, w)), 65535).astype(np.uint16)
    if kind == "constant":
        return np.full((h, w), 4321, np.uint16)
    if kind == "two_level":
        return np.where(rng.random((h, w)) < 0.3, 9000, 1200).astype(np.uint16)
    if kind == "bright_pixel":
        a = np.full((h, w), 150, np.uint16)
        a[rng.integers(h), rng.integers(w)] = 60000
        return a
    if kind == "ramp":
        yy, xx = np.mgrid[0:h, 0:w]
        return (200 + 40000 * (yy + xx) / max(h + w - 2, 1)).astype(np.uint16)
    if kind == "uint8":                       # 8-bit data in the uint16 buffer, intensity_inv = 1/255
        return rng.integers(0, 256, (h, w)).astype(np.uint16)
    if kind == "uint8_poisson":
        return np.minimum(rng.poisson(20 + 150 * _blob(h, w)), 255).astype(np.uint16)
    raise ValueError(kind)


# ---- batches -------------------------------------------------------------------------------
class Batch:
    """Fields [F, H, W] uint16 on the host plus cell records; bboxes are packed on shelves."""

    def __init__(self, H, W, fill=0):
        self.H, self.W = H, W
        self.fields = []
        self.fill = fill
        self.cells = []                       # dicts: field, minr, minc, h, w, kind, note
        self._x = self._y = self._shelf = 0

    def new_field(self, data=None):
        self.fields.append(np.full((self.H, self.W), self.fill, np.uint16) if data is None else data)
        self._x, self._y, self._shelf = 0, 0, 0
        return len(self.fields) - 1

    def add(self, field, minr, minc, h, w, kind, note=""):
        self.cells.append(dict(field=field, minr=minr, minc=minc, h=h, w=w, kind=kind, note=note))

    def pack(self, h, w, img, kind, gap=3):
        """Place ``img`` at the next free spot (shelf packing, tallest first works best)."""
        if not self.fields:
            self.new_field()
        if self._x + w > self.W:
            self._x, self._y, self._shelf = 0, self._y + self._shelf + gap, 0
        if self._y + h > self.H:
            self.new_field()
        f = len(self.fields) - 1
        self.fields[f][self._y:self._y + h, self._x:self._x + w] = img
        self.add(f, self._y, self._x, h, w, kind)
        self._x += w + gap
        self._shelf = max(self._shelf, h)

    def crop(self, i):
        c = self.cells[i]
        return self.fields[c["field"]][c["minr"]:c["minr"] + c["h"], c["minc"]:c["minc"] + c["w"]]

    def records(self, order=None):
        idx = range(len(self.cells)) if order is None else order
        from cell_image_analysis_b200 import _lib
        rec = np.zeros(len(idx), _lib.CELL_DTYPE)
        for j, i in enumerate(idx):
            c = self.cells[i]
            rec[j]["field"], rec[j]["label"] = c["field"], i + 1
            rec[j]["minr"], rec[j]["minc"] = c["minr"], c["minc"]
            rec[j]["maxr"], rec[j]["maxc"] = c["minr"] + c["h"], c["minc"] + c["w"]
            rec[j]["area"] = c["h"] * c["w"]
        return rec

    def describe(self, i):
        c = self.cells[i]
        s = f"cell {i} {c['h']}x{c['w']} [{c['kind']}] at field {c['field']} (r {c['minr']}, c {c['minc']})"
        return s + (f" {c['note']}" if c["note"] else "")


def device_images(eng, fields, pre):
    """The fields as an [F, H, W] view starting ``pre`` elements into a tensor whose margins
    before and after hold 65535."""
    flat = np.stack(fields).view(np.int16).ravel()
    big = torch.full((pre + flat.size + 64,), -1, dtype=torch.int16)
    big[pre:pre + flat.size] = torch.from_numpy(flat)
    big = big.to(eng.tdev)
    F, (H, W) = len(fields), fields[0].shape
    return big, big[pre:pre + flat.size].view(F, H, W)


def cells_tensor(eng, rec):
    return torch.from_numpy(rec.view(np.uint8).reshape(len(rec), 56).copy()).to(eng.tdev)


def params_for(clip_limit, intensity_inv):
    from cell_image_analysis_b200 import _lib
    p = _lib.default_params()
    p.clip_limit, p.intensity_inv = clip_limit, intensity_inv
    return p


def read_classes(eng, n):
    """Class of each of the n cells of the last crop call, from the device work lists."""
    stride = -(-n // 64) * 64
    counts = np.zeros(5, np.int32)
    eng._check(eng.lib.cia_debug_copy_workspace(eng.h, WS_CROP_SCRATCH, 0, C.c_void_p(counts.ctypes.data), 20))
    cls = np.full(n, -1, np.int64)
    for c in range(5):
        k = int(counts[c])
        if k == 0:
            continue
        lst = np.zeros(k, np.int32)
        eng._check(eng.lib.cia_debug_copy_workspace(eng.h, WS_CROP_SCRATCH, 256 + c * stride * 4,
                                                    C.c_void_p(lst.ctypes.data), 4 * k))
        assert (cls[lst] == -1).all() and ((lst >= 0) & (lst < n)).all(), f"class {CLASS_NAMES[c]}: bad list"
        cls[lst] = c
    return counts, cls


def status_code(eng):
    """What check_status raises since the last check (0: nothing)."""
    from cell_image_analysis_b200 import _lib
    try:
        eng.check_status()
    except _lib.CiaError as e:
        return e.code
    return 0


def run_crop(eng, images, rec, params):
    """crop_resize with the fp64 output; returns (c32, c64, device classes, status code)."""
    cells = cells_tensor(eng, rec)
    c32, c64 = eng.crop_resize(images, cells, len(rec), want64=True, params=params)
    counts, cls = read_classes(eng, len(rec))
    return c32.cpu().numpy(), c64.cpu().numpy(), cls, status_code(eng)


def run_levels(eng, images, rec, params):
    old = eng.params
    eng.params = params
    try:
        sizes = (rec["maxr"] - rec["minr"]) * (rec["maxc"] - rec["minc"])
        lv, offs = eng.debug_clahe_levels(images, cells_tensor(eng, rec), len(rec), sizes)
    finally:
        eng.params = old
    return [lv[offs[i]:offs[i + 1]].reshape(rec[i]["maxr"] - rec[i]["minr"], -1) for i in range(len(rec))]


def oracle_of(img, clip_limit, uint8):
    a = img.astype(np.uint8) if uint8 else img
    return oclahe.clahe_levels(a, clip_limit), oresize.resize(oclahe.equalize_adapthist(a, clip_limit))


def first_diff(got, ref, tol=0.0):
    bad = np.argwhere(~(np.abs(got.astype(np.float64) - ref.astype(np.float64)) <= tol))
    y, x = (int(v) for v in bad[0])
    return f"first differing (y, x) = ({y}, {x}): got {got[y, x]!r}, expected {ref[y, x]!r}"


# ---- the sweep: one call per clip limit / intensity scale, all classes mixed ----------------
CONTENT_CYCLE = ("constant", "two_level", "bright_pixel", "ramp")
# shapes re-run at the other clip limits: they move cells between the fast and the general path
CLIP_SHAPES = [(1, 7), (7, 1), (1, 97), (2, 50), (8, 8), (16, 16), (23, 23), (57, 93), (88, 59), (95, 95),
               (96, 96), (12, 90), (90, 12), (128, 128), (300, 1), (111, 40)]
UINT8_SHAPES = [(1, 50), (50, 1), (9, 9), (17, 17), (64, 64), (97, 97), (40, 700), (167, 93)]
REFUSED = [(1025, 40), (40, 1025)]


def build_group(shapes, kinds_of, seed, with_refused=False):
    rng = np.random.default_rng(seed)
    items = []
    for j, (h, w) in enumerate(shapes):
        for kind in kinds_of(j, h, w):
            items.append((h, w, kind))
    if with_refused:
        items += [(h, w, "noise") for h, w in REFUSED]
    b = Batch(1060, 1101)
    for h, w, kind in sorted(items, key=lambda t: (-t[0], -t[1])):
        b.pack(h, w, make_content(kind, h, w, rng), kind)
    # mixed order: neighbouring records belong to different classes
    order = np.random.default_rng(seed + 1).permutation(len(b.cells))
    b.cells = [b.cells[i] for i in order]
    return b


GROUPS = [
    # name, clip_limit, intensity_inv, builder
    ("clip 0.02", 0.02, 1.0 / 65535.0,
     lambda: build_group(SWEEP_SHAPES, lambda j, h, w: ("noise", "poisson", CONTENT_CYCLE[j % 4]), 11, True)),
    ("uint8", 0.02, 1.0 / 255.0,
     lambda: build_group(UINT8_SHAPES, lambda j, h, w: ("uint8", "uint8_poisson"), 12)),
    ("clip 0 (AHE)", 0.0, 1.0 / 65535.0,
     lambda: build_group(CLIP_SHAPES, lambda j, h, w: ("noise", "poisson"), 13)),
    ("clip 0.005", 0.005, 1.0 / 65535.0,
     lambda: build_group(CLIP_SHAPES, lambda j, h, w: ("noise", "poisson"), 14)),
    ("clip 0.05", 0.05, 1.0 / 65535.0,
     lambda: build_group(CLIP_SHAPES, lambda j, h, w: ("noise", "poisson"), 15)),
]


@pytest.fixture(scope="module")
def eng():
    from cell_image_analysis_b200.screening import Engine
    e = Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def module_clock():
    return time.perf_counter()


@pytest.fixture(scope="module")
def sweep(eng, module_clock):
    """Every group: the batch, device outputs and classes, and the oracle (computed once)."""
    out = []
    for gi, (name, clip_limit, inv, builder) in enumerate(GROUPS):
        b = builder()
        rec = b.records()
        big, images = device_images(eng, b.fields, pre=3 + gi)
        params = params_for(clip_limit, inv)
        c32, c64, cls, code = run_crop(eng, images, rec, params)
        refused = np.array([c["h"] > 1024 or c["w"] > 1024 for c in b.cells])
        ok = np.nonzero(~refused)[0]
        lv_ok = run_levels(eng, images, rec[ok], params)
        levels = {int(i): l for i, l in zip(ok, lv_ok)}
        ref = {int(i): oracle_of(b.crop(i), clip_limit, inv != 1.0 / 65535.0) for i in ok}
        out.append(dict(name=name, clip_limit=clip_limit, params=params, batch=b, rec=rec, big=big,
                        images=images, c32=c32, c64=c64, cls=cls, code=code, refused=refused,
                        levels=levels, ref=ref))
    return out


def _label(g, i):
    b = g["batch"]
    return f"{g['name']}: {b.describe(i)} class {CLASS_NAMES[g['cls'][i]]}"


def test_classes_match_mirror_and_cover_limits(sweep):
    bad = []
    for g in sweep:
        b = g["batch"]
        for i, c in enumerate(b.cells):
            want = expected_class(c["h"], c["w"], g["clip_limit"])
            if g["cls"][i] != want:
                got = CLASS_NAMES[g["cls"][i]] if g["cls"][i] >= 0 else "no list"
                bad.append(f"{g['name']}: {b.describe(i)}: device class {got}, mirror {CLASS_NAMES[want]} "
                           f"(fast_layout {fast_layout_total(c['h'], c['w'])} B, cell_bytes "
                           f"{cell_bytes(c['h'], c['w'])} B)")
    assert not bad, "\n".join(bad[:20])
    main = sweep[0]
    assert set(main["cls"].tolist()) == set(range(5)), "every class must get cells in the 0.02 sweep"
    shapes_by_class = {}
    for g in sweep:
        for i, c in enumerate(g["batch"].cells):
            shapes_by_class.setdefault(int(g["cls"][i]), set()).add((c["h"], c["w"], g["clip_limit"]))

    def need_in(cls_set, fn, lo, hi):
        return any(lo < fn(h, w) <= hi for h, w, _ in cls_set)
    # 26 KB: a fast-0 cell exactly at the limit and a fast-1 cell just above it
    assert need_in(shapes_by_class[0], fast_layout_total, FAST_LIMITS[0] - 1, FAST_LIMITS[0])
    assert need_in(shapes_by_class[1], fast_layout_total, FAST_LIMITS[0], FAST_LIMITS[0] + 64)
    # 42 KB: no cell the fast path accepts needs more (95 x 95 is the largest, 39808 B), so the limit
    # never sends a cell to the general path; the largest one runs in fast 1
    worst = max(fast_layout_total(h, w) for h in range(1, 97) for w in range(1, 97))
    assert worst == fast_layout_total(95, 95) <= FAST_LIMITS[1]
    assert (95, 95, 0.005) in shapes_by_class[1]
    # 92 KB and 206 KB: general cells exactly at each limit and 16 B (one alignment step) above it
    for c, lim in ((2, GENERAL_LIMITS[0]), (3, GENERAL_LIMITS[1])):
        assert need_in(shapes_by_class[c], cell_bytes, lim - 1, lim), CLASS_NAMES[c]
        assert need_in(shapes_by_class[c + 1], cell_bytes, lim, lim + 16), CLASS_NAMES[c + 1]


def test_levels_bit_exact(sweep):
    bad = []
    for g in sweep:
        for i, lv in g["levels"].items():
            ref = g["ref"][i][0]
            if lv.shape != ref.shape or not np.array_equal(lv, ref):
                n = int((lv != ref).sum()) if lv.shape == ref.shape else -1
                bad.append(f"{_label(g, i)} clip {g['clip_limit']}: {n} levels differ, "
                           + (first_diff(lv, ref) if n > 0 else f"shape {lv.shape} vs {ref.shape}"))
    assert not bad, f"{len(bad)} cells\n" + "\n".join(bad[:20])


def test_crop64_within_fp64_rounding(sweep):
    bad = []
    for g in sweep:
        for i in g["ref"]:
            got, ref = g["c64"][i], g["ref"][i][1]
            err = float(np.abs(got - ref).max())
            if not err <= CROP64_ATOL:
                bad.append(f"{_label(g, i)} clip {g['clip_limit']}: max |d| {err:.3e}, "
                           + first_diff(got, ref, CROP64_ATOL))
    assert not bad, f"{len(bad)} cells\n" + "\n".join(bad[:20])


def test_crop32_is_rounded_crop64(sweep):
    bad = []
    for g in sweep:
        want = g["c64"].astype(np.float32)        # c64 is already clipped to [lo, hi], exact in fp32
        for i in range(len(g["rec"])):
            if not np.array_equal(g["c32"][i].view(np.uint32), want[i].view(np.uint32)):
                bad.append(f"{_label(g, i)}: " + first_diff(g["c32"][i], want[i]))
    assert not bad, "\n".join(bad[:20])


def test_refused_cells(eng, sweep):
    """Sides > 1024: CIA_E_UNSUPPORTED from check_status, a zero crop, every other cell unchanged."""
    g = sweep[0]
    assert g["refused"].sum() == len(REFUSED)
    assert g["code"] == CIA_E_UNSUPPORTED
    for i in np.nonzero(g["refused"])[0]:
        assert (g["c32"][i] == 0).all() and (g["c64"][i] == 0).all(), g["batch"].describe(i)
        assert g["cls"][i] == 4
    keep = np.nonzero(~g["refused"])[0]
    c32, c64, cls, code = run_crop(eng, g["images"], g["rec"][keep], g["params"])
    assert code == 0
    assert np.array_equal(c64.view(np.uint64), g["c64"][keep].view(np.uint64))
    assert np.array_equal(c32.view(np.uint32), g["c32"][keep].view(np.uint32))


def test_row_order_single_cells_and_repeats(eng, sweep):
    """Row i is cell i (reversed records give reversed rows), a cell alone gives the bits it gives in
    the batch, and a repeated call gives the same bits."""
    for g in sweep:
        n = len(g["rec"])
        c32, c64, _, _ = run_crop(eng, g["images"], g["rec"], g["params"])
        assert np.array_equal(c64.view(np.uint64), g["c64"].view(np.uint64)), f"{g['name']}: repeat call"
        assert np.array_equal(c32.view(np.uint32), g["c32"].view(np.uint32)), f"{g['name']}: repeat call"
        rev = np.arange(n)[::-1]
        c32r, c64r, _, _ = run_crop(eng, g["images"], g["rec"][rev], g["params"])
        assert np.array_equal(c64r[::-1].view(np.uint64), g["c64"].view(np.uint64)), f"{g['name']}: reversed"
    g = sweep[0]
    picks = []
    for c in range(5):
        picks += [int(i) for i in np.nonzero(g["cls"] == c)[0][:3]]
    picks += [i for i, c in enumerate(g["batch"].cells) if min(c["h"], c["w"]) == 1][:6]
    for i in picks:
        c32, c64, _, code = run_crop(eng, g["images"], g["rec"][i:i + 1], g["params"])
        assert np.array_equal(c64[0].view(np.uint64), g["c64"][i].view(np.uint64)), _label(g, i)
        assert np.array_equal(c32[0].view(np.uint32), g["c32"][i].view(np.uint32)), _label(g, i)


def test_device_count_limits_cells(eng, sweep):
    """n_cells_dev < n: the cells before it are computed as in the full call, the rows after it are
    not written."""
    from cell_image_analysis_b200.screening import _ptr
    g = sweep[0]
    n = len(g["rec"])
    k = n // 2
    cells = cells_tensor(eng, g["rec"])
    n_dev = torch.tensor([k], dtype=torch.int32, device=eng.tdev)
    c32 = torch.full((n, 64, 64), float("nan"), dtype=torch.float32, device=eng.tdev)
    c64 = torch.full((n, 64, 64), float("nan"), dtype=torch.float64, device=eng.tdev)
    eng._check(eng.lib.cia_crop_resize(eng.h, _ptr(g["images"]), g["images"].shape[1], g["images"].shape[2],
                                       _ptr(cells), n, _ptr(n_dev), C.byref(g["params"]), _ptr(c32), _ptr(c64),
                                       eng._stream()))
    assert status_code(eng) == (CIA_E_UNSUPPORTED if g["refused"][:k].any() else 0)
    c32, c64 = c32.cpu().numpy(), c64.cpu().numpy()
    assert np.array_equal(c64[:k].view(np.uint64), g["c64"][:k].view(np.uint64))
    assert np.array_equal(c32[:k].view(np.uint32), g["c32"][:k].view(np.uint32))
    assert np.isnan(c64[k:]).all() and np.isnan(c32[k:]).all()


# ---- placement: field edges and corners, buffer ends, every alignment of the first pixel ----
PLACE_SHAPES = [(1, 1), (1, 9), (9, 1), (5, 13), (40, 33), (97, 120)]


@pytest.fixture(scope="module")
def placement():
    F, H, W = 3, 150, 203                      # W odd: each bbox row starts at another 16-byte phase
    rng = np.random.default_rng(21)
    b = Batch(H, W)
    for _ in range(F):
        b.new_field((np.minimum(rng.poisson(400 + 3000 * _blob(H, W)), 65535)
                     + rng.integers(0, 2000, (H, W))).astype(np.uint16))
    for f in (0, 1, F - 1):
        for h, w in PLACE_SHAPES:
            spots = {"top-left": (0, 0), "top-right": (0, W - w), "bottom-left": (H - h, 0),
                     "bottom-right": (H - h, W - w), "top": (0, (W - w) // 2), "bottom": (H - h, (W - w) // 3),
                     "left": ((H - h) // 2, 0), "right": ((H - h) // 3, W - w)}
            if f == 1:
                spots = {k: v for k, v in spots.items() if k in ("top-left", "bottom-right")}
            for where, (r, c) in spots.items():
                note = where + (" (buffer start)" if f == 0 and where == "top-left" else "") \
                    + (" (buffer end)" if f == F - 1 and where == "bottom-right" else "")
                b.add(f, r, c, h, w, "field", note)
    for h, w in ((1, 9), (3, 5), (17, 19), (6, 1)):    # every first-pixel phase through minc
        for minc in range(40, 48):
            b.add(1, 60, minc, h, w, "field", f"minc {minc}")
    ref = [oracle_of(b.crop(i), 0.02, False) for i in range(len(b.cells))]
    return b, ref


@pytest.mark.parametrize("pre", range(8))
def test_placement_and_alignment(eng, placement, pre):
    """The same cells with the image pointer ``pre`` elements past a 512-byte boundary."""
    b, ref = placement
    rec = b.records()
    big, images = device_images(eng, b.fields, pre)
    params = params_for(0.02, 1.0 / 65535.0)
    c32, c64, cls, code = run_crop(eng, images, rec, params)
    assert code == 0
    levels = run_levels(eng, images, rec, params)
    bad = []
    for i in range(len(rec)):
        c = b.cells[i]
        e00 = (pre + (c["field"] * b.H + c["minr"]) * b.W + c["minc"]) % 8
        what = f"pre {pre}: {b.describe(i)} e00 {e00} class {CLASS_NAMES[cls[i]]}"
        if not np.array_equal(levels[i], ref[i][0]):
            bad.append(f"{what}: levels, " + first_diff(levels[i], ref[i][0]))
        err = float(np.abs(c64[i] - ref[i][1]).max())
        if not err <= CROP64_ATOL:
            bad.append(f"{what}: crop64 max |d| {err:.3e}, " + first_diff(c64[i], ref[i][1], CROP64_ATOL))
        if not np.array_equal(c32[i], c64[i].astype(np.float32)):
            bad.append(f"{what}: crop32, " + first_diff(c32[i], c64[i].astype(np.float32)))
    assert not bad, f"{len(bad)} failures\n" + "\n".join(bad[:20])
    assert [int(c) for c in cls] == [expected_class(c["h"], c["w"], 0.02) for c in b.cells]


def test_report(sweep, module_clock):
    """Per class: cells, worst level mismatch, worst fp64 crop error (shown with pytest -rA)."""
    rows = {c: [0, 0, 0.0] for c in range(5)}
    for g in sweep:
        for i in g["ref"]:
            r = rows[int(g["cls"][i])]
            r[0] += 1
            r[1] = max(r[1], int((g["levels"][i] != g["ref"][i][0]).sum()))
            r[2] = max(r[2], float(np.abs(g["c64"][i] - g["ref"][i][1]).max()))
    print("\nclass      cells  worst level mismatch  worst |crop64 - oracle|")
    for c, (n, lv, e) in rows.items():
        print(f"{CLASS_NAMES[c]:<10} {n:5d}  {lv:20d}  {e:.3e}")
    print(f"refused (side > 1024): {int(sum(g['refused'].sum() for g in sweep))}")
    print(f"module time so far: {time.perf_counter() - module_clock:.1f} s")
    assert all(r[0] > 0 for r in rows.values())
