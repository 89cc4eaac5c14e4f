"""Layer-by-layer gate of the tensor-core autoencoder (csrc/cae_tc.cu, precisions 1 and 2).

The end-to-end tests judge the seven tcgen05 layers only through MSE / MAE (means over 4,096
pixels) and the features.  An error confined to one border, one phase of the L6 / L7 phase form
or one channel moves a cell's MSE by (affected pixels / 4096) x (relative error) and can hide
under a 1e-3 gate.  Here every layer is judged on its own:

* The kernel's input and output activations are read back through ``cia_debug_copy_workspace``
  (workspace 5 = ws_misc: A1h A1l A2h A2l A3h A4u A5u A6, each ``CH x per-cell halves``, laid out
  as in ``k_cae_forward_tc``; ``ws_layout`` below).
* Layer L is recomputed in fp64 from the DEVICE's layer L-1 output -- the fp16 values the MMAs
  read (hi, or hi + lo for the split layers) -- and from a numpy mirror of ``k_cae_tc_prepare``'s
  weight images (power-of-two scale, fp16 hi / lo, the phase-form and tap-sum images summed in
  fp32 in the same loop order, the layer-1 input scale 2^XSCALE_EXP, lo x lo dropped).  Errors do
  not compound, so every element gets its own bound.
* The bound is derived from the arithmetic, element by element, from the same data:
  - accumulation: tcgen05 adds each K16 step with ONE round-toward-zero (DESIGN.md section 5), an
    error below 2^-23 of the running sum, itself at most S = sum |a * w| (a second fp64 conv of
    absolute values); the accumulating kernels' fp32 flush additions (at most 18 per output) are
    counted as further steps;
  - the ``cae_l*_debias`` shift (debias x 2^-24 x S);
  - the fp32 epilogue roundings (fma / fma / mul / add, 2^-24 each of a magnitude bounded from S);
  - the fp16 storage: half an fp16 ulp for hi-only outputs, 2^-22 relative for hi + lo, and an
    absolute 2^-25 floor for subnormals;
  - 2x2 max-pool: the maximum bound over the window (max is 1-Lipschitz in the sup norm);
  - L7: the per-pixel error of the pre-sigmoid value, the intrinsics' documented error (see
    ``l7_reference``) and the fp32 reduction, propagated into per-cell MSE / MAE bounds.
* Assertion: |device - reference| <= bound for every element of every checked cell; the worst
  error / bound ratio of every layer is printed even when the test passes.

The CPU tests at the bottom check the reference itself (no GPU needed): chained without fp16
rounding or packing it must reproduce ``oracle.cae.forward``, the weight-image mirror must
reconstruct the weights and the up-sampled convolution, and the layer-2 gate must reject a layer 2
that leaves out one of the split-precision cross products.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from helpers import synth_cae_weights  # noqa: E402
from oracle import cae as ocae  # noqa: E402

U = 2.0 ** -24            # unit round-off of fp32 round-to-nearest
EPS = 2.0 ** -23          # bound of one round-toward-zero step, relative to the running sum
XSCALE_EXP = 6            # l1tc::XSCALE_EXP: layer 1 scales its input by 2^6 before the hi / lo split
DEBIAS = (0.5, 2.4, 1.2)  # cae_l1/l2/l3_debias in units of 2^-24 (handle defaults; set explicitly below)
PASS_CELLS = 18944        # default cae_pass_cells
SMS_ROUND = 148           # k_cae_forward_tc rounds a single pass up to a multiple of 148 cells
CIN = [1, 32, 64, 32, 32, 64, 32]
COUT = [32, 64, 32, 32, 64, 32, 1]
# ws_misc buffers in k_cae_forward_tc order: (name, channel chunks of 8, resolution)
WS_BUFFERS = (("A1h", 4, 32), ("A1l", 4, 32), ("A2h", 8, 16), ("A2l", 8, 16), ("A3h", 4, 8),
              ("A4u", 4, 8), ("A5u", 8, 16), ("A6", 4, 32))


# ---------------------------------------------------------------------------------------------
# workspace layout of k_cae_forward_tc
# ---------------------------------------------------------------------------------------------
def ws_layout(n: int, pass_cells: int = PASS_CELLS):
    """Cells per pass CH (the buffer stride), {buffer: (offset in halves, halves per cell, nch, R)} and
    the last pass (first cell, cells).  After a call the buffers hold only the last pass, its cells at
    chunk-relative positions 0 .. chunk-1."""
    ch = (n + SMS_ROUND - 1) // SMS_ROUND * SMS_ROUND if n < pass_cells else pass_cells
    off, bufs = 0, {}
    for name, nch, r in WS_BUFFERS:
        per = nch * r * r * 8
        bufs[name] = (off, per, nch, r)
        off += ch * per
    c0 = (n - 1) // ch * ch
    return ch, bufs, c0, n - c0


def planar_to_nchw(buf16: np.ndarray, n: int, nch: int, r: int) -> np.ndarray:
    """Chunk-planar [cell][C/8][y][x][8] -> [cell][C][y][x]."""
    return buf16.reshape(n, nch, r, r, 8).transpose(0, 1, 4, 2, 3).reshape(n, nch * 8, r, r)


# ---------------------------------------------------------------------------------------------
# numpy mirror of k_cae_tc_prepare
# ---------------------------------------------------------------------------------------------
def scale_exp(w) -> int:
    """Power-of-two exponent that puts max|w| in [2, 4) (cae_tc.cu scale_exp)."""
    m = float(np.max(np.abs(np.asarray(w, np.float32)))) if np.size(w) else 0.0
    if not m > 0:
        return 0
    return 2 - math.frexp(m)[1]


def split16(v):
    """fp16 hi + fp16 remainder lo of float32 values, both round-to-nearest-even (pack_image)."""
    v = np.asarray(v, np.float32)
    hi = v.astype(np.float16)
    return hi, (v - hi.astype(np.float32)).astype(np.float16)


def _phase_taps():
    """(py, px, dy, dx, low-res tap tl, neighbour ty, tx) in k_cae_tc_prepare's loop order: hi-res tap
    (dy, dx) of output phase (py, px) reads low-res pixel (y + oy, x + ox)."""
    out = []
    for py in range(2):
        for px in range(2):
            for dy in range(3):
                for dx in range(3):
                    oy, ox = (py + dy - 1) // 2, (px + dx - 1) // 2
                    out.append((py, px, dy, dx, (oy + 1) * 3 + (ox + 1), oy - (py - 1), ox - (px - 1)))
    return out


def phase_form(k, dtype=np.float32):
    """HWIO k [3,3,cin,cout] -> kp [9 low-res taps, cin, 4 phases, cout]: conv on the 2x nearest
    up-sampled input == 3x3 conv on the low-res input with four outputs.  float32: summed like the
    C++ loop (one fp32 add per contribution, in loop order); float64: exact."""
    k = np.asarray(k, dtype)
    kp = np.zeros((9, k.shape[2], 4, k.shape[3]), dtype)
    for py, px, dy, dx, tl, _, _ in _phase_taps():
        kp[tl, :, 2 * py + px, :] = kp[tl, :, 2 * py + px, :] + k[dy, dx]
    return kp


def tapsum_form(k, dtype=np.float32):
    """HWIO k [3,3,cin,1] -> kt [cin, 16]: column 4*(2py+px) + 2ty + tx = weight of low-res neighbour
    (Y + py - 1 + ty, X + px - 1 + tx) in output (2Y + py, 2X + px) (final_tapsum_kernel)."""
    k = np.asarray(k, dtype)
    kt = np.zeros((k.shape[2], 16), dtype)
    for py, px, dy, dx, _, ty, tx in _phase_taps():
        col = 4 * (2 * py + px) + 2 * ty + tx
        kt[:, col] = kt[:, col] + k[dy, dx, :, 0]
    return kt


def pack_weights(w: dict):
    """The tensor-core weight images of k_cae_tc_prepare, per layer: scale exponent, inverse scale and
    the fp16 hi / lo images (standard HWIO; layers 6 and 7 in phase form, whose scale layer 7 uses;
    layer 7 also in tap-sum form for final_tapsum_kernel, with the phase form's scale).  The sign of the BN
    scale that the pooling layers fold into their columns is left out: fp16 rounding is symmetric, so
    the folded products are the unfolded ones negated, and max(sign * c) undone equals the pooled f(c)."""
    packs = []
    for L in range(7):
        k = np.asarray(w["kernels"][L], np.float32)
        img = phase_form(k) if L >= 5 else k
        sw = scale_exp(img)
        hi, lo = split16(img * np.float32(2.0 ** sw))
        p = {"sw": sw, "inv": 2.0 ** (-sw - (XSCALE_EXP if L == 0 else 0)), "hi": hi, "lo": lo}
        if L == 6:
            p["t_hi"], p["t_lo"] = split16(tapsum_form(k) * np.float32(2.0 ** sw))
        packs.append(p)
    return packs


def bn_params(w: dict):
    return [ocae.bn_affine(*bn) for bn in w["bns"]]


# ---------------------------------------------------------------------------------------------
# fp64 reference operations (torch, on whatever device the inputs live)
# ---------------------------------------------------------------------------------------------
def _t(a, dev):
    return torch.as_tensor(np.asarray(a, np.float64), device=dev)


def conv(x, w):
    """'same' 3x3 cross-correlation: x [N,Cin,H,W], w HWIO [3,3,Cin,Cout]."""
    return F.conv2d(x, w.permute(3, 2, 0, 1).contiguous(), padding=1)


def phase_conv(x, kp):
    """x [N,Cin,R,R], kp [9,Cin,4,Cout] -> [N,Cout,2R,2R]: output (2y+py, 2x+px) from phase 2py+px."""
    n, cin, r, _ = x.shape
    cout = kp.shape[3]
    y = conv(x, kp.reshape(3, 3, cin, 4 * cout))
    return y.reshape(n, 2, 2, cout, r, r).permute(0, 3, 4, 1, 5, 2).reshape(n, cout, 2 * r, 2 * r)


def tapsum_conv(x, kt):
    """x [N,Cin,R,R], kt [Cin,16] -> [N,1,2R,2R]: the channel contraction per (phase, neighbour)
    column, then the shifted sum over the 2x2 low-res neighbours (zero outside the map)."""
    n, _, r, _ = x.shape
    p = F.pad(torch.einsum("nchw,cj->njhw", x, kt), (1, 1, 1, 1))
    out = torch.zeros((n, 1, 2 * r, 2 * r), dtype=x.dtype, device=x.device)
    for py in range(2):
        for px in range(2):
            for ty in range(2):
                for tx in range(2):
                    col = 4 * (2 * py + px) + 2 * ty + tx
                    out[:, 0, py::2, px::2] += p[:, col, py + ty:py + ty + r, px + tx:px + tx + r]
    return out


def up2(x):
    return F.interpolate(x, scale_factor=2, mode="nearest")


def pool2(x):
    return F.max_pool2d(x, 2)


def act(acc, S, inv, bias, s, t, rz_steps, debias, rn_steps):
    """bias -> ReLU -> BN of the exact accumulator ``acc`` (scaled units, x ``inv`` = conv output) and
    the bound of the device's fp32 value: rz_steps round-toward-zero steps (< 2^-23 x S each), the
    debias shift (debias x 2^-24 x S), rn_steps roundings of the pre-activation (fma's, or the fp32 FMA
    chain of the CUDA-core layer 1), then the BN product and sum (2^-24 each)."""
    dev = acc.device
    b, s, t = (_t(v, dev)[None, :, None, None] for v in (bias, s, t))
    z = acc * inv + b
    zmag = S * inv + b.abs()
    dz = S * inv * (rz_steps * EPS + debias * U) + rn_steps * U * zmag
    y = torch.relu(z) * s + t
    ymag = s.abs() * (zmag + dz)
    return y, s.abs() * dz + U * ymag + U * (ymag + t.abs())


def half_ulp16(mag):
    """Half an fp16 ulp at magnitude ``mag`` (2^-25 in the subnormal range)."""
    e = torch.floor(torch.log2(torch.clamp(mag, min=2.0 ** -14)))
    return torch.exp2(e - 11)


def store_bound(y, dy, split):
    mag = y.abs() + dy
    return dy + (2.0 ** -22 * mag + 2.0 ** -25 if split else half_ulp16(mag))


def split_store(y):
    """fp16 hi and lo of the fp32 value, as split_store8 stores an activation."""
    o = y.float()
    hi = o.half()
    return hi.double(), (o - hi.float()).half().double()


def split_conv(ahi, alo, whi, wlo, op=conv):
    """hi*hi + hi*lo + lo*hi (lo*lo dropped) and the same over absolute values."""
    acc = op(ahi, whi) + op(ahi, wlo) + op(alo, whi)
    S = op(ahi.abs(), whi.abs()) + op(ahi.abs(), wlo.abs()) + op(alo.abs(), whi.abs())
    return acc, S


def hi_conv(a, w, op=conv):
    return op(a, w), op(a.abs(), w.abs())


# L7: the intrinsics.  CUDA C++ Programming Guide, "Intrinsic Functions" (single precision):
#   __expf(x)        max error 2 + floor(|1.173 x|) ulp  (includes the x * log2(e) scaling)
#   __fdividef(x, y) max error 2 ulp for 2^-126 <= |y| <= 2^126 (0 above: the true value is < 2^-126)
# An fp32 ulp is at most 2^-23 of the value.  rec = 1 / (1 + e): a relative error r of e moves rec by
# rec (1 - rec) r; the add 1 + e (2^-24) and the division (2 x 2^-23) move it relatively.
SIG_EXP_ULP = (2.0, 1.173)
SIG_DIV_ULP = 2.0
# sequential fp32 additions a per-pixel term passes through on its way into MSE / MAE in
# final_tapsum_kernel: 8 per thread + 5 warp_sum levels + 16 per-warp sums
REDUCE_DEPTH = 29


def l7_reference(a6, X, pk, bias):
    """Per-cell (mse, mae, mse bound, mae bound) of layer 7 on the device's A6 (hi only)."""
    dev = a6.device
    # hi and lo weight columns: 2 RZ steps each, their sum and 3 tap-sum adds (2^-24 each)
    acc, S = split_conv(a6, torch.zeros_like(a6), _t(pk["t_hi"], dev), _t(pk["t_lo"], dev), tapsum_conv)
    steps = 2 + 4 * U / EPS
    b = float(bias[0])
    a = acc[:, 0] * pk["inv"] + b
    amag = S[:, 0] * pk["inv"] + abs(b)
    da = S[:, 0] * pk["inv"] * steps * EPS + U * amag                      # + fmaf(sum, inv, b)
    rec = torch.sigmoid(a)
    e_rel = (SIG_EXP_ULP[0] + torch.floor(SIG_EXP_ULP[1] * (a.abs() + da))) * EPS
    drec = da / 4 + rec * ((1 - rec) * e_rel + U + SIG_DIV_ULP * EPS) * 1.001 + 2.0 ** -126
    x = _t(X, dev)
    d = x - rec
    dd = drec + U * (d.abs() + drec)                                        # the fp32 subtraction
    g = REDUCE_DEPTH * U * 1.001
    sq_b = 2 * d.abs() * dd + dd * dd
    mse = (d * d).sum((1, 2)) / 4096
    mae = d.abs().sum((1, 2)) / 4096
    mse_b = (sq_b.sum((1, 2)) + g * ((d * d).sum((1, 2)) + sq_b.sum((1, 2)))) / 4096
    mae_b = (dd.sum((1, 2)) + g * (d.abs().sum((1, 2)) + dd.sum((1, 2)))) / 4096
    return mse, mae, mse_b, mae_b


# ---------------------------------------------------------------------------------------------
# the per-layer check
# ---------------------------------------------------------------------------------------------
class Report:
    """Worst error / bound ratio per layer and the located failures."""

    def __init__(self, tag):
        self.tag, self.ratio, self.failures = tag, {}, []

    def check(self, layer, got, ref, bound, cells, kind="act"):
        r = (got - ref).abs() / torch.clamp(bound, min=1e-300)
        r = torch.where(torch.isfinite(got), r, torch.full_like(r, math.inf))
        worst = float(r.max()) if r.numel() else 0.0
        self.ratio[layer] = max(self.ratio.get(layer, 0.0), worst)
        if not worst <= 1.0:
            i = np.unravel_index(int(torch.argmax(torch.nan_to_num(r, nan=math.inf))), tuple(r.shape))
            where = (f"cell {cells[i[0]]} channel {i[1]} (y, x) = ({i[2]}, {i[3]})" if kind == "act"
                     else f"cell {cells[i[0]]} feature {i[1]}" if kind == "feat" else f"cell {cells[i[0]]}")
            self.failures.append(f"[{self.tag}] {layer}: {where}: device {float(got[i]):.9g} reference "
                                 f"{float(ref[i]):.9g} |d| {float((got - ref).abs()[i]):.3e} bound "
                                 f"{float(bound[i]):.3e} ratio {float(r[i]):.3g}")

    def line(self):
        return f"[{self.tag}] worst |device - reference| / bound: " + "  ".join(
            f"{k} {v:.3g}" for k, v in self.ratio.items())

    def done(self):
        print(self.line())
        assert not self.failures, "\n".join(self.failures)


def read_taps(eng, n, pass_cells):
    """The last pass's activations from ws_misc as float64 [cell][C][y][x] (cells c0 .. n-1)."""
    ch, bufs, c0, chunk = ws_layout(n, pass_cells)
    out = {}
    for name, (off, per, nch, r) in bufs.items():
        dst = np.empty(chunk * per, np.float16)
        rc = eng.lib.cia_debug_copy_workspace(eng.h, 5, C.c_size_t(off * 2), C.c_void_p(dst.ctypes.data),
                                              C.c_size_t(dst.nbytes))
        assert rc == 0, rc
        out[name] = planar_to_nchw(dst, chunk, nch, r)
    return out, c0, chunk


def l1_reference(x, w, packs, bn, split):
    """Layer 1's pooled output and bound from the crops x [cell][1][64][64]: conv1_tc_split_kernel
    (split) or conv1_fp32_planar_kernel."""
    dev = x.device
    if split:    # the input scaled by 2^XSCALE_EXP and split into fp16 hi / lo, 3 MMAs of one K16 step
        v = (x * 2.0 ** XSCALE_EXP).float()
        xh = v.half().double()
        xl = (v - v.half().float()).half().double()
        acc, S = split_conv(xh, xl, _t(packs[0]["hi"], dev), _t(packs[0]["lo"], dev))
        y, dy = act(acc, S, packs[0]["inv"], w["biases"][0], *bn[0], 3, DEBIAS[0], 2)
    else:        # fp32 weights and crops, a 9-FMA chain started at the bias
        acc, S = hi_conv(x.double(), _t(w["kernels"][0], dev))
        y, dy = act(acc, S, 1.0, w["biases"][0], *bn[0], 0, 0.0, 9)
    return pool2(y), pool2(dy)


def check_l2(rep, w, packs, bn, a1h, a1l, a2, split, cells):
    """The layer-2 gate: the reference of layer 2 on the device's layer-1 output (a1h, and a1l on the
    split path) against the device's layer-2 output a2 (hi + lo on the split path).  The accumulating
    kernel of the split path: 3 x 9 x Cin/16 MMAs + at most 18 fp32 flush adds."""
    whi, wlo = _t(packs[1]["hi"], a1h.device), _t(packs[1]["lo"], a1h.device)
    if split:
        acc, S = split_conv(a1h, a1l, whi, wlo)
        y, dy = act(acc, S, packs[1]["inv"], w["biases"][1], *bn[1], 3 * 9 * 2 + 18, DEBIAS[1], 2)
    else:
        acc, S = hi_conv(a1h, whi)
        y, dy = act(acc, S, packs[1]["inv"], w["biases"][1], *bn[1], 9 * 2, 0.0, 2)
    y, dy = pool2(y), pool2(dy)
    rep.check("L2", a2, y, store_bound(y, dy, split), cells)


def check_layers(tag, w, packs, X, taps, mse, mae, feat, cells, path, dev="cuda"):
    """Judge L1..L7 of one tensor-core call.  path 1: split L1-L3 (features tapped from L3); path 2: the
    fp32 layer 1 and single-pass L2 / L3 (precision 2, and precision 1 with a separate encoder).
    X: the crops of ``cells``; taps: their activations (read_taps); mse / mae / feat: the call's outputs
    for these cells (feat None when they do not come from the tensor-core L3)."""
    rep = Report(tag)
    bn = bn_params(w)
    T = {k: torch.from_numpy(v.astype(np.float64)).to(dev) for k, v in taps.items()}
    x = torch.from_numpy(np.asarray(X, np.float32)).to(dev)[:, None]
    split = path == 1
    hw = [(_t(p["hi"], dev), _t(p["lo"], dev)) for p in packs]

    # L1
    y, dy = l1_reference(x, w, packs, bn, split)
    a1 = T["A1h"] + T["A1l"] if split else T["A1h"]
    rep.check("L1", a1, y, store_bound(y, dy, split), cells)

    # L2
    check_l2(rep, w, packs, bn, T["A1h"], T["A1l"], T["A2h"] + T["A2l"] if split else T["A2h"], split, cells)

    # L3
    if split:
        acc, S = split_conv(T["A2h"], T["A2l"], *hw[2])
        y, dy = act(acc, S, packs[2]["inv"], w["biases"][2], *bn[2], 3 * 9 * 4 + 18, DEBIAS[2], 2)
    else:
        acc, S = hi_conv(T["A2h"], hw[2][0])
        y, dy = act(acc, S, packs[2]["inv"], w["biases"][2], *bn[2], 9 * 4, 0.0, 2)
    y, dy = pool2(y), pool2(dy)
    rep.check("L3", T["A3h"], y, store_bound(y, dy, False), cells)
    if feat is not None:
        f = torch.from_numpy(np.asarray(feat, np.float64)).to(dev)
        rep.check("L3 features", f, y.permute(0, 2, 3, 1).reshape(len(cells), -1),
                  dy.permute(0, 2, 3, 1).reshape(len(cells), -1), cells, kind="feat")
        # the L3 epilogue writes both from the same registers
        a3_bits = taps["A3h"].transpose(0, 2, 3, 1).reshape(len(cells), -1).view(np.int16)
        f16_bits = np.asarray(feat, np.float32).astype(np.float16).view(np.int16)
        bad = np.argwhere(a3_bits != f16_bits)
        if len(bad):
            c, j = bad[0]
            rep.failures.append(f"[{tag}] L3: A3h != fp16_rn(features) at {len(bad)} elements, first cell "
                                f"{cells[c]} feature {j}")

    # L4 .. L6: single pass, hi operands, plain epilogue (one fma, ReLU, BN)
    acc, S = hi_conv(T["A3h"], hw[3][0])
    y, dy = act(acc, S, packs[3]["inv"], w["biases"][3], *bn[3], 9 * 2, 0.0, 1)
    rep.check("L4", T["A4u"], y, store_bound(y, dy, False), cells)
    acc, S = hi_conv(up2(T["A4u"]), hw[4][0])
    y, dy = act(acc, S, packs[4]["inv"], w["biases"][4], *bn[4], 9 * 2, 0.0, 1)
    rep.check("L5", T["A5u"], y, store_bound(y, dy, False), cells)
    acc, S = hi_conv(T["A5u"], hw[5][0], phase_conv)
    y, dy = act(acc, S, packs[5]["inv"], w["biases"][5], *bn[5], 9 * 4, 0.0, 1)
    rep.check("L6", T["A6"], y, store_bound(y, dy, False), cells)

    # L7: MSE / MAE
    rm, ra, bm, ba = l7_reference(T["A6"], X, packs[6], w["biases"][6])
    col = lambda v: torch.from_numpy(np.asarray(v, np.float64)).to(dev)  # noqa: E731
    rep.check("L7 mse", col(mse), rm, bm, cells, kind="cell")
    rep.check("L7 mae", col(mae), ra, ba, cells, kind="cell")
    return rep


# ---------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------
def constructed_crops(seed=5):
    """All-zero, all-one, single bright pixels in every corner and at every edge midpoint (non-zero
    values on the zero-padding borders of every layer), two checkerboards, uniform noise."""
    crops = [np.zeros((64, 64), np.float32), np.ones((64, 64), np.float32)]
    for y, x in ((0, 0), (0, 63), (63, 0), (63, 63), (0, 32), (63, 31), (31, 0), (32, 63)):
        c = np.zeros((64, 64), np.float32)
        c[y, x] = 1.0
        crops.append(c)
    cb = (np.add.outer(np.arange(64), np.arange(64)) % 2).astype(np.float32)
    crops += [cb, 1 - cb]
    rng = np.random.default_rng(seed)
    crops += [rng.uniform(0, 1, (64, 64)).astype(np.float32) for _ in range(3)]
    return np.stack(crops)


def model_sets(golden: dict):
    """Name -> CAE weights: the golden model, two held-out seeds, every gamma of the pooling layers
    negative (the sign fold on every channel), and channels whose gamma is -0.0."""
    def copy(w):
        return {"kernels": [k.copy() for k in w["kernels"]], "biases": [b.copy() for b in w["biases"]],
                "bns": [tuple(a.copy() for a in bn) for bn in w["bns"]]}
    neg = copy(golden)
    for L in range(3):
        neg["bns"][L][0][:] = -np.abs(neg["bns"][L][0])
    nz = copy(golden)
    for L, c in ((0, 5), (1, 17), (2, 3), (4, 40)):
        nz["bns"][L][0][c] = np.float32(-0.0)
    return {"golden": copy(golden), "seed101": synth_cae_weights(101), "seed202": synth_cae_weights(202),
            "neg_gamma": neg, "neg_zero_gamma": nz}


def load_cae(eng, which, w, n_conv):
    ks = [np.ascontiguousarray(k, np.float32) for k in w["kernels"][:n_conv]]
    bs = [np.ascontiguousarray(b, np.float32) for b in w["biases"][:n_conv]]
    bn = [np.ascontiguousarray(a, np.float32) for t in w["bns"][:min(n_conv, 6)] for a in t]
    K = (C.c_void_p * n_conv)(*[k.ctypes.data for k in ks])
    B = (C.c_void_p * n_conv)(*[b.ctypes.data for b in bs])
    N = (C.c_void_p * len(bn))(*[a.ctypes.data for a in bn])
    eng._check(eng.lib.cia_load_cae(eng.h, which, n_conv, K, B, N, C.c_float(ocae.BN_EPS)))


def make_engine(w, encoder=None):
    from cell_image_analysis_b200.screening import Engine
    eng = Engine(device=0, precision=1)
    load_cae(eng, 0, w, 7)
    if encoder is not None:
        load_cae(eng, 1, encoder, 3)
    eng.set_option("cae_pass_cells", PASS_CELLS)
    for i, v in enumerate(DEBIAS):
        eng.set_option(f"cae_l{i + 1}_debias", v)
    return eng


def run_and_check(eng, tag, w, packs, X, n, precision, path, n_dev=None, pass_cells=PASS_CELLS,
                  feat_from_tc=None):
    """One cae_forward call on the first n crops, then the per-layer check of its last pass."""
    x = torch.from_numpy(np.ascontiguousarray(X[:n])).to(eng.tdev)
    mse, mae, feat = eng.cae_forward(x, n, n_dev=n_dev, precision=precision)
    eng.check_status()
    mse, mae, feat = (t[:n].cpu().numpy() for t in (mse, mae, feat))
    taps, c0, chunk = read_taps(eng, n, pass_cells)
    cells = np.arange(c0, n)
    tc_feat = path == 1 if feat_from_tc is None else feat_from_tc
    rep = check_layers(tag, w, packs, X[c0:n], taps, mse[c0:], mae[c0:], feat[c0:] if tc_feat else None,
                       cells, path, dev=str(eng.tdev))
    return rep, (mse, mae, feat)


# ---------------------------------------------------------------------------------------------
# GPU tests
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def layer_crops(screener, golden_tiny):
    """~300 crops: the constructed ones, the golden tiny field's, then real crops of a synth field
    through the CUDA extraction path."""
    from cell_image_analysis_b200 import synth
    g, l = synth.make_field(0)
    real = np.array(screener.extract_quality_cells_from_labels(g, l)[0], np.float32)
    X = np.concatenate([constructed_crops(), golden_tiny["crops"].astype(np.float32), real])
    assert len(X) >= 300
    return np.ascontiguousarray(X[:300])


@pytest.fixture(scope="module")
def models(oracle_weights):
    return model_sets(oracle_weights)


@pytest.fixture(scope="module")
def engines(models):
    made = {}

    def get(name, encoder=None):
        key = (name, encoder)
        if key not in made:
            made[key] = make_engine(models[name], models[encoder] if encoder else None)
        return made[key]
    yield get
    for e in made.values():
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 147, 148, 149, 300])
def test_precision1_layers_golden(engines, models, layer_crops, n):
    """Default path (split L1-L3 with tapped features, single-pass L4-L7) at cell counts around a
    multiple of 148 (the single-pass buffer stride)."""
    w = models["golden"]
    rep, _ = run_and_check(engines("golden"), f"p1 golden n={n}", w, pack_weights(w), layer_crops, n, 1, 1)
    rep.done()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["seed101", "seed202", "neg_gamma", "neg_zero_gamma"])
def test_precision1_layers_models(engines, models, layer_crops, name):
    w = models[name]
    rep, _ = run_and_check(engines(name), f"p1 {name}", w, pack_weights(w), layer_crops, 300, 1, 1)
    rep.done()


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", [("golden", 1), ("golden", 149), ("golden", 300), ("seed101", 300),
                                    ("neg_gamma", 300), ("neg_zero_gamma", 149)])
def test_precision2_layers(engines, models, layer_crops, name, n):
    """Precision 2: fp32 layer 1, single-pass hi-only L2 / L3; its features come from the fp32 encoder on
    the side stream and must equal precision 0's bit for bit."""
    w = models[name]
    eng = engines(name)
    rep, (_, _, feat) = run_and_check(eng, f"p2 {name} n={n}", w, pack_weights(w), layer_crops, n, 2, 2)
    x = torch.from_numpy(np.ascontiguousarray(layer_crops[:n])).to(eng.tdev)
    f0 = eng.cae_forward(x, n, precision=0)[2][:n].cpu().numpy()
    eng.check_status()
    rep.done()
    assert np.array_equal(feat.view(np.int32), f0.view(np.int32)), "precision 2 features differ from precision 0's"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["golden", "seed202"])
def test_separate_encoder_layers(engines, models, layer_crops, name):
    """Precision 1 with a separately loaded encoder: the autoencoder takes the precision-2 branch and the
    features come from the fp32 encoder of the OTHER weights (equal to precision 0's bit for bit)."""
    w = models[name]
    eng = engines(name, "seed101")
    rep, (_, _, feat) = run_and_check(eng, f"p1 separate encoder {name}", w, pack_weights(w), layer_crops,
                                      300, 1, 2)
    x = torch.from_numpy(layer_crops).to(eng.tdev)
    f0 = eng.cae_forward(x, 300, precision=0)[2][:300].cpu().numpy()
    eng.check_status()
    rep.done()
    assert np.array_equal(feat.view(np.int32), f0.view(np.int32)), "separate-encoder features differ from precision 0's"
    enc_ref = ocae.forward(layer_crops[:8, :, :, None], models["seed101"], n_layers=3)[1].reshape(8, -1)
    np.testing.assert_allclose(feat[:8], enc_ref, rtol=1e-4, atol=1e-5)    # it IS the other encoder


@pytest.mark.gpu
def test_multipass_last_pass_rebased(engines, models, layer_crops):
    """cae_pass_cells = 148 and n = 300: passes of 148, 148 and 4 cells.  The ragged last pass sits at
    chunk-relative positions of the buffers; its layers must meet the gate, and every output of the
    three-pass call must equal the single-pass call's bit for bit."""
    w = models["golden"]
    eng = engines("golden")
    one = run_and_check(eng, "p1 single pass", w, pack_weights(w), layer_crops, 300, 1, 1)[1]
    eng.set_option("cae_pass_cells", 148)
    try:
        rep, many = run_and_check(eng, "p1 3 passes, last", w, pack_weights(w), layer_crops, 300, 1, 1,
                                  pass_cells=148)
    finally:
        eng.set_option("cae_pass_cells", PASS_CELLS)
    assert ws_layout(300, 148)[2:] == (296, 4)
    rep.done()
    for a, b, name in zip(one, many, ("mse", "mae", "features")):
        assert np.array_equal(a.view(np.int32), b.view(np.int32)), f"{name}: three passes differ from one"


@pytest.mark.gpu
def test_n_cells_dev_contract(engines, layer_crops):
    """cia_cae_forward with host bound n = 300 and a device count of 173: cells below 173 bit-equal to a
    call with n = 173, mse and mae zero from 173 on."""
    eng = engines("golden")
    x = torch.from_numpy(layer_crops).to(eng.tdev)
    n_dev = torch.tensor([173], dtype=torch.int32, device=eng.tdev)
    ref = [t[:173].cpu().numpy() for t in eng.cae_forward(x, 173, precision=1)]
    eng.check_status()
    for prec in (1, 2):
        mse = torch.full((300,), 7.0, device=eng.tdev)
        mae = torch.full((300,), 7.0, device=eng.tdev)
        feat = torch.full((300, 2048), 7.0, device=eng.tdev)
        eng._check(eng.lib.cia_cae_forward(eng.h, C.c_void_p(x.data_ptr()), 300, C.c_void_p(n_dev.data_ptr()),
                                           C.c_void_p(mse.data_ptr()), C.c_void_p(mae.data_ptr()),
                                           C.c_void_p(feat.data_ptr()), prec, eng._stream()))
        eng.check_status()
        got = [t.cpu().numpy() for t in (mse, mae, feat)]
        if prec == 1:
            for a, b, name in zip(got, ref, ("mse", "mae", "features")):
                assert np.array_equal(a[:173].view(np.int32), b.view(np.int32)), f"{name} of cells < 173"
        else:
            sub = [t[:173].cpu().numpy() for t in eng.cae_forward(x, 173, precision=2)]
            eng.check_status()
            for a, b, name in zip(got, sub, ("mse", "mae", "features")):
                assert np.array_equal(a[:173].view(np.int32), b.view(np.int32)), f"precision 2 {name} of cells < 173"
        assert not got[0][173:].any() and not got[1][173:].any(), f"precision {prec}: mse / mae beyond the device count"


@pytest.mark.gpu
def test_activation_outside_fp16_range(engines, oracle_weights, layer_crops):
    """A model whose BN scale drives a layer-4 activation far past 65504 (gamma 5e4 over a moving variance
    of 1e-3 on one channel) is finite in Keras and at precision 0.  Precision 1 stores activations as
    fp16: it must match the reference or report CIA_E_UNSUPPORTED, never a silent inf / NaN / wrong score."""
    from cell_image_analysis_b200 import _lib
    w = model_sets(oracle_weights)["golden"]
    g, b, m, v = w["bns"][3]
    g[0], v[0] = np.float32(5e4), np.float32(1e-3)
    eng = make_engine(w)
    try:
        n = 64
        X = layer_crops[:n]
        x = torch.from_numpy(np.ascontiguousarray(X)).to(eng.tdev)
        mse, mae, _ = eng.cae_forward(x, n, precision=1)
        code = 0
        try:
            eng.check_status()
        except _lib.CiaError as e:
            code = e.code
        mse1 = mse[:n].cpu().numpy()
        print(f"precision 1: status {code}, {int((~np.isfinite(mse1)).sum())} of {n} mse non-finite, "
              f"mse[:4] {mse1[:4]}")
        if code == 0:
            taps, c0, _ = read_taps(eng, n, PASS_CELLS)
            rep = check_layers("p1 fp16 overflow", w, pack_weights(w), X, taps, mse1, mae[:n].cpu().numpy(),
                               None, np.arange(n), 1, dev=str(eng.tdev))
            rep.done()
        else:
            assert code == _lib.CIA_E_UNSUPPORTED, code
        eng.check_status()                       # the status word was cleared by the check
        m0, a0, _ = eng.cae_forward(x, n, precision=0)
        eng.check_status()
        rec, _ = ocae.forward(X[:, :, :, None], w)
        rm, ra = ocae.recon_errors(X[:, :, :, None], rec)
        assert np.isfinite(rm).all()
        np.testing.assert_allclose(m0[:n].cpu().numpy(), rm, rtol=1e-3)
        np.testing.assert_allclose(a0[:n].cpu().numpy(), ra, rtol=1e-3)
    finally:
        eng.close()


# ---------------------------------------------------------------------------------------------
# CPU tests of the reference itself
# ---------------------------------------------------------------------------------------------
def _oracle_layers(X, w):
    """oracle.cae's layer chain with every intermediate (NCHW, float32)."""
    outs = []
    x = torch.from_numpy(np.ascontiguousarray(X))[:, None]
    for i in range(7):
        x = ocae._conv(x, w["kernels"][i], w["biases"][i], True)
        if i < 6:
            x = ocae._bn(torch.relu(x), w["bns"][i])
            if i < 3:
                x = F.max_pool2d(x, 2)
            outs.append(x.double())
            if i >= 3:
                x = F.interpolate(x, scale_factor=2, mode="nearest")
        else:
            outs.append(torch.sigmoid(x).double())
    return outs


def _exact_chain(X, w):
    """The reference operations above chained in fp64 with exact weights: no fp16, no packing, no
    scale.  L4 / L5 outputs stay at their low resolution (as the kernels store them); L6 runs in phase
    form and L7 in tap-sum form, from the low-resolution maps."""
    bn = bn_params(w)
    x = torch.from_numpy(np.asarray(X, np.float64))[:, None]
    outs = []
    for L in range(6):
        k = _t(w["kernels"][L], "cpu")
        if L == 4:
            acc = conv(up2(x), k)
        elif L == 5:
            acc = phase_conv(x, _t(phase_form(w["kernels"][L], np.float64), "cpu"))
        else:
            acc = conv(x, k)
        x = act(acc, acc.abs(), 1.0, w["biases"][L], *bn[L], 0, 0.0, 0)[0]
        if L < 3:
            x = pool2(x)
        outs.append(x)
    a = tapsum_conv(x, _t(tapsum_form(w["kernels"][6], np.float64), "cpu")) + float(w["biases"][6][0])
    outs.append(torch.sigmoid(a))
    return outs


@pytest.mark.parametrize("name", ["golden", "seed101", "neg_gamma", "neg_zero_gamma"])
def test_reference_chain_matches_oracle(oracle_weights, golden_tiny, name):
    """Without fp16 rounding and packing the per-layer reference is the oracle: every intermediate,
    the features and the reconstruction within fp32 noise, MSE / MAE too.  A wrong layout, phase,
    pooling or up-sampling in the reference fails here."""
    w = model_sets(oracle_weights)[name]
    X = np.concatenate([constructed_crops(), golden_tiny["crops"].astype(np.float32)])
    ref = _oracle_layers(X, w)
    got = _exact_chain(X, w)
    for L in range(7):          # the oracle's L4 / L5 outputs are taken before its up-sampling
        r, g = ref[L], got[L]
        assert g.shape == r.shape, (L, g.shape, r.shape)
        tol = 2e-5 * max(float(r.abs().max()), 1e-3)
        d = float((g - r).abs().max())
        assert d <= tol, f"layer {L + 1}: max |reference - oracle| {d:.3e} > {tol:.3e}"
    rec, enc = ocae.forward(X[:, :, :, None], w)
    np.testing.assert_allclose(got[2].permute(0, 2, 3, 1).numpy(), enc, rtol=0,
                               atol=2e-5 * max(np.abs(enc).max(), 1e-3))
    np.testing.assert_allclose(got[6][:, 0].numpy(), rec[:, :, :, 0], rtol=0, atol=2e-6)
    d = X - got[6][:, 0].numpy()
    rm, ra = ocae.recon_errors(X[:, :, :, None], rec)
    np.testing.assert_allclose((d * d).mean((1, 2)), rm, rtol=2e-5, atol=1e-12)
    np.testing.assert_allclose(np.abs(d).mean((1, 2)), ra, rtol=2e-5, atol=1e-12)


def test_weight_split_reconstructs(oracle_weights):
    """hi + lo reconstructs the scaled weights of every image to 2^-22 (2^-25 absolute for subnormal
    remainders), and the scale puts the largest weight in [2, 4)."""
    for name, w in model_sets(oracle_weights).items():
        for L, p in enumerate(pack_weights(w)):
            k = np.asarray(w["kernels"][L], np.float32)
            imgs = [(phase_form(k) if L >= 5 else k, p["hi"], p["lo"])]
            if L == 6:
                imgs.append((tapsum_form(k), p["t_hi"], p["t_lo"]))
            for img, hi, lo in imgs:
                v = img.astype(np.float64) * 2.0 ** p["sw"]
                assert 2 <= np.abs(phase_form(k) if L >= 5 else k).max() * 2.0 ** p["sw"] < 4
                err = np.abs(hi.astype(np.float64) + lo.astype(np.float64) - v)
                assert (err <= 2.0 ** -22 * np.abs(v) + 2.0 ** -25).all(), (name, L, err.max())
                assert (np.abs(hi.astype(np.float64) - v) <= 2.0 ** -11 * np.abs(v) + 2.0 ** -25).all()


@pytest.mark.parametrize("r,cin,cout", [(8, 32, 64), (16, 64, 32), (32, 32, 1)])
def test_phase_form_is_upsampled_conv(r, cin, cout):
    """The phase-form image (fp32-summed, as packed) applied at low resolution reproduces the 3x3 conv
    on the 2x nearest up-sampled map, borders included; so does the tap-sum image for one channel."""
    rng = np.random.default_rng(r + cin + cout)
    k = (rng.standard_normal((3, 3, cin, cout)) * 0.2).astype(np.float32)
    x = torch.from_numpy(rng.uniform(-1, 1, (3, cin, r, r)))
    x[:, :, 0, :] = 1.0                     # non-zero borders
    x[:, :, :, -1] = -1.0
    want = conv(up2(x), _t(k, "cpu"))
    mag = conv(up2(x.abs()), _t(np.abs(k), "cpu"))
    got = phase_conv(x, _t(phase_form(k), "cpu"))
    # kp's entries are fp32 sums of up to four taps: 2 roundings of 2^-24 relative
    assert ((got - want).abs() <= 2 * U * mag + 1e-12).all()
    exact = phase_conv(x, _t(phase_form(k, np.float64), "cpu"))
    assert float((exact - want).abs().max()) <= 1e-12 * float(mag.max())
    if cout == 1:
        got_t = tapsum_conv(x, _t(tapsum_form(k), "cpu"))
        assert ((got_t - want).abs() <= 2 * U * mag + 1e-12).all()
        # and a wrong neighbour / phase is caught: swap two phase columns of the image
        kt = tapsum_form(k)
        kt[:, [0, 4]] = kt[:, [4, 0]]
        assert float((tapsum_conv(x, _t(kt, "cpu")) - want).abs().max()) > 1e-3


def test_ws_layout_rule():
    """The pass size and buffer offsets of k_cae_forward_tc."""
    assert ws_layout(1)[0] == 148 and ws_layout(148)[0] == 148 and ws_layout(149)[0] == 296
    assert ws_layout(300)[0] == 444 and ws_layout(18943)[0] == 18944 and ws_layout(40000)[0] == 18944
    ch, bufs, c0, chunk = ws_layout(300, 148)
    assert (ch, c0, chunk) == (148, 296, 4)
    assert bufs["A1l"][0] == 148 * 4 * 32 * 32 * 8 and bufs["A6"][1] == 4 * 32 * 32 * 8
    assert ws_layout(40000)[2:] == (37888, 2112)
    total = sum(per for _, per, _, _ in bufs.values())
    assert total == 2 * 32768 + 2 * 16384 + 2048 + 2048 + 16384 + 32768     # per_cell halves



def test_l2_gate_catches_dropped_cross_term(oracle_weights, golden_tiny):
    """The layer-2 gate has teeth: a layer 2 that leaves out the A1l x W_hi products (one of the three
    split-precision MMAs per k-step) fails it by more than a factor 10, while the correct layer, stored
    as the device stores it, passes.  Layer 1's output is the reference of layer 1 on the golden tiny
    crops, stored as fp16 hi / lo."""
    w = model_sets(oracle_weights)["golden"]
    packs, bn = pack_weights(w), bn_params(w)
    X = golden_tiny["crops"].astype(np.float32)
    cells = np.arange(len(X))
    y1, _ = l1_reference(torch.from_numpy(X)[:, None], w, packs, bn, True)
    a1h, a1l = split_store(y1)

    def layer2(cross_lo_hi):
        whi, wlo = _t(packs[1]["hi"], "cpu"), _t(packs[1]["lo"], "cpu")
        acc = conv(a1h, whi) + conv(a1h, wlo) + (conv(a1l, whi) if cross_lo_hi else 0)
        y = pool2(act(acc, acc.abs(), packs[1]["inv"], w["biases"][1], *bn[1], 0, 0.0, 0)[0])
        return sum(split_store(y))

    good = Report("correct L2")
    check_l2(good, w, packs, bn, a1h, a1l, layer2(True), True, cells)
    print(good.line())
    assert not good.failures, "\n".join(good.failures)
    bad = Report("L2 without A1l x W_hi")
    check_l2(bad, w, packs, bn, a1h, a1l, layer2(False), True, cells)
    print(bad.line())
    assert bad.ratio["L2"] > 10.0, bad.line()
