"""The update block's own parts of rnc_conv2d_umma_fwd against fp64 references on the CPU: the GRU gate epilogues
(GRU_ZR, GRU_Q), the flow append (RELU_FLOW) and the coords update (FLOW_DELTA), the tile-blocked layouts, and the state the
loop carries from one step to the next (h and its split copy, the hoisted context share, coords1).  Everything runs through
the C ABI.  Next to every kernel error the tests print the fp32 CPU computation's own distance to fp64 as a yardstick.

Bars.  One tensor-core layer is within BAR * max(1, max |accumulation|) of fp64 (test_gpu_umma.py).  An epilogue's bar adds
the activation's derivative times that error, the activation's approximation error (sigmoid_fast / tanh_fast: ex2.approx and
rcp.approx, a few 1e-7; 2e-6 is allowed), fp32 rounding of the stored value (2^-24 relative per operation) and, for split
outputs, the hi/lo representation (2^-21 relative, 6e-8 absolute floor)."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT, build_model
from oracle import raft_oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

BAR = 2e-5                 # per-layer bar of the tensor-core convolution, relative to its accumulation's magnitude
ACT = 2e-6                 # allowance for the approximation error of sigmoid_fast / tanh_fast
ACT_EXACT = 1e-6           # the same, where the pre-activation is exact (measured bound of the approximations: ~4e-7)
EPS32 = 2.0 ** -24         # fp32 rounding, relative
SPLIT = 2.0 ** -21         # hi + lo split halves, relative (plus a 6e-8 absolute floor: half subnormals)
GUARD = 4096               # NaN-filled floats after every tile-blocked buffer

# rnc_conv_umma_desc.flags
NO_HALO, SPLIT_N, NO_PAIR, AUX_BLOCKED, OUT_BLOCKED, TF32 = 1, 4, 8, 16, 32, 64
FORMS = {"default": 0, "no_pair": NO_PAIR, "split_n": SPLIT_N}
KERNELS = {"1x5": (1, 5), "5x1": (5, 1)}

# (B, H8, W8) -> tile counts of the 1x5 and the 5x1 gate layers, and why the shape is here
SHAPES = {
    (1, 16, 32): (4, 4),        # the golden shape: 1x5 per tap (TW = 32), 4 tiles, even
    (1, 55, 128): (55, 56),     # 1x5 row halo, 55 tiles (odd: the CTA pair gets a ghost tile); 5x1 column halo, 56 tiles
    (1, 47, 156): (94, 60),     # KITTI at 1/8: row halo with a ragged second tile per row; column halo ragged both ways
    (1, 24, 64): (12, 12),      # W = 64, the edge of the row-halo condition (W > 64): per tap with TW = 64
    (3, 13, 37): (21, 18),      # per-tap 1x5, 21 tiles (odd); column-halo 5x1, 18 tiles; B > 1
    (1, 7, 9): (1, 1),          # H < 8: the 5x1 gates run per tap too; one tile, so the pair's second CTA is a ghost
    (8, 55, 128): (440, 448),   # the benchmarked step: a different column-tile width from B = 1
}
SHAPE_IDS = [f"{b}x{h}x{w}" for b, h, w in SHAPES]
B8 = (8, 55, 128)


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def split(t):
    hi = t.half()
    return hi, (t - hi.float()).half()


def to_cl(x):
    """[B, C, H, W] -> [B*H*W, C]"""
    return x.permute(0, 2, 3, 1).reshape(-1, x.shape[1]).contiguous()


def to_nchw(x, B, H, W):
    return x.reshape(B, H, W, -1).permute(0, 3, 1, 2)


def dsig(x):
    s = torch.sigmoid(x)
    return s * (1 - s)


def report(case, what, err, bar, yard=None):
    y = f"{yard:.2e}" if yard is not None else "-"
    print(f"UB| {case} | {what} | kernel {err:.2e} | fp32 {y} | bar {bar:.2e}")


# ----------------------------------------------------------------------------- tiling and the tile-blocked layout


def tile_shape(kh, kw, H, W, flags):
    """The documented tiling of a stride-1 layer (rnc.h, rnc_conv_umma_tiles): row halo (kw > 1, W > 64) -> 128 x 1 px,
    column halo (kw == 1 < kh, W >= 16, H >= 8) -> 16 x 8 px, otherwise per tap: TW = the smallest power of two >= W in
    [8, 128], TH = 128 / TW.  RNC_CONV_NO_HALO forces per tap."""
    if not flags & NO_HALO and kw > 1 and W > 64:
        return 128, 1
    if not flags & NO_HALO and kw == 1 and kh > 1 and W >= 16 and H >= 8:
        return 16, 8
    tw = 8
    while tw < W and tw < 128:
        tw *= 2
    return tw, 128 // tw


def tiling(kh, kw, B, H, W, flags):
    from rnc import native
    TW, TH = tile_shape(kh, kw, H, W, flags)
    tiles = B * -(-W // TW) * -(-H // TH)
    assert native.lib().rnc_conv_umma_tiles(kh, kw, 1, B, H, W, flags) == tiles, (kh, kw, B, H, W, flags)
    return tiles, TW, TH


def from_blocked(buf, ld, kh, kw, B, H, W, flags):
    """Tile-blocked [tile][channel][128 px] -> ([B*H*W, ld] channel-last, entries of the out-of-image rows).
    Tile t = (b * tiles_y + ty) * tiles_x + tx, row r = (y - ty*TH) * TW + (x - tx*TW) (rnc.h)."""
    tiles, TW, TH = tiling(kh, kw, B, H, W, flags)
    ty, tx = -(-H // TH), -(-W // TW)
    full = buf[:tiles * ld * 128].reshape(B, ty, tx, ld, TH, TW).permute(0, 1, 4, 2, 5, 3).reshape(B, ty * TH, tx * TW, ld)
    outside = torch.cat([full[:, H:].reshape(-1), full[:, :H, W:].reshape(-1)])
    return full[:, :H, :W].reshape(-1, ld), outside


def to_blocked(t, kh, kw, B, H, W, flags):
    """[B*H*W, ld] channel-last -> tile-blocked (NaN in the out-of-image rows) + a NaN guard."""
    tiles, TW, TH = tiling(kh, kw, B, H, W, flags)
    ty, tx = -(-H // TH), -(-W // TW)
    ld = t.shape[1]
    full = torch.full((B, ty * TH, tx * TW, ld), float("nan"))
    full[:, :H, :W] = t.reshape(B, H, W, ld)
    body = full.reshape(B, ty, TH, tx, TW, ld).permute(0, 1, 3, 5, 2, 4).reshape(-1)
    return torch.cat([body, torch.full((GUARD,), float("nan"))])


def blocked_buf(ld, kh, kw, B, H, W, flags):
    """Exactly rnc_conv_umma_tiles(...) * ld * 128 floats, then a guard; NaN everywhere."""
    tiles, _, _ = tiling(kh, kw, B, H, W, flags)
    return torch.full((tiles * ld * 128 + GUARD,), float("nan"), device=DEV)


def test_shapes_cover_the_tilings_they_are_listed_for():
    for (B, H, W), (t15, t51) in SHAPES.items():
        assert tiling(1, 5, B, H, W, 0)[0] == t15 and tiling(5, 1, B, H, W, 0)[0] == t51
        for kh, kw in KERNELS.values():
            tiling(kh, kw, B, H, W, NO_HALO)                        # the per-tap tiling agrees too
    assert tile_shape(1, 5, 55, 128, 0) == (128, 1) and tile_shape(5, 1, 55, 128, 0) == (16, 8)
    assert tile_shape(1, 5, 24, 64, 0) == (64, 2) and tile_shape(5, 1, 7, 9, 0) == (16, 8)
    assert sum(1 for t in SHAPES.values() if t[0] % 2) >= 2                       # odd counts: ghost tiles


# ----------------------------------------------------------------------------- GRU gates with random operands

_GATES = {}               # (shape, kernel) -> GateCase, kept for the module: the fp64 parts are the expensive bit


class GateCase:
    """One SepConvGRU half step at a shape: h | inp | x as the engine holds them in hx (update.py:45-50), the gate weights
    split as PackedUpdateUmma.gate does (K = h and x in the layer, the context share inp hoisted with the biases), and the
    fp64 parts of the reference that do not depend on the kernel's output."""

    def __init__(self, shape, kern):
        from rnc.engine_umma import SplitBuf, UmmaWeights
        B, H, W = shape
        kh, kw = KERNELS[kern]
        self.shape, self.k = shape, (kh, kw)
        g = torch.Generator().manual_seed(1000 * B + 10 * H + W + 7 * kh)
        self.h = torch.tanh(2 * torch.randn(B, 128, H, W, generator=g))
        self.inp = torch.relu(torch.randn(B, 128, H, W, generator=g))
        self.x = torch.relu(torch.randn(B, 128, H, W, generator=g))
        fan = (384 * kh * kw) ** 0.5
        self.wzr = torch.randn(256, 384, kh, kw, generator=g) / fan
        self.bzr = torch.linspace(-40, 40, 256)[torch.randperm(256, generator=g)]    # pre-activations over about +-40
        self.wq = torch.randn(128, 384, kh, kw, generator=g) / fan
        self.bq = torch.linspace(-24, 24, 128)[torch.randperm(128, generator=g)]     # across |x| = 0.25, into saturation
        M = B * H * W
        self.hx = SplitBuf(M, 384, DEV)
        for i, t in enumerate((self.h, self.inp, self.x)):
            self.hx.hi[:, 128 * i:128 * (i + 1)], self.hx.lo[:, 128 * i:128 * (i + 1)] = split(to_cl(t).to(DEV))

        def gate(w, b):
            return (UmmaWeights(torch.cat([w[:, :128], w[:, 256:]], 1).to(DEV), None, [128, 128]),
                    UmmaWeights(w[:, 128:256].to(DEV), b.to(DEV), [128]))
        self.zr, self.zr_c = gate(self.wzr, self.bzr)
        self.q, self.q_c = gate(self.wq, self.bq)
        # fp64 reference parts
        self.pad = (kh // 2, kw // 2)
        d = torch.float64
        acc_it = F.conv2d(torch.cat([self.h, self.x], 1).to(d), torch.cat([self.wzr[:, :128], self.wzr[:, 256:]], 1).to(d), padding=self.pad)
        self.czr_acc = F.conv2d(self.inp.to(d), self.wzr[:, 128:256].to(d), padding=self.pad)
        self.pre_zr = acc_it + self.czr_acc + self.bzr.to(d).view(1, -1, 1, 1)
        self.e_zr = BAR * (max(1.0, acc_it.abs().max().item()) + max(1.0, self.czr_acc.abs().max().item())) \
            + 4 * EPS32 * self.pre_zr.abs()
        self.cq_acc = F.conv2d(self.inp.to(d), self.wq[:, 128:256].to(d), padding=self.pad)
        self.qx_acc = F.conv2d(self.x.to(d), self.wq[:, 256:].to(d), padding=self.pad)
        pre32 = F.conv2d(torch.cat([self.h, self.inp, self.x], 1), self.wzr, self.bzr, padding=self.pad)
        self.yard_z = (torch.sigmoid(pre32[:, :128]).double() - torch.sigmoid(self.pre_zr[:, :128])).abs().max().item()
        self.q_ref = None


def gate_case(shape, kern):
    key = (shape, kern)
    if key not in _GATES:
        _GATES[key] = GateCase(shape, kern)
    return _GATES[key]


def run_gates(eng, d, form, blocked):
    """Hoisted context share (EPI_LINEAR, OUT_BLOCKED when blocked) -> GRU_ZR -> GRU_Q, as _update_iter issues them.
    Returns channel-last CPU tensors."""
    from rnc import native
    from rnc.engine_umma import SplitBuf
    B, H, W = d.shape
    kh, kw = d.k
    M = B * H * W
    if blocked:
        czr, cq, z = (blocked_buf(ld, kh, kw, B, H, W, form) for ld in (256, 128, 128))
    else:
        czr, cq, z = (torch.full((M, ld), float("nan"), device=DEV) for ld in (256, 128, 128))
    for wt, buf in ((d.zr_c, czr), (d.q_c, cq)):
        eng.uconv(B, H, W, d.hx.ptrs(128), 128, 384, wt, native.EPI_LINEAR, out_f32=buf.data_ptr(), ldo_f32=wt.coutpad,
                  flags=form | (OUT_BLOCKED if blocked else 0))
    fl = form | (AUX_BLOCKED if blocked else 0)
    h = to_cl(d.h).to(DEV)                                  # fp32 master of the state, updated in place by GRU_Q
    rh = SplitBuf(M, 128, DEV)
    eng.uconv(B, H, W, d.hx.ptrs(), 128, 384, d.zr, native.EPI_GRU_ZR, in1=d.hx.ptrs(256), c1=128, ld1=384,
              out_split=rh.ptrs(), ldo_split=128, h=h.data_ptr(), ldh=128, aux0=z.data_ptr(), ldaux=128,
              add=czr.data_ptr(), ldadd=256, flags=fl)
    hs = SplitBuf(M, 384, DEV)                              # the split copy lands in channels [0, 128); the rest is a sentinel
    hs.hi.fill_(-7.0)
    hs.lo.fill_(0.125)
    eng.uconv(B, H, W, rh.ptrs(), 128, 128, d.q, native.EPI_GRU_Q, in1=d.hx.ptrs(256), c1=128, ld1=384,
              out_split=hs.ptrs(), ldo_split=384, h=h.data_ptr(), ldh=128, aux0=z.data_ptr(), ldaux=128,
              add=cq.data_ptr(), ldadd=128, flags=fl)
    torch.cuda.synchronize()
    r = {"rh": (rh.hi.float() + rh.lo.float()).cpu(), "h": h.cpu(), "hs": (hs.hi[:, :128].float() + hs.lo[:, :128].float()).cpu(),
         "sentinel_ok": bool((hs.hi[:, 128:] == -7.0).all() and (hs.lo[:, 128:] == 0.125).all())}
    for name, buf, ld in (("czr", czr, 256), ("cq", cq, 128), ("z", z, 128)):
        buf = buf.cpu()
        if blocked:
            assert torch.isnan(buf[-GUARD:]).all(), f"{name}: write past rnc_conv_umma_tiles(...) * {ld} * 128 floats"
            buf, outside = from_blocked(buf, ld, kh, kw, B, H, W, form)
            assert torch.isnan(outside).all(), f"{name}: write into the out-of-image rows of a tile"
        assert torch.isfinite(buf).all(), f"{name}: entries left unwritten"
        r[name] = buf
    return r


@pytest.fixture(scope="module")
def ueng():
    from rnc.engine_umma import UmmaEngine
    return UmmaEngine()


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("kern", list(KERNELS))
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
def test_gru_gates_vs_fp64(ueng, shape, kern, form):
    """GRU_ZR then GRU_Q (update.py:45-50) over K = h | x with the hoisted context share as the `add` operand, in the
    channel-last and the tile-blocked layouts: z = sigmoid, r*h as split halves, h updated in place and its split copy; the
    hoisted form agrees with fp64 of the full 384-channel convolution (linearity)."""
    d = gate_case(shape, kern)
    B, H, W = shape
    case = f"gates {kern} {B}x{H}x{W} {form}"
    fl = FORMS[form]
    cl, bl = run_gates(ueng, d, fl, False), run_gates(ueng, d, fl, True)
    for k in cl:                       # the same products and adds in the same order: bit-identical
        assert cl[k] == bl[k] if k == "sentinel_ok" else torch.equal(cl[k], bl[k]), f"{case}: {k} blocked != channel-last"
    if fl:
        ref = run_gates(ueng, d, 0, False)
        same = all(torch.equal(ref[k], cl[k]) for k in ("z", "rh", "h", "hs"))
        print(f"UB| {case}: bit-identical to the default form: {same}")
        if fl & NO_PAIR:
            assert same, f"{case}: the single-CTA form differs from the pair form"
    assert cl["sentinel_ok"], f"{case}: GRU_Q wrote outside channels [0, 128) of its split output"
    # the hoisted layer itself
    c_ref = to_cl(d.czr_acc + d.bzr.double().view(1, -1, 1, 1))
    e = (cl["czr"].double() - c_ref).abs()
    bar = BAR * max(1.0, d.czr_acc.abs().max().item()) + EPS32 * c_ref.abs()
    report(case, "hoisted zr share", e.max().item(), bar.max().item())
    assert (e <= bar).all()
    # z = sigmoid(pre[:128])
    pre = to_cl(d.pre_zr)
    ez = to_cl(d.e_zr)
    zr = torch.sigmoid(pre[:, :128])
    bar = dsig((pre[:, :128].abs() - ez[:, :128]).clamp(min=0)) * ez[:, :128] + ACT
    e = (cl["z"].double() - zr).abs()
    report(case, "z", e.max().item(), bar.max().item(), d.yard_z)
    assert (e <= bar).all(), f"{case}: z off by {e.max().item():.2e}"
    # r * h, written as split halves
    hv = to_cl(d.h).double()
    rhr = torch.sigmoid(pre[:, 128:]) * hv
    bar = (dsig((pre[:, 128:].abs() - ez[:, 128:]).clamp(min=0)) * ez[:, 128:] + ACT) * hv.abs() + (EPS32 + SPLIT) * rhr.abs() + 6e-8
    e = (cl["rh"].double() - rhr).abs()
    report(case, "r*h", e.max().item(), bar.max().item())
    assert (e <= bar).all(), f"{case}: r*h off by {e.max().item():.2e}"
    # q gate on the kernel's r*h and z: h' = (1-z) h + z tanh(q), in place, and its split copy
    rh_k = to_nchw(cl["rh"], B, H, W).double()
    acc_it = F.conv2d(rh_k, d.wq[:, :128].double(), padding=d.pad) + d.qx_acc
    pre_q = to_cl(acc_it + d.cq_acc + d.bq.double().view(1, -1, 1, 1))
    eq = BAR * (max(1.0, acc_it.abs().max().item()) + max(1.0, d.cq_acc.abs().max().item())) + 4 * EPS32 * pre_q.abs()
    zk = cl["z"].double()
    href = (1 - zk) * hv + zk * torch.tanh(pre_q)
    dtanh = 1 - torch.tanh((pre_q.abs() - eq).clamp(min=0)) ** 2
    bar = zk * (dtanh * eq + ACT) + 4 * EPS32 * (hv.abs() + 1)
    e = (cl["h"].double() - href).abs()
    q32 = F.conv2d(torch.cat([to_nchw(cl["rh"], B, H, W), d.inp, d.x], 1), d.wq, d.bq, padding=d.pad)
    z32 = cl["z"]
    h32 = (1 - z32) * to_cl(d.h) + z32 * torch.tanh(to_cl(q32))
    report(case, "h (q gate)", e.max().item(), bar.max().item(), (h32.double() - href).abs().max().item())
    assert (e <= bar).all(), f"{case}: h off by {e.max().item():.2e}"
    hk = cl["h"]
    e = (cl["hs"] - hk).abs()
    assert (e <= hk.abs() * SPLIT + 6e-8).all(), f"{case}: split copy of h off by {e.max().item():.2e}"


# ----------------------------------------------------------------------------- gate activations on exact pre-activations


@pytest.mark.parametrize("kern", list(KERNELS))
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
def test_gate_activations_on_exact_pre_activations(ueng, shape, kern):
    """With zero input planes the pre-activation is exactly the `add` operand (multiples of 2^-12, bias 0), so the epilogue's
    arithmetic is measured alone: z and r over +-44, q densely across the polynomial / exponential switch of tanh_fast at
    |x| = 0.25 and into the clamp at |x| = 20.  The add operand is encoded into the tile-blocked layout here, from the
    formula of rnc.h, independently of the OUT_BLOCKED store."""
    from rnc import native
    from rnc.engine_umma import SplitBuf
    d = gate_case(shape, kern)
    B, H, W = shape
    kh, kw = d.k
    M = B * H * W
    case = f"exact {kern} {B}x{H}x{W}"
    g = torch.Generator().manual_seed(M + kh)
    q = 4096.0

    def grid(lo, hi, n):
        return torch.randint(int(lo * q), int(hi * q) + 1, (M, n), generator=g).float() / q
    a_zr = torch.cat([grid(0, 44, 64), grid(-44, 0, 64), grid(-44, 44, 128)], 1)       # z >= 0.5 where q sweeps 0.25
    a_q = torch.cat([grid(-0.6, 0.6, 64), grid(-30, 30, 64)], 1)
    a_q[:, 0], a_q[:, 1] = 0.25, -0.25
    zero = SplitBuf(M, 384, DEV)
    h0 = to_cl(d.h)
    outs = {}
    for blocked in (False, True):
        fl = AUX_BLOCKED if blocked else 0
        if blocked:
            add_zr, add_q = (to_blocked(a, kh, kw, B, H, W, 0).to(DEV) for a in (a_zr, a_q))
            z = blocked_buf(128, kh, kw, B, H, W, 0)
        else:
            add_zr, add_q = a_zr.to(DEV), a_q.to(DEV)
            z = torch.full((M, 128), float("nan"), device=DEV)
        h = h0.to(DEV)
        rh = SplitBuf(M, 128, DEV)
        ueng.uconv(B, H, W, zero.ptrs(), 128, 384, d.zr, native.EPI_GRU_ZR, in1=zero.ptrs(256), c1=128, ld1=384,
                   out_split=rh.ptrs(), ldo_split=128, h=h.data_ptr(), ldh=128, aux0=z.data_ptr(), ldaux=128,
                   add=add_zr.data_ptr(), ldadd=256, flags=fl)
        hs = SplitBuf(M, 128, DEV)
        ueng.uconv(B, H, W, zero.ptrs(), 128, 384, d.q, native.EPI_GRU_Q, in1=zero.ptrs(256), c1=128, ld1=384,
                   out_split=hs.ptrs(), ldo_split=128, h=h.data_ptr(), ldh=128, aux0=z.data_ptr(), ldaux=128,
                   add=add_q.data_ptr(), ldadd=128, flags=fl)
        torch.cuda.synchronize()
        zc = z.cpu()
        if blocked:
            assert torch.isnan(zc[-GUARD:]).all()
            zc, _ = from_blocked(zc, 128, kh, kw, B, H, W, 0)
        outs[blocked] = (zc, (rh.hi.float() + rh.lo.float()).cpu(), h.cpu())
    for a, b in zip(outs[False], outs[True]):
        assert torch.equal(a, b), f"{case}: blocked != channel-last"
    zk, rhk, hk = outs[False]
    pz, pq, hv = a_zr.double(), a_q.double(), h0.double()
    e = (zk.double() - torch.sigmoid(pz[:, :128])).abs().max().item()
    report(case, "z", e, ACT_EXACT, (torch.sigmoid(a_zr[:, :128]).double() - torch.sigmoid(pz[:, :128])).abs().max().item())
    assert e <= ACT_EXACT
    rr = torch.sigmoid(pz[:, 128:]) * hv
    e = (rhk.double() - rr).abs()
    assert (e <= ACT_EXACT * hv.abs() + (EPS32 + SPLIT) * rr.abs() + 6e-8).all(), f"{case}: r*h off by {e.max().item():.2e}"
    zd = zk.double()
    href = (1 - zd) * hv + zd * torch.tanh(pq)
    e = (hk.double() - href).abs()
    bar = zd * ACT_EXACT + 4 * EPS32 * (hv.abs() + 1)
    report(case, "h", e.max().item(), bar.max().item(), (((1 - zk) * h0 + zk * torch.tanh(a_q)).double() - href).abs().max().item())
    assert (e <= bar).all(), f"{case}: h off by {e.max().item():.2e}"


# ----------------------------------------------------------------------------- OUT_BLOCKED layout contract


@pytest.mark.parametrize("flags", [0, NO_HALO], ids=["halo", "no_halo"])
@pytest.mark.parametrize("kern", list(KERNELS))
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
def test_out_blocked_layout_contract(ueng, shape, kern, flags):
    """EPI_LINEAR with RNC_CONV_OUT_BLOCKED into exactly rnc_conv_umma_tiles(...) * ld * 128 floats: nothing past the end,
    nothing in the out-of-image rows, and the buffer decoded with rnc.h's formula equals fp64 of the layer."""
    from rnc import native
    d = gate_case(shape, kern)
    B, H, W = shape
    kh, kw = d.k
    buf = blocked_buf(128, kh, kw, B, H, W, flags)
    ueng.uconv(B, H, W, d.hx.ptrs(128), 128, 384, d.q_c, native.EPI_LINEAR, out_f32=buf.data_ptr(), ldo_f32=128,
               flags=flags | OUT_BLOCKED)
    torch.cuda.synchronize()
    buf = buf.cpu()
    assert torch.isnan(buf[-GUARD:]).all(), "write past the end of the tile-blocked tensor"
    got, outside = from_blocked(buf, 128, kh, kw, B, H, W, flags)
    assert torch.isnan(outside).all(), "write into the out-of-image rows"
    ref = to_cl(d.cq_acc + d.bq.double().view(1, -1, 1, 1))
    e = (got.double() - ref).abs()
    bar = BAR * max(1.0, d.cq_acc.abs().max().item()) + EPS32 * ref.abs()
    report(f"out_blocked {kern} {B}x{H}x{W} flags {flags}", "linear", e.max().item(), bar.max().item())
    assert (e <= bar).all()


# ----------------------------------------------------------------------------- RELU_FLOW and FLOW_DELTA


def flow_field(B, H, W, g):
    """Smooth flow plus a patch moving 40 px left and 40 px down (coordinates below zero at the left edge)."""
    yy, xx = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    flow = torch.stack([3 * torch.sin(yy / 7) + 0.05 * xx - 2, 2 * torch.cos(xx / 11) - 0.04 * yy + 1], 0)[None].repeat(B, 1, 1, 1)
    flow = flow + 0.1 * torch.randn(B, 2, H, W, generator=g)
    y0, x0 = H // 3, W // 4
    flow[:, 0, y0:y0 + max(1, H // 4), x0:x0 + max(1, W // 4)] = -40.0
    flow[:, 1, y0:y0 + max(1, H // 4), x0:x0 + max(1, W // 4)] = 40.0
    return flow


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
def test_relu_flow_epilogue(ueng, shape, form):
    """BasicMotionEncoder.conv + the flow append (update.py:96-97): 3x3, 256 -> 126 with ReLU, channels 126 and 127 =
    coords1 - grid, written at channel 256 of an hx-like row of 384 halves; channels [0, 256) keep their sentinel."""
    from rnc import native
    from rnc.engine_umma import SplitBuf, UmmaWeights
    B, H, W = shape
    M = B * H * W
    g = torch.Generator().manual_seed(M + 5)
    x = torch.relu(torch.randn(B, 256, H, W, generator=g))
    w = torch.randn(126, 256, 3, 3, generator=g) / 48.0
    b = 0.5 * torch.randn(126, generator=g)
    flow = flow_field(B, H, W, g)
    coords1 = orc.coords_grid(B, H, W) + flow
    xin = SplitBuf(M, 256, DEV)
    xin.hi[:], xin.lo[:] = split(to_cl(x).to(DEV))
    wt = UmmaWeights(w.to(DEV), b.to(DEV), [256], extra_cout=2)
    out = SplitBuf(M, 384, DEV)
    out.hi.fill_(-7.0)
    out.lo.fill_(0.125)
    c1 = coords1.to(DEV)
    ueng.uconv(B, H, W, xin.ptrs(), 256, 256, wt, native.EPI_RELU_FLOW, out_split=out.ptrs(256), ldo_split=384,
               aux0=c1.data_ptr(), flags=FORMS[form])
    torch.cuda.synchronize()
    assert (out.hi[:, :256] == -7.0).all() and (out.lo[:, :256] == 0.125).all(), "sentinel channels overwritten"
    got = (out.hi[:, 256:].double() + out.lo[:, 256:].double()).cpu()
    acc = F.conv2d(x.double(), w.double(), padding=1)
    ref = to_cl(F.relu(acc + b.double().view(1, -1, 1, 1)))
    e = (got[:, :126] - ref).abs()
    bar = BAR * max(1.0, acc.abs().max().item()) + (EPS32 + SPLIT) * ref.abs() + 6e-8
    y32 = to_cl(F.relu(F.conv2d(x, w, b, padding=1))).double()
    case = f"relu_flow {B}x{H}x{W} {form}"
    report(case, "relu", e.max().item(), bar.max().item(), (y32 - ref).abs().max().item())
    assert (e <= bar).all()
    fref = to_cl(coords1.double() - orc.coords_grid(B, H, W).double())      # coords1 as stored (fp32) minus the grid
    e = (got[:, 126:] - fref).abs()
    report(case, "flow", e.max().item(), ((EPS32 + SPLIT) * fref.abs() + 6e-8).max().item())
    assert (e <= (EPS32 + SPLIT) * fref.abs() + 6e-8).all()
    assert fref[:, 0].min() <= -30 and fref[:, 1].max() >= 39 and coords1[:, 0].min() < 0


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
def test_flow_delta_epilogue(ueng, shape, form):
    """RNC_EPI_FLOW_DELTA (rnc.h): FlowHead.conv2 (3x3, 256 -> 2, update.py:10,14) fused with coords1 += delta
    (raft_nc_dbl.py:157), delta also written NCHW to out_f32."""
    from rnc import native
    from rnc.engine_umma import SplitBuf, UmmaWeights
    B, H, W = shape
    M = B * H * W
    g = torch.Generator().manual_seed(M + 9)
    x = torch.relu(torch.randn(B, 256, H, W, generator=g))
    w = torch.randn(2, 256, 3, 3, generator=g) / 48.0
    b = torch.randn(2, generator=g)
    c0 = orc.coords_grid(B, H, W) + flow_field(B, H, W, g)
    xin = SplitBuf(M, 256, DEV)
    xin.hi[:], xin.lo[:] = split(to_cl(x).to(DEV))
    wt = UmmaWeights(w.to(DEV), b.to(DEV), [256])
    coords = c0.to(DEV)
    delta = torch.full((B, 2, H, W), float("nan"), device=DEV)
    ueng.uconv(B, H, W, xin.ptrs(), 256, 256, wt, native.EPI_FLOW_DELTA, out_f32=delta.data_ptr(), aux0=coords.data_ptr(),
               flags=FORMS[form])
    torch.cuda.synchronize()
    acc = F.conv2d(x.double(), w.double(), padding=1)
    dref = acc + b.double().view(1, -1, 1, 1)
    e_acc = BAR * max(1.0, acc.abs().max().item())
    e = (delta.cpu().double() - dref).abs()
    case = f"flow_delta {B}x{H}x{W} {form}"
    report(case, "delta", e.max().item(), e_acc + EPS32 * dref.abs().max().item(),
           (F.conv2d(x, w, b, padding=1).double() - dref).abs().max().item())
    assert (e <= e_acc + EPS32 * dref.abs()).all()
    cref = c0.double() + dref
    e = (coords.cpu().double() - cref).abs()
    report(case, "coords1", e.max().item(), (e_acc + 2 * EPS32 * cref.abs()).max().item())
    assert (e <= e_acc + 2 * EPS32 * cref.abs()).all()


# ----------------------------------------------------------------------------- argument checks


def test_launcher_rejects_unsupported_epilogue_requests(ueng):
    """Each rejected request is checked against the same request without its defect, which must launch."""
    from rnc import native
    from rnc.engine_umma import SplitBuf, UmmaWeights
    B, H, W = 1, 16, 32
    M = B * H * W
    g = torch.Generator().manual_seed(2)
    hx, rh, o = SplitBuf(M, 384, DEV), SplitBuf(M, 128, DEV), SplitBuf(M, 384, DEV)
    h, z, f = torch.zeros(M, 128, device=DEV), torch.zeros(M, 128, device=DEV), torch.zeros(M, 256, device=DEV)
    fb = blocked_buf(256, 1, 5, B, H, W, 0)
    coords = orc.coords_grid(B, H, W).to(DEV)

    def wts(cout, cin, kh, kw, segs, **kw_):
        return UmmaWeights(torch.randn(cout, cin, kh, kw, generator=g).to(DEV) / 40, torch.randn(cout, generator=g).to(DEV), segs, **kw_)
    zr, zr96, q = wts(256, 256, 1, 5, [128, 128]), wts(96, 256, 1, 5, [128, 128]), wts(128, 256, 1, 5, [128, 128])
    lin = wts(256, 128, 1, 5, [128])
    flow_ok, flow_bad = wts(126, 256, 3, 3, [256], extra_cout=2), wts(128, 256, 3, 3, [256])

    def gru_zr(wt, flags=0):
        ueng.uconv(B, H, W, hx.ptrs(), 128, 384, wt, native.EPI_GRU_ZR, in1=hx.ptrs(256), c1=128, ld1=384, out_split=rh.ptrs(),
                   ldo_split=128, h=h.data_ptr(), ldh=128, aux0=z.data_ptr(), ldaux=128, flags=flags)

    def gru_q(out_f32=0):
        ueng.uconv(B, H, W, rh.ptrs(), 128, 128, q, native.EPI_GRU_Q, in1=hx.ptrs(256), c1=128, ld1=384, out_split=o.ptrs(),
                   ldo_split=384, h=h.data_ptr(), ldh=128, aux0=z.data_ptr(), ldaux=128, out_f32=out_f32, ldo_f32=128)

    def linear(epi, flags=0, split_out=False):
        ueng.uconv(B, H, W, hx.ptrs(128), 128, 384, lin, epi, out_f32=(fb if flags & OUT_BLOCKED else f).data_ptr(), ldo_f32=256,
                   out_split=o.ptrs() if split_out else (0, 0), ldo_split=384 if split_out else 0, flags=flags)

    def relu_flow(wt):
        ueng.uconv(B, H, W, hx.ptrs(), 256, 384, wt, native.EPI_RELU_FLOW, out_split=o.ptrs(256), ldo_split=384,
                   aux0=coords.data_ptr())
    cases = [
        ("GRU_ZR with cout % 64 != 0", lambda: gru_zr(zr), lambda: gru_zr(zr96)),
        ("AUX_BLOCKED with EPI_RELU", lambda: linear(native.EPI_RELU), lambda: linear(native.EPI_RELU, AUX_BLOCKED)),
        ("OUT_BLOCKED with a split output", lambda: linear(native.EPI_LINEAR, OUT_BLOCKED),
         lambda: linear(native.EPI_LINEAR, OUT_BLOCKED, split_out=True)),
        ("TF32 with GRU_ZR", lambda: gru_zr(zr), lambda: gru_zr(zr, TF32)),
        ("RELU_FLOW with coutpad < cout + 2", lambda: relu_flow(flow_ok), lambda: relu_flow(flow_bad)),
        ("GRU_Q with out_f32", lambda: gru_q(), lambda: gru_q(f.data_ptr())),
    ]
    for what, good, bad in cases:
        good()
        with pytest.raises((ValueError, native.RncError)):
            bad()
        torch.cuda.synchronize()
        print(f"UB| rejects {what}")


# ----------------------------------------------------------------------------- the update block, step after step

VARIANTS = {
    "default": {},
    "no_halo": {"RNC_CONV_FLAGS": "1"},
    "split_n": {"RNC_CONV_FLAGS": "4"},
    "no_pair": {"RNC_CONV_FLAGS": "8"},
    "channel_last": {"RNC_BLOCKED": "0"},
    "convf1_ffma": {"RNC_CONVF1": "ffma"},
}
ENGINE_ENV = ("RNC_CONV", "RNC_LOOKUP", "RNC_CONVF1", "RNC_FORK", "RNC_BLOCKED", "RNC_CONV_FLAGS")
MODELS = ("raft_nc_dbl", "raft")
BLOCK_BAR = 5e-5           # net, delta, coords1 (the bar test_update_block_teacher_forced holds against the fp32 reference)


def fresh_engine(monkeypatch, env):
    """A new UmmaEngine reading `env` (engine_for would hand back a cached engine built under other switches)."""
    for k in ENGINE_ENV:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    from rnc.engine_umma import UmmaEngine
    return UmmaEngine()


def steps_for(shape):
    """(steps, step at which load_state brings a new inp): three carried steps, then a new context; one step at B = 8."""
    return (1, None) if shape == B8 else (4, 3)


def block_inputs(shape, corr_std):
    B, H, W = shape
    steps, _ = steps_for(shape)
    g = torch.Generator().manual_seed(31 * B + 7 * H + W)
    net = torch.tanh(torch.randn(B, 128, H, W, generator=g))
    inp = torch.relu(torch.randn(B, 128, H, W, generator=g))
    inp2 = torch.relu(torch.randn(B, 128, H, W, generator=g))
    corrs = [torch.randn(B, 324, H, W, generator=g) * corr_std for _ in range(steps)]
    return dict(net=net, inp=inp, inp2=inp2, corrs=corrs, flow=flow_field(B, H, W, g))


def run_kernel_steps(eng, model, x, shape, batch=None):
    """load_state, coords_init, then update_iter step after step with a teacher-forced corr each time; `batch` selects
    pairs.  Returns per step: net, delta, coords1 (NCHW), hx[:, :128] as hi + lo, h (the fp32 master), mask (CL)."""
    from rnc import native
    B, H, W = shape
    sel = (lambda t: t) if batch is None else (lambda t: t[batch:batch + 1])
    if batch is not None:
        B = 1
    ub = model.update_block
    pk = eng.packed_update(ub)
    ws = eng.workspace(torch.device(DEV), B, H, W, pk.has_mask, False)
    eng.load_state(ws, sel(x["net"]).to(DEV).contiguous(), sel(x["inp"]).to(DEV).contiguous())
    flow = sel(x["flow"]).to(DEV).contiguous()
    native.check(eng.L.rnc_coords_init(C.c_void_p(ws.coords1.data_ptr()), C.c_void_p(flow.data_ptr()), B, H, W, stream()),
                 "coords_init")
    steps, reload = steps_for(shape)
    out = []
    for k in range(steps):
        if k == reload:
            eng.load_state(ws, eng.net_nchw(ws), sel(x["inp2"]).to(DEV).contiguous())
        eng.begin_iter(ws, pk)
        eng.load_corr(ws, sel(x["corrs"][k]).to(DEV).contiguous())
        eng.update_iter(ws, pk, want_mask=pk.has_mask, want_delta=True)
        r = {"net": eng.net_nchw(ws), "delta": ws.delta.clone(), "coords1": ws.coords1.clone(),
             "hx": ws.hx.hi[:, :128].float() + ws.hx.lo[:, :128].float(), "h": ws.h.clone()}
        if pk.has_mask:
            r["mask"] = ws.mask.clone()
        torch.cuda.synchronize()
        out.append({k_: v.cpu() for k_, v in r.items()})
    return out


def run_oracle_steps(sd, x, shape, with_mask, dtype):
    """orc.update_block iterated: flow = coords1 - coords0, coords1 += delta; coords1 starts from its fp32 value."""
    B, H, W = shape
    steps, reload = steps_for(shape)
    cv = lambda t: t.to(dtype)
    coords0 = orc.coords_grid(B, H, W)
    c1 = cv(coords0 + x["flow"])
    coords0 = cv(coords0)
    net, inp = cv(x["net"]), cv(x["inp"])
    out = []
    for k in range(steps):
        if k == reload:
            inp = cv(x["inp2"])
        net, mask, delta = orc.update_block(sd, net, inp, cv(x["corrs"][k]), c1 - coords0, with_mask)
        c1 = c1 + delta
        out.append({"net": net, "delta": delta, "coords1": c1, "mask": mask})
    return out


_MODELS, _ORACLE = {}, {}


def model_for(name):
    if name not in _MODELS:
        m = build_model(name)
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        _MODELS[name] = (m.to(DEV), sd)
    return _MODELS[name]


def oracle_for(name, shape, gold):
    key = (name, shape)
    if key not in _ORACLE:
        _, sd = model_for(name)
        x = block_inputs(shape, float(torch.cat([gold["corr_it0"].flatten(), gold["corr_it3"].flatten()]).std()))
        t0 = time.time()
        r64 = run_oracle_steps({k: v.double() for k, v in sd.items()}, x, shape, name == "raft", torch.float64)
        t64 = time.time() - t0
        r32 = run_oracle_steps({k: v.float() for k, v in sd.items()}, x, shape, name == "raft", torch.float32)
        print(f"UB| fp64 oracle {name} {shape}: {t64:.1f} s for {len(r64)} step(s) on the CPU ({torch.get_num_threads()} threads)")
        _ORACLE[key] = (x, r64, r32)
    return _ORACLE[key]


def check_steps(case, got, r64, r32, shape, with_mask):
    B, H, W = shape
    cmax = 0.0
    for k, (g_, o, y) in enumerate(zip(got, r64, r32)):
        cmax = max(cmax, o["coords1"].abs().max().item())
        bars = {"net": BLOCK_BAR, "delta": BLOCK_BAR,
                # + one fp32 rounding of the stored coords1 per step (the oracle keeps it in fp64)
                "coords1": BLOCK_BAR + (k + 1) * EPS32 * cmax}
        if with_mask:
            bars["mask"] = BLOCK_BAR * max(1.0, o["mask"].abs().max().item())
        for key, bar in bars.items():
            kv = to_nchw(g_[key], B, H, W) if key == "mask" else g_[key]
            e = (kv.double() - o[key]).abs().max().item()
            report(f"{case} step {k}", key, e, bar, (y[key].double() - o[key]).abs().max().item())
            assert e <= bar, f"{case} step {k}: {key} off by {e:.2e} (bar {bar:.2e})"
        e = (g_["hx"] - g_["h"]).abs()
        assert (e <= g_["h"].abs() * SPLIT + 6e-8).all(), f"{case} step {k}: hx[:, :128] is not the split copy of h"
        assert torch.equal(to_nchw(g_["h"], B, H, W), g_["net"])


@pytest.mark.parametrize("variant", list(VARIANTS))
@pytest.mark.parametrize("shape", list(SHAPES), ids=SHAPE_IDS)
@pytest.mark.parametrize("name", MODELS)
def test_update_block_steps_vs_fp64_oracle(gold, monkeypatch, name, shape, variant):
    """Steps of the tensor-core update block on carried state (no load_state in between: the hoisted context share, h and
    its split copy, coords1 are what earlier steps left), then load_state with a different inp and one more step (the
    hoisted share must be recomputed).  One step at B = 8, where every pair must also match that pair run alone."""
    m, _ = model_for(name)
    x, r64, r32 = oracle_for(name, shape, gold)
    B, H, W = shape
    case = f"block {name} {B}x{H}x{W} {variant}"
    eng = fresh_engine(monkeypatch, VARIANTS[variant])
    got = run_kernel_steps(eng, m, x, shape)
    check_steps(case, got, r64, r32, shape, name == "raft")
    if variant in ("no_pair", "channel_last"):
        ref = run_kernel_steps(fresh_engine(monkeypatch, {}), m, x, shape)
        for k, (a, b) in enumerate(zip(got, ref)):
            for key in a:
                assert torch.equal(a[key], b[key]), f"{case} step {k}: {key} differs from the default form"
    if shape == B8:
        eng = fresh_engine(monkeypatch, VARIANTS[variant])
        worst, identical = 0.0, True
        for b in range(B):
            alone = run_kernel_steps(eng, m, x, shape, batch=b)
            for a, s in zip(got, alone):
                for key in a:
                    # mask: CL rows of pair b; the others NCHW (net, delta, coords1) or CL (hx, h)
                    rows = a[key].reshape(B, -1)[b] if key in ("mask", "hx", "h") else a[key][b:b + 1]
                    e = (rows.reshape(-1) - s[key].reshape(-1)).abs().max().item()
                    if key == "mask":
                        e /= max(1.0, s[key].abs().max().item())
                    worst, identical = max(worst, e), identical and e == 0.0
        print(f"UB| {case}: pairs vs alone max diff {worst:.2e}, bit-identical {identical}")
        assert worst <= 1e-6


def dump_default_run(name, out_path):
    """The default engine's B = 8 step of the test above, saved with torch.save.  The engine switches must be unset."""
    from rnc.engine_umma import UmmaEngine
    assert not any(k in os.environ for k in ENGINE_ENV)
    m, _ = model_for(name)
    z = np.load(os.path.join(ROOT, "tests", "golden", "cfg1.npz"))
    corr_std = float(torch.cat([torch.from_numpy(z["corr_it0"]).flatten(), torch.from_numpy(z["corr_it3"]).flatten()]).std())
    got = run_kernel_steps(UmmaEngine(), m, block_inputs(B8, corr_std), B8)
    torch.save(got, out_path)
    return got


def test_update_block_same_without_programmatic_dependent_launch(tmp_path, monkeypatch):
    """Every tensor-core convolution triggers its dependents at entry and orders itself with griddepcontrol.wait.  The same
    step at B = 8 with RNC_PDL=0 (plain stream order, read once per process: a subprocess) must give the same bits."""
    assert os.environ.get("RNC_PDL", "1") != "0", "this process must run with PDL on"
    out = tmp_path / "no_pdl.pt"
    env = {k: v for k, v in os.environ.items() if k not in ENGINE_ENV}
    env["RNC_PDL"] = "0"
    code = (f"import sys; sys.path[:0] = [{os.path.join(ROOT, 'tests')!r}, {ROOT!r}, {os.path.join(ROOT, 'raft-ncup_b200')!r}]\n"
            f"import test_gpu_update_block as t; t.dump_default_run('raft', {str(out)!r})\n")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    res = subprocess.run(cmd, env=env, cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    for k in ENGINE_ENV:
        monkeypatch.delenv(k, raising=False)
    on = dump_default_run("raft", str(tmp_path / "pdl.pt"))
    off = torch.load(str(out))
    for k, (a, b) in enumerate(zip(on, off)):
        for key in a:
            assert torch.equal(a[key], b[key]), f"step {k}: {key} differs with PDL off"
    print("UB| PDL on vs off at B=8: bit-identical")
