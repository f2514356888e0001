"""Training path of RAFT / RAFT-NCUP (SURVEY.md §8f-3, Appendix G; BASELINE config #5): the forward of
``RAFT.forward`` in train mode (raft_nc_dbl.py:115-173, raft.py:87-143) as an autograd graph whose heavy nodes are
``torch.autograd.Function``s running librnc's exact-fp32 kernels forward AND backward:

    ConvCL          every nn.Conv2d (update.py, extractor.py, interp_weights_est.py): rnc_conv2d_cl_fwd; data gradient = the same
                    kernel on the (zero-dilated, for stride 2) output gradient with flipped / transposed weights; weight and bias
                    gradient = rnc_conv2d_cl_wgrad
    CorrPyramid     CorrBlock.__init__ on features (corr.py:7-21): rnc_fmap_pyramid / adjoint rnc_pyramid_pool_bwd
    CorrLookup      CorrBlock.__call__ (corr.py:23-44): rnc_corr_lookup_fwd / rnc_corr_lookup_bwd (d fmap1, d fmap2 pyramid; coords
                    are detached, raft_nc_dbl.py:149)
    NConv2dFn       NConv2d.forward (nconv_modules.py:164-199): rnc_nconv2d_fwd / rnc_nconv2d_bwd (quotient rule, confidence path)

Activations stay channel-last ([B, H, W, C] fp32) between convolutions.  Pointwise glue (ReLU / sigmoid / tanh / gate blend,
cat, nearest x2, zero-stuffing, the loss) and the normalisation layers (InstanceNorm / BatchNorm: library kernels, like cuDNN
in the reference) are plain torch ops — plumbing around the kernels above.  `sequence_loss`, `fetch_optimizer` and
`train_step` restate train.py:46-71, :83-99, :203-227; `ddp_model` replaces nn.DataParallel (train.py:169-175) with one
process per GPU and a bucketed NCCL all-reduce of the 4.9 M fp32 gradients.
"""
import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import native
from .engine import CORR_CH, ConvDesc, _ptr, _require_cuda, _stream, engine_for, pack_conv

_PACK_CACHE = {}          # (id(weight), version, kind, cin_pad) -> (weight, packed); flushed at the start of every training forward


def _packed(weight, kind, cin_pad):
    """Kernel-ready copy of a convolution weight ('fwd') or of its flipped transpose ('dgrad'), cached for the 12 iterations of a
    step.  The entry keeps the weight tensor alive, so neither its id nor its storage can be recycled while the entry exists."""
    key = (id(weight), weight._version, kind, cin_pad)
    hit = _PACK_CACHE.get(key)
    if hit is None or hit[0] is not weight:
        if len(_PACK_CACHE) > 512:
            _PACK_CACHE.clear()
        w = weight.detach()
        if kind == "dgrad":          # Wd[ci, co, ky, kx] = W[co, ci, kh-1-ky, kw-1-kx]
            w = w.flip(2, 3).transpose(0, 1)
        hit = _PACK_CACHE[key] = (weight, pack_conv(w.contiguous(), None, cin_pad=cin_pad))
    return hit[1]


def _ceil4(c):
    return (c + 3) // 4 * 4


def _conv_mode():
    """RNC_TRAIN_CONV selects how the training path's convolutions (forward and data gradient) run:
      ffma (default)  exact fp32 on CUDA cores (rnc_conv2d_cl_fwd): per-layer error 1.5e-7; every non-fnet parameter's gradient
                      within 1e-3 of the reference's autograd (cfg 5 step on B200: 149 ms)
      tf32            tcgen05 kind::tf32 on TF32 hi/lo operand planes, 3 MMAs per K step (x_hi*w_hi + x_hi*w_lo + x_lo*w_hi):
                      ~2^-21 per product (per-layer 1e-6 .. 5e-6) with fp32's exponent range, so output gradients of 1e-9
                      survive; 112 ms per step, ill-conditioned parameters (cnet.conv1) move to 5e-3
      umma            fp16 hi/lo split operands (the inference kernels): output gradients underflow the split's normal range —
                      per-parameter gradient errors of 5e-3 (forward only) to 4e-2 (with RNC_TRAIN_DGRAD=umma)
    The weight gradient runs on the CUDA cores (rnc_conv2d_cl_wgrad) unless RNC_TRAIN_WGRAD=tf32 qualifies the tf32 form: then
    the layers _wgrad_umma_ok names run it as rnc_conv2d_umma_wgrad (tcgen05 TF32x3, K = pixels in chunks of 512), so that every
    wide convolution of the step runs on the tensor cores.  RNC_TRAIN_WGRAD has no effect under ffma or umma.
    Parity first: the default is the exact path; the tensor-core forms are opt-in and reported beside it by bench.py."""
    import os
    return os.environ.get("RNC_TRAIN_CONV", "ffma")


def _umma_ok(eng, Cx, cout, dgrad=False):
    """Can this layer run on the tensor-core convolution?  The kernel stores whole 32-channel chunks of fp32 output, so the
    output row must not need wider padding than the channel-last tensors use; the fp16 form also needs a pitch of 8 halves."""
    import os
    mode = _conv_mode()
    if eng.mode != "umma" or mode == "ffma" or (cout + 31) // 32 * 32 != _ceil4(cout):
        return None
    if mode == "tf32":
        return "tf32" if Cx % 4 == 0 else None
    if dgrad and os.environ.get("RNC_TRAIN_DGRAD", "ffma") != "umma":
        return None
    return "f16" if Cx % 8 == 0 and Cx >= 32 and cout >= 32 else None


def _wgrad_umma_ok(eng, Cx, cout):
    """Does this layer's weight gradient run on the tensor cores (rnc_conv2d_umma_wgrad)?  Only when RNC_TRAIN_WGRAD=tf32 and the
    layer's forward runs in the TF32 form.  The rule is a function of the layer's shape: narrow layers (FlowHead.conv2 256->2,
    Simple.out 32->2, the 4-channel 7x7 stems and convf1) would fill a fraction of a 128 x N tile and stay on the CUDA cores;
    every layer it sends to the tensor cores is faster there at config 5 (tools/wgrad_probe.py, profiles/r03_wgrad.json)."""
    import os
    if os.environ.get("RNC_TRAIN_WGRAD", "ffma") != "tf32" or _umma_ok(eng, Cx, cout) != "tf32":
        return False
    return cout >= 32 and Cx >= 16


class _WeightsTF32:
    """[Cout,Cin,KH,KW] -> TF32 hi/lo planes of floats [CoutPad][taps * blocks * 32] (hi = round-to-nearest TF32, lo = w - hi), the
    operand format of RNC_CONV_TF32 layers; no scaling is needed (fp32 exponent range)."""

    def __init__(self, w, cin_pad):
        from .engine_umma import _coutpad
        cout, cin, kh, kw = w.shape
        nblk = (cin_pad + 31) // 32
        self.cout, self.kh, self.kw = cout, kh, kw
        self.coutpad = _coutpad(cout)
        self.ktot = kh * kw * nblk * 32
        wp = torch.zeros(self.coutpad, kh * kw, nblk * 32, dtype=torch.float32, device=w.device)
        wp[:cout, :, :cin] = w.permute(0, 2, 3, 1).reshape(cout, kh * kw, cin)
        ws = wp.reshape(self.coutpad, self.ktot)
        self.w_hi = ((ws.view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32).contiguous()
        self.w_lo = (ws - self.w_hi).contiguous()
        self.unscale = 1.0
        self.bias = torch.zeros(self.coutpad, dtype=torch.float32, device=w.device)


def _packed_umma(weight, kind, cin_pad, fmt="f16"):
    from .engine_umma import UmmaWeights
    key = (id(weight), weight._version, kind + "_" + fmt, cin_pad)
    hit = _PACK_CACHE.get(key)
    if hit is None or hit[0] is not weight:
        w = weight.detach().float()
        if kind == "dgrad":
            w = w.flip(2, 3).transpose(0, 1)
        if fmt == "tf32":
            packed = _WeightsTF32(w.contiguous(), cin_pad)
        else:
            if w.shape[1] != cin_pad:
                w = F.pad(w, (0, 0, 0, 0, 0, cin_pad - w.shape[1]))
            # fixed scale 2^10 (no device sync per pack): exact for |w| < 32; a lo part below the half normal range only costs an
            # absolute 2^-34 per weight
            packed = UmmaWeights(w.contiguous(), None, [cin_pad], scale_log2=10)
        hit = _PACK_CACHE[key] = (weight, packed)
    return hit[1]


def _conv_launch_umma(eng, x, wt, cout, stride=1, bias=None, fmt="f16"):
    """Same contract as _conv_launch on the tcgen05 path: x fp32 CL -> hi/lo operand planes (halves or TF32 words) ->
    rnc_conv2d_umma_fwd with an fp32 channel-last output; stride 2 is native (TMA element strides), no subsampling pass."""
    B, H, W, Cx = x.shape
    Ho, Wo = (H + stride - 1) // stride, (W + stride - 1) // stride
    M = B * H * W
    dt = torch.float32 if fmt == "tf32" else torch.float16
    hi = torch.empty(M, Cx, dtype=dt, device=x.device)
    lo = torch.empty(M, Cx, dtype=dt, device=x.device)
    split = eng.L.rnc_f32_to_tf32_split if fmt == "tf32" else eng.L.rnc_f32_to_split
    native.check(split(_ptr(x), Cx, Cx, M, _ptr(hi), _ptr(lo), Cx, 0, _stream()), "operand split")
    ldo = _ceil4(cout)
    out = torch.empty(B, Ho, Wo, ldo, dtype=torch.float32, device=x.device)
    if bias is not None:
        wt = _WithBias(wt, bias)
    eng.uconv(B, Ho, Wo, (hi.data_ptr(), lo.data_ptr()), Cx, Cx, wt, native.EPI_LINEAR, out_f32=out.data_ptr(), ldo_f32=ldo,
              stride=stride, hin=H, win=W, flags=eng.conv_flags | (native.CONV_TF32 if fmt == "tf32" else 0))
    return out


class _WithBias:
    """A packed weight with this call's bias vector (the pack is cached per weight; biases are tiny and change with it)."""

    def __init__(self, wt, bias):
        self.__dict__.update(wt.__dict__)
        b = torch.zeros_like(wt.bias)
        b[:wt.cout] = bias.detach()
        self.bias = b


def _conv_launch(eng, x, packed, cout, kh, kw, bias=None):
    """x CL [B,H,W,C] contiguous (C % 4 == 0) -> CL [B,H,W,ceil4(cout)] (pad channels zero), stride 1, zero padding k/2."""
    B, H, W, Cx = x.shape
    ldo = _ceil4(cout)
    alloc = torch.empty if ldo == cout else torch.zeros          # pad channels must read as zero downstream
    out = alloc(B, H, W, ldo, dtype=torch.float32, device=x.device)
    w, b = packed
    if bias is not None:
        b = torch.zeros_like(b)
        b[:cout] = bias.detach()
    d = ConvDesc()
    d.in0, d.c0, d.ld0 = x.data_ptr(), Cx, Cx
    d.in1, d.c1, d.ld1 = 0, 0, 0
    d.weight, d.bias = w.data_ptr(), b.data_ptr()
    d.out, d.ldo = out.data_ptr(), ldo
    d.B, d.H, d.W = B, H, W
    d.cout, d.kh, d.kw, d.epilogue = cout, kh, kw, native.EPI_LINEAR
    native.check(eng.L.rnc_conv2d_cl_fwd(C.byref(d), _stream()), "conv2d_cl")
    return out


class ConvCL(torch.autograd.Function):
    """y = conv2d(x, weight, bias, stride, padding = k // 2) on channel-last tensors.
    x [B,H,W,Cx] (Cx = ceil4(Cin); channels beyond Cin must be zero), weight [Cout,Cin,kh,kw] -> y [B,Ho,Wo,ceil4(Cout)]."""

    @staticmethod
    def forward(ctx, x, weight, bias, stride):
        x = x.contiguous()
        eng = engine_for(x.device)
        cout, cin, kh, kw = weight.shape
        Cx = x.shape[-1]
        if Cx % 4 or Cx < cin:
            raise ValueError("ConvCL: input must be channel-last with ceil4(Cin) channels")
        if stride not in (1, 2):
            raise NotImplementedError("stride 1 or 2")
        fmt = _umma_ok(eng, Cx, cout)
        if fmt:
            y = _conv_launch_umma(eng, x, _packed_umma(weight, "fwd", Cx, fmt), cout, stride, bias, fmt)
        else:
            y = _conv_launch(eng, x, _packed(weight, "fwd", Cx), cout, kh, kw, bias)
            if stride == 2:
                y = y[:, ::2, ::2].contiguous()      # same padding: out(y, x) of the strided conv = full(2y, 2x)
        ctx.save_for_backward(x, weight)
        ctx.stride, ctx.has_bias = stride, bias is not None
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight = ctx.saved_tensors
        eng = engine_for(x.device)
        cout, cin, kh, kw = weight.shape
        B, H, W, Cx = x.shape
        gy = gy.contiguous()
        ldg = gy.shape[-1]
        gx = gw = gb = None
        with torch.cuda.device(x.device):
            if ctx.needs_input_grad[0]:
                g_full = gy
                if ctx.stride == 2:
                    g_full = torch.zeros(B, H, W, ldg, dtype=torch.float32, device=x.device)
                    g_full[:, ::2, ::2] = gy
                fmt = _umma_ok(eng, ldg, cin, dgrad=True)
                if fmt:
                    gx = _conv_launch_umma(eng, g_full, _packed_umma(weight, "dgrad", ldg, fmt), cin, fmt=fmt)
                else:
                    gx = _conv_launch(eng, g_full, _packed(weight, "dgrad", ldg), cin, kh, kw)
                if gx.shape[-1] != Cx:               # Cx > ceil4(cin) never happens; equal by construction
                    gx = F.pad(gx, (0, Cx - gx.shape[-1]))
            if ctx.needs_input_grad[1] or (ctx.has_bias and ctx.needs_input_grad[2]):
                gwp = torch.zeros(kh * kw, Cx, cout, dtype=torch.float32, device=x.device)
                gbp = torch.zeros(cout, dtype=torch.float32, device=x.device) if ctx.has_bias else None
                if _wgrad_umma_ok(eng, Cx, cout):
                    nbytes = eng.L.rnc_conv2d_umma_wgrad_workspace_bytes(Cx, cout, B, H, W, kh, kw, ctx.stride)
                    ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=x.device)
                    native.check(eng.L.rnc_conv2d_umma_wgrad(_ptr(x), Cx, Cx, _ptr(gy), ldg, cout, B, H, W, kh, kw, ctx.stride,
                                                             _ptr(gwp), cout, _ptr(gbp), _ptr(ws), ws.numel() * 4, _stream()),
                                 "conv2d_umma_wgrad")
                else:
                    native.check(eng.L.rnc_conv2d_cl_wgrad(_ptr(x), Cx, Cx, _ptr(gy), ldg, cout, B, H, W, kh, kw, ctx.stride,
                                                           _ptr(gwp), cout, _ptr(gbp), _stream()), "conv2d_cl_wgrad")
                gw = gwp.view(kh, kw, Cx, cout)[:, :, :cin].permute(3, 2, 0, 1).contiguous()
                gb = gbp
        return gx, gw, gb, None


def conv_cl(x, conv, stride=None):
    """nn.Conv2d `conv` (zero padding k // 2, as every convolution of the reference) on a channel-last tensor."""
    s = conv.stride[0] if stride is None else stride
    y = ConvCL.apply(x, conv.weight, conv.bias, s)
    return y


def to_cl(x, pad_to=None):
    """NCHW -> contiguous channel-last, channels zero-padded to a multiple of 4 (or to pad_to)."""
    y = x.permute(0, 2, 3, 1)
    c = y.shape[-1]
    tgt = pad_to or _ceil4(c)
    if tgt != c:
        y = F.pad(y, (0, tgt - c))
    return y.contiguous()


def to_nchw(x, c=None):
    y = x if c is None else x[..., :c]
    return y.permute(0, 3, 1, 2).contiguous()


# --------------------------------------------------------------------------------------------- correlation


class CorrPyramid(torch.autograd.Function):
    """fmap2 (CL) -> pooled feature pyramid (corr.py:18-21 on features; SURVEY.md finding 7).  Output: flat pyramid buffer."""

    @staticmethod
    def forward(ctx, fmap2_cl, levels):
        eng = engine_for(fmap2_cl.device)
        B, H, W, D = fmap2_cl.shape
        total = eng.L.rnc_pyramid_offset(B, D, H, W, levels)
        pyr = torch.empty(total, dtype=torch.float32, device=fmap2_cl.device)
        pyr[:B * H * W * D] = fmap2_cl.reshape(-1)
        native.check(eng.L.rnc_fmap_pyramid(_ptr(pyr), B, D, H, W, levels, _stream()), "fmap_pyramid")
        ctx.dims = (B, H, W, D, levels)
        return pyr

    @staticmethod
    def backward(ctx, g_pyr):
        B, H, W, D, levels = ctx.dims
        eng = engine_for(g_pyr.device)
        g = g_pyr.clone()
        with torch.cuda.device(g.device):
            native.check(eng.L.rnc_pyramid_pool_bwd(_ptr(g), B, D, H, W, levels, _stream()), "pyramid_pool_bwd")
        return g[:B * H * W * D].view(B, H, W, D), None


class CorrLookup(torch.autograd.Function):
    """corr.py:23-44 on (fmap1 CL, fmap2 pyramid): -> CL [B,H,W,324] in the reference channel order."""

    @staticmethod
    def forward(ctx, f1_cl, f2_pyr, coords, levels):
        eng = engine_for(f1_cl.device)
        B, H, W, D = f1_cl.shape
        coords = coords.detach().float().contiguous()
        out = torch.empty(B, H, W, CORR_CH, dtype=torch.float32, device=f1_cl.device)
        native.check(eng.L.rnc_corr_lookup_fwd(_ptr(f1_cl), _ptr(f2_pyr), _ptr(coords), B, D, H, W, levels, 4, _ptr(out), 1, CORR_CH,
                                               _stream()), "corr_lookup")
        ctx.save_for_backward(f1_cl, f2_pyr, coords)
        ctx.levels = levels
        return out

    @staticmethod
    def backward(ctx, g_out):
        f1_cl, f2_pyr, coords = ctx.saved_tensors
        eng = engine_for(f1_cl.device)
        B, H, W, D = f1_cl.shape
        g_out = g_out.contiguous()
        with torch.cuda.device(f1_cl.device):
            g_f1 = torch.empty_like(f1_cl)
            g_f2 = torch.zeros_like(f2_pyr)
            native.check(eng.L.rnc_corr_lookup_bwd(_ptr(f1_cl), _ptr(f2_pyr), _ptr(coords), _ptr(g_out), g_out.shape[-1], B, D, H, W,
                                                   ctx.levels, 4, _ptr(g_f1), _ptr(g_f2), _stream()), "corr_lookup_bwd")
        return g_f1, g_f2, None, None


def corr_lookup_autograd(corr_block, coords):
    """Seam CorrBlock.__call__ with gradients to the NCHW feature maps it was built from."""
    f1 = to_cl(corr_block.fmap1.float())
    pyr = CorrPyramid.apply(to_cl(corr_block.fmap2.float()), corr_block.num_levels)
    out = CorrLookup.apply(f1, pyr, coords, corr_block.num_levels)
    return to_nchw(out)


# --------------------------------------------------------------------------------------------- normalized convolution


class NConv2dFn(torch.autograd.Function):
    """(data, conf, W > 0) -> (nconv, conf_out), nconv_modules.py:164-199."""

    @staticmethod
    def forward(ctx, data, conf, weight, eps):
        eng = engine_for(data.device)
        data, conf, weight = data.contiguous(), conf.contiguous(), weight.contiguous()
        N, Cin, H, W = data.shape
        Cout, _, kh, kw = weight.shape
        y = torch.empty(N, Cout, H, W, dtype=torch.float32, device=data.device)
        c = torch.empty_like(y)
        native.check(eng.L.rnc_nconv2d_fwd(_ptr(data), _ptr(conf), _ptr(weight), N, Cin, Cout, H, W, kh, kw, eps, _ptr(y), _ptr(c),
                                           _stream()), "nconv2d")
        ctx.save_for_backward(data, conf, weight, y, c)
        ctx.eps = eps
        return y, c

    @staticmethod
    def backward(ctx, gy, gc):
        data, conf, weight, y, c = ctx.saved_tensors
        eng = engine_for(data.device)
        N, Cin, H, W = data.shape
        Cout, _, kh, kw = weight.shape
        with torch.cuda.device(data.device):
            nbytes = eng.L.rnc_nconv2d_bwd_workspace_bytes(N, Cout, H, W)
            ws = torch.zeros((nbytes + 7) // 8, dtype=torch.float64, device=data.device)
            g_data = torch.empty_like(data) if ctx.needs_input_grad[0] else None
            g_conf = torch.empty_like(conf) if ctx.needs_input_grad[1] else None
            g_w = torch.empty_like(weight) if ctx.needs_input_grad[2] else None
            native.check(eng.L.rnc_nconv2d_bwd(_ptr(data), _ptr(conf), _ptr(weight), _ptr(y), _ptr(c),
                                               _ptr(gy.contiguous()) if gy is not None else None,
                                               _ptr(gc.contiguous()) if gc is not None else None, N, Cin, Cout, H, W, kh, kw, ctx.eps,
                                               _ptr(g_data), _ptr(g_conf), _ptr(g_w), _ptr(ws), ws.numel() * 8, _stream()), "nconv2d_bwd")
        return g_data, g_conf, g_w, None


def nconv2d_autograd(data, conf, weight, eps=1e-20):
    _require_cuda(data, conf, weight)
    return NConv2dFn.apply(data.float(), conf.float(), weight.float(), eps)


# --------------------------------------------------------------------------------------------- module graphs (channel-last)


def _norm_cl(x, norm):
    """InstanceNorm2d / BatchNorm2d / identity on a channel-last tensor (library kernels on a strided NCHW view)."""
    if isinstance(norm, nn.Sequential) and len(norm) == 0:
        return x
    v = x.permute(0, 3, 1, 2)
    if isinstance(norm, nn.InstanceNorm2d):
        v = F.instance_norm(v, eps=norm.eps)
    elif isinstance(norm, nn.BatchNorm2d):
        v = F.batch_norm(v, norm.running_mean, norm.running_var, norm.weight, norm.bias, norm.training, norm.momentum, norm.eps)
    else:
        raise NotImplementedError(type(norm).__name__)
    return v.permute(0, 2, 3, 1).contiguous()


def res_block_cl(blk, x):
    """extractor.py:6-56."""
    y = F.relu(_norm_cl(conv_cl(x, blk.conv1), blk.norm1))
    y = F.relu(_norm_cl(conv_cl(y, blk.conv2), blk.norm2))
    if blk.downsample is not None:
        x = _norm_cl(conv_cl(x, blk.downsample[0]), blk.downsample[1])
    return F.relu(x + y)


def encoder_cl(enc, x_cl):
    """BasicEncoder.forward (extractor.py:160-192) on a channel-last image batch [N,H,W,4] (3 channels + 1 zero)."""
    x = F.relu(_norm_cl(conv_cl(x_cl, enc.conv1), enc.norm1))
    for layer in (enc.layer1, enc.layer2, enc.layer3):
        for blk in layer:
            x = res_block_cl(blk, x)
    x = conv_cl(x, enc.conv2)
    if enc.training and enc.dropout is not None:
        x = enc.dropout(x.permute(0, 3, 1, 2)).permute(0, 2, 3, 1).contiguous()
    return x


def motion_encoder_cl(e, flow_cl, corr_cl):
    """update.py:89-97; flow_cl [B,H,W,4] (2 + 2 zero channels) -> [B,H,W,128] = cat(conv out 126, flow 2)."""
    cor = F.relu(conv_cl(corr_cl, e.convc1))
    cor = F.relu(conv_cl(cor, e.convc2))
    flo = F.relu(conv_cl(flow_cl, e.convf1))
    flo = F.relu(conv_cl(flo, e.convf2))
    out = F.relu(conv_cl(torch.cat([cor, flo], -1), e.conv))          # [B,H,W,128]: channels 126, 127 are zero pads
    return torch.cat([out[..., :126], flow_cl[..., :2]], -1)


def sep_conv_gru_cl(g, h, x):
    """update.py:45-60 on channel-last h [.,128], x [.,256]."""
    for tag in ("1", "2"):
        hx = torch.cat([h, x], -1)
        z = torch.sigmoid(conv_cl(hx, getattr(g, "convz" + tag)))
        r = torch.sigmoid(conv_cl(hx, getattr(g, "convr" + tag)))
        q = torch.tanh(conv_cl(torch.cat([r * h, x], -1), getattr(g, "convq" + tag)))
        h = (1 - z) * h + z * q
    return h


def flow_head_cl(fh, net):
    """update.py:13-14 -> [B,H,W,4] (delta in channels 0, 1)."""
    return conv_cl(F.relu(conv_cl(net, fh.conv1)), fh.conv2)


def update_block_cl(ub, net, inp, corr, flow_cl):
    """update.py:130-141 on channel-last tensors: returns (net, mask or None, delta [B,H,W,4])."""
    motion = motion_encoder_cl(ub.encoder, flow_cl, corr)
    net = sep_conv_gru_cl(ub.gru, net, torch.cat([inp, motion], -1))
    delta = flow_head_cl(ub.flow_head, net)
    mask = None
    if len(ub.mask) > 0:
        mask = 0.25 * conv_cl(F.relu(conv_cl(net, ub.mask[0])), ub.mask[2])
    return net, mask, delta


def simple_cl(wn, x_cl):
    """Simple.forward (interp_weights_est.py:39-47) on channel-last input [B,h,w,132] -> NCHW [B,2,h,w] after final_act."""
    x = x_cl
    for blk in wn.conv:
        x = conv_cl(x, blk[0])
        if len(blk) == 3:
            x = _norm_cl(x, blk[1])
        x = F.relu(x)
    x = conv_cl(x, wn.out)
    return wn.final_act(to_nchw(x, wn.out.out_channels))


def nconv_unet_train(net, data, conf):
    """NConvUNet.forward live path (nconv_modules.py:106-136, SURVEY.md Appendix A.3) with autograd."""
    x, c = NConv2dFn.apply(data, conf, net.nconv_in.weight, net.nconv_in.eps)
    x, c = NConv2dFn.apply(x, c, net.nconv_x2[0].weight, net.nconv_x2[0].eps)
    x, c = NConv2dFn.apply(torch.cat((x, x), 1), torch.cat((c, c), 1), net.decoder[0].weight, net.decoder[0].eps)
    return NConv2dFn.apply(x, c, net.nconv_out.weight, net.nconv_out.eps)


def zero_stuff(x, scale=4):
    """upsampler.py:179-210: zeros [B,C,s*h,s*w] with out[..., s//2::s, s//2::s] = x."""
    b, c, h, w = x.shape
    out = torch.zeros(b, c, h * scale, w * scale, dtype=x.dtype, device=x.device)
    out[:, :, scale // 2::scale, scale // 2::scale] = x
    return out


def ncup_upsampler_train(up, x_lowres, x_guidance, out_scale=1.0):
    """NConvUpsampler.forward (upsampler.py:143-177) with autograd: x_lowres NCHW [B,2,h,w], guidance NCHW [B,128,h/2,w/2]."""
    _require_cuda(x_lowres, x_guidance)
    with torch.cuda.device(x_lowres.device):
        g4 = F.interpolate(x_guidance, x_lowres.shape[2:], mode="area")           # integer x2 'area' upscale = replication
        w4 = simple_cl(up.weights_est_net, to_cl(torch.cat([x_lowres, g4], 1), pad_to=136))     # pitch % 8 == 0: tensor-core layer
        xh, wh = zero_stuff(x_lowres), zero_stuff(w4)
        b, c, oh, ow = xh.shape
        out, _ = nconv_unet_train(up.interpolation_net, xh.view(b * c, 1, oh, ow), wh.view(b * c, 1, oh, ow))
        out = out.view(b, c, oh, ow)
        return out * out_scale if out_scale != 1.0 else out


def simple_train(wn, x):
    with torch.cuda.device(x.device):
        return simple_cl(wn, to_cl(x.float()))


def flow_head_train(fh, x):
    with torch.cuda.device(x.device):
        return to_nchw(flow_head_cl(fh, to_cl(x.float())), 2)


def sep_conv_gru_train(g, h, x):
    with torch.cuda.device(h.device):
        return to_nchw(sep_conv_gru_cl(g, to_cl(h.float()), to_cl(x.float())))


def motion_encoder_train(e, flow, corr):
    with torch.cuda.device(flow.device):
        return to_nchw(motion_encoder_cl(e, to_cl(flow.float()), to_cl(corr.float())))


def update_block_train(ub, net, inp, corr, flow):
    """BasicUpdateBlock.forward (update.py:130-141) with autograd, NCHW in / out."""
    with torch.cuda.device(net.device):
        n, m, d = update_block_cl(ub, to_cl(net.float()), to_cl(inp.float()), to_cl(corr.float()), to_cl(flow.float()))
        net_out = to_nchw(n)
        ub.net = net_out
        mask = to_nchw(m) if m is not None else 0.25 * net_out
        return net_out, mask, to_nchw(d, 2)


def convex_upsample_train(flow, mask):
    """raft.py:73-84 (model `raft`), pointwise torch ops: softmax over the 9 neighbours x unfold(8 * flow)."""
    n, _, h, w = flow.shape
    m = torch.softmax(mask.view(n, 1, 9, 8, 8, h, w), dim=2)
    nb = F.unfold(8 * flow, [3, 3], padding=1).view(n, 2, 9, 1, 1, h, w)
    up = torch.sum(m * nb, dim=2).permute(0, 1, 4, 2, 5, 3)
    return up.reshape(n, 2, 8 * h, 8 * w)


def raft_forward_train(model, image1, image2, iters=12, flow_init=None, test_mode=False):
    """RAFT.forward with autograd (raft_nc_dbl.py:115-173 / raft.py:87-143): returns the list of `iters` full-resolution
    predictions (or (flow_low, flow_up) in test_mode)."""
    _PACK_CACHE.clear()
    B, _, Him, Wim = image1.shape
    H8, W8 = Him // 8, Wim // 8
    dev = image1.device
    im1 = 2 * (image1.float() / 255.0) - 1.0
    im2 = 2 * (image2.float() / 255.0) - 1.0
    fmaps = encoder_cl(model.fnet, to_cl(torch.cat([im1, im2], 0))).float()       # [2B,H8,W8,256]
    f1, f2 = fmaps[:B].contiguous(), fmaps[B:].contiguous()
    pyr = CorrPyramid.apply(f2, 4)
    cnet = encoder_cl(model.cnet, to_cl(im1))
    net, inp = torch.tanh(cnet[..., :128]), torch.relu(cnet[..., 128:])
    ys, xs = torch.meshgrid(torch.arange(H8, device=dev), torch.arange(W8, device=dev), indexing="ij")
    coords0 = torch.stack([xs, ys], 0).float()[None].repeat(B, 1, 1, 1)
    coords1 = coords0.clone()
    if flow_init is not None:
        coords1 = coords1 + flow_init
    preds = []
    ub = model.update_block
    for _ in range(iters):
        coords1 = coords1.detach()                                                  # raft_nc_dbl.py:149
        corr = CorrLookup.apply(f1, pyr, coords1, 4)
        flow = coords1 - coords0
        net, mask, delta = update_block_cl(ub, net, inp, corr, to_cl(flow))
        ub.net = net                                                                # guidance tap (update.py:135), channel-last here
        coords1 = coords1 + to_nchw(delta, 2)
        flow_lr = coords1 - coords0
        if model.ncup:
            x4 = F.interpolate(flow_lr, scale_factor=2, mode="nearest")             # raft_nc_dbl.py:110
            flow_up = 8 * ncup_upsampler_train(model.upsampler, x4, to_nchw(net))   # raft_nc_dbl.py:161
        else:
            flow_up = convex_upsample_train(flow_lr, to_nchw(mask))
        preds.append(flow_up)
    ub.net = to_nchw(net)
    if test_mode:
        return coords1 - coords0, preds[-1]
    return preds


# --------------------------------------------------------------------------------------------- loss / optimiser / step (train.py)

MAX_FLOW = 400


def sequence_loss(flow_preds, flow_gt, valid, gamma=0.8, max_flow=MAX_FLOW):
    """train.py:46-71 — gamma-weighted L1 over the prediction sequence; invalid pixels count in the mean's denominator."""
    n = len(flow_preds)
    mag = torch.sum(flow_gt ** 2, dim=1).sqrt()
    valid = (valid >= 0.5) & (mag < max_flow)
    loss = 0.0
    for i, pred in enumerate(flow_preds):
        loss = loss + gamma ** (n - i - 1) * (valid[:, None] * (pred - flow_gt).abs()).mean()
    epe = torch.sum((flow_preds[-1] - flow_gt) ** 2, dim=1).sqrt().view(-1)[valid.view(-1)]
    metrics = {"epe": epe.mean().item(), "1px": (epe < 1).float().mean().item(), "3px": (epe < 3).float().mean().item(),
               "5px": (epe < 5).float().mean().item()}
    return loss, metrics


def fetch_optimizer(model, lr=2e-5, wdecay=5e-5, epsilon=1e-8, num_steps=100000):
    """train.py:83-99 (the shipped scripts: AdamW + OneCycleLR, linear anneal, pct_start 0.05, no momentum cycling)."""
    opt = torch.optim.AdamW(model.parameters(), lr=lr, weight_decay=wdecay, eps=epsilon)
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, lr, num_steps + 100, pct_start=0.05, cycle_momentum=False, anneal_strategy="linear")
    return opt, sched


def train_step(model, optimizer, scheduler, image1, image2, flow_gt, valid, iters=12, gamma=0.85, clip=1.0, return_metrics=True):
    """One optimisation step exactly as train.py:203-227 without AMP: zero_grad, forward (list of predictions), sequence_loss,
    backward (under DistributedDataParallel: gradient all-reduce overlapped with it), clip_grad_norm_(clip), step."""
    optimizer.zero_grad()
    preds = model(image1, image2, iters=iters)
    loss, metrics = sequence_loss(preds, flow_gt, valid, gamma)
    loss.backward()
    torch.nn.utils.clip_grad_norm_(model.parameters(), clip)
    optimizer.step()
    if scheduler is not None:
        scheduler.step()
    return loss.detach(), (metrics if return_metrics else None)


def ddp_model(model, device, bucket_cap_mb=8):
    """train.py:169-175 wraps the model in single-process nn.DataParallel; here: one process per GPU, replicas kept in sync by
    DistributedDataParallel's bucketed NCCL all-reduce of the gradients (19.6 MB fp32; every parameter receives a gradient,
    SURVEY.md Appendix G, so no unused-parameter search).  The NConv encoder aliases are one Parameter object: DDP sees it once."""
    from torch.nn.parallel import DistributedDataParallel as DDP
    return DDP(model.to(device), device_ids=[device.index], bucket_cap_mb=bucket_cap_mb, broadcast_buffers=False,
               gradient_as_bucket_view=True)
