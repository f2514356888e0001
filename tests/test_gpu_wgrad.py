"""Tensor-core weight gradient of the training path (rnc_conv2d_umma_wgrad, tcgen05 TF32x3, K = pixels) against fp64, through the
C ABI.  Each error test prints the CUDA-core kernel's (rnc_conv2d_cl_wgrad, exact fp32) own distance to fp64 beside the new
kernel's as a yardstick."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from conftest import build_model
from oracle import raft_oracle as orc
from oracle.make_golden_r2 import GRAD_ITERS, tied_leaves, train_inputs

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def L():
    from rnc import native
    return native.lib()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def p(t):
    return C.c_void_p(t.data_ptr() if t is not None else 0)


def rel(a, b):
    return ((a.double().cpu() - b.double().cpu()).norm() / (b.double().cpu().norm() + 1e-300)).item()


def ws_bytes(cin, cout, B, H, W, kh, kw, s):
    return L().rnc_conv2d_umma_wgrad_workspace_bytes(cin, cout, B, H, W, kh, kw, s)


def call(kind, x, cin, gy, cout, kh, kw, s, gw, gb, ldw=None, ws=None, nbytes=None):
    """x [B,H,W,ldx], gy [B,Ho,Wo,ldg] CL fp32 on the GPU; gw [taps,cin,ldw] and gb [cout] accumulate."""
    B, H, W, ldx = x.shape
    ldg = gy.shape[-1]
    ldw = gw.shape[-1] if ldw is None else ldw
    if kind == "ffma":
        return L().rnc_conv2d_cl_wgrad(p(x), ldx, cin, p(gy), ldg, cout, B, H, W, kh, kw, s, p(gw), ldw, p(gb), stream())
    if ws is None:
        n = ws_bytes(cin, cout, B, H, W, kh, kw, s)
        ws = torch.empty((n + 15) // 16 * 4, dtype=torch.float32, device=DEV)
        nbytes = n
    return L().rnc_conv2d_umma_wgrad(p(x), ldx, cin, p(gy), ldg, cout, B, H, W, kh, kw, s, p(gw), ldw, p(gb), p(ws), nbytes, stream())


def problem(cin, cout, kh, kw, s, B, H, W, seed, positive=False, gscale=1.0):
    g = torch.Generator().manual_seed(seed)
    Ho, Wo = (H + s - 1) // s, (W + s - 1) // s
    if positive:
        x, gy = torch.rand(B, cin, H, W, generator=g), torch.rand(B, cout, Ho, Wo, generator=g)
    else:
        x, gy = torch.randn(B, cin, H, W, generator=g), torch.randn(B, cout, Ho, Wo, generator=g)
    return x, gy * gscale


def reference(x, gy, cout, kh, kw, s, device="cpu"):
    """fp64 autograd of conv2d (zero padding k // 2): d loss / d w, d loss / d b."""
    cin = x.shape[1]
    xr = x.double().to(device)
    wr = torch.zeros(cout, cin, kh, kw, dtype=torch.float64, device=device, requires_grad=True)
    br = torch.zeros(cout, dtype=torch.float64, device=device, requires_grad=True)
    F.conv2d(xr, wr, br, stride=s, padding=(kh // 2, kw // 2)).backward(gy.double().to(device))
    return wr.grad.cpu(), br.grad.cpu()


def to_cl(t, ld=None):
    y = t.permute(0, 2, 3, 1)
    if ld is not None and ld != y.shape[-1]:
        y = F.pad(y, (0, ld - y.shape[-1]))
    return y.contiguous().to(DEV)


def unpack(gw, cout, kh, kw):
    taps, cin, ldw = gw.shape
    return gw.view(kh, kw, cin, ldw)[..., :cout].permute(3, 2, 0, 1).cpu()


def both(x, gy, cout, kh, kw, s):
    """(dw, db) of both kernels, from zero-filled outputs."""
    cin = x.shape[1]
    xc, gc = to_cl(x), to_cl(gy, (cout + 3) // 4 * 4)           # gy rows padded to 4 floats, as ConvCL passes them
    out = {}
    for kind in ("ffma", "tf32"):
        gw = torch.zeros(kh * kw, cin, cout, device=DEV)
        gb = torch.zeros(cout, device=DEV)
        assert call(kind, xc, cin, gc, cout, kh, kw, s, gw, gb) == 0, kind
        torch.cuda.synchronize()
        out[kind] = (unpack(gw, cout, kh, kw), gb.cpu())
    return out


# every wide convolution shape of the training graph (cin, cout, kh, kw, stride)
LAYERS = [(324, 256, 1, 1, 1), (256, 192, 3, 3, 1), (128, 64, 3, 3, 1), (256, 126, 3, 3, 1), (384, 128, 1, 5, 1), (384, 128, 5, 1, 1),
          (128, 256, 3, 3, 1), (64, 64, 3, 3, 1), (64, 96, 3, 3, 2), (64, 96, 1, 1, 2), (96, 128, 3, 3, 2), (128, 256, 1, 1, 1),
          (136, 64, 3, 3, 1), (64, 32, 3, 3, 1), (256, 576, 1, 1, 1), (192, 128, 1, 1, 1)]
# odd H and W with Wo a ragged multiple of 32 (B = 3), and Wo < 32
SIZES = [(3, 13, 77), (2, 9, 21)]


@pytest.mark.parametrize("size", SIZES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("cin,cout,kh,kw,s", LAYERS, ids=lambda v: str(v))
def test_layer_matches_fp64(cin, cout, kh, kw, s, size):
    B, H, W = size
    x, gy = problem(cin, cout, kh, kw, s, B, H, W, seed=cin * 31 + cout + kh * 7 + s + H)
    rw, rb = reference(x, gy, cout, kh, kw, s)
    out = both(x, gy, cout, kh, kw, s)
    e = {k: (rel(v[0], rw), rel(v[1], rb)) for k, v in out.items()}
    print(f"{cin}->{cout} {kh}x{kw} s{s} {B}x{H}x{W}: tf32x3 dw {e['tf32'][0]:.2e} db {e['tf32'][1]:.2e} | "
          f"CUDA cores dw {e['ffma'][0]:.2e} db {e['ffma'][1]:.2e}")
    assert e["tf32"][0] <= 1e-5 and e["tf32"][1] <= 1e-5


@pytest.mark.parametrize("positive", [False, True], ids=["random_sign", "all_positive"])
def test_long_k_fnet_layer1(positive):
    """config 5's fnet layer 1: 4 frames of 192 x 256 = 196,608 output pixels, 64 -> 64 3x3.  All-positive operands are the
    worst case for the truncating accumulate (no cancellation of the per-add bias)."""
    cin = cout = 64
    B, H, W = 4, 192, 256
    x, gy = problem(cin, cout, 3, 3, 1, B, H, W, seed=77, positive=positive)
    rw, rb = reference(x, gy, cout, 3, 3, 1, device=DEV)          # fp64 on the GPU: the same arithmetic, faster than the CPU
    out = both(x, gy, cout, 3, 3, 1)
    e = {k: (rel(v[0], rw), rel(v[1], rb)) for k, v in out.items()}
    print(f"long K ({B * H * W} px, {'all positive' if positive else 'random sign'}): tf32x3 dw {e['tf32'][0]:.2e} db {e['tf32'][1]:.2e} | "
          f"CUDA cores dw {e['ffma'][0]:.2e} db {e['ffma'][1]:.2e}")
    bar = 2e-5 if positive else 1e-5
    assert e["tf32"][0] <= bar and e["tf32"][1] <= bar


def test_exponent_range():
    """Output gradients span 1e-9..1e-2: the TF32 hi/lo planes keep fp32's exponent range, so scaling gy by 1e-9 or 1e2 leaves
    the relative error where it is (an fp16 split would underflow at 1e-9)."""
    cin, cout, kh, kw, s = 128, 64, 3, 3, 1
    errs = []
    for scale in (1e-9, 1e2):
        x, gy = problem(cin, cout, kh, kw, s, 2, 24, 40, seed=5, gscale=scale)
        rw, rb = reference(x, gy, cout, kh, kw, s)
        out = both(x, gy, cout, kh, kw, s)
        errs.append((rel(out["tf32"][0], rw), rel(out["tf32"][1], rb)))
        print(f"gy x {scale:g}: tf32x3 dw {errs[-1][0]:.2e} db {errs[-1][1]:.2e} | CUDA cores dw {rel(out['ffma'][0], rw):.2e}")
    assert all(e <= 1e-5 for pair in errs for e in pair)
    assert 0.5 <= errs[0][0] / errs[1][0] <= 2.0


def test_accumulation_padded_strides_and_sentinels():
    """gw / gb are accumulated; ldx > cin, ldg > cout, ldw > cout work and columns beyond cout in gw stay untouched; gb may be
    NULL."""
    cin, cout, kh, kw, s = 96, 72, 3, 3, 2
    B, H, W = 2, 17, 35
    x, gy = problem(cin, cout, kh, kw, s, B, H, W, seed=9)
    rw, rb = reference(x, gy, cout, kh, kw, s)
    ldx, ldg, ldw = cin + 8, cout + 4, cout + 12
    xc, gc = to_cl(x, ldx), to_cl(gy, ldg)
    g = torch.Generator().manual_seed(10)
    pre_w = torch.randn(kh * kw, cin, cout, generator=g)
    pre_b = torch.randn(cout, generator=g)
    gw = torch.full((kh * kw, cin, ldw), 12345.0, device=DEV)
    gw[..., :cout] = pre_w.to(DEV)
    gb = pre_b.to(DEV)
    assert call("tf32", xc, cin, gc, cout, kh, kw, s, gw, gb) == 0
    torch.cuda.synchronize()
    assert (gw[..., cout:] == 12345.0).all()
    dw = unpack(gw, cout, kh, kw) - pre_w.view(kh, kw, cin, cout).permute(3, 2, 0, 1)
    e_w, e_b = rel(dw, rw), rel(gb.cpu() - pre_b, rb)
    print(f"prefilled, padded strides: dw {e_w:.2e} db {e_b:.2e}")
    assert e_w <= 1e-5 and e_b <= 1e-5
    gw2 = torch.zeros(kh * kw, cin, ldw, device=DEV)
    assert call("tf32", xc, cin, gc, cout, kh, kw, s, gw2, None) == 0          # gb = NULL
    torch.cuda.synchronize()
    assert rel(unpack(gw2, cout, kh, kw), rw) <= 1e-5 and (gw2[..., cout:] == 0).all()


def test_invalid_requests_are_rejected_before_any_launch():
    from rnc import native
    cin, cout, B, H, W = 64, 64, 2, 12, 20
    x = torch.randn(B * H * W * cin + 4, device=DEV)
    xv = x[:B * H * W * cin].view(B, H, W, cin)
    xmis = x[1:1 + B * H * W * cin].view(B, H, W, cin)                   # 4-byte offset: not 16-byte aligned
    gy = torch.randn(B, H, W, cout, device=DEV)
    gw = torch.zeros(9, cin, cout, device=DEV)
    gb = torch.zeros(cout, device=DEV)
    n = ws_bytes(cin, cout, B, H, W, 3, 3, 1)
    assert n > 0 and ws_bytes(cin, cout, B, H, W, 3, 3, 3) == 0
    ws = torch.empty((n + 15) // 16 * 4, device=DEV)
    gy2 = torch.randn(B, (H + 1) // 2, (W + 1) // 2, cout, device=DEV)
    cases = [  # (name, defective call, the same call minus the defect, expected status)
        ("workspace one byte short", lambda: call("tf32", xv, cin, gy, cout, 3, 3, 1, gw, gb, ws=ws, nbytes=n - 1),
         lambda: call("tf32", xv, cin, gy, cout, 3, 3, 1, gw, gb, ws=ws, nbytes=n), -5),
        ("stride 3", lambda: call("tf32", xv, cin, gy2, cout, 3, 3, 3, gw, gb, ws=ws, nbytes=n),
         lambda: call("tf32", xv, cin, gy2, cout, 3, 3, 2, gw, gb), -1),
        ("even kernel", lambda: call("tf32", xv, cin, gy, cout, 2, 3, 1, gw, gb, ws=ws, nbytes=n),
         lambda: call("tf32", xv, cin, gy, cout, 3, 3, 1, gw, gb, ws=ws, nbytes=n), -1),
        ("misaligned x", lambda: call("tf32", xmis, cin, gy, cout, 3, 3, 1, gw, gb, ws=ws, nbytes=n),
         lambda: call("tf32", xv, cin, gy, cout, 3, 3, 1, gw, gb, ws=ws, nbytes=n), -2),
        ("ldw < cout", lambda: call("tf32", xv, cin, gy, cout, 3, 3, 1, gw, gb, ldw=cout - 4, ws=ws, nbytes=n),
         lambda: call("tf32", xv, cin, gy, cout, 3, 3, 1, gw, gb, ldw=cout, ws=ws, nbytes=n), -1),
    ]
    for name, bad, good, want in cases:
        native.launch_count_reset()
        assert bad() == want, name
        assert native.launch_count() == 0, name                               # host-side rejection: nothing launched
        assert good() == 0, name
        assert native.launch_count() > 0, name
    torch.cuda.synchronize()


def _wide_layers(monkeypatch, conv, wgrad):
    """Run one small training forward + backward; return the (Cx, cout) of every weight-gradient call per entry point."""
    from rnc import native
    monkeypatch.setenv("RNC_TRAIN_CONV", conv)
    monkeypatch.setenv("RNC_TRAIN_WGRAD", wgrad)
    lib = native.lib()
    calls = {"rnc_conv2d_umma_wgrad": [], "rnc_conv2d_cl_wgrad": []}
    for name, seen in calls.items():
        orig = getattr(lib, name)

        def wrap(*a, _orig=orig, _seen=seen):
            _seen.append((a[2], a[5], a[9], a[10], a[11]))
            return _orig(*a)
        monkeypatch.setattr(lib, name, wrap)
    from rnc.train import sequence_loss
    m = build_model("raft_nc_dbl").to(DEV).train()
    m.freeze_bn()
    im1, im2, gt, valid = (t.to(DEV) for t in train_inputs())
    loss, _ = sequence_loss(m(im1, im2, iters=2), gt, valid, gamma=0.85)
    loss.backward()
    torch.cuda.synchronize()
    return calls


def test_routing_follows_the_rule(monkeypatch):
    from rnc.engine import engine_for
    from rnc.train import _umma_ok, _wgrad_umma_ok
    calls = _wide_layers(monkeypatch, "tf32", "tf32")
    eng = engine_for(torch.device(DEV))
    tc, cc = calls["rnc_conv2d_umma_wgrad"], calls["rnc_conv2d_cl_wgrad"]
    print(f"tensor-core weight gradients: {len(tc)} calls, {len(set(tc))} shapes; CUDA cores: {len(cc)} calls {sorted(set(cc))}")
    assert len(tc) > 0
    for cx, cout, *_ in tc:
        assert _wgrad_umma_ok(eng, cx, cout) and cout >= 32 and cx >= 16 and _umma_ok(eng, cx, cout) == "tf32"
    for cx, cout, *_ in cc:
        assert not _wgrad_umma_ok(eng, cx, cout)
    # the narrow layers stay on the CUDA cores: FlowHead.conv2 (256 -> 2), Simple.out (32 -> 2), the 4-channel 7x7 stems
    assert (256, 2, 3, 3, 1) in cc and (32, 2, 1, 1, 1) in cc and any(c[0] == 4 and c[2] == 7 for c in cc)


def test_wgrad_switch_needs_the_tf32_forward(monkeypatch):
    calls = _wide_layers(monkeypatch, "ffma", "tf32")
    assert len(calls["rnc_conv2d_umma_wgrad"]) == 0 and len(calls["rnc_conv2d_cl_wgrad"]) > 0


def _grad_errors(m, name, im1, im2, gt, valid, leaves, gmax):
    from rnc.train import sequence_loss
    m.zero_grad(set_to_none=True)
    preds = m(im1.to(DEV), im2.to(DEV), iters=GRAD_ITERS)
    loss, _ = sequence_loss(preds, gt.to(DEV), valid.to(DEV), gamma=0.85)
    loss.backward()
    errs = {}
    for k, prm in m.named_parameters():
        assert prm.grad is not None, k
        ref = leaves[k].grad
        errs[k] = float((prm.grad.cpu() - ref).norm() / (ref.norm() + 1e-5 * gmax))
    return float(loss.detach()), errs


@pytest.mark.parametrize("name", ["raft_nc_dbl", "raft"])
def test_whole_model_gradients_against_the_oracle(name, monkeypatch):
    """The metric of test_gpu_train.py::test_training_loss_and_gradients_match_the_oracle, with RNC_TRAIN_CONV=tf32 alone and
    with RNC_TRAIN_WGRAD=tf32 added: the tensor-core weight gradient may not move any parameter's gradient materially further
    from the CPU oracle than the tf32 forward / data gradient already do."""
    m = build_model(name)
    im1, im2, gt, valid = train_inputs()
    sd, leaves = tied_leaves(m)
    _, _, ups = orc.raft_forward_graph(sd, im1, im2, iters=GRAD_ITERS, model=name)
    oloss = orc.sequence_loss(ups, gt, valid, gamma=0.85)
    oloss.backward()
    gmax = max(float(q.grad.norm()) for q in leaves.values())
    m = m.to(DEV).train()
    m.freeze_bn()
    monkeypatch.setenv("RNC_TRAIN_CONV", "tf32")
    monkeypatch.setenv("RNC_TRAIN_WGRAD", "ffma")
    loss_a, ea = _grad_errors(m, name, im1, im2, gt, valid, leaves, gmax)
    monkeypatch.setenv("RNC_TRAIN_WGRAD", "tf32")
    loss_b, eb = _grad_errors(m, name, im1, im2, gt, valid, leaves, gmax)
    worst = max(ea, key=lambda k: eb[k] - 1.5 * ea[k])
    print(f"{name}: loss tf32 {loss_a:.6f} +wgrad {loss_b:.6f} oracle {float(oloss):.6f}; worst per-parameter error tf32 "
          f"{max(ea.values()):.2e}, +wgrad {max(eb.values()):.2e}; tightest {worst}: {ea[worst]:.2e} -> {eb[worst]:.2e}")
    assert abs(loss_b - float(oloss)) < 1e-4
    for k in ea:
        assert eb[k] <= 1.5 * ea[k] + 1e-3, (k, ea[k], eb[k])


def test_train_step_in_the_new_mode(monkeypatch):
    from rnc.train import fetch_optimizer, train_step
    monkeypatch.setenv("RNC_TRAIN_CONV", "tf32")
    monkeypatch.setenv("RNC_TRAIN_WGRAD", "tf32")
    m = build_model("raft_nc_dbl").to(DEV).train()
    m.freeze_bn()
    im1, im2, gt, valid = (t.to(DEV) for t in train_inputs())
    opt, sched = fetch_optimizer(m, lr=1e-4, num_steps=20)
    before = {k: q.detach().clone() for k, q in m.named_parameters()}
    losses = [float(train_step(m, opt, sched, im1, im2, gt, valid, iters=2)[0]) for _ in range(3)]
    print("losses", losses)
    assert all(torch.isfinite(torch.tensor(losses))) and losses[-1] < losses[0]
    assert all(not torch.equal(before[k], q.detach()) for k, q in m.named_parameters())
