"""Weight gradient of the training path on the CUDA cores (rnc_conv2d_cl_wgrad) vs the tensor cores (rnc_conv2d_umma_wgrad), at
config 5 (B = 2 pairs, 384x512, 12 iterations; encoders, update block, weights net):

  0. the error of the tensor-core form against fp64 vs the TMEM accumulation chunk, on the longest K of the step;
  1. every distinct convolution shape of one step (recorded from a real step): time per call of both kernels (CUDA events,
     3 warm-up + 20 timed launches), TFLOP/s (2 * P * cin * cout * taps), relative error of dw / db against fp64 on the CPU,
     whether the routing rule (rnc.train._wgrad_umma_ok) sends the layer to the tensor cores, calls per step;
  2. full train_steps for RNC_TRAIN_CONV=ffma, =tf32, and =tf32 with RNC_TRAIN_WGRAD=tf32, alternating the three forms over
     several rounds in the same process.

    python tools/wgrad_probe.py OUTDIR [--rounds 3] [--steps 5] [--no-steps]

Writes OUTDIR/r03_wgrad.json (committed as profiles/r03_wgrad.json) with the GPU's name, power limit and max SM clock."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "raft-ncup_b200")]
from rnc import native  # noqa: E402
from rnc.engine import engine_for  # noqa: E402
from rnc.synth import build_model  # noqa: E402
from rnc.train import _wgrad_umma_ok, fetch_optimizer, train_step  # noqa: E402

DEV = torch.device("cuda", 0)
FORMS = {"ffma": {"RNC_TRAIN_CONV": "ffma", "RNC_TRAIN_WGRAD": "ffma"},
         "tf32": {"RNC_TRAIN_CONV": "tf32", "RNC_TRAIN_WGRAD": "ffma"},
         "tf32+wgrad_tf32": {"RNC_TRAIN_CONV": "tf32", "RNC_TRAIN_WGRAD": "tf32"}}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def step_inputs():
    g = torch.Generator().manual_seed(1)
    B, H, W = 2, 384, 512
    im1, im2 = (torch.rand(B, 3, H, W, generator=g) * 255).to(DEV), (torch.rand(B, 3, H, W, generator=g) * 255).to(DEV)
    gt, valid = (torch.randn(B, 2, H, W, generator=g) * 5).to(DEV), torch.ones(B, H, W, device=DEV)
    return im1, im2, gt, valid


def set_form(name):
    os.environ.update(FORMS[name])


def record_shapes(m, opt, sched, inputs):
    """(Cx, cout, B, Hin, Win, kh, kw, stride, ldg) -> calls per step, from one step whose weight gradients all run on the CUDA
    cores (RNC_TRAIN_CONV=tf32: the forms' routing rule is evaluated per shape below)."""
    L = native.lib()
    orig = L.rnc_conv2d_cl_wgrad
    seen = {}

    def wrap(*a):
        key = (a[2], a[5], a[6], a[7], a[8], a[9], a[10], a[11], a[4])
        seen[key] = seen.get(key, 0) + 1
        return orig(*a)
    L.rnc_conv2d_cl_wgrad = wrap
    try:
        set_form("tf32")
        train_step(m, opt, sched, *inputs, iters=12, return_metrics=False)
        torch.cuda.synchronize()
    finally:
        L.rnc_conv2d_cl_wgrad = orig
    return seen


def time_layer(key, calls):
    cx, cout, B, H, W, kh, kw, s, ldg = key
    L = native.lib()
    Ho, Wo = (H + s - 1) // s, (W + s - 1) // s
    g = torch.Generator().manual_seed(cx * 1000 + cout)
    x = torch.randn(B, cx, H, W, generator=g)
    gy = torch.randn(B, cout, Ho, Wo, generator=g) * 1e-4
    xr = x.double()
    wr = torch.zeros(cout, cx, kh, kw, dtype=torch.float64, requires_grad=True)
    br = torch.zeros(cout, dtype=torch.float64, requires_grad=True)
    F.conv2d(xr, wr, br, stride=s, padding=(kh // 2, kw // 2)).backward(gy.double())
    xc = x.permute(0, 2, 3, 1).contiguous().to(DEV)
    gc = F.pad(gy.permute(0, 2, 3, 1), (0, ldg - cout)).contiguous().to(DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nbytes = L.rnc_conv2d_umma_wgrad_workspace_bytes(cx, cout, B, H, W, kh, kw, s)
    ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=DEV)
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def run(kind, gw, gb):
        if kind == "ffma":
            return L.rnc_conv2d_cl_wgrad(P(xc), cx, cx, P(gc), ldg, cout, B, H, W, kh, kw, s, P(gw), cout, P(gb), st)
        return L.rnc_conv2d_umma_wgrad(P(xc), cx, cx, P(gc), ldg, cout, B, H, W, kh, kw, s, P(gw), cout, P(gb), P(ws), nbytes, st)

    out = {"cin": cx, "cout": cout, "B": B, "Hin": H, "Win": W, "kh": kh, "kw": kw, "stride": s, "calls_per_step": calls,
           "routed_to_tensor_cores": None}
    flops = 2.0 * B * Ho * Wo * cx * cout * kh * kw
    for kind in ("ffma", "tf32"):
        gw = torch.zeros(kh * kw, cx, cout, device=DEV)
        gb = torch.zeros(cout, device=DEV)
        native.check(run(kind, gw, gb), kind)
        torch.cuda.synchronize()
        dw = gw.view(kh, kw, cx, cout).permute(3, 2, 0, 1).double().cpu()
        e_w = float((dw - wr.grad).norm() / wr.grad.norm())
        e_b = float((gb.double().cpu() - br.grad).norm() / br.grad.norm())
        for _ in range(3):
            run(kind, gw, gb)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 20
        e0.record()
        for _ in range(n):
            run(kind, gw, gb)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out[kind] = {"us_per_call": round(ms * 1e3, 2), "tflops": round(flops / (ms * 1e-3) / 1e12, 2), "rel_err_dw": e_w, "rel_err_db": e_b}
    return out


def kc_sweep():
    """Error of the tensor-core weight gradient against fp64 vs the TMEM accumulation chunk (RNC_WGRAD_KC, in 32-px K blocks)
    on config 5's longest K: fnet layer 1, 64 -> 64 3x3 over 4 x 192 x 256 = 196,608 output pixels.  A chunk never outlasts
    its work item's K split (about 6,100 px here), so the largest setting stands for "no chunking"."""
    L = native.lib()
    cin = cout = 64
    B, H, W = 4, 192, 256
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nbytes = L.rnc_conv2d_umma_wgrad_workspace_bytes(cin, cout, B, H, W, 3, 3, 1)
    ws = torch.empty((nbytes + 15) // 16 * 4, dtype=torch.float32, device=DEV)
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    out = []
    for positive in (False, True):
        g = torch.Generator().manual_seed(77)
        rnd = torch.rand if positive else torch.randn
        x, gy = rnd(B, cin, H, W, generator=g), rnd(B, cout, H, W, generator=g)
        wr = torch.zeros(cout, cin, 3, 3, dtype=torch.float64, device=DEV, requires_grad=True)
        F.conv2d(x.double().to(DEV), wr, padding=1).backward(gy.double().to(DEV))
        ref = wr.grad.cpu()
        xc, gc = x.permute(0, 2, 3, 1).contiguous().to(DEV), gy.permute(0, 2, 3, 1).contiguous().to(DEV)

        def err(kind):
            gw = torch.zeros(9, cin, cout, device=DEV)
            if kind == "ffma":
                native.check(L.rnc_conv2d_cl_wgrad(P(xc), cin, cin, P(gc), cout, cout, B, H, W, 3, 3, 1, P(gw), cout, None, st))
            else:
                native.check(L.rnc_conv2d_umma_wgrad(P(xc), cin, cin, P(gc), cout, cout, B, H, W, 3, 3, 1, P(gw), cout, None, P(ws),
                                                     nbytes, st))
            dw = gw.view(3, 3, cin, cout).permute(3, 2, 0, 1).double().cpu()
            return float((dw - ref).norm() / ref.norm())
        row = {"operands": "all positive" if positive else "random sign", "cuda_cores": err("ffma"), "tensor_cores": {}}
        for kc in (1, 4, 16, 64, 256):
            os.environ["RNC_WGRAD_KC"] = str(kc)
            row["tensor_cores"][str(kc * 32)] = err("tf32")
        os.environ.pop("RNC_WGRAD_KC")
        print(f"KC sweep ({row['operands']}): CUDA cores {row['cuda_cores']:.2e}; tensor cores by chunk px "
              + " ".join(f"{k}:{v:.2e}" for k, v in row["tensor_cores"].items()), flush=True)
        out.append(row)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("outdir")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--no-steps", action="store_true", help="per-layer and chunk measurements only")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "wgrad_probe measures on the GPU"
    os.makedirs(args.outdir, exist_ok=True)
    info = gpu_info()
    print("GPU (name, power limit, max SM clock):", info, flush=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sweep = kc_sweep()
    m = build_model("raft_nc_dbl").to(DEV).train()
    m.freeze_bn()
    opt, sched = fetch_optimizer(m, lr=1e-5, num_steps=1000)
    inputs = step_inputs()
    set_form("ffma")
    train_step(m, opt, sched, *inputs, iters=12, return_metrics=False)
    shapes = record_shapes(m, opt, sched, inputs)
    eng = engine_for(DEV)
    os.environ.update(FORMS["tf32+wgrad_tf32"])
    layers = []
    for key, calls in sorted(shapes.items(), key=lambda kv: -kv[0][2] * kv[0][3] * kv[0][4] * kv[0][0] * kv[0][1] * kv[0][5] * kv[0][6]):
        r = time_layer(key, calls)
        r["routed_to_tensor_cores"] = bool(_wgrad_umma_ok(eng, key[0], key[1]))
        layers.append(r)
        print(f"{r['cin']:>4}->{r['cout']:<4} {r['kh']}x{r['kw']} s{r['stride']} B{r['B']} {r['Hin']}x{r['Win']} x{calls:<3} "
              f"routed {int(r['routed_to_tensor_cores'])} | CUDA cores {r['ffma']['us_per_call']:8.1f} us {r['ffma']['tflops']:6.1f} TF/s "
              f"err {r['ffma']['rel_err_dw']:.1e} | tensor cores {r['tf32']['us_per_call']:8.1f} us {r['tf32']['tflops']:6.1f} TF/s "
              f"err {r['tf32']['rel_err_dw']:.1e} db {r['tf32']['rel_err_db']:.1e}", flush=True)
    per_step = {k: sum(r[k]["us_per_call"] * r["calls_per_step"] for r in layers) / 1e3 for k in ("ffma", "tf32")}
    routed = sum((r["tf32"] if r["routed_to_tensor_cores"] else r["ffma"])["us_per_call"] * r["calls_per_step"] for r in layers) / 1e3
    print(f"weight gradients per step (sum of per-call times x calls): CUDA cores {per_step['ffma']:.1f} ms, with the routing "
          f"rule {routed:.1f} ms", flush=True)

    times = {k: [] for k in FORMS}
    for rnd in range(0 if args.no_steps else args.rounds):
        for name in FORMS:
            set_form(name)
            for _ in range(2):
                train_step(m, opt, sched, *inputs, iters=12, return_metrics=False)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                train_step(m, opt, sched, *inputs, iters=12, return_metrics=False)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / args.steps)
            print(f"round {rnd} {name:>16}: {times[name][-1]:.1f} ms per step", flush=True)
    steps = {k: {"ms_per_step_rounds": v, "ms_per_step_median": sorted(v)[len(v) // 2] if v else None} for k, v in times.items()}
    res = {"gpu": info, "config": "cfg 5: raft_nc_dbl, B=2, 384x512, 12 iterations, frozen BN, AdamW + clip",
           "chunk_pixels": 512, "error_vs_chunk_pixels": sweep, "layers": layers,
           "wgrad_ms_per_step": {"cuda_cores": per_step["ffma"], "routing_rule": routed},
           "train_step": steps, "time": time.strftime("%Y-%m-%d %H:%M:%S")}
    with open(os.path.join(args.outdir, "r03_wgrad.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v["ms_per_step_median"] for k, v in steps.items()}))


if __name__ == "__main__":
    main()
