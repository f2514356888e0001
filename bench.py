"""bench.py — image-pairs/s of the RAFT-NCUP hot path at 1024x436, 32 iterations (BASELINE.json metric), with the
corr-lookup kernel's HBM roofline and the CPU baseline beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference|reference_gpu] [--model raft_nc_dbl|raft]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

--impl reference      the UNMODIFIED reference (oracle/_ref, copied there by oracle/install_reference.py) on the host CPU cores
--impl reference_gpu  the same reference modules in eager PyTorch on the GPU, TF32 off (SURVEY.md §0.1: "the bar"); the native
                      arm runs this leg in a subprocess (the reference's module names clash with the drop-in's) and reports it
                      as `gpu_eager_baseline`
--dump-outputs DIR    after the timed steps, write the flows (flow_lo, flow_up; `loss` in --mode train) the last timed step
                      returned as DIR/<name>.npy; the inputs and weights are seeded, so two builds compare output for output

A "step" = one RAFT.forward over one batch of synthetic pairs (BASELINE configs[2]: batch 8 per GPU, 1024x436 padded to
440, 32 iterations, model raft_nc_dbl = full path incl. the NCUP upsampler; configs[1]'s corr-lookup kernel is timed
inside the same steps).  Weak scaling: every rank runs an independent replica on its own 8 pairs, no data-path collective.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "raft-ncup_b200")
REF_CORE = os.path.join(ROOT, "oracle", "_ref", "core")          # copy of the unmodified reference (git-ignored)

import torch  # noqa: E402


def use_product_path():
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)


def use_reference_path():
    """The reference is a directory of scripts that does `sys.path.append('core')` (evaluate.py:2): same here."""
    if not os.path.isdir(REF_CORE):
        return False
    if REF_CORE not in sys.path:
        sys.path.insert(0, REF_CORE)
    return True

H_IMG, W_IMG, ITERS, BATCH = 436, 1024, 32, 8
K2_BYTES_PER_PAIR_ITER = 25_891_840      # SURVEY.md §8(d): fmap1 + coords + out + fmap2 pyramid, fp32
K4_BYTES_PER_PAIR_CALL = 3_886_080       # SURVEY.md §8(d): flow_lr + conf read, 2x64xP fp32 written
K4_FMA_PER_PIXEL = 2 * (4 * 2 + 2 * 25 * 2 + 2 * 9 * 2 + 2)    # num + den streams: nconv_in (<= 4 live taps), x2, decoder, out
K5_BYTES_PER_PAIR_CALL = 19_880_960      # SURVEY.md §8(d): mask 16,220,160 + flow 56,320 + out 3,604,480
# same formula at the storage width the tensor-core lookup uses: fp16 fmap1/fmap2 pyramid, fp32 coords, 2 x fp16 outputs
K2_STORAGE_BYTES_PER_PAIR_ITER = 2 * 7040 * 256 + 8 * 7040 + 4 * 7040 * 324 + 2 * 256 * 9280


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full summary of this round."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get(kernel_key, {}).get("dram_bytes_per_launch")
    return None
METRIC = "image-pairs/sec @ 1024x436, 32 iters"
TRAIN_METRIC = "training image-pairs/sec @ 512x384, 12 iters (BASELINE configs[4])"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def synth_frames(b, seed):
    g = torch.Generator().manual_seed(seed)
    im1 = torch.rand(b, 3, H_IMG, W_IMG, generator=g) * 255
    im2 = torch.rand(b, 3, H_IMG, W_IMG, generator=g) * 255
    ph = (8 - H_IMG % 8) % 8                                        # InputPadder 'sintel' (utils.py:12-15): 436 -> 440, split evenly
    return [torch.nn.functional.pad(x, [0, 0, ph // 2, ph - ph // 2], mode="replicate") for x in (im1, im2)]


def ref_args(dataset="sintel"):
    """The flag values every reference script ships (eval_raft_nc_sintel.sh:12-34)."""
    return argparse.Namespace(
        small=False, mixed_precision=False, load_pretrained=None, freeze_raft=False, dataset=dataset, align_corners=True,
        final_upsampling="NConvUpsampler", final_upsampling_scale=4, final_upsampling_use_data_for_guidance=True,
        final_upsampling_channels_to_batch=True, final_upsampling_use_residuals=False, final_upsampling_est_on_high_res=False,
        interp_net="NConvUNet", interp_net_channels_multiplier=2, interp_net_num_downsampling=1,
        interp_net_data_pooling="conf_based", interp_net_encoder_filter_sz=5, interp_net_decoder_filter_sz=3,
        interp_net_out_filter_sz=1, interp_net_shared_encoder=True, interp_net_use_double_conv=False, interp_net_use_bias=False,
        weights_est_net="Simple", weights_est_net_num_ch=[64, 32], weights_est_net_filter_sz=[3, 3, 1],
        weights_est_net_dilation=[1, 1, 1])


def reference_model(name):
    """RAFT(args) of the unmodified reference (oracle/_ref/core/raft_nc_dbl.py:26 / raft.py:24), seed 1234 (train.py:345)."""
    import importlib
    import warnings
    warnings.filterwarnings("ignore")
    torch.manual_seed(1234)
    return importlib.import_module(name).RAFT(ref_args()).eval()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_cores():
    """Cores this process may actually use: scheduler affinity capped by the cgroup CPU quota (the GPU boxes expose
    128 logical CPUs but a 16-core quota; oversubscribing them makes the CPU path several times slower)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def cpu_reference_pairs_per_s(steps, warmup, model_name="raft_nc_dbl"):
    """The reference's own CPU path on the host cores: RAFT(args).eval() from oracle/_ref under torch.no_grad(), fp32, all
    the cores the cgroup allows.  One step = ONE pair at the full 1024x436 / 32-iteration shape (a bounded sample of the 8-pair
    batch: ~7 s).  Falls back to the oracle port (pinned to the reference by tests/golden) when oracle/_ref is absent.
    Returns (pairs/s, s/step, kind)."""
    torch.set_num_threads(host_cores())
    p1, p2 = synth_frames(1, 7)
    if use_reference_path():
        model = reference_model(model_name)
        kind = "reference"

        def step():
            with torch.no_grad():
                return model(p1, p2, iters=ITERS, test_mode=True)     # upsamples every iteration (raft_nc_dbl.py:161)
    else:
        use_product_path()
        from oracle import raft_oracle as orc
        from rnc.synth import build_model
        sd = {k: v.detach() for k, v in build_model(model_name).state_dict().items()}
        kind = "port"

        def step():
            return orc.raft_forward(sd, p1, p2, iters=ITERS, model=model_name)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return 1.0 / dt, dt, kind


CPU_SAMPLE = "1 pair per step at 1024x436 (pad 440), 32 iters, NCUP upsampling every iteration as the reference does"


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warmup = args.steps, min(args.warmup, 1)
    v, dt, kind = cpu_reference_pairs_per_s(steps, warmup, args.model)
    cores = torch.get_num_threads()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"cfg2/3: 1024x436 (pad 440), 32 iters, {args.model} full path incl. the upsampler, B=1 per step "
                               "(bounded sample of the B=8 batch)", "device": "host CPU",
                   "implementation": "unmodified reference modules from oracle/_ref" if kind == "reference" else "oracle port"},
        "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": cores, "kind": kind, "sample": CPU_SAMPLE},
        "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_reference_gpu(args):
    """SURVEY.md §0.1 / BASELINE.md §3.5: the reference's eager PyTorch path on the same B200 (cuBLAS bmm volume + grid_sample
    + cuDNN convolutions), TF32 off so that it computes what its CPU path computes.  CUDA events, warm-up, one JSON line."""
    if not use_reference_path() or not torch.cuda.is_available():
        print(json.dumps({"impl": "reference_gpu", "unavailable": "oracle/_ref or GPU missing"}))
        return
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda", 0)
    if args.mode == "train":
        return run_reference_gpu_train(args, dev)
    model = reference_model(args.model).to(dev)
    p1, p2 = synth_frames(args.batch, 7)
    d1, d2 = p1.to(dev), p2.to(dev)
    times = []
    with torch.no_grad():
        for i in range(max(1, args.warmup) + args.steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            lo, up = model(d1, d2, iters=ITERS, test_mode=True)
            e1.record()
            torch.cuda.synchronize()
            if i >= max(1, args.warmup):
                times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    print(json.dumps({"impl": "reference_gpu", "metric": METRIC, "value": args.batch / (ms * 1e-3), "unit": "pairs/s",
                      "ms_per_step": ms, "steps": args.steps, "batch": args.batch, "model": args.model, "dtype": "f32",
                      "tf32": False, "checksum_flow_up_abs_mean": float(up.abs().mean()),
                      "note": "unmodified reference modules (oracle/_ref) .cuda(), eager PyTorch, cudnn/matmul TF32 disabled, "
                              "inputs resident, CUDA events"}))


def run_reference_gpu_train(args, dev):
    """The reference's own training step in eager PyTorch on the GPU (train.py:203-227 without AMP): unmodified modules from
    oracle/_ref, train mode + freeze_bn, sequence loss (train.py:46-71 restated: train.py itself does not import), AdamW,
    clip 1.0 — the comparator of `--mode train`."""
    B, H, W, iters = args.train_batch, 384, 512, 12
    model = reference_model(args.model).to(dev).train()
    model.freeze_bn()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-4, weight_decay=5e-5, eps=1e-8)
    g = torch.Generator().manual_seed(100)
    im1, im2 = (torch.rand(B, 3, H, W, generator=g) * 255).to(dev), (torch.rand(B, 3, H, W, generator=g) * 255).to(dev)
    gt, valid = (torch.randn(B, 2, H, W, generator=g) * 5).to(dev), torch.ones(B, H, W, device=dev)
    times = []
    for i in range(3 + args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        opt.zero_grad()
        preds = model(im1, im2, iters=iters)
        mag = torch.sum(gt ** 2, dim=1).sqrt()
        val = (valid >= 0.5) & (mag < 400)
        loss = sum(0.85 ** (len(preds) - k - 1) * (val[:, None] * (p - gt).abs()).mean() for k, p in enumerate(preds))
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            times.append(e0.elapsed_time(e1))
    ms = sum(times) / len(times)
    print(json.dumps({"impl": "reference_gpu", "mode": "train", "metric": TRAIN_METRIC, "value": B / (ms * 1e-3), "unit": "pairs/s",
                      "ms_per_step": ms, "steps": args.steps, "batch": B, "model": args.model, "dtype": "f32", "tf32": False,
                      "loss_last": float(loss),
                      "note": "unmodified reference modules (oracle/_ref) in eager PyTorch, cuDNN/cuBLAS TF32 disabled"}))


def gpu_eager_baseline(args):
    """Run the reference_gpu leg in a fresh process (module names `raft_nc_dbl`, `update`, `corr`, ... clash with the drop-in)."""
    if not os.path.isdir(REF_CORE):
        return {"unavailable": "oracle/_ref not installed (run oracle/install_reference.py)"}
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference_gpu", "--steps", "2", "--warmup", "1",
           "--batch", str(args.batch), "--model", args.model, "--mode", args.mode, "--train-batch", str(args.train_batch)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=900,
                             env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        return json.loads(line)
    except Exception as e:     # noqa: BLE001 — the baseline leg must never take the bench down
        return {"unavailable": f"{type(e).__name__}: {e}"}


def mean_ms(pairs):
    return sum(a.elapsed_time(b) for a, b in pairs) / max(len(pairs), 1)


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays):
    """--dump-outputs: what the timed path returned in its last timed step, one DIR/<name>.npy per array (float64 stays
    float64, anything else is stored as float32), so that two builds can be compared output for output on the same seeded
    inputs.  Batched outputs over 64 MiB in all keep the same leading pairs of the batch."""
    import numpy as np
    arrays = {k: v.detach().cpu().numpy() for k, v in arrays.items()}
    arrays = {k: a if a.dtype == np.float64 else a.astype(np.float32) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        n = DUMP_BYTES // (total // min(a.shape[0] for a in arrays.values()))
        arrays = {k: a[:n] for k, a in arrays.items()}
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), a)


def run_native(args, rank, world, local_rank):
    import torch.distributed as dist
    use_product_path()
    from rnc import native
    from rnc.synth import build_model, motion_boundary_flow_init
    assert torch.cuda.is_available(), "bench.py --impl native needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    model = build_model(args.model).to(dev)
    p1, p2 = synth_frames(args.batch, 7 + rank)
    h1, h2 = p1.pin_memory(), p2.pin_memory()                      # host buffers of the e2e arm
    d1, d2 = h1.to(dev), h2.to(dev)                                # resident inputs of the `value` arm
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    out_lo = torch.empty(args.batch, 2, 55, 128).pin_memory()
    out_up = torch.empty(args.batch, 2, 440, 1024).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident():
        with torch.no_grad():
            return model(d1, d2, iters=ITERS, test_mode=True)

    # e2e: every step copies ITS inputs from pinned host memory and reads ITS flows back, inside the timed region.  Like any
    # input pipeline, the H2D copy of step i+1 is issued on a copy stream while step i computes (double-buffered staging).
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [(torch.empty_like(d1), torch.empty_like(d2), torch.cuda.Event()) for _ in range(2)]
    state = {"i": 0, "primed": False}

    def prefetch(slot):
        a, b, ev = stage[slot]
        copy_stream.wait_stream(torch.cuda.current_stream())      # the slot's previous consumer has finished
        with torch.cuda.stream(copy_stream):
            a.copy_(h1, non_blocking=True)
            b.copy_(h2, non_blocking=True)
            ev.record(copy_stream)

    def step_e2e():
        with torch.no_grad():
            i = state["i"]
            if not state["primed"]:
                prefetch(i & 1)
                state["primed"] = True
            a, b, ev = stage[i & 1]
            torch.cuda.current_stream().wait_event(ev)
            prefetch((i + 1) & 1)                                    # next step's inputs travel during this step's compute
            lo, up = model(a, b, iters=ITERS, test_mode=True)
            out_lo.copy_(lo, non_blocking=True)
            out_up.copy_(up, non_blocking=True)
            state["i"] = i + 1
        return lo, up

    def timed(fn, steps):
        evs = []
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            flush.zero_()                                           # L2 flush between timed iterations (not timed)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            evs.append((e0, e1))
        barrier()
        wall = time.perf_counter() - t0
        dev_ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                # max over ranks
        return t.item(), wall, out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    step_e2e()
    torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    eng = model.engine()
    eng.profile = {}
    native.launch_count_reset()
    ms_total, wall, (flow_lo, flow_up) = timed(step_resident, args.steps)
    launches = native.launch_count()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"flow_lo": flow_lo, "flow_up": flow_up})    # before later calls reuse the buffers
    prof, eng.profile = eng.profile, None
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    # the lookup kernel alone (in the timed region convf1 runs underneath it on a side stream): 32 back-to-back launches
    iso_ms = None
    if hasattr(eng, "lookup_resident"):
        ws = next(w for k, w in eng._ws.items() if k[0] == eng.mode and w.B == args.batch)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(ITERS):
            eng.lookup_resident(ws)
        e1.record()
        torch.cuda.synchronize()
        iso_ms = e0.elapsed_time(e1) / ITERS
    # (tile, level) units of the LAST lookup launch that the fixed boxes could not cover (recomputed by the exact kernel),
    # and the same kernel on the motion-boundary stimulus (flow discontinuities of 24 px at 1/8 resolution)
    fb_units = mb_ms = mb_units = None
    if hasattr(eng, "lookup_resident") and getattr(eng, "lookup_mode", "") == "umma":
        fb_units = int((ws.lookup_flags != 0).sum().item())
        keep = ws.coords1.clone()
        ws.coords1.add_(motion_boundary_flow_init(args.batch, ws.H8, ws.W8).to(dev))
        for _ in range(2):
            eng.lookup_resident(ws)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(ITERS):
            eng.lookup_resident(ws)
        e1.record()
        torch.cuda.synchronize()
        mb_ms = e0.elapsed_time(e1) / ITERS
        mb_units = int((ws.lookup_flags != 0).sum().item())
        ws.coords1.copy_(keep)
    # K5 (convex upsampler of model `raft`) alone on cfg-2/3 shaped buffers: 20 launches
    k5_ms = None
    if rank == 0:
        mk = torch.randn(args.batch * 55 * 128, 576, device=dev)
        fl = torch.randn(args.batch, 2, 55, 128, device=dev)
        dims = type("D", (), {"B": args.batch, "H8": 55, "W8": 128})()
        for _ in range(3):
            eng.convex_upsample(dims, fl, mk, 576)
        flush.zero_()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            eng.convex_upsample(dims, fl, mk, 576)
        e1.record()
        torch.cuda.synchronize()
        k5_ms = e0.elapsed_time(e1) / 20
        del mk, fl
    # single pair latency (the reference's evaluate.py usage: B = 1)
    b1_ms = None
    if rank == 0:
        with torch.no_grad():
            for _ in range(2):
                model(d1[:1], d2[:1], iters=ITERS, test_mode=True)
            torch.cuda.synchronize()
            ts = []
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                model(d1[:1], d2[:1], iters=ITERS, test_mode=True)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
        b1_ms = statistics.median(ts)
    clocks = sampler.stop() if rank == 0 else None

    pairs = world * args.batch * args.steps
    value = pairs / (ms_total * 1e-3)
    e2e = pairs / (ms_e2e * 1e-3)
    if rank != 0:
        return
    peak, peak_src = peaks()
    k2_ms = mean_ms(prof.get("corr_lookup", []))
    k2_bytes = K2_BYTES_PER_PAIR_ITER * args.batch
    k2_gbs = k2_bytes / (k2_ms * 1e-3) / 1e9 if k2_ms else 0.0
    k4_ms = mean_ms(prof.get("ncup", []))
    k4_gbs = K4_BYTES_PER_PAIR_CALL * args.batch / (k4_ms * 1e-3) / 1e9 if k4_ms else 0.0
    ub_ms = mean_ms(prof.get("update_block", []))
    ub_tflops = 37.7e9 * args.batch / (ub_ms * 1e-3) / 1e12 if ub_ms else 0.0
    line = {
        "metric": METRIC, "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"cfg2/3: batch={args.batch}/GPU 1024x436 (pad 440), 32 iters, {args.model} full path "
                               "(encoders + corr lookup + update block + NCUP upsampler), random-init weights seed 1234",
                   "parallelism": f"replicas x{world} (batch-sharded, no collective)",
                   "l2": "flushed with a 256 MiB write between timed steps", "timing": "CUDA events per step, max over ranks",
                   "wall_s_incl_flush": wall},
        "e2e": {"value": e2e, "unit": "pairs/s", "h2d_bytes_per_step": int(h1.numel() + h2.numel()) * 4,
                "d2h_bytes_per_step": int(out_lo.numel() + out_up.numel()) * 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"kernel": "corr_lookup_umma_kernel (tcgen05 fused corr lookup, K2; incoherent units recomputed exactly inside the same launch)", "bound": "hbm",
                     "achieved": k2_gbs, "peak": peak, "unit": "GB/s", "frac": k2_gbs / peak, "traffic": ncu_traffic("corr_lookup"),
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": k2_bytes,
                     "algorithmic_bytes_note": "SURVEY §8d contract figure (fp32 storage: 25,891,840 B/pair-iter); at the storage "
                                               "width actually used (fp16 features, 4 B hi/lo outputs) one launch moves "
                                               f"{K2_STORAGE_BYTES_PER_PAIR_ITER * args.batch} B",
                     "avg_launch_ms": k2_ms, "launches_timed": len(prof.get("corr_lookup", [])),
                     "storage_width": {"bytes_per_launch": K2_STORAGE_BYTES_PER_PAIR_ITER * args.batch,
                                       "frac": (K2_STORAGE_BYTES_PER_PAIR_ITER * args.batch / (k2_ms * 1e-3) / 1e9 / peak) if k2_ms else None},
                     "fallback_units_per_launch": fb_units, "units_per_launch": args.batch * 56 * 4,
                     "motion_boundary": {"avg_launch_ms": mb_ms, "fallback_units_per_launch": mb_units,
                                         "frac": (k2_bytes / (mb_ms * 1e-3) / 1e9 / peak) if mb_ms else None,
                                         "note": "same launch with a 24 px (1/8-res) flow discontinuity added to coords1: boundary "
                                                 "tiles go through the exact CUDA-core kernel"},
                     "isolated": {"avg_launch_ms": iso_ms, "achieved": (k2_bytes / (iso_ms * 1e-3) / 1e9) if iso_ms else None,
                                  "frac": (k2_bytes / (iso_ms * 1e-3) / 1e9 / peak) if iso_ms else None,
                                  "note": "same kernel, 32 back-to-back launches outside the timed region (warm L2, no "
                                          "neighbouring kernels)"}},
        "roofline_ncup": {"kernel": "ncup_fused_kernel (K4)", "bound": "hbm", "achieved": k4_gbs, "peak": peak, "unit": "GB/s",
                          "frac": k4_gbs / peak, "avg_launch_ms": k4_ms,
                          "algorithmic_bytes_per_launch": K4_BYTES_PER_PAIR_CALL * args.batch,
                          "fma_pipe": {"tflops_fp32": (K4_FMA_PER_PIXEL * 2 * args.batch * 2 * 440 * 1024 / (k4_ms * 1e-3) / 1e12) if k4_ms else None,
                                       "peak_tflops_fp32": 74.5,
                                       "note": "the chain is ~300 multiply-adds per output pixel (4 normalized convolutions, num and den "
                                               "streams): bound by the FP32 FMA pipe (148 SMs x 128 lanes x 2 x 1.965 GHz), not by HBM"}},
        "roofline_convex": {"kernel": "convex_upsample_kernel (K5, model raft)", "bound": "hbm",
                            "achieved": (K5_BYTES_PER_PAIR_CALL * args.batch / (k5_ms * 1e-3) / 1e9) if k5_ms else None, "peak": peak,
                            "unit": "GB/s", "frac": (K5_BYTES_PER_PAIR_CALL * args.batch / (k5_ms * 1e-3) / 1e9 / peak) if k5_ms else None,
                            "avg_launch_ms": k5_ms, "algorithmic_bytes_per_launch": K5_BYTES_PER_PAIR_CALL * args.batch,
                            "note": "20 back-to-back launches on cfg-2/3 shaped buffers (mask 130 MB > L2)"},
        "update_block": {"avg_iter_ms": ub_ms, "tflops_fp32_equiv": ub_tflops, "flop_per_pair_iter": 37.7e9},
        "latency_b1_ms": b1_ms,
    }
    if world == 1 and not args.no_cpu_baseline:
        del model, d1, d2, stage, flush
        torch.cuda.empty_cache()
        line["gpu_eager_baseline"] = gpu_eager_baseline(args)
        ge = line["gpu_eager_baseline"].get("value")
        if ge:
            line["gpu_eager_baseline"]["speedup_value_over_eager"] = value / ge
        line["cpu_baseline"] = cpu_baseline_subprocess(args)
    print(json.dumps(line))


def cpu_baseline_subprocess(args):
    """The reference's CPU path, one bounded step, in a fresh process (same module-name clash as the GPU leg)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "0", "--model", args.model]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600,
                             env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        ref = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        cb = ref["cpu_baseline"]
        cb["sample"] += f"; 1 run, {ref['ms_per_step'] / 1e3:.1f} s"
        return cb
    except Exception as e:     # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}


def run_train(args, rank, world, local_rank):
    """BASELINE configs[4] / SURVEY.md §8e: one optimisation step of raft_nc_dbl per timed step — batch 2 per GPU (16 on 8 GPUs),
    384x512 synthetic frames, 12 iterations, sequence loss, AdamW + OneCycle, gradient clipping; under torchrun the replicas are
    DistributedDataParallel over NCCL (one bucketed all-reduce of the 19.6 MB of fp32 gradients per step, overlapped with the
    backward pass).  Train mode with frozen BatchNorm, as every stage but `chairs` (train.py:185-186)."""
    import torch.distributed as dist
    use_product_path()
    from rnc import native
    from rnc.synth import build_model
    from rnc.train import ddp_model, fetch_optimizer, train_step
    assert torch.cuda.is_available(), "bench.py --mode train needs a GPU"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B, H, W, iters = args.train_batch, 384, 512, 12
    model = build_model(args.model).to(dev).train()
    model.freeze_bn()
    nparams = sum(p.numel() for p in model.parameters())
    net = ddp_model(model, dev) if world > 1 else model
    opt, sched = fetch_optimizer(net, lr=1e-4, num_steps=10000)
    g = torch.Generator().manual_seed(100 + rank)
    h1 = (torch.rand(B, 3, H, W, generator=g) * 255).pin_memory()
    h2 = (torch.rand(B, 3, H, W, generator=g) * 255).pin_memory()
    hgt = (torch.randn(B, 2, H, W, generator=g) * 5).pin_memory()
    hval = torch.ones(B, H, W).pin_memory()

    def step():
        im1, im2, gt, val = (t.to(dev, non_blocking=True) for t in (h1, h2, hgt, hval))     # the step's inputs come from the host
        loss, _ = train_step(net, opt, sched, im1, im2, gt, val, iters=iters, gamma=0.85, clip=1.0, return_metrics=False)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    native.launch_count_reset()
    barrier()
    evs = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step()
        e1.record()
        evs.append((e0, e1))
    barrier()
    launches = native.launch_count()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss})
    ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    # the collective alone: all-reduce of a flat fp32 buffer of the gradients' size
    ar_ms = None
    if world > 1:
        flat = torch.zeros(nparams, dtype=torch.float32, device=dev)
        for _ in range(3):
            dist.all_reduce(flat)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            dist.all_reduce(flat)
        e1.record()
        torch.cuda.synchronize()
        ar_ms = e0.elapsed_time(e1) / 10
    # the TF32x3 tensor-core form of the forward / data-gradient convolutions (opt-in: RNC_TRAIN_CONV=tf32), same steps
    tc_ms = None
    if world == 1:
        os.environ["RNC_TRAIN_CONV"] = "tf32"
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        tc_ms = e0.elapsed_time(e1) / args.steps
        os.environ["RNC_TRAIN_CONV"] = "ffma"
    clocks = sampler.stop() if rank == 0 else None
    if rank != 0:
        return
    pairs = world * B * args.steps
    # forward flops per pair at 384x512 (SURVEY.md Appendix C scaled by the pixel count): 12 x (update block 37.7 + NCUP 6.1)
    # + encoders 184 GFLOP at 440x1024; backward ~ 2x forward
    scale = (H * W) / (440.0 * 1024.0)
    fwd_gflop = (iters * (37.7 + 6.1) + 184.0) * scale
    print(json.dumps({
        "mode": "train", "metric": TRAIN_METRIC, "value": pairs / (ms * 1e-3), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"cfg5: batch={B}/GPU ({B * world} global) 384x512, 12 iters, {args.model}, sequence loss gamma 0.85, AdamW + "
                               "OneCycleLR, clip 1.0, train mode with frozen BatchNorm; forward AND backward through librnc's exact fp32 "
                               "kernels (conv fwd/dgrad/wgrad, corr lookup fwd/bwd, NConv fwd/bwd)",
                   "parallelism": f"ddp x{world} (one process per GPU, NCCL gradient all-reduce, bucket 8 MB)" if world > 1 else "single GPU",
                   "timing": "CUDA events per step incl. H2D of the step's inputs, max over ranks"},
        "loss_last": float(loss), "parameters": nparams, "grad_bytes": nparams * 4,
        "allreduce": {"alone_ms": ar_ms, "bytes": nparams * 4,
                      "bus_GBps": (2 * (world - 1) / world * nparams * 4 / (ar_ms * 1e-3) / 1e9) if ar_ms else None,
                      "note": "all-reduce of a flat fp32 buffer of the gradients' size, 10 back-to-back; inside the step it is "
                              "bucketed and overlapped with the backward pass"},
        "tflops_fp32": 3 * fwd_gflop * B * 1e9 / (ms / args.steps * 1e-3) / 1e12,
        "gpu_launches": int(launches), "clocks": clocks,
        "tf32x3_convs": {"ms_per_step": tc_ms, "value": (B / (tc_ms * 1e-3)) if tc_ms else None,
                         "note": "RNC_TRAIN_CONV=tf32: forward and data-gradient convolutions on tcgen05 kind::tf32 (hi/lo operand "
                                 "planes, 3 MMAs per K step); per-layer error 1e-6..5e-6 instead of 1.5e-7, opt-in"},
        "gpu_eager_baseline": gpu_eager_baseline(args) if world == 1 and not args.no_cpu_baseline else None}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "reference_gpu"])
    ap.add_argument("--model", default="raft_nc_dbl", choices=["raft_nc_dbl", "raft"])
    ap.add_argument("--batch", type=int, default=BATCH, help="pairs per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"], help="train: one optimisation step per timed step (cfg 5)")
    ap.add_argument("--train-batch", type=int, default=2, help="pairs per GPU in --mode train")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes what the native path computed: use it with --impl native")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.impl == "reference_gpu":
        if rank == 0:
            run_reference_gpu(args)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.mode == "train":
            run_train(args, rank, world, local_rank)
        else:
            run_native(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
