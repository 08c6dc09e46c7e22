#!/usr/bin/env python
"""bench.py -- images/sec (forward + backward) of the hot path
ERFNet -> activation/mask -> weighted least squares -> backprojection loss.

    python bench.py --gpus N --steps K --warmup W            # our arm (sm_100a kernels via the C ABI)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own modules on the host cores, rank 0 only

Workload (BASELINE.json configs[1]): egolane 2-lane, order 2, batch 32 per GPU, 256x512, fp32 I/O,
model.train() with dropout, `zero_grad -> forward -> loss -> backward` (optimizer excluded, SURVEY.md 8d).
Multi-GPU = weak scaling: 32 images per GPU, per-replica BN statistics, one flat-gradient all-reduce
(NCCL) per step inside the timed region.

One JSON line on stdout (rank 0).  `value`: inputs resident in HBM.  `e2e`: through the public modules
with HOST (pinned) inputs copied in every step and the loss read back every step.

`--dump-outputs DIR` (this project's arm) writes what the last timed step handed its caller (the loss, every
parameter gradient, the BatchNorm running statistics) as DIR/<name>.npy.  Inputs, weights and dropout draws are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    1: dict(name="egolane_2lane_b1_256x512_fp32", nclasses=2, order=2, mask=0.3, resize=256, batch=1),
    2: dict(name="egolane_2lane_b32_256x512_fp32", nclasses=2, order=2, mask=0.3, resize=256, batch=32),
    3: dict(name="tusimple_4lane_b64_256x512", nclasses=4, order=3, mask=0.2, resize=256, batch=64),
    4: dict(name="tusimple_4lane_b32pergpu_320x640", nclasses=4, order=3, mask=0.2, resize=320, batch=32),
}
MODE_DTYPE = {"tf32x3": "fp32 (storage fp32; products 3xTF32 on tcgen05 = fp32-grade; fp32 accumulate)",
              "tf32": "tf32 (storage fp32; single-pass TF32 products on tcgen05; fp32 accumulate)",
              "fp32": "fp32 (CUDA-core FFMA)"}
MODE_TEXT = {"tf32x3": "3xTF32 on tcgen05 (a_hi*w_hi + a_hi*w_lo + a_lo*w_hi, TMEM fp32 accumulators) for every convolution but the "
                       "3->13 stem and the 16->L output ConvTranspose2d (fp32 FFMA): 3-tap convs conv_tc_x3.cu (C=16 as 4-pixel "
                       "super-pixels), stride-2 layers conv_tcg.cu, weight gradients wgrad_tc_x3.cu / wgrad_tcg.cu",
             "tf32": "single-pass TF32 on tcgen05 for the same layers (what cuDNN's default does for the reference's fp32 convs)",
             "fp32": "every convolution on the CUDA-core FFMA kernels (conv_f32.cu, wgrad_f32.cu)"}
MODE_ACCURACY = {"tf32x3": "meets the reference-fp32 gates: on the reference's golden inputs |ours - fp64| <= 4 |reference fp32 - fp64| + "
                           "1e-4 for every block output, beta and the loss (tests/test_net_gpu.py, __graft_entry__.smoke(); measured "
                           "numbers in profiles/r02/accuracy_*.json)",
                 "tf32": "beta 1.1e-3 (2 lanes, order 2) / 2.1e-3 (4 lanes, order 3) norm-wise from fp64 on the golden inputs -- OUTSIDE "
                         "the 1e-4 gate; labelled extra only (profiles/r01/tf32_accuracy_*.json)",
                 "fp32": "meets the same gates as tf32x3 (tests/test_net_gpu.py)"}
FWD_GFLOP_PER_IMG = {(2, 256): 13.231, (4, 256): 13.239, (4, 320): 20.686, (2, 320): 20.673}   # SURVEY.md 8d
FWD_GFLOP_PER_IMG_CLAS = {(4, 256): 15.497}        # + the two Classification heads
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_MAX_BYTES = 64 * 10 ** 6


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            d["_source"] = "measured"
            return d
        except Exception:
            pass
    d = dict(FALLBACK_PEAKS)
    d["_source"] = "fallback"
    return d


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, smax, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def build_args(cfg, no_cuda=False):
    from lanedetection_end2end_b200.Networks.utils import define_args
    argv = ["--image_dir", "x", "--gt_dir", "y", "--nclasses", str(cfg["nclasses"]), "--order", str(cfg["order"]),
            "--batch_size", str(cfg["batch"]), "--mask_percentage", str(cfg["mask"]), "--resize", str(cfg["resize"]),
            "--loss_policy", "backproject", "--end_to_end", "True"]
    if cfg.get("clas"):
        argv += ["--clas", "1"]          # line-type + horizon heads on the shared encoder output (BP/train.sh:1)
    if no_cuda:
        argv.append("--no_cuda")
    return define_args().parse_args(argv)


def host_batch(cfg, seed, pinned):
    import torch
    g = torch.Generator().manual_seed(seed)
    B, R = cfg["batch"], cfg["resize"]
    x = torch.rand(B, 3, R, 2 * R, generator=g)
    xgt = torch.rand(B, 4, 56, generator=g, dtype=torch.float64) * 500.0
    valid = torch.ones(B, 4, 56, dtype=torch.float64)
    valid[:, :, :8] = 0
    if pinned:
        x, xgt, valid = x.pin_memory(), xgt.pin_memory(), valid.pin_memory()
    return x, xgt, valid


# ----------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's OWN modules (unmodified; byte-compiled into oracle/_ref/ by build() --
# oracle/reference_import.py) on the host cores, kind "reference"; only if they are not installed, the oracle's CPU
# restatement (kind "port").
# ----------------------------------------------------------------------------------------------
def _pick_threads(one_step_probe, cores):
    """ "all the host threads it can use": the thread count that is actually fastest on this host (128 threads on
    these small convolutions are far slower than 16-32), found on a 2-image probe."""
    import torch
    best_nt, best_t = cores, None
    for nt in sorted({n for n in (8, 16, 32, 64, cores) if n <= cores}):
        torch.set_num_threads(nt)
        one_step_probe()
        t0 = time.perf_counter()
        one_step_probe()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best_nt, best_t = nt, dt
    torch.set_num_threads(best_nt)
    return best_nt


def _time_cpu_steps(one_step, steps, warmup):
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        one_step()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return statistics.median(times)


def cpu_reference_run(cfg, steps, warmup, sample_images):
    """The unmodified reference: Networks.LSQ_layer.Net + Loss_crit.backprojection_loss, model.train(),
    zero_grad -> forward -> per-lane loss -> backward (BP/main.py:286-305,338-339), fp32, CPU."""
    import contextlib
    import io
    import torch
    from oracle import reference_import as ri
    if cfg["resize"] != 256:
        # the reference's own grid has +-inf in row 34 at --resize 320 and returns NaN (SURVEY.md 7.2 #10); it still
        # executes the same work, so it is timed; its outputs are not used
        pass
    ns = ri.import_reference("Backprojection_Loss")
    cores = os.cpu_count() or 1
    L, order, R = cfg["nclasses"], cfg["order"], cfg["resize"]
    Bs = max(1, min(cfg["batch"], sample_images))
    args = ri.make_args(ns, ["--nclasses", str(L), "--order", str(order), "--batch_size", str(Bs), "--mask_percentage",
                             str(cfg["mask"]), "--resize", str(R), "--loss_policy", "backproject", "--end_to_end", "True"]
                       + (["--clas", "1"] if cfg.get("clas") else []))
    torch.manual_seed(0)
    model = ns.LSQ_layer.Net(args)
    with contextlib.redirect_stdout(io.StringIO()):
        ns.utils.define_init_weights(model, "kaiming")
    model.train()
    crit = ns.Loss_crit.backprojection_loss(args)
    g = torch.Generator().manual_seed(0)
    x = torch.rand(Bs, 3, R, 2 * R, generator=g)
    xgt = torch.rand(Bs, 4, 56, generator=g, dtype=torch.float64) * 500.0
    valid = torch.ones(Bs, 4, 56, dtype=torch.float64)
    valid[:, :, :8] = 0
    gt_line = torch.zeros(Bs, 4)

    bce = torch.nn.BCEWithLogitsLoss()
    gt_cls = torch.ones(Bs, 4)
    gt_hor = torch.zeros(Bs, R)
    gt_hor[:, 80] = 1.0

    def one_step(n=Bs):
        model.zero_grad()
        out = model(x[:n], gt_line[:n], True)
        loss = sum(crit(out[l], xgt[:n, l], valid[:n, l])[0] for l in range(L)) / L
        if cfg.get("clas"):      # BP/main.py:321-326
            loss = loss + (bce(out[6], gt_cls[:n]) + bce(out[7], gt_hor[:n])).double()
        loss.backward()

    # the reference sizes its grid / constants for args.batch_size: the probe uses the full sample
    cores_used = _pick_threads(one_step, cores)
    med = _time_cpu_steps(one_step, steps, warmup)
    ri.purge()
    return {"value": Bs / med, "unit": "images/sec", "cores": cores_used, "kind": "reference",
            "sample": "%d steps x %d images (of the %d-image batch), fwd+bwd fp32, the reference's own Networks.LSQ_layer.Net + "
                      "Loss_crit.backprojection_loss (unmodified, from %s), torch %s CPU, %d threads (fastest of the tried "
                      "counts; host has %d), median step %.3f s"
                      % (steps, Bs, cfg["batch"], ri.REFERENCE_ROOT, torch.__version__, cores_used, cores, med),
            "ms_per_step": med * 1e3, "images_per_step": Bs}


def gpu_stock_reference_run(cfg, steps, warmup, allow_tf32):
    """Labelled extra (BASELINE.md section 2, "library-kernel comparison point"): the reference's OWN modules, unmodified, on
    the same B200 through stock PyTorch (cuDNN / cuBLAS / torch.inverse), `cudnn.benchmark = True` as BP/main.py:62 sets it,
    with torch's default TF32 convolutions (allow_tf32 True: 1e-3-accurate) or strict fp32 (False).  Eager launches, the
    way the reference runs.  None of this repo's kernels is on that path."""
    import contextlib
    import io
    import torch
    from oracle import reference_import as ri
    ns = ri.import_reference("Backprojection_Loss")
    L, order, R, B = cfg["nclasses"], cfg["order"], cfg["resize"], cfg["batch"]
    args = ri.make_args(ns, ["--nclasses", str(L), "--order", str(order), "--batch_size", str(B), "--mask_percentage",
                             str(cfg["mask"]), "--resize", str(R), "--loss_policy", "backproject", "--end_to_end", "True"], no_cuda=False)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32 = bool(allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    try:
        torch.manual_seed(0)
        model = ns.LSQ_layer.Net(args)
        with contextlib.redirect_stdout(io.StringIO()):
            ns.utils.define_init_weights(model, "kaiming")
        model = model.cuda().train()
        crit = ns.Loss_crit.backprojection_loss(args)
        g = torch.Generator().manual_seed(0)
        x = torch.rand(B, 3, R, 2 * R, generator=g).cuda()
        xgt = (torch.rand(B, 4, 56, generator=g, dtype=torch.float64) * 500.0).cuda()
        valid = torch.ones(B, 4, 56, dtype=torch.float64)
        valid[:, :, :8] = 0
        valid = valid.cuda()
        gt_line = torch.zeros(B, 4)

        def one_step():
            model.zero_grad()
            out = model(x, gt_line, True)
            loss = sum(crit(out[l], xgt[:, l], valid[:, l])[0] for l in range(L)) / L
            loss.backward()

        for _ in range(max(3, warmup)):
            one_step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one_step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
        ri.purge()
    return {"value": B / ms * 1e3, "unit": "images/sec", "ms_per_step": ms, "steps": steps,
            "what": "the reference's unmodified Networks.LSQ_layer.Net + backprojection_loss on this GPU through stock PyTorch %s "
                    "(cuDNN convolutions %s, cudnn.benchmark, eager launches)" % (torch.__version__, "TF32 (torch default)" if allow_tf32 else "fp32"),
            "accuracy": "convolutions in TF32: ~1e-3 from fp64 on beta (tests/test_tf32_emulation_cpu.py)" if allow_tf32 else "fp32"}


def cpu_port_run(cfg, steps, warmup, sample_images):
    import torch
    from oracle import erfnet_oracle as eo, lsq_oracle as lo, inputs
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    L, order, R = cfg["nclasses"], cfg["order"], cfg["resize"]
    Bs = max(1, min(cfg["batch"], sample_images))
    P = {k[4:]: torch.from_numpy(v).requires_grad_(True) for k, v in inputs.make_erfnet_params(3, L, seed=0).items()}
    M, Minv = lo.get_homography(R)
    grid = lo.projective_grid(R, 2 * R, M.astype("float32"))
    crit = lo.BackprojectionLoss(order, R, M=M, M_inv=Minv)
    zero_rows = lo.mask_rows(R, cfg["mask"])
    g = torch.Generator().manual_seed(0)
    x = torch.rand(Bs, 3, R, 2 * R, generator=g)
    xgt = torch.rand(Bs, 4, 56, generator=g, dtype=torch.float64) * 500.0
    valid = torch.ones(Bs, 4, 56, dtype=torch.float64)
    valid[:, :, :8] = 0
    drop_p = {p: (0.03 if p.startswith("encoder.layers.") and int(p.split(".")[-1]) < 6 else 0.3) for p, _ in eo.ENC_NB}

    def one_step(xb, xgtb, validb):
        for p in P.values():
            p.grad = None
        nb = xb.shape[0]
        masks = {k: (torch.rand(nb, P[k + ".bn2.weight"].numel()) >= pr).float() / (1 - pr) for k, pr in drop_p.items()}
        # masked rows are skipped (identical to multiplying by zero for finite grids; at resize 320 the
        # reference itself yields NaN, SURVEY.md 7.2 #10)
        loss, _, _, _ = eo.full_step(xb, P, grid, order, L, zero_rows, xgtb, validb, drop_masks=masks, loss_obj=crit,
                                     resize=R, skip_rows=zero_rows if R != 256 else 0)
        loss.backward()

    cores_used = _pick_threads(lambda: one_step(x[:2], xgt[:2], valid[:2]), cores)
    med = _time_cpu_steps(lambda: one_step(x, xgt, valid), steps, warmup)
    return {"value": Bs / med, "unit": "images/sec", "cores": cores_used, "kind": "port",
            "sample": "%d steps x %d images (of the %d-image batch), fwd+bwd fp32, torch-CPU oracle port of the "
                      "reference modules, %d threads (fastest of the tried counts; host has %d), median step %.3f s"
                      % (steps, Bs, cfg["batch"], cores_used, cores, med),
            "ms_per_step": med * 1e3, "images_per_step": Bs}


def cpu_baseline_run(cfg, steps, warmup, sample_images):
    """Real reference if it is reachable (kind "reference"), else the oracle port (kind "port")."""
    try:
        from oracle import reference_import as ri
        if ri.available():
            return cpu_reference_run(cfg, steps, warmup, sample_images)
    except Exception as e:      # missing dependency on this host, ...: say so and fall back
        sys.stderr.write("reference arm: the reference modules could not be run (%s: %s); timing the oracle port\n"
                         % (type(e).__name__, e))
    return cpu_port_run(cfg, steps, warmup, sample_images)


def run_reference_arm(a, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_baseline_run(cfg, a.steps, a.warmup, a.cpu_sample)
    line = {"impl": "reference", "metric": "images/sec (fwd+bwd)", "value": r["value"], "unit": "images/sec",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": {"workload": cfg["name"], "per_gpu_batch": cfg["batch"], "images_per_step": r["images_per_step"],
                       "resolution": "%dx%d" % (cfg["resize"], 2 * cfg["resize"])},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------
def _arm_watchdog(seconds):
    """A hung collective must not burn the box: after `seconds` of wall clock dump the stacks and exit non-zero."""
    import faulthandler
    import signal

    def on_alarm(signum, frame):
        sys.stderr.write("bench.py watchdog: no result after %d s, aborting\n" % seconds)
        faulthandler.dump_traceback(file=sys.stderr, all_threads=True)
        sys.stderr.flush()
        os._exit(3)

    signal.signal(signal.SIGALRM, on_alarm)
    signal.alarm(seconds)
    # SIGALRM handlers only run between bytecodes: a main thread blocked inside a C++ call (NCCL teardown, a hung
    # collective) never gets there.  faulthandler's watchdog is a C thread that needs neither the GIL nor the main thread.
    faulthandler.dump_traceback_later(seconds + 15, exit=True, file=sys.stderr)


def dump_outputs(outdir, model, loss):
    """The loss (float64), every parameter gradient and the BatchNorm running statistics (float32) of the step just run,
    one DIR/<name>.npy each."""
    import numpy as np
    import torch
    arrays = {"loss": loss}
    arrays.update(("grad." + n, p.grad) for n, p in model.named_parameters() if p.grad is not None)
    arrays.update(("buffer." + n, b) for n, b in model.named_buffers() if n.endswith(("running_mean", "running_var")))
    arrays = {n: t.detach().cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)
              for n, t in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes of outputs exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(outdir, exist_ok=True)
    for n, v in arrays.items():
        np.save(os.path.join(outdir, n + ".npy"), v)


def run_ours(a, cfg):
    import torch
    import torch.distributed as dist
    from lanedetection_end2end_b200 import _capi
    from lanedetection_end2end_b200.Networks.LSQ_layer import Net
    from lanedetection_end2end_b200.Networks.utils import define_init_weights
    from lanedetection_end2end_b200.Loss_crit import backprojection_loss
    from lanedetection_end2end_b200.ddp import FlatGradAllReduce, broadcast_parameters

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _capi.lib()     # fail loudly if the extension is missing
    from lanedetection_end2end_b200 import ops_net
    ops_net.set_conv_mode(a.conv_mode)

    args = build_args(cfg)
    L, B = cfg["nclasses"], cfg["batch"]
    torch.manual_seed(0)
    model = Net(args)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        define_init_weights(model, "kaiming")
    model = model.cuda().train()
    model.defer_status_check = True
    crit = backprojection_loss(args)
    broadcast_parameters(model)
    reducer = FlatGradAllReduce(model) if world > 1 else None

    hx, hxgt, hvalid = host_batch(cfg, 1234 + rank, pinned=True)
    dx, dxgt, dvalid = hx.to(dev), hxgt.to(dev), hvalid.to(dev)
    gt_line = torch.zeros(B, 4)

    clas = bool(cfg.get("clas"))
    if clas:
        # BP/main.py:109-110,321-326: BCEWithLogits on the two heads, added with weight_class = weight_fit = 1
        bce = torch.nn.BCEWithLogitsLoss()
        gt_cls = torch.ones(B, 4, device=dev)
        gt_hor = torch.zeros(B, cfg["resize"], device=dev)
        gt_hor[:, 80] = 1.0

    extra_loss = (lambda out: (bce(out[6], gt_cls) + bce(out[7], gt_hor)).double()) if clas else None

    def step(x, xgt, valid):
        model.zero_grad(set_to_none=True)
        out = model(x, gt_line, True)
        loss = 0
        for l in range(L):
            ll, _ = crit(out[l], xgt[:, l], valid[:, l])
            loss = loss + ll
        loss = loss / L
        if clas:
            loss = loss + extra_loss(out)
        loss.backward()
        if reducer is not None:
            reducer()
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    for _ in range(max(a.warmup, 3)):
        step(dx, dxgt, dvalid)
    barrier()
    st = int(model.lsq_status.item())
    if st:
        raise RuntimeError("LSQ status %d during warm-up" % st)
    l0 = _capi.LAUNCHES
    step(dx, dxgt, dvalid)
    launches = _capi.LAUNCHES - l0

    gstep = None
    if a.graph:
        from lanedetection_end2end_b200.engine import GraphedTrainStep
        ok = 1
        try:
            gstep = GraphedTrainStep(model, crit, L, dx, dxgt, dvalid, reducer,
                                     capture_error_mode="thread_local" if world > 1 else "global", extra_loss=extra_loss)
        except Exception as e:        # capture failed: report it and measure eagerly instead
            sys.stderr.write("CUDA graph capture failed (%s: %s); falling back to eager launches\n" % (type(e).__name__, e))
            ok = 0
            torch.cuda.synchronize()
        if world > 1:                 # every rank must take the same path (the graph holds the all-reduce)
            flag = torch.tensor([ok], device=dev, dtype=torch.int32)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            ok = int(flag.item())
        if ok:
            for _ in range(max(a.warmup, 3)):
                gstep()
            barrier()
        else:
            gstep = None
            a.graph = False

    def dev_step():
        if gstep is not None:
            gstep()
        else:
            step(dx, dxgt, dvalid)

    if gstep is not None:
        gstep.prefetch(hx, hxgt, hvalid)          # batch 0 of the e2e loop

    last_loss = [None]

    def e2e_step():
        if gstep is not None:
            # double-buffered loader: every step copies one batch host->device (pinned, copy stream) — the
            # batch of the NEXT step, overlapped with this step's compute — and reads the loss back
            gstep.swap_in()
            gstep.prefetch(hx, hxgt, hvalid)
            loss = gstep()
        else:
            loss = step(hx.to(dev, non_blocking=True), hxgt.to(dev, non_blocking=True), hvalid.to(dev, non_blocking=True))
        last_loss[0] = loss
        v = float(loss.item())                    # D2H read of the step's result
        st = int(model.lsq_status.item())
        if st:
            raise RuntimeError("status word %d (1 singular / 2 non-finite / 4 not positive definite normal matrix)" % st)
        return v

    sampler = ClockSampler(local) if rank == 0 else None
    ms_dev = timed(dev_step, a.steps)
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, a.steps)
    clocks = sampler.stop() if sampler is not None else None
    if a.dump_outputs and rank == 0:
        # the end-to-end loop is the last timed loop; the extra arms and the traced step below overwrite the gradients
        dump_outputs(a.dump_outputs, model, last_loss[0])

    # extra arms (N=1 only: single-GPU diagnostics, and a second graph capture with NCCL inside is not worth the risk of
    # ranks diverging on a capture error): the same step in the other two convolution modes, timed the same way and
    # reported next to the headline as LABELLED extras -- never the headline
    extras = {}
    if a.parity_arm and world == 1:
        for mode, label in (("fp32", "fp32_ffma_mode"), ("tf32", "tf32_single_pass_mode")):
            if mode == a.conv_mode:
                continue
            ops_net.set_conv_mode(mode)
            try:
                psteps = max(3, a.steps // 2)
                pg = None
                if a.graph:
                    from lanedetection_end2end_b200.engine import GraphedTrainStep
                    try:
                        pg = GraphedTrainStep(model, crit, L, dx, dxgt, dvalid, None, extra_loss=extra_loss)
                    except Exception as e:
                        sys.stderr.write("%s: graph capture failed (%s: %s); timing eager launches\n" % (label, type(e).__name__, e))
                        pg = None
                        torch.cuda.synchronize()
                if pg is not None:
                    for _ in range(3):
                        pg()
                    pms = timed(lambda: pg(), psteps)
                    del pg
                else:
                    for _ in range(3):
                        step(dx, dxgt, dvalid)
                    pms = timed(lambda: step(dx, dxgt, dvalid), psteps)
                extras[label] = {"dtype": MODE_DTYPE[mode], "conv_mode": MODE_TEXT[mode], "accuracy": MODE_ACCURACY[mode],
                                 "value": world * B * psteps / (pms * 1e-3), "unit": "images/sec",
                                 "ms_per_step": pms / psteps, "steps": psteps, "inputs": "resident in HBM"}
            finally:
                ops_net.set_conv_mode(a.conv_mode)
        # experiment: 3xTF32 forward / input gradients with single-pass TF32 weight gradients (ops_net.WGRAD_SINGLE_PASS)
        ops_net.WGRAD_SINGLE_PASS = True
        try:
            psteps = max(3, a.steps // 2)
            from lanedetection_end2end_b200.engine import GraphedTrainStep
            pg = GraphedTrainStep(model, crit, L, dx, dxgt, dvalid, None, extra_loss=extra_loss) if a.graph else None
            fn = (lambda: pg()) if pg is not None else (lambda: step(dx, dxgt, dvalid))
            for _ in range(3):
                fn()
            pms = timed(fn, psteps)
            del pg
            extras["tf32x3_with_single_pass_tf32_weight_gradients"] = {
                "value": world * B * psteps / (pms * 1e-3), "unit": "images/sec", "ms_per_step": pms / psteps, "steps": psteps,
                "accuracy": "activations, beta, loss and input gradients as the default mode; PARAMETER gradients carry TF32 rounding "
                            "noise (~5e-4 norm-wise): above the 1e-4 the north star names, so never the headline",
                "inputs": "resident in HBM"}
        except Exception as e:
            extras["tf32x3_with_single_pass_tf32_weight_gradients"] = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
        finally:
            ops_net.WGRAD_SINGLE_PASS = False
        if cfg["resize"] == 256 and not cfg.get("clas"):
            for tf32, label in ((True, "stock_pytorch_reference_gpu_tf32"), (False, "stock_pytorch_reference_gpu_fp32")):
                try:
                    extras[label] = gpu_stock_reference_run(cfg, max(3, a.steps // 2), 3, tf32)
                except Exception as e:      # the reference's GPU path is not ours to fix: report why it did not run
                    extras[label] = {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
                torch.cuda.empty_cache()

    # one traced step: CUDA events around every C-ABI launch on the launching stream
    table, roofline, roofline_lsq, roofline_kernels = None, None, None, None
    peaks = load_peaks()
    # every rank runs the step (it contains the gradient all-reduce); only rank 0 records the events
    if rank == 0:
        _capi.TRACE = []
    step(dx, dxgt, dvalid)
    torch.cuda.synchronize()
    if rank == 0:
        trace, _capi.TRACE = _capi.TRACE, None
        agg = {}
        for name, e0, e1, flops, nbytes in trace:
            d = agg.setdefault(name, {"launches": 0, "ms": 0.0, "flops": 0, "bytes": 0})
            d["launches"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += flops
            d["bytes"] += nbytes
        tot = sum(d["ms"] for d in agg.values())
        table = {k: dict(v, share=v["ms"] / tot if tot else 0.0) for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}
        dom = next(iter(table))
        d = table[dom]
        hbm_peak = peaks.get("hbm_gbs", FALLBACK_PEAKS["hbm_gbs"])
        bf16_peak = peaks.get("bf16_tflops_sustained", FALLBACK_PEAKS["bf16_tflops_sustained"])
        tf32_peak = bf16_peak / 2.0     # MEASURED_PEAKS.json has no TF32 entry: dense TF32 = half the dense bf16 rate
        TENSOR_KERNELS = {"lf_conv1d_tc_x3": 3, "lf_conv1d_tc": 1, "lf_wgrad3_tc_x3": 3, "lf_wgrad3_tc": 1, "lf_conv_tcg": None,
                          "lf_wgrad_tcg": None}

        def kernel_roofline(name, dd):
            """SURVEY.md 8(d): the conv / weight-gradient kernels are judged against the TENSOR roof (algorithmic FLOPs, i.e.
            one multiply-add per product, over the TF32 dense rate), everything else against HBM; the other roof is kept
            beside it."""
            ach_b = dd["bytes"] / (dd["ms"] * 1e-3) / 1e9 if dd["bytes"] else None
            ach_f = dd["flops"] / (dd["ms"] * 1e-3) / 1e12 if dd["flops"] else None
            base = {"kernel": name, "launches_per_step": dd["launches"], "avg_launch_ms": dd["ms"] / dd["launches"],
                    "share_of_step": dd["share"]}
            hbm = None if ach_b is None else {"bound": "hbm", "achieved": ach_b, "peak": hbm_peak, "unit": "GB/s", "frac": ach_b / hbm_peak}
            tens = None if ach_f is None else {"bound": "tensor", "achieved": ach_f, "peak": tf32_peak, "unit": "TFLOP/s",
                                               "frac": ach_f / tf32_peak}
            if name in TENSOR_KERNELS and tens is not None:
                passes = TENSOR_KERNELS[name] or (3 if a.conv_mode == "tf32x3" else 1)
                return dict(base, **tens, other_roof=hbm,
                            peak_source=peaks["_source"] + ": 1/2 of the sustained dense bf16 rate (no TF32 entry in MEASURED_PEAKS.json)",
                            algorithmic="2 * pixels * taps * Cin * Cout FLOPs per launch (one multiply-add per product)",
                            tensor_passes_per_product=passes,
                            tensor_pipe_work_frac=passes * tens["frac"])
            if hbm is not None:
                return dict(base, **hbm, other_roof=tens, peak_source=peaks["_source"] + " (copy bandwidth)",
                            algorithmic="every input / output tensor of the launch once, 4 B per element")
            return None

        roofline = kernel_roofline(dom, d)
        # DRAM traffic per launch of the dominant kernel: a STATIC figure from the committed `ncu --set full` capture of this
        # kernel (profiles/r02), taken on this workload's shapes -- not measured in this run; null for other workloads
        if roofline is not None:
            roofline["traffic"], roofline["traffic_source"] = None, None
            try:
                cap = json.load(open(os.path.join(ROOT, "profiles", "r02", "ncu_%s.json" % dom)))
                if cap.get("workload") == cfg["name"] and cap.get("batch") == B:
                    roofline["traffic"] = cap["mean_traffic_bytes_per_launch"]
                    roofline["traffic_source"] = "static: profiles/r02/ncu_%s.json (%s)" % (dom, cap.get("how", ""))
            except (OSError, ValueError, KeyError):
                pass
        roofline_kernels = [r for r in (kernel_roofline(k, v) for k, v in list(table.items())[:10]) if r is not None]
        for k in ("lf_lsq_fwd", "lf_lsq_bwd"):
            if k in table:
                dd = table[k]
                ach = dd["bytes"] / (dd["ms"] * 1e-3) / 1e9
                roofline_lsq = roofline_lsq or {}
                roofline_lsq[k] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                                   "frac": ach / hbm_peak, "avg_launch_ms": dd["ms"] / dd["launches"],
                                   "note": "algorithmic bytes (SURVEY.md 8d: no credit for the masked rows the kernel skips); "
                                           "launch-latency regime at this size; see tools/bench_lsq.py for the stress config"}

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        cpu = cpu_baseline_run(cfg, 4, 1, a.cpu_sample)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        imgs = world * B * a.steps
        h2d = hx.numel() * 4 + hxgt.numel() * 8 + hvalid.numel() * 8
        gflop = (FWD_GFLOP_PER_IMG_CLAS if cfg.get("clas") else FWD_GFLOP_PER_IMG).get((L, cfg["resize"]))
        line = {"metric": "images/sec (fwd+bwd)", "value": imgs / (ms_dev * 1e-3), "unit": "images/sec",
                "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_dev / a.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": MODE_DTYPE[a.conv_mode], "data": "synthetic",
                "config": {"workload": cfg["name"], "per_gpu_batch": B, "global_batch": world * B,
                           "resolution": "%dx%d" % (cfg["resize"], 2 * cfg["resize"]), "nclasses": L,
                           "order": cfg["order"], "parallelism": "dp%d" % world,
                           "l2": "no flush needed: ~6 GB of activations per step >> 126 MB L2",
                           "conv_mode": a.conv_mode + ": " + MODE_TEXT[a.conv_mode],
                           "init": "kaiming, torch.manual_seed(0)",
                           "launch": "one CUDA graph replay per step" if a.graph else "eager launches"},
                "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/sec", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": 12, "ms_per_step": ms_e2e / a.steps,
                        "h2d": ("double-buffered: each step copies the next step's batch from pinned host memory on a "
                                "copy stream while this step computes" if a.graph else "synchronous with the step")},
                "gpu_launches": launches * a.steps, "gpu_launches_per_step": launches,
                "clocks": clocks,
                "algorithmic_tflops": (3 * gflop * imgs / 1e3) / (ms_dev * 1e-3) if gflop else None,
                "roofline": roofline, "roofline_kernels": roofline_kernels, "roofline_lsq": roofline_lsq, "cpu_baseline": cpu,
                "extra_modes": extras or None, "accuracy": MODE_ACCURACY[a.conv_mode]}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without ProcessGroupNCCL's teardown: with a captured graph still referencing the communicator
        # destroy_process_group() blocked until the launcher's timeout (session 15: the JSON line was out, the process
        # never exited).  Every rank is past its last collective here.
        gstep = None
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None, help="per-GPU batch override")
    ap.add_argument("--clas", action="store_true",
                    help="add the Classification heads (--clas 1 of BP/train.sh:1; SURVEY.md 8f-2) and their BCE losses to the step")
    ap.add_argument("--cpu-sample", dest="cpu_sample", type=int, default=32,
                    help="images per CPU-baseline / reference-arm step (default: the whole 32-image batch of config 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="launch every kernel eagerly instead of replaying the whole step as one CUDA graph")
    ap.add_argument("--no-parity-arm", "--no-extra-arms", dest="parity_arm", action="store_false",
                    help="skip the two labelled extra timings (fp32 FFMA mode, single-pass TF32 mode) reported next to the headline")
    ap.add_argument("--conv-mode", dest="conv_mode", default=os.environ.get("LANEFIT_CONV_MODE", "tf32x3"),
                    choices=["fp32", "tf32", "tf32x3"],
                    help="tf32x3 = tcgen05 with 3xTF32 operand splits (fp32-grade, default); tf32 = single-pass TF32 on tcgen05 "
                         "(labelled extra, 1e-3 accuracy); fp32 = CUDA-core FFMA kernels")
    ap.add_argument("--max-seconds", dest="max_seconds", type=int, default=int(os.environ.get("LANEFIT_BENCH_MAX_SECONDS", "900")),
                    help="wall-clock watchdog: abort (exit 3, stacks on stderr) instead of hanging the box")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the loss, parameter gradients and BatchNorm running statistics of the last timed step "
                         "as DIR/<name>.npy (--impl ours only)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to this project's arm only (--impl ours)")
    if a.max_seconds > 0:
        _arm_watchdog(a.max_seconds)
    cfg = dict(CONFIGS[a.config])
    if a.batch:
        cfg["batch"] = a.batch
    if a.clas:
        cfg["clas"] = True
        cfg["name"] += "_clas"
    if a.impl == "reference":
        run_reference_arm(a, cfg)
    else:
        run_ours(a, cfg)


if __name__ == "__main__":
    main()
