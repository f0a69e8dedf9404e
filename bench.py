#!/usr/bin/env python
"""bench.py -- images/sec of the PackNet01 640x192 self-supervised training step on N B200s (one process
per GPU, NCCL), plus the roofline numbers of the hot kernels and the CPU baseline (BASELINE.json metric).

  python bench.py --gpus 1 --steps K --warmup W          our arm (sm_100a kernels)
  python bench.py --impl reference ...                   the reference's algorithm on the host CPU cores
                                                         (oracle port: the Python reference cannot travel)
For N>1 the driver launches `python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...`.
A step = forward (PackNet01 + PoseNet) + photometric loss + backward + gradient all-reduce + Adam."""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


_T0 = time.time()


def log(msg):
    """progress to stderr (stdout carries exactly one JSON line)"""
    sys.stderr.write("[bench %7.1fs] %s\n" % (time.time() - _T0, msg))
    sys.stderr.flush()


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4, help="images per GPU (BASELINE configs[1]: 4)")
    ap.add_argument("--height", type=int, default=192)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "tf32x3", "tf32x1"],
                    help="tensor-core GEMM mode; bf16x3 and tf32x3 meet the 1e-3 depth parity bar, tf32x1 does not")
    ap.add_argument("--no-graph", action="store_true",
                    help="enqueue every step eagerly instead of replaying the captured whole-step CUDA graphs (flip / no flip)")
    ap.add_argument("--set", action="append", default=[], metavar="KEY=0|1",
                    help="A/B switch of a kernel variant against its library default: pack_fold, loss_grouped, im2col_first, "
                         "stage_flat, gn_tree, unpack_tiled, pack_tiled (e.g. --set pack_fold=0 --set loss_grouped=0 = the round-1 path)")
    ap.add_argument("--no-overlap", action="store_true",
                    help="A/B (N > 1): ONE gradient all-reduce after the backward instead of buckets launched from the backward")
    ap.add_argument("--torch-adam", action="store_true",
                    help="A/B: torch.optim.Adam(fused) + per-call weight packing instead of packnet_sfm_b200.optim.FlatAdam")
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-stock-torch", action="store_true", help="skip the stock-PyTorch-on-the-GPU leg (oracle step on cuda)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what one more step of the timed path computes from the initial weights "
                         "(loss, metrics, depth maps, poses, a fixed sample of the updated parameters) as DIR/<name>.npy, "
                         "float32: identical inputs from run to run, to compare two builds output for output")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    def __init__(self, index):
        self.rows, self.stop, self.index = [], threading.Event(), index
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None, "reasons": reasons,
                "samples": len(self.rows)}


def make_host_batch(B, H, W, rank):
    from packnet_sfm_b200 import synthetic
    fr = synthetic.make_frames(B, H, W, seed=1234 + rank)
    pin = (lambda t: t.pin_memory()) if torch.cuda.is_available() else (lambda t: t)
    return {"rgb": pin(fr["rgb"]), "rgb_context": [pin(c) for c in fr["rgb_context"]], "intrinsics": pin(fr["intrinsics"])}


def to_device(hb, dev):
    b = {"rgb": hb["rgb"].to(dev, non_blocking=True), "rgb_context": [c.to(dev, non_blocking=True) for c in hb["rgb_context"]],
         "intrinsics": hb["intrinsics"].to(dev, non_blocking=True)}
    b["rgb_original"], b["rgb_context_original"] = b["rgb"], b["rgb_context"]   # synthetic frames: no colour jitter
    return b


def usable_cpus():
    """Host threads the process can really use: min(affinity, cgroup CPU quota).  The GPU box reports 128 logical
    CPUs but its cgroup grants 16 (cpu.max = "1600000 100000"); 128 OpenMP threads on 16 CPUs ran 10x slower."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return int(os.environ.get("PN_CPU_THREADS", n))


def cpu_baseline(args, steps, batch=1, budget_s=150.0):
    """The oracle port of the reference step on the host cores on a `batch`-image sample of the workload (batch = the
    workload's own batch in the --impl reference arm, 1 in the cpu_baseline leg of our arm); the number of timed steps is
    cut so that the leg stays inside `budget_s`."""
    from oracle.step_oracle import StepOracle
    from packnet_sfm_b200 import synthetic
    cores = usable_cpus()
    torch.set_num_threads(cores)
    fr = synthetic.make_frames(batch, args.height, args.width, seed=1234)
    orc = StepOracle()
    t0 = time.perf_counter()
    orc.step(fr)                                     # warm-up (allocations, oneDNN primitive caches)
    warm = time.perf_counter() - t0
    log("cpu baseline warm-up step (B=%d): %.1f s on %d threads" % (batch, warm, cores))
    steps = max(1, min(steps, int(budget_s / max(warm, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        orc.step(fr)
    dt = (time.perf_counter() - t0) / steps
    return {"value": batch / dt, "unit": "images/sec", "cores": cores, "kind": "port",
            "sample": "B=%d %dx%d full step (PackNet01+PoseNet fwd, loss, bwd, Adam), %d timed after 1 warm-up, "
                      "torch %s CPU fp32" % (batch, args.height, args.width, steps, torch.__version__),
            "ms_per_step": dt * 1e3, "steps": steps}


METRIC = "images/sec PackNet01 640x192 self-sup step (fwd+loss+bwd+allreduce+Adam)"


def workload_name(H, W, B):
    return ("PackNet01(1A)+PoseNet+MultiViewPhotometricLoss, synthetic %dx%d 3-frame triplets, batch=%d/GPU, "
            "4 scales upsampled, Adam lr 2e-4" % (H, W, B))


GRAD_BYTES = 129886704 * 4      # PackNet01 (128 294 020) + PoseNet (1 592 684) fp32 gradients, SURVEY.md 8(a21)


def bench_config(H, W, B, world):
    return {"workload": workload_name(H, W, B), "global_batch": B * world, "parallelism": "dp%d" % world,
            "l2": "no flush between steps: weights (0.5 GB) + activations (GBs) exceed the 126 MB L2",
            "grad_allreduce_bytes": GRAD_BYTES}


def ncu_metrics(tag):
    """Counters that only a profiler run can give (DRAM traffic, tensor-pipe activity) come from profiles/ncu_metrics.json,
    written by tools/ncu_extract.py from an `ncu --set full` capture and stamped with the commit it was taken at -- never
    from literals in this file (VERDICT r1 / ADVICE r1: they go stale when a kernel changes)."""
    p = os.path.join(ROOT, "profiles", "ncu_metrics.json")
    try:
        return json.load(open(p)).get(tag)
    except Exception:
        return None


def stock_torch_gpu(args, dev, steps=5):
    """BASELINE.md: "the stock PyTorch on B200 images/s to beat" -- the plain-PyTorch restatement of the reference step
    (oracle/step_oracle.py: the reference's own op sequence) on CUDA tensors, i.e. cuDNN / cuBLAS / ATen kernels, same
    batch and image size, with cudnn.allow_tf32 as PyTorch defaults it (True) and off (what the 1e-3 parity bar needs)."""
    from oracle.step_oracle import StepOracle
    from packnet_sfm_b200 import synthetic
    out = {}
    fr = synthetic.make_frames(args.batch, args.height, args.width, seed=1234)
    fr = {"rgb": fr["rgb"].to(dev), "rgb_context": [c.to(dev) for c in fr["rgb_context"]], "intrinsics": fr["intrinsics"].to(dev)}
    prev = torch.backends.cudnn.allow_tf32
    try:
        for tag, tf32 in (("tf32_default", True), ("fp32", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            orc = StepOracle(device=dev)
            for _ in range(3):
                orc.step(fr)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                orc.step(fr)           # float(loss) inside: one D2H read per step, like our e2e leg
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[tag] = {"images_per_sec": args.batch / (ms * 1e-3), "ms_per_step": ms, "cudnn_allow_tf32": tf32}
            del orc
            torch.cuda.empty_cache()
    except Exception as e:      # an OOM of the unfused program must not cost the main result
        out["failed"] = repr(e)[:300]
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    out["what"] = ("oracle/step_oracle.py (the reference's op sequence in plain PyTorch) on cuda, torch %s, B=%d %dx%d, %d steps "
                   "after 3 warm-ups" % (torch.__version__, args.batch, args.height, args.width, steps))
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B, H, W = args.batch, args.height, args.width
    # same metric / unit / config as the GPU arm: the whole per-GPU batch per step on the host cores (VERDICT r1: the B=1,
    # 3-step sample made the driver's comparison `same_config: false`); the step count is bounded to ~2.5 minutes
    cb = cpu_baseline(args, max(1, min(args.steps, 8)), batch=B)
    steps = cb["steps"]
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"],
            "unit": "images/sec", "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": cb["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(H, W, B, args.gpus),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def time_kernels(args, dev, pk):
    """Roofline numbers of the two hot kernels, timed alone with CUDA events on the launching stream."""
    from packnet_sfm_b200 import functional as PF, synthetic, _lib
    from packnet_sfm_b200.losses import MultiViewPhotometricLoss
    from packnet_sfm_b200.geometry import Pose
    from packnet_sfm_b200.models import YACS_LOSS_DEFAULTS
    B, H, W = args.batch, args.height, args.width
    res = {}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > L2 (126 MB)

    def timed(fn, iters=10):
        ts = []
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2]

    # fused warp + SSIM + L1 + automask-min + smoothness (HBM bound). Algorithmic bytes: SURVEY.md §8(d)
    fr = synthetic.make_frames(B, H, W, seed=5)
    # as the step calls it: the four maps at their own resolution, read nearest-upsampled by the kernel (a8 fused)
    inv = [d.to(dev).requires_grad_(True) for d in synthetic.make_inv_depths(B, H, W, seed=6, full_res=False)]
    vec = synthetic.make_pose_vecs(B, seed=7).to(dev)
    mats = [Pose.from_vec(vec[:, j], "euler").mat.requires_grad_(True) for j in range(2)]
    loss_fn = MultiViewPhotometricLoss(**YACS_LOSS_DEFAULTS)
    img, ctx, K = fr["rgb"].to(dev), [c.to(dev) for c in fr["rgb_context"]], fr["intrinsics"].to(dev)
    out = {}

    def fwd():
        out["o"] = loss_fn(img, ctx, inv, K, K, [Pose(m) for m in mats], nearest_upsample=True)

    def bwd():
        torch.autograd.grad(out["o"]["loss"], inv + mats, retain_graph=True)

    for _ in range(3):
        fwd(); bwd()
    torch.cuda.synchronize()
    # as in the step: replayed CUDA graphs (the eager calls carry ~60 us of host enqueue gaps per call, which is not kernel time)
    loss_timing = "cuda graph replay, L2 flushed before every replay"
    try:
        gf, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(gf):
            fwd()
        with torch.cuda.graph(gb, pool=gf.pool()):
            bwd()
        torch.cuda.synchronize()
        t_f, t_b = timed(gf.replay), timed(gb.replay)
    except Exception as e:
        log("loss graph capture failed (%s): eager timing" % repr(e)[:200])
        loss_timing = "eager calls, L2 flushed before every call"
        torch.cuda.synchronize()
        t_f, t_b = timed(fwd), timed(bwd)
    P_s = B * H * W * 4
    bytes_f, bytes_b = 48 * P_s, 44 * P_s
    from packnet_sfm_b200 import losses as _losses
    grouped = bool(_losses._grouped)
    shape_tag = "%dx%dx%d" % (B, H, W)
    nm_loss = ncu_metrics("loss_%s_%s" % ("grouped" if grouped else "tile", shape_tag))
    res["roofline_loss"] = {"bound": "hbm", "kernel": ("loss_group_kernel" if grouped else "loss_tile_kernel") + " fwd+bwd (incl. prep / finish launches)",
                            "achieved": (bytes_f + bytes_b) / ((t_f + t_b) * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                            "frac": (bytes_f + bytes_b) / ((t_f + t_b) * 1e-3) / 1e9 / pk["hbm_gbs"],
                            "traffic": (nm_loss or {}).get("dram_bytes"), "traffic_source": (nm_loss or {}).get("source"),
                            "traffic_commit": (nm_loss or {}).get("commit"),
                            "fwd_ms": t_f, "bwd_ms": t_b, "algorithmic_bytes": bytes_f + bytes_b, "peak_source": pk["source"],
                            "timing": loss_timing,
                            "calls": ("training call: pn_loss_forward_backward (loss + unit gradients in one tile launch) then pn_loss_backward_finish"
                                      if (grouped and _losses._fused_training) else "pn_loss_forward then pn_loss_backward")}
    # pack1 (tensor bound).  Reference formulation: Conv2d(2048 -> 64, 5x5) over the Conv3d-inflated tensor at H/2 x W/2
    # (201.3 GFLOP per image, SURVEY.md 8d).  What the step launches for it since round 2 is the FOLDED 7x7 convolution
    # 256 -> 64 of the space-to-depth tensor (12544/51200 of those MACs) -- the dominant conv_igemm launch of the step.
    h2, w2, cin, cout, k = H // 2, W // 2, 2048, 64, 5
    prec = PF.get_precision()
    flops_ref = 2.0 * B * h2 * w2 * cout * cin * k * k
    tf32_peak = pk["bf16_tflops"] / (1.0 if PF.is_bf16(prec) else 2.0)
    peak_source = pk["source"] + (" cuBLAS bf16" if PF.is_bf16(prec) else " cuBLAS bf16 / 2 (tf32 dense rate is half the bf16 rate)")
    w = (torch.rand(cout, cin, k, k, device=dev) - 0.5) * 0.01
    folded_path = PF.pack_fold_enabled(h2 * w2)
    if folded_path:
        kf, cf = k + 2, cin // 8
        xs = torch.rand(B, h2, w2, cf, device=dev) - 0.5
        wf = (torch.rand(cout, cf, kf, kf, device=dev) - 0.5) * 0.01
        with torch.no_grad():
            wp, wlo = PF._pack_weight(wf, False, prec)
            xh, xlo = PF._operands(xs, prec)
            for _ in range(2):
                PF._conv_raw(xh, xlo, wp, wlo, None, cout, kf, prec)
            t_c = timed(lambda: PF._conv_raw(xh, xlo, wp, wlo, None, cout, kf, prec), iters=5)
        flops = 2.0 * B * h2 * w2 * cout * cf * kf * kf
        kernel_name, tag = "conv_igemm_kernel (pack1 folded: %d -> %d, %dx%d at %dx%d, %s)" % (cf, cout, kf, kf, h2, w2, args.precision), "folded"
        # the whole block as the step runs it: nine weight folds + space-to-depth + operand split + weight packing +
        # conv_igemm + frame terms, against the REFERENCE formulation's FLOPs
        from packnet_sfm_b200 import folded
        x1 = torch.rand(B, H, W, 64, device=dev) - 0.5
        w3 = torch.rand(8, 1, 3, 3, 3, device=dev) - 0.5
        b3, b2 = torch.rand(8, device=dev) - 0.5, torch.rand(cout, device=dev) - 0.5
        with torch.no_grad():
            for _ in range(2):
                folded.pack_conv_folded(x1, w, b2, w3, b3, PF.conv2d)
            t_fold = timed(lambda: folded.pack_conv_folded(x1, w, b2, w3, b3, PF.conv2d), iters=5)
        res["roofline_pack1_block"] = {"bound": "tensor", "kernel": "pack1 block forward as launched: folds + s2d + split + pack + "
                                       "conv_igemm 7x7 + frame terms (%s)" % args.precision,
                                       "achieved": flops_ref / (t_fold * 1e-3) / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                                       "frac": flops_ref / (t_fold * 1e-3) / 1e12 / tf32_peak, "traffic": None, "ms": t_fold,
                                       "algorithmic_flops": flops_ref, "executed_mac_ratio": 12544.0 / 51200.0,
                                       "note": "achieved counts the REFERENCE formulation's FLOPs (Conv2d over the 8x-inflated "
                                               "channel count); the folded convolution executes 12544/51200 of them"}
    else:
        x = torch.rand(B, h2, w2, cin, device=dev) - 0.5
        with torch.no_grad():
            wp, wlo = PF._pack_weight(w, False, prec)
            xh, xlo = PF._operands(x, prec)
            for _ in range(2):
                PF._conv_raw(xh, xlo, wp, wlo, None, cout, k, prec)
            t_c = timed(lambda: PF._conv_raw(xh, xlo, wp, wlo, None, cout, k, prec), iters=5)
        flops = flops_ref
        kernel_name, tag = "conv_igemm_kernel (pack1 conv2d 2048 -> 64, 5x5, %s)" % args.precision, "pack1"
    nm_conv = ncu_metrics("conv_%s_%s_%s" % (tag, args.precision, shape_tag))
    res["roofline"] = {"bound": "tensor", "kernel": kernel_name,
                       "achieved": flops / (t_c * 1e-3) / 1e12, "peak": tf32_peak, "unit": "TFLOP/s",
                       "frac": flops / (t_c * 1e-3) / 1e12 / tf32_peak,
                       "traffic": (nm_conv or {}).get("dram_bytes"), "traffic_source": (nm_conv or {}).get("source"),
                       "traffic_commit": (nm_conv or {}).get("commit"),
                       "tensor_pipe_active_pct_ncu": (nm_conv or {}).get("tensor_pipe_active_pct"),
                       "ms": t_c, "algorithmic_flops": flops,
                       "mma_products_per_flop": 3 if PF.is_split(prec) else 1, "peak_source": peak_source,
                       # the same launch counted in executed MMA work (bf16x3 issues three products per algorithmic product)
                       "executed_mma_frac": flops / (t_c * 1e-3) / 1e12 / tf32_peak * (3 if PF.is_split(prec) else 1)}
    return res


def dump_outputs(directory, out, model, max_elems=1 << 21):
    """What a caller of the training step receives from a call: the loss, its metrics, the four inverse-depth maps, the two
    context poses, and the updated parameters.  The parameters (130 M) and any array of more than `max_elems` elements are
    stored as a fixed, seeded sample of `max_elems` of them, which bounds the files to about 40 MB."""
    import numpy as np
    arrays = {"loss": out["loss"], **out["metrics"]}
    arrays.update({"inv_depth%d" % i: d for i, d in enumerate(out["inv_depths"])})
    arrays.update({"pose%d" % j: p.mat for j, p in enumerate(out["poses"])})
    arrays["parameters"] = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > max_elems:
            idx = torch.randint(t.numel(), (max_elems,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(directory, name + ".npy"), t.cpu().numpy())
    log("outputs of the step from the initial state written to %s (%s)" % (directory, ", ".join(sorted(arrays))))


def apply_variants(settings, PF, _lib, _losses):
    """--set KEY=0|1 overrides; returns the EFFECTIVE setting of every variant (library defaults where not overridden)."""
    setters = {"pack_fold": lambda v: PF.set_pack_fold(v), "loss_grouped": _losses.set_grouped_kernel,
               "im2col_first": PF.set_im2col_first, "unpack_tiled": PF.set_unpack_tiled, "pack_tiled": PF.set_pack_tiled,
               "stage_flat": lambda v: _lib.set_tuning(_lib.PN_TUNE_STAGE_FLAT, int(v)),
               "gn_tree": lambda v: _lib.set_tuning(_lib.PN_TUNE_GN_TREE, int(v))}
    eff = {"pack_fold": PF.pack_fold_enabled(), "loss_grouped": bool(_losses._grouped), "im2col_first": PF.im2col_first_enabled(),
           "unpack_tiled": PF._state["unpack_tiled"], "pack_tiled": PF._state["pack_tiled"],
           "stage_flat": os.environ.get("PN_STAGE_FLAT", "1") != "0", "gn_tree": os.environ.get("PN_GN_TREE", "1") != "0"}
    for kv in settings:
        k, _, v = kv.partition("=")
        if k not in setters or v not in ("0", "1"):
            raise SystemExit("--set %s: expected one of %s with =0 or =1" % (kv, sorted(setters)))
        setters[k](v == "1")
        eff[k] = v == "1"
    return eff


def run_ours(args):
    args.graph = not args.no_graph
    import torch.distributed as dist
    from packnet_sfm_b200 import _lib, functional as PF, parallel
    from packnet_sfm_b200.models import SelfSupModel
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # Everything runs on ONE non-default stream from the first kernel on.  Autograd binds a parameter's AccumulateGrad node to
    # the stream of the first forward; nodes born on the legacy default stream make the later whole-step capture fail
    # ("operation would make the legacy stream depend on a capturing blocking stream", gpurun r02a).
    main_stream = torch.cuda.Stream(dev)
    torch.cuda.set_stream(main_stream)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    PF.set_precision({"bf16x3": PF.PRECISION_BF16X3, "tf32x3": PF.PRECISION_TF32X3, "tf32x1": PF.PRECISION_TF32X1}[args.precision])
    _lib.lib()          # fail loudly if the extension is missing
    torch.manual_seed(42)
    import random
    random.seed(42)
    log("building model")
    model = SelfSupModel().to(dev).train()
    log("model on device")
    parallel.broadcast_parameters(model)
    from packnet_sfm_b200 import losses as _losses, optim
    from packnet_sfm_b200.networks import gradient_buckets, native_conv_weights
    variants = apply_variants(args.set, PF, _lib, _losses)
    B, H, W = args.batch, args.height, args.width
    groups = [{"name": "Depth", "params": list(model.depth_net.parameters()), "lr": 2e-4},
              {"name": "Pose", "params": list(model.pose_net.parameters()), "lr": 2e-4}]
    if args.torch_adam:      # A/B: ATen's fused multi-tensor Adam + per-call weight packing + flat gradient bucket (round 1)
        bucket = parallel.FlatBucket(model.parameters())
        opt = torch.optim.Adam(groups, fused=True, capturable=bool(args.graph))
        zero_grad, reduce_grads = bucket.zero_grad, bucket.allreduce_mean
    else:                    # flat parameters / gradients / moments, one Adam launch that also writes the engine's weight tiles
        opt = optim.FlatAdam(groups, native=native_conv_weights(model.depth_net, (H, W)),
                             buckets=gradient_buckets(model.depth_net, (H, W)) if world > 1 and not args.no_overlap else None)
        zero_grad, reduce_grads = opt.zero_grad, opt.allreduce_mean
    hb = make_host_batch(B, H, W, rank)
    dbatch = to_device(hb, dev)
    state = {}
    if args.dump_outputs:
        # Two runs of the same steps drift apart (split-K partial sums land in any order, and Adam's first updates are
        # +-lr for every gradient that is only rounding noise): the dumped step starts again from this initial state.
        start = ([p.detach().clone() for p in model.parameters()], None if args.torch_adam else opt.state_dict())

    def restore_start():
        with torch.no_grad():
            for p, v in zip(model.parameters(), start[0]):
                p.copy_(v)
        if args.torch_adam:
            for st in opt.state.values():
                for v in st.values():
                    if torch.is_tensor(v):
                        v.zero_()
        else:
            opt.load_state_dict(start[1])
            opt.repack()            # the forward tiles of the stored weights (a replayed graph does not check them)

    def step(batch):
        zero_grad()
        out = model(batch)
        out["loss"].backward()
        reduce_grads()
        opt.step()
        state["out"] = out

    def timed_region(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for i in range(max(args.warmup, 3)):
        t_w = time.time()
        step(dbatch)
        torch.cuda.synchronize()
        log("warm-up step %d: %.1f ms (loss %.5f)" % (i, (time.time() - t_w) * 1e3, float(state["out"]["loss"].item())))
    eager_step = step
    graph_info = None
    graphs = None
    if args.graph:
        # Whole-step capture: the only host-side decision of a step is the random left-right flip of the depth
        # network (SfmModel.py:81-90) -> one graph per outcome, chosen every step by the same random.random() draw.
        # Gradients are freed before each capture so that the backward allocates them from the graph's pool.
        flip_prob = model.flip_lr_prob
        graphs = {}
        for fl in (False, True):
            model.flip_lr_prob = 1.0 if fl else 0.0
            eager_step(dbatch)
        torch.cuda.synchronize()
        per_graph_launches = 0
        try:
            for fl in (False, True):
                model.flip_lr_prob = 1.0 if fl else 0.0
                zero_grad()
                g = torch.cuda.CUDAGraph()
                l0 = _lib.launch_count()
                with torch.cuda.graph(g):
                    out = model(dbatch)
                    out["loss"].backward()
                    reduce_grads()
                    opt.step()
                per_graph_launches = _lib.launch_count() - l0
                # the loss module keeps ONE metrics dict, refilled by every call: hold this graph's own metric tensors
                graphs[fl] = (g, dict(out, metrics=dict(out["metrics"])))
        except Exception as e:      # a failed capture is not sticky: fall back to eager enqueue and say so in the JSON line
            log("whole-step capture failed (%s): falling back to eager steps" % repr(e)[:300])
            graphs = None
            try:
                torch.cuda.synchronize()
            except Exception:
                pass
        model.flip_lr_prob = flip_prob
        torch.cuda.synchronize()
        if graphs is not None:
            log("captured 2 step graphs (%d library launches each)" % per_graph_launches)
            graph_info = {"graphs": 2, "library_launches_per_graph": int(per_graph_launches)}

            def step(batch):
                # `batch` must be the static device batch the graphs were captured on (dbatch); e2e copies into it
                g, out = graphs[random.random() < flip_prob]
                g.replay()
                state["out"] = out

        for _ in range(2):
            step(dbatch)
        torch.cuda.synchronize()
        log("graph replay ok (loss %.5f)" % float(state["out"]["loss"].item()))
    # host time to ENQUEUE one step on an idle GPU (no sync inside): step time close to this = launch-bound
    torch.cuda.synchronize()
    t_q = time.perf_counter()
    step(dbatch)
    enqueue_ms = (time.perf_counter() - t_q) * 1e3
    torch.cuda.synchronize()
    log("host enqueue of one step: %.1f ms" % enqueue_ms)
    launches0 = _lib.launch_count()
    cpu0 = time.process_time()
    prof = os.environ.get("PN_CUDA_PROFILER") == "1"   # ncu --profile-from-start off: capture the timed region only
    if prof:
        torch.cuda.profiler.start()
    with ClockSampler(local) as clk:
        ms = timed_region(lambda: step(dbatch), args.steps)
    if prof:
        torch.cuda.profiler.stop()
    cpu_ms = (time.process_time() - cpu0) * 1e3 / args.steps     # host CPU time (all threads) per step
    launches = _lib.launch_count() - launches0
    if graph_info is not None:
        launches = graph_info["library_launches_per_graph"] * args.steps     # replayed kernel nodes of our library
    log("timed region: %.1f ms/step (host CPU %.1f ms/step), %d library launches" % (ms / args.steps, cpu_ms, launches))
    if args.dump_outputs:
        # one more step of the timed path (the same graphs, or eager steps) from the initial weights and optimizer state
        restore_start()
        random.seed(42)             # the same left-right flip draw whatever ran before (graphs, eager steps, warm-up count)
        step(dbatch)
        torch.cuda.synchronize()
        if rank == 0:
            dump_outputs(args.dump_outputs, state["out"], model)

    def e2e_step():
        if graph_info is not None:
            # H2D from pinned memory INTO the static tensors the graphs read
            dbatch["rgb"].copy_(hb["rgb"], non_blocking=True)
            for dst, src in zip(dbatch["rgb_context"], hb["rgb_context"]):
                dst.copy_(src, non_blocking=True)
            dbatch["intrinsics"].copy_(hb["intrinsics"], non_blocking=True)
            step(dbatch)
        else:
            step(to_device(hb, dev))
        state["loss_host"] = float(state["out"]["loss"].item())     # D2H read of the step's result

    e2e_step()
    ms_e2e = timed_region(e2e_step, args.steps)
    log("e2e region: %.1f ms/step" % (ms_e2e / args.steps))
    h2d = sum(t.numel() * 4 for t in [hb["rgb"], hb["intrinsics"]] + hb["rgb_context"])

    if rank == 0:
        pk = peaks()
        extra = time_kernels(args, dev, pk) if world == 1 else {}
        log("kernel rooflines done")
        imgs = B * world * args.steps
        line = {"metric": METRIC,
                "value": imgs / (ms * 1e-3), "unit": "images/sec", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 (tensor-core GEMMs: %s)" % args.precision, "data": "synthetic",
                "config": bench_config(H, W, B, world),
                "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": int(launches), "host_cpu_ms_per_step": cpu_ms, "host_enqueue_ms_per_step": enqueue_ms, "clocks": clk.summary(),
                "loss": state.get("loss_host"), "cuda_graph": graph_info, "variants": variants,
                "optimizer": "torch.optim.Adam(fused)" if args.torch_adam else "packnet_sfm_b200.optim.FlatAdam"}
        line.update(extra)
        if world == 1 and not args.no_stock_torch:
            line["stock_torch_gpu"] = stock_torch_gpu(args, dev)
            log("stock torch on the GPU: %s" % json.dumps(line["stock_torch_gpu"])[:300])
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, args.cpu_steps)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        # NCCL wants every CUDA graph that captured one of its collectives destroyed before the communicator (gpurun r02i: with
        # the step graphs alive destroy_process_group never returned and the ranks sat until the launcher's timeout)
        step = None
        if graphs is not None:
            graphs.clear()
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        bye = threading.Timer(20.0, lambda: os._exit(0))      # the JSON line is out: never let teardown hold the launcher
        bye.daemon = True
        bye.start()
        dist.destroy_process_group()
        bye.cancel()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
