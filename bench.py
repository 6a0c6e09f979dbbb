#!/usr/bin/env python
"""bench.py -- TANTE hot-path throughput on B200 (driver contract: one JSON line on rank 0).

    python bench.py --gpus N --steps K --warmup W            # the B200-native arm
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (oracle port)

Workload `train` (default; BASELINE.json configs[1], the configuration the metric is quoted on): one bf16
training step of TANTE (configs/tante.yaml: fixed-step, K=1, THWTHWTHW, patch 8) on the synthetic Active Matter
shape (11 fields, 256x256), batch 16 per GPU: 4 chained model calls with BPTT through the window
(trainer/trainer.py:144-159), MSE, backward, clip_grad_norm_(1.0), AdamW(lr 5e-5, wd 1e-5).  N > 1: data parallel,
one NCCL all-reduce of the flat gradient bucket per step (weak scaling).  value = training samples/s (whole job).

Workload `rollout` (BASELINE.json configs[2]): adaptive-step rollout inference on the synthetic
Rayleigh-Benard shape (4 fields, 512x128), n_steps_rollout frames per trajectory, trajectories sharded
over the ranks with NO data-path collective (weak scaling: fixed trajectories per GPU).
A "step" = one rollout pass over one batch of trajectories.  value = trajectories/s (whole job).

Timed regions use CUDA events on the launching stream, W >= 3 warm-up steps, inputs far larger than
L2 per step (stated in `config`), barrier + synchronize on both sides, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES = {  # SURVEY.md 8: (D, H, W)
    "trl": (4, 128, 384), "active_matter": (11, 256, 256), "rayleigh_benard": (4, 512, 128),
    "viscoelastic": (8, 512, 512),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "rollout"])
    ap.add_argument("--shape", default=None, choices=sorted(SHAPES))
    ap.add_argument("--batch", type=int, default=None, help="samples (train) / trajectories (rollout) per GPU per step")
    ap.add_argument("--n-steps-output", type=int, default=4, help="chained model calls per training sample")
    ap.add_argument("--n-roll", type=int, default=8)
    ap.add_argument("--taylor-order", type=int, default=1)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--rt-bias", type=float, default=0.0)
    ap.add_argument("--cpu-seconds", type=float, default=20.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the gpu_eager_baseline legs")
    ap.add_argument("--no-extras", action="store_true",
                    help="default line only: skip the rollout / head_sweep sub-records of the default (train) run")
    ap.add_argument("--amp-mix", action="store_true", help="rollout: per-trajectory input amplitudes (different step sequences)")
    ap.add_argument("--dropout", type=float, default=0.0, help="train: dropout probability (configs/tante.yaml:29 uses 0.1)")
    ap.add_argument("--global-batch", type=int, default=None,
                    help="strong scaling: total samples / trajectories per step, split evenly over the ranks")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32, rank 0)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if a.shape is None:
        a.shape = "active_matter" if a.workload == "train" else "rayleigh_benard"
    if a.batch is None:
        a.batch = 16 if a.workload == "train" else 64
    a.scaling = "weak"
    if a.global_batch:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if a.global_batch % world:
            raise SystemExit("--global-batch must be divisible by the number of ranks")
        a.batch = a.global_batch // world
        a.scaling = "strong"
    return a


def model_axes(K):
    return "-".join(["THWTHWTHW"] + ["THW"] * (K - 1))


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_setup(args):
    import torch
    from oracle import tante_oracle as O
    D, H, W = SHAPES[args.shape]
    cfg = O.OracleConfig(n_fields=D, H=H, W=W, taylor_order=args.taylor_order, attn_axes=model_axes(args.taylor_order),
                         deg=False)
    return O, cfg


def cpu_leg(args, seconds, state_dict=None):
    """The reference's CPU implementation of the path (oracle port of models/tante.py + r_evaler.py:87-105)
    on all host threads, on a bounded sample of the same workload: single-trajectory rollouts."""
    import torch
    O, cfg = oracle_setup(args)
    torch.set_num_threads(os.cpu_count() or 1)
    sd = state_dict if state_dict is not None else O.make_state_dict(cfg, 211, args.rt_bias)
    x = O.make_input(cfg, 1, 212)
    with torch.inference_mode():
        O.rollout_eval(sd, cfg, x, args.n_roll)            # warm-up
        t0 = time.perf_counter()
        n = 0
        while True:
            O.rollout_eval(sd, cfg, x, args.n_roll)
            n += 1
            el = time.perf_counter() - t0
            if el > seconds or n >= 64:
                break
    return {"value": n / el, "unit": "trajectories/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} single-trajectory rollouts (B=1, {args.n_roll} frames, {args.shape} shape, fp32, "
                      f"torch {torch.__version__} CPU) in {el:.1f}s"}, el / max(n, 1)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm = max(args.warmup, 1)
    steps = args.steps
    import torch
    O, cfg = oracle_setup(args)
    torch.set_num_threads(os.cpu_count() or 1)
    sd = O.make_state_dict(cfg, 211, args.rt_bias)
    x = O.make_input(cfg, 1, 212)
    # each step = a bounded sample of the workload: ONE trajectory rollout (the b200 arm does `batch` per step)
    with torch.inference_mode():
        for _ in range(min(warm, 2)):
            O.rollout_eval(sd, cfg, x, args.n_roll)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.rollout_eval(sd, cfg, x, args.n_roll)
        el = time.perf_counter() - t0
    val = steps / el
    D, H, W = SHAPES[args.shape]
    line = {
        "impl": "reference", "metric": "rollout_trajectories_per_s", "value": val, "unit": "trajectories/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * el / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(bench_config(args, 1), reference_arm=(
            "CPU port (oracle/tante_oracle.py, pinned to the live reference) of R_Evaler.rollout_model, one trajectory per "
            "step in fp32 as a bounded sample of the b200 arm's 64-trajectory bf16 workload (DESIGN.md 1); the same-GPU "
            "stock-PyTorch number is the b200 line's gpu_eager_baseline.")),
        "cpu_baseline": {"value": val, "unit": "trajectories/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{steps} single-trajectory rollouts, one per step"},
        "e2e": {"value": val, "unit": "trajectories/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def bench_config(args, batch):
    D, H, W = SHAPES[args.shape]
    return {"workload": f"adaptive rollout inference, synthetic {args.shape} shape ({D} fields, {H}x{W}), "
                        f"{args.n_roll} frames/trajectory (BASELINE.json configs[2])",
            "trajectories_per_gpu_per_step": batch, "n_steps_rollout": args.n_roll, "taylor_order": args.taylor_order,
            "attn_axes": model_axes(args.taylor_order), "patch_scale": 8, "embed_dim": 256, "deg": False,
            "weights": "random init, torch.manual_seed(211), reference initialisers", "rt_bias": args.rt_bias,
            "l2_hygiene": "per-step working set (latents+activations) >> 126 MB L2; no explicit flush",
            "parallelism": f"trajectory-sharded x{args.gpus}, no collective"}


CLASS_NAMES = {0: "gemm_tc_kernel, bf16/activation epilogue (QKV, MLP-in, convs, input gradients; K=64..768: below the ridge)",
               1: "gemm_tc_kernel, fp32 residual + LayerNorm / embedding epilogue (out-proj, MLP-out, conv3)",
               2: "wgrad_tc_kernel (weight gradients)",
               3: "block_tail_kernel (out-proj + residual + LN2 + MLP + residual + next LN1 fused: three chained tcgen05 GEMMs)",
               4: "mlp_bwd_kernel (input-gradient chain of the MLP fused: dY W2 -> gelu' -> W1, two chained tcgen05 GEMMs)"}


def ncu_traffic(workload, cls):
    """DRAM bytes of one representative launch of the class from the committed ncu capture (profiles/traffic_*.json)."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "traffic_*.json")), reverse=True):
        try:
            d = json.load(open(path))
            e = d.get(workload, {}).get(str(cls))
            if e:
                return e["traffic"], (f"static ncu --set full capture committed as profiles/{os.path.basename(path)} "
                                      f"({d.get('captured', 'round 1u')}; not measured in this run): {e['kernel']} "
                                      f"(algorithmic {e['algorithmic_bytes']} B)")
        except Exception:
            pass
    return None, None


def roofline_object(classes, gemm_ms, gemm_flops, gemm_n, K_, ms_prof, peaks, tensor_mode, workload="train"):
    """BASELINE roofline of the dominant kernel family.  The tcgen05 GEMM launches fall into classes with different
    bounds (tante_profile_read_class): the top-level numbers are those of the class with the largest share of the step;
    every class is listed under `classes` (tensor classes in TFLOP/s vs the measured bf16 peak, HBM classes in
    algorithmic GB/s vs the measured copy bandwidth)."""
    if tensor_mode:
        tpeak = peaks.get("bf16_tflops_sustained") or 1400.0
        tsrc = ("MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained")
    else:
        tpeak, tsrc = 72.0, "nominal fp32 FFMA 72 TFLOP/s (no measured fp32 peak in MEASURED_PEAKS.json)"
    hpeak = peaks.get("hbm_gbs") or 6650.0
    hsrc = "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"
    out_cls = {}
    for cls, (ms, fl, by, n) in classes.items():
        if n == 0 or ms <= 0:
            continue
        tf = fl / (ms * 1e-3) / 1e12
        gb = by / (ms * 1e-3) / 1e9
        # classes 1 and 2 are HBM-bound by construction; class 0 (K = 64..768 GEMMs streaming their operands from HBM)
        # is HBM-bound too whenever its arithmetic intensity is below the ridge point of the measured peaks
        hbm_bound = cls != 0 or (by > 0 and fl / by < (tpeak * 1e12) / (hpeak * 1e9))
        out_cls[cls] = {
            "kernel": CLASS_NAMES[cls] if tensor_mode else CLASS_NAMES[cls].replace("_tc_", "_simt_"),
            "bound": "hbm" if hbm_bound else "tensor",
            "achieved": gb if hbm_bound else tf, "peak": hpeak if hbm_bound else tpeak,
            "unit": "GB/s" if hbm_bound else "TFLOP/s", "frac": (gb / hpeak) if hbm_bound else (tf / tpeak),
            "tflops": tf, "algorithmic_GBps": gb, "flop_per_byte": (fl / by) if by > 0 else None,
            "frac_of_tensor_peak": tf / tpeak, "frac_of_hbm_peak": gb / hpeak, "launches": int(n), "avg_us_per_launch": 1e3 * ms / n,
            "ms_per_step": ms / K_, "share_of_step": ms / ms_prof,
        }
    all_tf = (gemm_flops / (gemm_ms * 1e-3)) / 1e12 if gemm_ms > 0 else None
    dom = max(out_cls, key=lambda c: out_cls[c]["ms_per_step"]) if out_cls else None
    top = dict(out_cls[dom]) if dom is not None else {"kernel": "gemm", "bound": "tensor", "achieved": all_tf, "peak": tpeak,
                                                        "unit": "TFLOP/s", "frac": (all_tf / tpeak) if all_tf else None}
    traffic, traffic_src = ncu_traffic(workload, dom) if dom is not None else (None, None)
    top.update({
        "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": f"{hsrc}; {tsrc}",
        "all_gemm_launches": int(gemm_n), "all_gemm_ms_per_step": gemm_ms / K_, "all_gemm_share_of_step": gemm_ms / ms_prof,
        "all_gemm_tflops": all_tf, "all_gemm_frac_of_tensor_peak": (all_tf / tpeak) if all_tf else None,
        "algorithmic_flops_per_step": gemm_flops / K_,
        "classes": {str(c): v for c, v in out_cls.items()},
        "note": ("per launch: algorithmic bytes (operands + outputs once; weights excluded, L2-resident) or 2*M*N*K flops / "
                 "CUDA-event time on the launch stream, summed over every launch of the class in K steps; the top-level "
                 "entry is the class with the largest share of the step"),
    })
    return top


def _dist_helpers(dev, world):
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms
    return barrier, max_over_ranks


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


DUMP_MAX_ELEMS = 6 << 20      # per array: a dump holds at most two arrays this large, so it stays under 64 MB


def flat(tensors):
    """One 1-D tensor of the given tensors' elements; complex tensors contribute (re, im) pairs."""
    import torch
    return torch.cat([(torch.view_as_real(t) if t.is_complex() else t).detach().reshape(-1) for t in tensors])


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy in float32.  A tensor of more than DUMP_MAX_ELEMS elements is replaced by
    the same seeded sample of its flattened elements on every run, so that two builds run with the same arguments can be
    compared output for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


AMP_MIX = (0.25, 1.0, 2.0, 4.0)      # per-trajectory input amplitudes of the `adaptive` rollout record


def rollout_measure(args, dev, world, rank, with_cpu_baseline=True, dump_dir=None):
    """BASELINE configs[2]: per-sample adaptive rollout, `args.batch` trajectories per GPU per step.  Returns the JSON
    record on rank 0 (None elsewhere).  args.rt_bias shifts the interprators' last bias (SURVEY F7); args.amp_mix scales
    trajectory i's window by AMP_MIX[i % 4] so that trajectories of one batch take different step sequences."""
    import torch
    from tante_b200 import TANTE, TanteMetadata
    barrier, max_over_ranks = _dist_helpers(dev, world)
    D, H, W = SHAPES[args.shape]
    B, n_roll = args.batch, args.n_roll

    torch.manual_seed(211)                                 # configs/tante.yaml:1
    model = TANTE(4, TanteMetadata(spatial_resolution=(H, W), n_fields=D), taylor_order=args.taylor_order,
                  attn_axes=model_axes(args.taylor_order), patch_scale=8, deg=False, dropout=0.0,
                  precision=args.precision)
    if args.rt_bias:
        with torch.no_grad():
            for ip in model.interprators:
                ip.interprete[4].bias.add_(args.rt_bias)
    model = model.to(dev).eval()

    g = torch.Generator().manual_seed(212 + rank)
    host_in = torch.randn(B, 4, D, H, W, generator=g)
    if getattr(args, "amp_mix", False):
        host_in *= torch.tensor([AMP_MIX[i % len(AMP_MIX)] for i in range(B)]).view(B, 1, 1, 1, 1)
    host_in = host_in.pin_memory()
    host_out = torch.empty(B, n_roll, H, W, D).pin_memory()
    dev_in = host_in.to(dev)
    calib = None
    if getattr(args, "amp_mix", False):
        # Random-init interprators give R_t = 1.0x for every trajectory (SURVEY F7), so a constant bias only moves all
        # trajectories together.  Calibrate: shift the bias so that the MEDIAN first-call R_t of this batch sits exactly on an
        # integer boundary (4.0) -- about half of the trajectories then emit 3 frames per call and half 4, each with its own
        # step sequence, which is what per-sample adaptive stepping is for.
        with torch.inference_mode():
            _, rts0, _, _ = model.rollout(dev_in, n_roll, per_sample=True)
        r0 = rts0[0].float().cpu()
        shift = 4.0 - float(r0.median())
        with torch.no_grad():
            for ip in model.interprators:
                ip.interprete[4].bias.add_(shift)
        calib = {"first_call_Rt_before": [float(r0.min()), float(r0.median()), float(r0.max())], "bias_shift": shift}
    cpu_sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}

    W_, K_ = max(args.warmup, 3), args.steps
    with torch.inference_mode():
        for _ in range(W_):
            y, rts, ns, steps = model.rollout(dev_in, n_roll, per_sample=True, sync=False)
        barrier()
        # ---- timed region 1: device-resident inputs (value) ----
        sampler = ClockSampler(dev.index or 0)
        sampler.start()
        l0 = model.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(K_):
            y, rts, ns, steps = model.rollout(dev_in, n_roll, per_sample=True, sync=False)
        e1.record()
        barrier()
        ms_total = max_over_ranks(e0.elapsed_time(e1))
        launches = model.launch_count() - l0
        clocks = sampler.stop()
        if dump_dir and rank == 0:
            dump_outputs(dump_dir, {"frames": y, "rts": rts, "frames_per_call": ns, "model_calls": steps})
        steps_h = steps.tolist()
        model_calls = int(max(steps_h))
        ns_first = ns[0].tolist()
        if launches and model_calls > 1:
            # the WHILE-graph body is counted once per rollout by the library (the device decides how often it runs)
            launches = int(launches + (model_calls - 1) * K_ * (launches // K_ - 2))

        # ---- timed region 2: end to end through the public API with host buffers ----
        # Every step copies its pinned HOST window to the device and the whole predicted history back;
        # tante_b200.pipeline.HostPrefetcher (the repo's staging API) runs those copies on dedicated streams, so window
        # i+1 travels in and history i-1 travels out while rollout i is computed.  Two host output buffers alternate.
        from tante_b200.pipeline import HostPrefetcher
        pf = HostPrefetcher(dev)
        host_out2 = torch.empty_like(host_out).pin_memory()

        def e2e_run(n):
            pf.put(host_in)
            for i in range(n):
                (d,) = pf.get()
                if i + 1 < n:
                    pf.put(host_in)
                y, *_ = model.rollout(d, n_roll, per_sample=True, sync=False)
                pf.done()
                pf.download(y, host_out if i % 2 == 0 else host_out2)
            pf.join()
        e2e_run(2)
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        e2e_run(K_)
        e3.record()
        barrier()
        ms_e2e = max_over_ranks(e2.elapsed_time(e3))

        # ---- live per-kernel timing of the dominant kernel class (GEMMs) over the same K steps ----
        model.profile_gemms(True)
        e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e4.record()
        for _ in range(K_):
            model.rollout(dev_in, n_roll, per_sample=True, sync=False)
        e5.record()
        torch.cuda.synchronize(dev)
        prof_classes = model.profile_read_classes()
        gemm_ms, gemm_flops, gemm_n = model.profile_read()
        model.profile_gemms(False)
        ms_prof = e4.elapsed_time(e5)
    del model
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    peaks = load_peaks()
    tensor_mode = args.precision == "bf16"
    traj = B * world
    line = {
        "metric": "rollout_trajectories_per_s", "value": traj * K_ / (ms_total * 1e-3), "unit": "trajectories/s",
        "n_gpus": world, "steps": K_, "warmup": W_, "ms_per_step": ms_total / K_, "higher_is_better": True,
        "scaling": getattr(args, "scaling", "weak"), "vs_baseline": None, "dtype": "bf16" if tensor_mode else "f32", "data": "synthetic",
        "config": bench_config(args, B),
        "model_calls_per_trajectory": {"max": model_calls, "min": int(min(steps_h)), "mean": sum(steps_h) / len(steps_h)},
        "frames_first_call": {str(k): ns_first.count(k) for k in sorted(set(ns_first))},
        "adaptive_calibration": calib,
        "frames_per_s": traj * n_roll * K_ / (ms_total * 1e-3),
        "e2e": {"value": traj * K_ / (ms_e2e * 1e-3), "unit": "trajectories/s",
                "h2d_bytes_per_step": host_in.numel() * 4, "d2h_bytes_per_step": host_out.numel() * 4,
                "ms_per_step": ms_e2e / K_},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline_object(prof_classes, gemm_ms, gemm_flops, gemm_n, K_, ms_prof, peaks, tensor_mode, "rollout"),
    }
    if world == 1 and with_cpu_baseline and not args.no_cpu_baseline:
        cb, _ = cpu_leg(args, args.cpu_seconds, cpu_sd)
        line["cpu_baseline"] = cb
    return line


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    line = rollout_measure(args, dev, world, rank, dump_dir=args.dump_outputs)
    if rank == 0:
        if world == 1 and not args.no_eager:
            try:
                line["gpu_eager_baseline"] = eager_rollout_leg(args, dev)
            except Exception as e:   # the eager leg is a reported baseline; never lose the product's line to it
                line["gpu_eager_baseline"] = {"error": repr(e)[:300]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# =====================================================================================================
# gpu_eager_baseline: the reference module's op sequence in stock PyTorch on the same GPU (SURVEY.md §2, §8(d))
# =====================================================================================================
class _RefCudaFlags:
    """utils.set_seed_device on CUDA (utils.py:19-34): cudnn.benchmark, TF32 matmuls ("high")."""

    def __enter__(self):
        import torch
        self.prev = (torch.backends.cudnn.benchmark, torch.get_float32_matmul_precision())
        torch.backends.cudnn.benchmark = True
        torch.set_float32_matmul_precision("high")

    def __exit__(self, *a):
        import torch
        torch.backends.cudnn.benchmark = self.prev[0]
        torch.set_float32_matmul_precision(self.prev[1])


def _eager_model(cfg, dev, torch_seed=211, rt_bias=0.0):
    import torch
    from oracle.eager_module import EagerTANTE
    torch.manual_seed(torch_seed)
    m = EagerTANTE(cfg, dropout=0.0)
    if rt_bias and not cfg.deg:
        with torch.no_grad():
            for ip in m.interprators:
                ip.interprete[4].bias.add_(rt_bias)
    return m.to(dev)


def eager_rollout_leg(args, dev, steps=3):
    """R_Evaler.rollout_model around the stock nn.Module (oracle/eager_module.py) on `dev`: inference_mode, bf16
    autocast, TF32, whole batch per call with sample 0's R_t governing n -- the reference's own GPU path.  torch 2.11's fused
    attention kernels refuse the T-axis layer at the product's batch (64 x 1024 sequences x 8 heads of length 4: first the
    cuDNN graph, then the grid limit of the flash / memory-efficient kernels), so the leg falls back to the largest batch the
    stock module runs at and reports it -- trajectories/s is a per-trajectory rate either way."""
    import torch
    from oracle import tante_oracle as O
    from oracle.eager_module import eager_rollout
    D, H, W = SHAPES[args.shape]
    cfg = O.OracleConfig(n_fields=D, H=H, W=W, taylor_order=args.taylor_order, attn_axes=model_axes(args.taylor_order),
                         deg=False)
    n_roll = args.n_roll
    notes = []
    with _RefCudaFlags():
        model = _eager_model(cfg, dev, rt_bias=args.rt_bias).eval()
        g = torch.Generator().manual_seed(212)
        x_all = torch.randn(args.batch, 4, D, H, W, generator=g).to(dev)
        B, ms = args.batch, None
        while B >= 1 and ms is None:
            x = x_all[:B]
            try:
                with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
                    for _ in range(2):
                        eager_rollout(model, x, n_roll)
                    torch.cuda.synchronize(dev)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(steps):
                        eager_rollout(model, x, n_roll)
                    e1.record()
                    torch.cuda.synchronize(dev)
                ms = e0.elapsed_time(e1) / steps
            except RuntimeError as e:
                notes.append(f"batch {B}: {str(e).splitlines()[0][:90]}")
                try:
                    torch.cuda.synchronize(dev)
                except RuntimeError:
                    pass
                B //= 2
    del model, x_all
    torch.cuda.empty_cache()
    if ms is None:
        raise RuntimeError("the stock module did not run at any batch size: " + "; ".join(notes))
    return {"value": B / (ms * 1e-3), "unit": "trajectories/s", "ms_per_step": ms, "steps": steps, "batch": B,
            "batches_refused_by_stock_torch": notes,
            "what": "oracle/eager_module.py (stock torch.nn restatement of the reference module, pinned to the reference "
                    "goldens) on the same GPU: inference_mode + bf16 autocast + TF32 + cudnn.benchmark (utils.py:19-34), "
                    f"R_Evaler loop, batch {B}, sample 0's R_t governs n (tante.py:163)"}


def eager_train_leg(args, dev, steps=3):
    """Trainer.train_one_epoch body (trainer.py:178-198) around the stock nn.Module on `dev`: bf16 autocast, TF32,
    4 chained forwards with BPTT, MSE, backward, clip_grad_norm_(1.0), torch.optim.AdamW(lr 5e-5, wd 1e-5)."""
    import torch
    from einops import rearrange
    from oracle import tante_oracle as O
    D, H, W = SHAPES[args.shape]
    cfg = O.OracleConfig(n_fields=D, H=H, W=W, taylor_order=1, attn_axes="THWTHWTHW", deg=True)
    B, n_out = args.batch, args.n_steps_output
    with _RefCudaFlags():
        model = _eager_model(cfg, dev).train()
        opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=1e-5)
        g = torch.Generator().manual_seed(212)
        x = torch.randn(B, 4, D, H, W, generator=g).to(dev)
        y_ref = torch.randn(B, n_out, H, W, D, generator=g).to(dev)

        def step():
            with torch.autocast("cuda", dtype=torch.bfloat16):
                moving, ys, cum = x, [], 0
                while cum < n_out:
                    y = model(moving)
                    cum += y.shape[1]
                    if cum < n_out:
                        moving = torch.cat([moving[:, y.shape[1]:], y], dim=1)
                    ys.append(rearrange(y, "b t c h w -> b t h w c"))
                y_pred = torch.cat(ys, dim=1)[:, :n_out]
                loss = torch.mean((y_pred - y_ref) ** 2, dim=(-3, -2)).mean()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=1.0)
            opt.step()
            opt.zero_grad()
            return loss
        for _ in range(2):
            step()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = step()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        peak_mem = torch.cuda.max_memory_allocated(dev)
    del model, opt, x, y_ref
    torch.cuda.empty_cache()
    return {"value": B / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": steps, "final_loss": float(loss),
            "peak_memory_bytes": int(peak_mem),
            "what": "oracle/eager_module.py (stock torch.nn restatement of the reference module, pinned to the reference "
                    "goldens) on the same GPU: bf16 autocast + TF32 + cudnn.benchmark (utils.py:19-34), Trainer step "
                    f"(trainer.py:178-198) at batch {B}: {n_out} chained forwards with BPTT, MSE, clip_grad_norm_, AdamW"}


# =====================================================================================================
# head sweep (BASELINE.json configs[4]): K x patch x n of the fused Taylor head vs the measured HBM copy bandwidth
# =====================================================================================================
def head_sweep_leg(dev, precision="bf16", full=False):
    import torch
    from tante_b200 import TANTE, TanteMetadata
    peaks = load_peaks()
    peak = peaks.get("hbm_gbs") or 6650.0
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    cases = []
    shapes = {"trl": (4, 128, 384, 64), "active_matter": (11, 256, 256, 32)}   # batch: > 2x the 126 MB L2 per launch
    patches = (2, 4, 8, 16, 32) if full else (4, 8, 16)
    for sname, (D, H, W, B) in shapes.items():
        x = torch.randn(B, 4, D, H, W, device=dev)
        for P in patches:
            for K in (1, 2, 3, 4):
                try:
                    m = TANTE(4, TanteMetadata(spatial_resolution=(H, W), n_fields=D), taylor_order=K,
                              attn_axes="-".join(["T"] * K), patch_scale=P, deg=False, precision=precision).to(dev).eval()
                except Exception as e:
                    cases.append({"shape": sname, "P": P, "K": K, "skipped": str(e)[:100]})
                    continue
                k0 = m.patch_kernels[0]
                for n in (1, 4, 8):
                    try:
                        ms = m.bench_head(x, n, iters=10)
                    except Exception as e:
                        cases.append({"shape": sname, "P": P, "K": K, "n": n, "skipped": str(e)[:100]})
                        continue
                    s_act = 2 if precision == "bf16" else 4
                    if k0 == 4:
                        # patch_scale >= 16: the bilinear resize after the last transposed conv blends neighbouring patches,
                        # so the head is the Horner emit over the decoded derivative fields: boundary C of SURVEY.md 8(d)
                        boundary, by = "C", (K + 1 + n) * B * D * H * W * 4
                    else:
                        rows = B * H * W // (k0 * k0)
                        boundary, by = "B", rows * K * 64 * s_act + B * D * H * W * 4 * (1 + n)
                    gbs = by / (ms * 1e-3) / 1e9
                    cases.append({"shape": sname, "P": P, "K": K, "n": n, "boundary": boundary, "us": 1e3 * ms, "bytes": by,
                                  "GBps": gbs, "frac": gbs / peak})
                del m
        del x
        torch.cuda.empty_cache()
    clocks = sampler.stop()
    ok = [c for c in cases if "frac" in c]
    per_shape = {}
    for sname in shapes:
        fr = [c["frac"] for c in ok if c["shape"] == sname]
        if fr:
            worst = min((c for c in ok if c["shape"] == sname), key=lambda c: c["frac"])
            per_shape[sname] = {"min": min(fr), "mean": sum(fr) / len(fr), "max": max(fr), "cells": len(fr),
                                "cells_ge_0.70": sum(f >= 0.70 for f in fr),
                                "worst_cell": {k: worst[k] for k in ("P", "K", "n", "us", "frac")}}
    return {"what": "stand-alone fused Taylor head (tante_bench_head): last deconv + Horner sum + residual + emit; algorithmic "
                    "bytes per launch = rows*K*64*s_act + B*D*H*W*4*(1+n) (boundary B of SURVEY.md 8(d)), rows = B*H*W/k0^2",
            "boundary": "B for patch_scale <= 8 (last deconv + Horner + emit fused), C for patch_scale >= 16 (Horner + emit over "
                        "decoded fields, bytes = (K+1+n)*B*D*H*W*4)", "bound": "hbm", "peak": peak, "unit": "GB/s",
            "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
            "patch_scales": list(patches), "K": [1, 2, 3, 4], "n": [1, 4, 8], "per_shape": per_shape, "clocks": clocks,
            "skipped": [c for c in cases if "skipped" in c][:8], "cases": ok}


# =====================================================================================================
# workload `train` (BASELINE.json configs[1])
# =====================================================================================================
def train_config(args, batch):
    D, H, W = SHAPES[args.shape]
    return {"workload": f"TANTE training step, synthetic {args.shape} shape ({D} fields, {H}x{W}), batch {batch}/GPU "
                        f"(BASELINE.json configs[1])",
            "samples_per_gpu_per_step": batch, "n_steps_output": args.n_steps_output,
            "step": "4 chained forwards with BPTT + MSE + backward + clip_grad_norm_(1.0) + AdamW(lr 5e-5, wd 1e-5)",
            "taylor_order": 1, "attn_axes": "THWTHWTHW", "patch_scale": 8, "embed_dim": 256, "deg": True,
            "dropout": args.dropout, "weights": "random init, torch.manual_seed(211), reference initialisers",
            "l2_hygiene": "per-step working set (saved activations ~4 GB per model call) >> 126 MB L2; no explicit flush",
            "parallelism": (f"dp{args.gpus}: one NCCL all-reduce of the flat fp32 gradient bucket per step" if args.gpus > 1
                            else "single GPU, no collective")}


def oracle_train_setup(args):
    import torch
    from oracle import tante_oracle as O
    D, H, W = SHAPES[args.shape]
    cfg = O.OracleConfig(n_fields=D, H=H, W=W, taylor_order=1, attn_axes="THWTHWTHW", deg=True)
    return O, cfg


def cpu_train_leg(args, seconds, max_steps=8, state_dict=None):
    """The reference's CPU training step (oracle port of models/tante.py + trainer/trainer.py:178-198 with torch
    autograd and torch AdamW) on all host threads, on a bounded sample of the workload: batches of ONE sample."""
    import torch
    O, cfg = oracle_train_setup(args)
    torch.set_num_threads(os.cpu_count() or 1)
    sd = state_dict if state_dict is not None else O.make_state_dict(cfg, 211)
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.AdamW(list(sd.values()), lr=5e-5, weight_decay=1e-5)
    g = torch.Generator().manual_seed(212)
    D, H, W = SHAPES[args.shape]
    x = torch.randn(1, 4, D, H, W, generator=g)
    y_ref = torch.randn(1, args.n_steps_output, H, W, D, generator=g)

    def step():
        y, _, _ = O.rollout_eval(sd, cfg, x, args.n_steps_output)
        loss = O.train_loss(y, y_ref, None)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(sd.values()), 1.0)
        opt.step()
        return float(loss.detach())

    step()                                                  # warm-up
    t0 = time.perf_counter()
    n = 0
    while True:
        step()
        n += 1
        el = time.perf_counter() - t0
        if el > seconds or n >= max_steps:
            break
    return {"value": n / el, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n} training steps of batch 1 ({args.n_steps_output} chained forwards + backward + clip + AdamW, "
                      f"{args.shape} shape, fp32, torch {torch.__version__} CPU autograd) in {el:.1f}s"}


def run_reference_train(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    steps = args.steps
    warm = max(args.warmup, 1)
    O, cfg = oracle_train_setup(args)
    torch.set_num_threads(os.cpu_count() or 1)
    sd = {k: v.clone().requires_grad_(True) for k, v in O.make_state_dict(cfg, 211).items()}
    opt = torch.optim.AdamW(list(sd.values()), lr=5e-5, weight_decay=1e-5)
    g = torch.Generator().manual_seed(212)
    D, H, W = SHAPES[args.shape]
    x = torch.randn(1, 4, D, H, W, generator=g)
    y_ref = torch.randn(1, args.n_steps_output, H, W, D, generator=g)

    def step():
        y, _, _ = O.rollout_eval(sd, cfg, x, args.n_steps_output)
        loss = O.train_loss(y, y_ref, None)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(sd.values()), 1.0)
        opt.step()

    for _ in range(min(warm, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    el = time.perf_counter() - t0
    val = steps / el
    line = {
        "impl": "reference", "metric": "training_samples_per_s", "value": val, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * el / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(train_config(args, 1), reference_arm=(
            "CPU port (oracle/tante_oracle.py, pinned to the live reference) of the reference's training step: the reference is "
            "pure Python with missing dependencies and cannot travel to the GPU box (DESIGN.md 1).  fp32 (the reference's CPU "
            "path has no autocast), batch 1 per step as a bounded sample of the b200 arm's batch-16 bf16 workload; samples/s is "
            "per-sample throughput, so the two values are comparable, the configs are not identical by construction.  The "
            "same-GPU stock-PyTorch number is the b200 line's gpu_eager_baseline.")),
        "cpu_baseline": {"value": val, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": f"{steps} training steps of batch 1, one per bench step (the b200 arm does "
                                   f"{args.batch} samples per step)"},
        "e2e": {"value": val, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_b200_train(args):
    import torch
    import torch.distributed as dist
    from tante_b200 import TANTE, TanteMetadata
    from tante_b200.trainer import GradBucket, train_step

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    D, H, W = SHAPES[args.shape]
    B, n_out = args.batch, args.n_steps_output

    torch.manual_seed(211)                                 # configs/tante.yaml:1 -- identical weights on every rank
    model = TANTE(4, TanteMetadata(spatial_resolution=(H, W), n_fields=D), taylor_order=1, attn_axes="THWTHWTHW",
                  patch_scale=8, deg=True, dropout=args.dropout, precision=args.precision)
    cpu_sd = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(dev).train()
    bucket = GradBucket(model)
    if os.environ.get("TANTE_TORCH_OPTIMIZER", "0") != "0":
        opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=1e-5, fused=True)    # tante.yaml:38-41 (torch's fused kernel)
    else:
        # same update rule, one launch over the flat gradient with the clip folded in (tante_optimizer_step); under
        # torchrun the bucket is all-reduced by the library's own NCCL communicator (tante_allreduce_grads)
        from tante_b200 import FusedAdamW
        opt = FusedAdamW(model.parameters(), lr=5e-5, weight_decay=1e-5, model=model)
        bucket.init_native_comm(model)

    g = torch.Generator().manual_seed(212 + rank)
    host_x = torch.randn(B, 4, D, H, W, generator=g).pin_memory()
    host_y = torch.randn(B, n_out, H, W, D, generator=g).pin_memory()
    host_loss = torch.zeros(1).pin_memory()
    dev_x, dev_y = host_x.to(dev), host_y.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    W_, K_ = max(args.warmup, 3), args.steps
    for _ in range(W_):
        train_step(model, opt, dev_x, dev_y, n_out, bucket)
    barrier()
    # ---- timed region 1: inputs resident in HBM (value) ----
    sampler = ClockSampler(local)
    sampler.start()
    l0 = model.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(K_):
        loss = train_step(model, opt, dev_x, dev_y, n_out, bucket)
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = model.launch_count() - l0
    clocks = sampler.stop()
    final_loss = float(loss)
    if args.dump_outputs and rank == 0:
        # the caller of train_step receives the loss; the step leaves the updated weights and their gradients in the module
        params = [p for _, p in model.named_parameters()]
        dump_outputs(args.dump_outputs, {"loss": loss.reshape(1), "params": flat(params), "grads": flat(p.grad for p in params)})

    # ---- timed region 2: end to end with HOST batches (H2D of inputs+targets, D2H of the loss every step) ----
    # Every step copies its pinned HOST batch to the device and its loss back; tante_b200.pipeline.HostPrefetcher (the
    # repo's staging API) runs those copies on dedicated streams, so batch i+1 travels while batch i is computed.
    from tante_b200.pipeline import HostPrefetcher
    pf = HostPrefetcher(dev)

    def e2e_run(n):
        pf.put(host_x, host_y)
        for i in range(n):
            x, y = pf.get()
            if i + 1 < n:
                pf.put(host_x, host_y)
            ls = train_step(model, opt, x, y, n_out, bucket)
            pf.done()
            pf.download(ls.reshape(1), host_loss)
        pf.join()
    e2e_run(2)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    e2e_run(K_)
    e3.record()
    barrier()
    ms_e2e = max_over_ranks(e2.elapsed_time(e3))

    # ---- live per-kernel timing of the dominant kernel class (forward/input-gradient/weight-gradient GEMMs) ----
    model.profile_gemms(True)
    e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e4.record()
    for _ in range(K_):
        train_step(model, opt, dev_x, dev_y, n_out, bucket)
    e5.record()
    torch.cuda.synchronize(dev)
    prof_classes = model.profile_read_classes()
    gemm_ms, gemm_flops, gemm_n = model.profile_read()
    model.profile_gemms(False)
    ms_prof = e4.elapsed_time(e5)

    grad_bytes = bucket.flat.numel() * 4
    # free the training state before the sub-records run in the same process
    del model, opt, bucket, dev_x, dev_y, pf
    import gc
    gc.collect()
    torch.cuda.empty_cache()

    # ---- sub-records: every other BASELINE config, measured in the same driver run --------------------------------
    extras = {}
    if not args.no_extras:
        import copy
        ra = copy.copy(args)
        ra.workload, ra.shape, ra.batch, ra.taylor_order = "rollout", "rayleigh_benard", 64, 1
        ra.steps, ra.warmup = min(args.steps, 10), 3
        for key, rt_bias, amp in (("rollout", 0.0, False), ("rollout_adaptive", 0.0, True)):
            ra.rt_bias, ra.amp_mix = rt_bias, amp
            try:
                rec = rollout_measure(ra, dev, world, rank, with_cpu_baseline=False)
            except Exception as e:      # a sub-record must never cost the headline line
                rec = {"error": repr(e)[:300]}
            if rank == 0:
                if world == 1 and not args.no_eager and isinstance(rec, dict) and "error" not in rec:
                    try:
                        if rec.get("adaptive_calibration"):
                            ra.rt_bias = rec["adaptive_calibration"]["bias_shift"]     # same weights for the eager module
                        rec["gpu_eager_baseline"] = eager_rollout_leg(ra, dev)
                        rec["vs_gpu_eager"] = rec["value"] / rec["gpu_eager_baseline"]["value"]
                    except Exception as e:
                        rec["gpu_eager_baseline"] = {"error": repr(e)[:300]}
                extras[key] = rec
        if rank == 0 and world == 1:
            try:
                extras["head_sweep"] = head_sweep_leg(dev, args.precision)
            except Exception as e:
                extras["head_sweep"] = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    tensor_mode = args.precision == "bf16"
    samples = B * world
    line = {
        "metric": "training_samples_per_s", "value": samples * K_ / (ms_total * 1e-3), "unit": "samples/s",
        "n_gpus": world, "steps": K_, "warmup": W_, "ms_per_step": ms_total / K_, "higher_is_better": True,
        "scaling": getattr(args, "scaling", "weak"), "vs_baseline": None, "dtype": "bf16" if tensor_mode else "f32", "data": "synthetic",
        "config": train_config(args, B),
        "final_loss": final_loss,
        "model_calls_per_step": n_out,
        "allreduce_bytes_per_step": grad_bytes if world > 1 else 0,
        "e2e": {"value": samples * K_ / (ms_e2e * 1e-3), "unit": "samples/s",
                "h2d_bytes_per_step": (host_x.numel() + host_y.numel()) * 4, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / K_},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline_object(prof_classes, gemm_ms, gemm_flops, gemm_n, K_, ms_prof, peaks, tensor_mode),
    }
    if world == 1 and not args.no_eager:
        try:
            line["gpu_eager_baseline"] = eager_train_leg(args, dev)
            line["vs_gpu_eager"] = line["value"] / line["gpu_eager_baseline"]["value"]
        except Exception as e:
            line["gpu_eager_baseline"] = {"error": repr(e)[:300]}
    line.update(extras)
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_train_leg(args, args.cpu_seconds, state_dict=cpu_sd)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    # the benchmark writes nothing into the source tree: it imports modules that build() does not (tante_b200.pipeline,
    # oracle.eager_module), whose bytecode caches would otherwise appear there
    sys.dont_write_bytecode = True
    args = parse()
    if args.workload == "train":
        if args.impl == "reference":
            run_reference_train(args)
        else:
            run_b200_train(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
