"""Cost of one R_Trainer optimizer step (r_trainer.py:145-157: rollout, MSE + rt penalty, backward, clip_grad_value_, AdamW) on
the adaptive model (deg=False), per-sample loops (TANTE_BPTT_WINDOWS=0) against the batched rollout, alternating in one process.
Shape: BASELINE configs[1] (Active Matter 11 x 256 x 256, batch 16, 4 output steps, bf16, patch_scale 8, K = 1 THWTHWTHW).
Prints one JSON line: samples/s and ms/step of both paths per round, launches per step, the rel-L2 between the two paths' loss and
gradients on the same weights, and the GPU's name and power limit.
usage: python tools/adaptive_train_probe.py [--batch 16] [--steps 4] [--iters 5] [--rounds 3] [--precision bf16] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tante_b200 import TANTE, TanteMetadata  # noqa: E402
from tante_b200.trainer import mse_loss, rollout_train  # noqa: E402

PATHS = {"loop": "0", "batched": "1"}


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except Exception as e:      # the number is still valid; say why the limit is missing
        info["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=4, help="n_steps_output")
    ap.add_argument("--iters", type=int, default=5, help="timed optimizer steps per path and round")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--precision", default="bf16")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("adaptive_train_probe needs a CUDA device")
    D, H, W = 11, 256, 256
    dev = torch.device("cuda:0")
    torch.manual_seed(211)
    model = TANTE(4, TanteMetadata(spatial_resolution=(H, W), n_fields=D), taylor_order=1, attn_axes="THWTHWTHW",
                  patch_scale=8, deg=False, dropout=0.0, precision=a.precision).to(dev).train()
    opt = torch.optim.AdamW(model.parameters(), lr=5e-5, weight_decay=1e-5)
    g = torch.Generator().manual_seed(212)
    x = torch.randn(a.batch, 4, D, H, W, generator=g).to(dev)
    y_ref = torch.randn(a.batch, a.steps, H, W, D, generator=g).to(dev)

    def set_path(p):
        os.environ["TANTE_BPTT_WINDOWS"] = PATHS[p]

    def loss_and_grads():
        y, rts = rollout_train(model, x, a.steps, 1.5)
        loss = mse_loss(y, y_ref, rts, 0.5, 2)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        return loss

    def step():
        loss = loss_and_grads()
        torch.nn.utils.clip_grad_value_(model.parameters(), 1.0)
        opt.step()
        opt.zero_grad()
        return loss

    # parity on the same weights, before any optimizer step
    par = {}
    for p in PATHS:
        set_path(p)
        loss = loss_and_grads()
        par[p] = (loss.detach().double(), torch.cat([q.grad.detach().double().reshape(-1) for q in model.parameters()]))
    rel = lambda u, v: float((u - v).norm() / v.norm().clamp_min(1e-30))
    parity = {"loss_rel": rel(par["batched"][0], par["loop"][0]), "grad_rel_l2": rel(par["batched"][1], par["loop"][1]),
              "loss_loop": float(par["loop"][0]), "loss_batched": float(par["batched"][0])}

    launches = {}
    for p in PATHS:            # warm-up of both paths, and the launches of one step
        set_path(p)
        step()
        torch.cuda.synchronize()
        n0 = model.launch_count()
        step()
        torch.cuda.synchronize()
        launches[p] = model.launch_count() - n0

    rounds = []
    for r in range(a.rounds):
        row = {}
        for p in PATHS:
            set_path(p)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(a.iters):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.iters
            row[p] = {"ms_per_step": round(ms, 3), "samples_per_s": round(a.batch / ms * 1e3, 2)}
        rounds.append(row)
    best = {p: max(r[p]["samples_per_s"] for r in rounds) for p in PATHS}
    out = {"probe": "adaptive_train", "shape": "active_matter 11x256x256", "batch": a.batch, "n_steps_output": a.steps,
           "precision": a.precision, "model": "deg=False K=1 THWTHWTHW patch_scale 8 embed 256", "iters": a.iters,
           "rounds": rounds, "best_samples_per_s": best, "speedup_best": round(best["batched"] / best["loop"], 3),
           "launches_per_step": launches, "parity": parity, "gpu": gpu_info(),
           "max_mem_gib": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2)}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
