"""Generate tests/golden/*.npz from the LIVE upstream reference (TEST INFRASTRUCTURE).

Needs an upstream TANTE checkout:

    TANTE_REFERENCE_ROOT=<upstream checkout> python -m oracle.make_golden

The reference ships no golden vectors (SURVEY.md §4); these files are outputs of the
reference's own `models.TANTE` (+ the `deg=False` repair in oracle/ref_shim.py) and
`trainer.metrics.MSE`, driven by restatements of `R_Evaler.rollout_model`
(trainer/r_evaler.py:87-105) and `R_Trainer.rollout_model` + loss/backward
(trainer/r_trainer.py:112-159) that call the reference module unchanged.  Weights
and inputs are the deterministic synthetic ones of `oracle.tante_oracle.make_state_dict`
/ `make_input`, so a fixture only stores (config, seeds) + reference outputs.
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import ref_shim, tante_oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def build_ref(ns, cfg: O.OracleConfig, sd):
    md = ref_shim.make_metadata(cfg.n_fields, cfg.H, cfg.W)
    m = ns.TANTE(in_T=cfg.in_T, dset_metadata=md, taylor_order=cfg.taylor_order,
                 frame_interval=cfg.frame_interval, output_length=cfg.output_length,
                 attn_axes=cfg.attn_axes, expanded_channel=cfg.expanded_channel, n_head=cfg.n_head,
                 mlp_ratio=cfg.mlp_ratio, dropout=0.0,
                 enc_dec_type=cfg.enc_dec_type, embed_dim=cfg.embed_dim, modes1=cfg.modes1, modes2=cfg.modes2,
                 patch_scale=cfg.patch_scale, overlap_ratio=cfg.overlap_ratio, deg=cfg.deg)
    m.load_state_dict(sd)
    m.t_seq = m.t_seq.cpu()
    return m


def ref_rollout_eval(m, cfg, window, n_roll, out_T=None):
    """R_Evaler.rollout_model (r_evaler.py:87-105) around the reference module."""
    out_T = n_roll if out_T is None else out_T
    moving, ys, Rts, ns, cum = window, [], [], [], 0
    while cum < n_roll:
        if cfg.deg:
            y, rt = m(moving), None
        else:
            y, rt = m(moving, out_T)
        cum += y.shape[1]
        if cum < n_roll:
            moving = torch.cat([moving[:, y.shape[1]:, ...], y], dim=1)
        ys.append(y.permute(0, 1, 3, 4, 2))
        ns.append(y.shape[1])
        if rt is not None:
            Rts.append(rt)
    return torch.cat(ys, dim=1)[:, :n_roll], (torch.cat(Rts, 0) if Rts else None), ns


def ref_rollout_train(m, cfg, batch, n_steps, out_T=1.5):
    """R_Trainer.rollout_model (r_trainer.py:112-133): per-sample loops, BPTT window."""
    outs, Rts, all_ns = [], [], []
    for i in range(batch.shape[0]):
        y, r, ns = ref_rollout_eval(m, cfg, batch[i:i + 1], n_steps, out_T)
        outs.append(y)
        all_ns.append(ns)
        if r is not None:
            Rts.append(r)
    return torch.cat(outs, 0), (torch.cat(Rts, 0) if Rts else None), all_ns


def sub(t: torch.Tensor, stride: int):
    return t.detach().reshape(-1)[::stride].numpy().copy()


def save(name, cfg, meta, arrays):
    meta = dict(meta)
    meta["cfg"] = cfg.__dict__
    arrays = {k: (v.detach().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in arrays.items()}
    arrays["meta_json"] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}: {os.path.getsize(path)/1024:.1f} KiB")


def case_forward(ns, name, cfg, B, out_T, rt_bias, seed=211, stride=1, stages=False, n_roll=0):
    sd = O.make_state_dict(cfg, seed, rt_bias)
    m = build_ref(ns, cfg, sd).eval()
    x = O.make_input(cfg, B, seed + 1)
    arrays = {}
    hooks, cap = [], {}
    if stages:
        hooks.append(m.encoder.register_forward_hook(lambda mod, i, o: cap.__setitem__("enc", o.detach().clone())))
        for k in range(cfg.taylor_order):
            hooks.append(m.blocks[k].register_forward_hook(
                lambda mod, i, o, k=k: cap.__setitem__(f"backbone{k}", o.detach().clone())))
            hooks.append(m.blocks[k].register_forward_pre_hook(
                lambda mod, i, k=k: cap.__setitem__(f"backbone{k}_in", i[0].detach().clone())))
            hooks.append(m.decoders[k].register_forward_hook(
                lambda mod, i, o, k=k: cap.__setitem__(f"deriv{k}", o.detach().clone())))
            for j in range(len(cfg.segments[k])):
                hooks.append(m.blocks[k].blocks[j].register_forward_hook(
                    lambda mod, i, o, k=k, j=j: cap.__setitem__(f"block{k}_{j}", (i[0].detach().clone(), o.detach().clone()))))
    with torch.inference_mode():
        out = m(x, out_T)
    for h in hooks:
        h.remove()
    if cfg.deg:
        y, rt = out, None
    else:
        y, rt = out
        arrays["R_t"] = rt
    arrays["frames"] = sub(y, stride)
    arrays["frame_norms"] = torch.linalg.vector_norm(y.reshape(B, y.shape[1], -1), dim=-1)
    arrays["deriv_norms"] = torch.linalg.vector_norm((y - x[:, -1:]).reshape(B, y.shape[1], -1), dim=-1)
    meta = dict(kind="forward", B=B, out_T=out_T, rt_bias=rt_bias, seed=seed, input_seed=seed + 1,
                n=int(y.shape[1]), stride=stride, frames_shape=list(y.shape), n_roll=n_roll)
    if stages:
        arrays["stage_enc"] = cap["enc"]
        for k in range(cfg.taylor_order):
            arrays[f"stage_backbone{k}_in"] = cap[f"backbone{k}_in"]
            arrays[f"stage_backbone{k}"] = cap[f"backbone{k}"]
            arrays[f"stage_deriv{k}"] = cap[f"deriv{k}"]
            # first transformer block of each backbone: input (after propagators) and output, in (N,S,C) layout
            arrays[f"stage_block{k}_0_in"] = cap[f"block{k}_0"][0]
            arrays[f"stage_block{k}_0_out"] = cap[f"block{k}_0"][1]
    if n_roll:
        with torch.inference_mode():
            yr, Rts, nseq = ref_rollout_eval(m, cfg, x, n_roll)
            arrays["roll_frames"] = sub(yr, stride)
            arrays["roll_frame_norms"] = torch.linalg.vector_norm(yr.reshape(B, n_roll, -1), dim=-1)
            arrays["roll_ns"] = np.asarray(nseq, dtype=np.int32)
            if Rts is not None:
                arrays["roll_Rts"] = Rts
            if not cfg.deg:
                yp, Rp, nsp = ref_rollout_train(m, cfg, x, n_roll, out_T=n_roll)
                arrays["psroll_frames"] = sub(yp, stride)
                arrays["psroll_frame_norms"] = torch.linalg.vector_norm(yp.reshape(B, n_roll, -1), dim=-1)
                arrays["psroll_Rts"] = Rp
                meta["psroll_ns"] = nsp
    save(name, cfg, meta, arrays)


def case_train(ns, name, cfg, B, n_steps, rt_bias=0.0, seed=211, stride=17):
    """One reference training step's loss and gradients (r_trainer.py:145-155 / trainer.py:178-193)."""
    sd = O.make_state_dict(cfg, seed, rt_bias)
    m = build_ref(ns, cfg, sd).train()
    x = O.make_input(cfg, B, seed + 1)
    g = torch.Generator().manual_seed(seed + 2)
    y_ref = torch.randn(B, n_steps, cfg.H, cfg.W, cfg.n_fields, generator=g)
    x = x.clone().requires_grad_(True)
    loss_fn = ns.metrics.MSE()
    if cfg.deg:
        y_pred, _, nseq = ref_rollout_eval(m, cfg, x, n_steps)
        loss = loss_fn(y_pred, y_ref, None).mean()
        Rts = None
    else:
        y_pred, Rts, nseq = ref_rollout_train(m, cfg, x, n_steps, 1.5)
        loss = loss_fn(y_pred, y_ref, Rts, 0.5, 2)
    loss.backward()
    arrays = {"loss": loss.detach(), "y_pred": sub(y_pred, stride), "grad_input": sub(x.grad, stride),
              "grad_input_norm": x.grad.norm()}
    if Rts is not None:
        arrays["Rts"] = Rts.detach()
    names, norms = [], []
    for k, p in m.named_parameters():
        names.append(k)
        gp = p.grad if p.grad is not None else torch.zeros_like(p)
        norms.append(float(gp.norm()))
        if gp.numel() <= 4096:
            arrays["grad::" + k] = gp
        else:
            arrays["gradsub::" + k] = sub(gp, stride)
    arrays["grad_norms"] = np.asarray(norms, dtype=np.float64)
    meta = dict(kind="train", B=B, n_steps=n_steps, rt_bias=rt_bias, seed=seed, input_seed=seed + 1,
                target_seed=seed + 2, stride=stride, param_names=names)
    save(name, cfg, meta, arrays)


def main_round2(ns):
    """Round-2 fixtures: patch_scale 16 / 32 / 64 (shifted 4x4 windows + bilinear resize, enc_dec_cnn.py:75-81,93-95,
    176-184) and the long / composite attention axes L, Y, A (attn_backbone.py:164-182) -- written by the live reference."""
    C = O.OracleConfig
    case_forward(ns, "fwd_adp_k2_p16", C(n_fields=3, H=64, W=96, taylor_order=2, attn_axes="THW-WT", deg=False,
                                          patch_scale=16), B=2, out_T=6, rt_bias=2.7, stages=True, n_roll=6, stride=5)
    case_forward(ns, "fwd_deg_k1_p32", C(n_fields=4, H=128, W=192, taylor_order=1, attn_axes="THW", deg=True,
                                          patch_scale=32), B=2, out_T=1, rt_bias=0.0, n_roll=3, stride=13)
    case_forward(ns, "fwd_adp_k1_p64", C(n_fields=2, H=256, W=128, taylor_order=1, attn_axes="HWT", deg=False,
                                          patch_scale=64), B=1, out_T=4, rt_bias=1.3, n_roll=4, stride=11)
    case_forward(ns, "fwd_adp_k1_p16_d11", C(n_fields=11, H=64, W=64, taylor_order=1, attn_axes="TW", deg=False,
                                              patch_scale=16), B=2, out_T=4, rt_bias=1.3, n_roll=4, stride=13)
    # axes L / Y / A and an axis longer than 64 tokens (W_p = 96 at patch 4)
    case_forward(ns, "fwd_adp_k2_axes_lya", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="LTY-AW", deg=False),
                 B=2, out_T=6, rt_bias=2.7, stages=True, n_roll=6)
    case_forward(ns, "fwd_deg_k1_w96", C(n_fields=2, H=32, W=384, taylor_order=1, attn_axes="WHT", deg=True,
                                          patch_scale=4), B=2, out_T=1, rt_bias=0.0, n_roll=2)
    if "--fno" in sys.argv:
        main_fno(ns)


def main_mlp(ns):
    """mlp_ratio != 1 (attn_backbone.py:52-56: hidden = int(embed_dim * mlp_ratio)): forward / rollout and one training step."""
    C = O.OracleConfig
    case_forward(ns, "fwd_adp_k2_mlp2", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="THW-HWT", deg=False, mlp_ratio=2.0),
                 B=2, out_T=6, rt_bias=2.7, stages=True, n_roll=6)
    case_forward(ns, "fwd_deg_k1_mlp05", C(n_fields=3, H=32, W=32, taylor_order=1, attn_axes="THW", deg=True, mlp_ratio=0.5),
                 B=2, out_T=1, rt_bias=0.0, n_roll=3)
    case_train(ns, "train_deg_k1_mlp4", C(n_fields=3, H=32, W=32, taylor_order=1, attn_axes="THW", deg=True, mlp_ratio=4.0),
               B=2, n_steps=3)


def main_axisc(ns):
    """Attention axis 'C' (attn_backbone.py:124-130,184-189): every latent token becomes a sequence of embed_dim channel
    tokens, lifted 1 -> expanded_channel by a two-layer MLP, run through a TransformerBlock(expanded_channel); the last
    feature is the new latent."""
    C = O.OracleConfig
    case_forward(ns, "fwd_adp_k2_axes_c", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="TCW-HC", deg=False),
                 B=2, out_T=6, rt_bias=2.7, stages=True, n_roll=6)
    case_forward(ns, "fwd_deg_k1_axes_c64", C(n_fields=3, H=32, W=32, taylor_order=1, attn_axes="HC", deg=True,
                                               expanded_channel=256, mlp_ratio=0.5),
                 B=1, out_T=1, rt_bias=0.0, n_roll=2)


def main_train_long(ns):
    """One training step (r_trainer.py:112-159) with the composite attention axes L / Y / A (sequences of 96 / 32 / 384 tokens)."""
    C = O.OracleConfig
    case_train(ns, "train_adp_k2_lya", C(n_fields=2, H=64, W=96, taylor_order=2, attn_axes="LTY-AW", deg=False), B=2, n_steps=3,
               rt_bias=0.0)


def main_train_wide(ns):
    """Training steps at patch_scale 16 / 32 (shifted 4x4 windows + bilinear resize, enc_dec_cnn.py:75-81,93-95,176-184)."""
    C = O.OracleConfig
    case_train(ns, "train_adp_k2_p16", C(n_fields=3, H=64, W=96, taylor_order=2, attn_axes="THW-WT", deg=False, patch_scale=16),
               B=2, n_steps=3, rt_bias=0.0)
    case_train(ns, "train_deg_k1_p32", C(n_fields=4, H=128, W=192, taylor_order=1, attn_axes="THW", deg=True, patch_scale=32),
               B=2, n_steps=3)


def main_train_fno(ns):
    """Training steps with enc_dec_type='fno' (enc_dec_fno.py:184-323): gradients of the complex spectral weights included."""
    C = O.OracleConfig
    case_train(ns, "train_deg_k1_fno_p8", C(n_fields=3, H=64, W=96, taylor_order=1, attn_axes="THW", deg=True, enc_dec_type="fno",
                                             patch_scale=8, modes1=16, modes2=16), B=2, n_steps=2)
    case_train(ns, "train_adp_k2_fno_p4", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="TH-W", deg=False, enc_dec_type="fno",
                                             patch_scale=4, modes1=8, modes2=8), B=2, n_steps=3, rt_bias=0.0)


def main_c512(ns):
    """embed_dim = 512 (models/tante.py:53): head_dim 64 at n_head 8, head_dim 32 at n_head 16."""
    C = O.OracleConfig
    case_forward(ns, "fwd_adp_k2_c512", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="THW-HW", deg=False, embed_dim=512),
                 B=2, out_T=6, rt_bias=2.7, n_roll=6, stride=3)
    case_train(ns, "train_deg_k1_c512", C(n_fields=3, H=32, W=32, taylor_order=1, attn_axes="THW", deg=True, embed_dim=512, n_head=16),
               B=2, n_steps=3)


def main_fno_wide(ns):
    """enc_dec_type='fno' at patch_scale 32 / 64: 8x8 patch stages (windows shifted by 3, transposed convs resized from 8h - 6)."""
    C = O.OracleConfig
    case_forward(ns, "fwd_deg_k1_fno_p32", C(n_fields=3, H=128, W=128, taylor_order=1, attn_axes="THW", deg=True,
                                              enc_dec_type="fno", patch_scale=32, modes1=16, modes2=16),
                 B=2, out_T=1, rt_bias=0.0, n_roll=2, stride=11)
    case_forward(ns, "fwd_adp_k1_fno_p64", C(n_fields=2, H=128, W=192, taylor_order=1, attn_axes="WT", deg=False,
                                              enc_dec_type="fno", patch_scale=64, modes1=8, modes2=16),
                 B=1, out_T=4, rt_bias=1.3, n_roll=4, stride=7)
    case_train(ns, "train_deg_k1_fno_p32", C(n_fields=3, H=128, W=128, taylor_order=1, attn_axes="TH", deg=True,
                                              enc_dec_type="fno", patch_scale=32, modes1=16, modes2=16), B=1, n_steps=2)


def main_train_axisc(ns):
    """One training step through axis-'C' layers (channel attention, attn_backbone.py:124-130,184-189)."""
    C = O.OracleConfig
    case_train(ns, "train_deg_k1_axes_c", C(n_fields=2, H=32, W=32, taylor_order=1, attn_axes="TCH", deg=True), B=2, n_steps=2)


def main_overlap(ns):
    """overlap_ratio != 0 (enc_dec_cnn.py:64-66,109,130-132,176-184): strided overlapping windows + adaptive average pooling in the
    encoder, overlap-add transposed convs + bilinear resize in the decoder."""
    C = O.OracleConfig
    case_forward(ns, "fwd_adp_k2_ov50_p8", C(n_fields=3, H=64, W=96, taylor_order=2, attn_axes="THW-WT", deg=False,
                                              overlap_ratio=0.5), B=2, out_T=6, rt_bias=2.7, stages=True, n_roll=6, stride=5)
    case_forward(ns, "fwd_deg_k1_ov25_p16", C(n_fields=2, H=64, W=64, taylor_order=1, attn_axes="HWT", deg=True, patch_scale=16,
                                               overlap_ratio=0.25), B=2, out_T=1, rt_bias=0.0, n_roll=3, stride=7)
    case_forward(ns, "fwd_deg_k1_ov70_p32", C(n_fields=4, H=128, W=128, taylor_order=1, attn_axes="TW", deg=True, patch_scale=32,
                                               overlap_ratio=0.7), B=1, out_T=1, rt_bias=0.0, n_roll=2, stride=11)
    case_train(ns, "train_deg_k1_ov50_p8", C(n_fields=3, H=32, W=32, taylor_order=1, attn_axes="THW", deg=True, overlap_ratio=0.5),
               B=2, n_steps=2)
    case_forward(ns, "fwd_adp_k1_fno_ov50_p8", C(n_fields=3, H=64, W=96, taylor_order=1, attn_axes="TW", deg=False, enc_dec_type="fno",
                                                  patch_scale=8, modes1=16, modes2=16, overlap_ratio=0.5), B=2, out_T=4, rt_bias=1.3,
                 n_roll=4, stride=7)
    case_train(ns, "train_deg_k1_fno_ov30_p16", C(n_fields=2, H=64, W=64, taylor_order=1, attn_axes="TH", deg=True, enc_dec_type="fno",
                                                   patch_scale=16, modes1=8, modes2=8, overlap_ratio=0.3), B=1, n_steps=2)
    case_train(ns, "train_adp_k1_ov40_p16", C(n_fields=2, H=64, W=64, taylor_order=1, attn_axes="TH", deg=False, patch_scale=16,
                                               overlap_ratio=0.4), B=2, n_steps=2, rt_bias=0.0)


def main_fno(ns):
    """enc_dec_type='fno' (enc_dec_fno.py:184-323): spectral layers (rfft2 / low modes / irfft2 + 1x1 conv) between the patch convs."""
    C = O.OracleConfig
    case_forward(ns, "fwd_deg_k1_fno_p8", C(n_fields=3, H=64, W=96, taylor_order=1, attn_axes="THW", deg=True,
                                             enc_dec_type="fno", patch_scale=8, modes1=16, modes2=16),
                 B=2, out_T=1, rt_bias=0.0, n_roll=3, stride=7, stages=True)
    case_forward(ns, "fwd_adp_k2_fno_p4", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="TH-W", deg=False,
                                             enc_dec_type="fno", patch_scale=4, modes1=8, modes2=8),
                 B=2, out_T=6, rt_bias=2.7, n_roll=6, stride=3)
    case_forward(ns, "fwd_deg_k1_fno_p16", C(n_fields=4, H=64, W=128, taylor_order=1, attn_axes="WT", deg=True,
                                              enc_dec_type="fno", patch_scale=16, modes1=12, modes2=20),
                 B=1, out_T=1, rt_bias=0.0, n_roll=2, stride=5)


# ---- the live-reference comparisons of tests/test_oracle_vs_reference.py and tests/test_abi_cpu.py, stored --------------
LIVE_CASES = {   # name -> (cfg, B, out_T, rt_bias); weights O.make_state_dict(cfg, 7, rt_bias), input O.make_input(cfg, B, 8)
    "ref_live_deg_k1": (O.OracleConfig(n_fields=4, H=64, W=64, taylor_order=1, deg=True), 2, 1, 0.0),
    "ref_live_adp_k2_lya": (O.OracleConfig(n_fields=3, H=32, W=32, taylor_order=2, attn_axes="THWLA-TYW", deg=False,
                                           patch_scale=4, frame_interval=0.5), 2, 8, 5.2),
    "ref_live_adp_k1_p16": (O.OracleConfig(n_fields=2, H=64, W=128, taylor_order=1, attn_axes="THW", deg=False,
                                           patch_scale=16), 1, 8, 1.3),
}
LIVE_STRIDE = 7
# default initialisation under torch.manual_seed(211): in_T 4, 3 fields on 64x96, patch_scale 8, dropout 0.1
INIT_CASES = (dict(taylor_order=1, attn_axes="THWTHW", deg=True), dict(taylor_order=2, attn_axes="THW-HW", deg=False),
              dict(taylor_order=2, attn_axes="TH-W", deg=False, enc_dec_type="fno", modes1=16, modes2=16),
              dict(taylor_order=2, attn_axes="TCW-CH", deg=False, expanded_channel=256, mlp_ratio=2.0))
INIT_SAMPLE = 128   # values stored per tensor (evenly strided); the float64 sum and sum of squares cover every element


def init_summary(t: torch.Tensor):
    """(strided sample, float64 sum, float64 sum of squares) of one state_dict tensor (complex as (re, im) pairs)."""
    a = (torch.view_as_real(t) if t.is_complex() else t).detach().reshape(-1).numpy().astype(np.float64)
    step = max(1, a.size // INIT_SAMPLE)
    return a[::step][:INIT_SAMPLE].astype(np.float32), float(a.sum()), float(np.square(a).sum())


def main_live(ns, source="the live reference module"):
    """tests/golden/ref_live_*.npz (the reference's frames / R_t for LIVE_CASES) and ref_init.npz (the reference module's
    default initialisation for INIT_CASES)."""
    for name, (cfg, B, out_T, bias) in LIVE_CASES.items():
        sd = O.make_state_dict(cfg, 7, bias)
        m = build_ref(ns, cfg, sd).eval()
        with torch.inference_mode():
            out = m(O.make_input(cfg, B, 8), out_T)
        y, rt = (out, None) if cfg.deg else out
        arrays = {"frames": sub(y, LIVE_STRIDE)}
        if rt is not None:
            arrays["R_t"] = rt
        save(name, cfg, {"B": B, "out_T": out_T, "rt_bias": bias, "seed": 7, "input_seed": 8, "stride": LIVE_STRIDE,
                         "frames_shape": list(y.shape), "keys": sorted(m.state_dict().keys()), "source": source}, arrays)
    arrays, cases = {}, []
    md = ref_shim.make_metadata(3, 64, 96)
    for i, kw in enumerate(INIT_CASES):
        torch.manual_seed(211)
        sd = ns.TANTE(in_T=4, dset_metadata=md, patch_scale=8, dropout=0.1, **kw).state_dict()
        sums = {}
        for j, (k, v) in enumerate(sd.items()):
            arrays[f"c{i}_{j}"], s, s2 = init_summary(v)
            sums[k] = [list(v.shape), s, s2]
        cases.append({"kw": kw, "keys": list(sd.keys()), "sums": sums})
    arrays["meta_json"] = np.frombuffer(json.dumps({"source": source, "init": cases}).encode(), dtype=np.uint8)
    path = os.path.join(OUT, "ref_init.npz")
    np.savez_compressed(path, **arrays)
    print(f"wrote {path}: {os.path.getsize(path)/1024:.1f} KiB")


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    ns = ref_shim.load_reference()
    if "--live" in sys.argv:
        main_live(ns)
        return
    if "--round2" in sys.argv:
        main_round2(ns)
        return
    if "--fno" in sys.argv:
        main_fno(ns)
        return
    if "--mlp" in sys.argv:
        main_mlp(ns)
        return
    if "--overlap" in sys.argv:
        main_overlap(ns)
        return
    if "--trainaxisc" in sys.argv:
        main_train_axisc(ns)
        return
    if "--fnowide" in sys.argv:
        main_fno_wide(ns)
        return
    if "--c512" in sys.argv:
        main_c512(ns)
        return
    if "--trainfno" in sys.argv:
        main_train_fno(ns)
        return
    if "--trainwide" in sys.argv:
        main_train_wide(ns)
        return
    if "--trainlong" in sys.argv:
        main_train_long(ns)
        return
    if "--axisc" in sys.argv:
        main_axisc(ns)
        return
    C = O.OracleConfig
    # 1. fixed-step (what configs/tante.yaml selects), full outputs on a small grid
    case_forward(ns, "fwd_deg_k1_p8", C(n_fields=4, H=64, W=96, taylor_order=1, deg=True), B=2, out_T=1,
                 rt_bias=0.0, n_roll=4)
    # 2. tiny all-stages case for kernel bring-up (adaptive, K=2)
    case_forward(ns, "fwd_stages_k2_p8", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="THW-HWT", deg=False),
                 B=2, out_T=8, rt_bias=2.7, stages=True, n_roll=8)
    # 3. adaptive K=2 with steps [3,3,..]
    case_forward(ns, "fwd_adp_k2_p8_b27", C(n_fields=3, H=64, W=96, taylor_order=2, attn_axes="THWTHW-THW", deg=False),
                 B=2, out_T=8, rt_bias=2.7, n_roll=8)
    # 4. adaptive K=3, patch 4, frame_interval 0.5
    case_forward(ns, "fwd_adp_k3_p4", C(n_fields=3, H=32, W=64, taylor_order=3, attn_axes="THW-WH-T", deg=False,
                                         patch_scale=4, frame_interval=0.5), B=3, out_T=8, rt_bias=5.2, n_roll=8)
    # 5. BASELINE config 1: TRL shape, B=1, K in {1,2}, rollout 8, bias shifts of SURVEY §8(c) (subsampled)
    for K, axes in ((1, "THWTHWTHW"), (2, "THWTHW-THW")):
        for b in (0.0, 1.3, 5.2):
            case_forward(ns, f"trl_k{K}_b{str(b).replace('.', '')}",
                         C(n_fields=4, H=128, W=384, taylor_order=K, attn_axes=axes, deg=False),
                         B=1, out_T=8, rt_bias=b, stride=97, n_roll=8)
    # 6. patch_scale 2 (kernels (2,1,1))
    case_forward(ns, "fwd_adp_k1_p2", C(n_fields=2, H=16, W=24, taylor_order=1, attn_axes="THW", deg=False,
                                         patch_scale=2), B=2, out_T=4, rt_bias=1.3, n_roll=4)
    # 7. training step goldens (loss + grads)
    case_train(ns, "train_adp_k2", C(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="THW-HWT", deg=False),
               B=2, n_steps=4, rt_bias=0.0)
    case_train(ns, "train_deg_k1", C(n_fields=3, H=32, W=32, taylor_order=1, attn_axes="THWTHW", deg=True),
               B=2, n_steps=4)


if __name__ == "__main__":
    main()
