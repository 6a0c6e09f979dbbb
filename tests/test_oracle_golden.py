"""The CPU oracle restatement vs the committed reference outputs (tests/golden, written by
oracle/make_golden.py from the live upstream module).  CPU only."""
import glob
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, golden_cfg, load_golden, rel_l2
from oracle import tante_oracle as O

FWD = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "*.npz"))
             if not os.path.basename(p).startswith(("train_", "ref_")))
FAST = [n for n in FWD if not n.startswith("trl_")] + ["trl_k1_b52", "trl_k2_b13"]
TOL = 2e-6   # fp32 CPU restatement vs fp32 CPU reference: measured <= 6e-7 (summation order only)


@pytest.mark.parametrize("name", FAST)
def test_forward_matches_reference_golden(name):
    z, meta = load_golden(name)
    cfg = golden_cfg(meta)
    sd = O.make_state_dict(cfg, meta["seed"], meta["rt_bias"])
    x = O.make_input(cfg, meta["B"], meta["input_seed"])
    with torch.inference_mode():
        out = O.forward(sd, cfg, x, meta["out_T"])
    if cfg.deg:
        y = out
    else:
        y, rt = out
        np.testing.assert_allclose(rt.numpy(), z["R_t"], rtol=0, atol=5e-6)
    assert y.shape[1] == meta["n"], "adaptive step count differs from the reference"
    assert list(y.shape) == meta["frames_shape"]
    s = meta["stride"]
    assert rel_l2(y.reshape(-1)[::s].numpy(), z["frames"]) < TOL
    u0 = x[:, -1:]
    d = (y - u0).reshape(meta["B"], y.shape[1], -1).norm(dim=-1).numpy()
    np.testing.assert_allclose(d, z["deriv_norms"], rtol=1e-5)


@pytest.mark.parametrize("name", ["fwd_stages_k2_p8", "fwd_adp_k3_p4", "fwd_deg_k1_p8", "fwd_adp_k1_p2"])
def test_rollout_matches_reference_golden(name):
    z, meta = load_golden(name)
    cfg = golden_cfg(meta)
    sd = O.make_state_dict(cfg, meta["seed"], meta["rt_bias"])
    x = O.make_input(cfg, meta["B"], meta["input_seed"])
    with torch.inference_mode():
        y, Rts, ns = O.rollout_eval(sd, cfg, x, meta["n_roll"])
    assert ns == z["roll_ns"].tolist()
    s = meta["stride"]
    assert rel_l2(y.reshape(-1)[::s].numpy(), z["roll_frames"]) < 5e-6
    if not cfg.deg:
        np.testing.assert_allclose(Rts.numpy(), z["roll_Rts"], atol=1e-5)
        with torch.inference_mode():
            yp, Rp, nsp = O.rollout_per_sample(sd, cfg, x, meta["n_roll"], meta["n_roll"])
        assert nsp == meta["psroll_ns"]
        assert rel_l2(yp.reshape(-1)[::s].numpy(), z["psroll_frames"]) < 5e-6


def test_stage_tensors_match_reference_golden():
    z, meta = load_golden("fwd_stages_k2_p8")
    cfg = golden_cfg(meta)
    sd = O.make_state_dict(cfg, meta["seed"], meta["rt_bias"])
    x = O.make_input(cfg, meta["B"], meta["input_seed"])
    with torch.inference_mode():
        enc = O.encoder(sd, cfg, x)
        assert rel_l2(enc.numpy(), z["stage_enc"]) < TOL
        e = O.embed(sd, cfg, x)
        assert rel_l2(e.numpy(), z["stage_backbone0_in"]) < TOL
        frames, R_t, parts = O.forward(sd, cfg, x, meta["out_T"], return_parts=True)
        assert rel_l2(parts["latent"].numpy(), z["stage_backbone1"]) < TOL
        for k in range(cfg.taylor_order):
            assert rel_l2(parts["derivatives"][k].numpy(), z[f"stage_deriv{k}"][:, 0]) < 5e-6
        blk = O.transformer_block(sd, "blocks.0.blocks.0.", torch.from_numpy(z["stage_block0_0_in"]), cfg.n_head, True)
        assert rel_l2(blk.numpy(), z["stage_block0_0_out"]) < TOL


@pytest.mark.parametrize("name", ["train_adp_k2", "train_deg_k1", "train_deg_k1_mlp4", "train_adp_k2_lya", "train_adp_k2_p16", "train_deg_k1_p32", "train_deg_k1_fno_p8",
                                  "train_adp_k2_fno_p4", "train_deg_k1_c512", "train_deg_k1_fno_p32",
                                  "train_deg_k1_axes_c", "train_deg_k1_ov50_p8", "train_adp_k1_ov40_p16",
                                  "train_deg_k1_fno_ov30_p16"])
def test_training_step_grads_match_reference_golden(name):
    z, meta = load_golden(name)
    cfg = golden_cfg(meta)
    sd = O.make_state_dict(cfg, meta["seed"], meta["rt_bias"])
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    x = O.make_input(cfg, meta["B"], meta["input_seed"]).requires_grad_(True)
    g = torch.Generator().manual_seed(meta["target_seed"])
    y_ref = torch.randn(meta["B"], meta["n_steps"], cfg.H, cfg.W, cfg.n_fields, generator=g)
    if cfg.deg:
        y, _, _ = O.rollout_eval(sd, cfg, x, meta["n_steps"])
        loss = O.train_loss(y, y_ref, None)
    else:
        y, Rts, _ = O.rollout_per_sample(sd, cfg, x, meta["n_steps"], 1.5)
        loss = O.train_loss(y, y_ref, Rts, 0.5, 2)
    loss.backward()
    assert abs(float(loss) - float(z["loss"])) < 1e-6 * max(1.0, abs(float(z["loss"])))
    s = meta["stride"]
    assert rel_l2(x.grad.reshape(-1)[::s].numpy(), z["grad_input"]) < 2e-5
    norms = z["grad_norms"]
    for name_, gn in zip(meta["param_names"], norms):
        gp = sd[name_].grad
        got = 0.0 if gp is None else float(gp.norm())
        assert abs(got - gn) <= 2e-5 * max(gn, 1e-6) + 1e-9, name_
        key = "grad::" + name_
        if key in z and gn > 0:
            assert rel_l2(gp.numpy(), z[key]) < 5e-5, name_


@pytest.mark.parametrize("name", ["fwd_deg_k1_p8", "fwd_stages_k2_p8", "fwd_adp_k3_p4", "fwd_adp_k1_p2"])
def test_eager_module_matches_reference_golden(name):
    """oracle/eager_module.py (the stock-torch nn.Module bench.py times on the GPU as `gpu_eager_baseline`) loads the
    reference state_dict unchanged and reproduces the reference's frames, R_t and rollout."""
    from oracle.eager_module import EagerTANTE, eager_rollout
    z, meta = load_golden(name)
    cfg = golden_cfg(meta)
    sd = O.make_state_dict(cfg, meta["seed"], meta["rt_bias"])
    m = EagerTANTE(cfg).eval()
    m.load_state_dict(sd, strict=True)
    x = O.make_input(cfg, meta["B"], meta["input_seed"])
    with torch.inference_mode():
        out = m(x, meta["out_T"])
        y = out if cfg.deg else out[0]
        if not cfg.deg:
            np.testing.assert_allclose(out[1].numpy(), z["R_t"], rtol=0, atol=5e-6)
        yr = eager_rollout(m, x, meta["n_roll"])
    s = meta["stride"]
    assert list(y.shape) == meta["frames_shape"]
    assert rel_l2(y.reshape(-1)[::s].numpy(), z["frames"]) < TOL
    assert rel_l2(yr.reshape(-1)[::s].numpy(), z["roll_frames"]) < 5e-6
