"""GPU parity of the training path (taped forward + hand-written backward, through the C ABI and the autograd
Function) against the reference's own loss/gradient goldens and against autograd over the CPU oracle.

The drivers below are the reference trainers' rollouts restated around the drop-in module:
R_Trainer.rollout_model (trainer/r_trainer.py:112-133: per-sample B=1 loops, out_T=1.5, window NOT detached => BPTT)
and Trainer.rollout_model (trainer/trainer.py:144-159: whole batch, fixed step), loss = trainer/metrics.py MSE.
"""
import numpy as np
import pytest
import torch

from conftest import golden_cfg, load_golden, rel_l2
from oracle import tante_oracle as O

pytestmark = pytest.mark.gpu

FP32_GRAD_TOL = 2e-4       # fp32 CUDA vs fp32 CPU reference gradients (different summation orders, atomics)
BF16_GRAD_TOL = 6e-2       # bf16 tensor mode: per-tensor gradient rel-L2 (activations/gradients rounded to bf16)


def _rollout_train(model, cfg, x, n_steps, out_T):
    """The reference trainers' rollout around `model` (channels-first in, channels-last out)."""
    def roll(win):
        moving, ys, rts, cum = win, [], [], 0
        while cum < n_steps:
            if cfg.deg:
                y, rt = model(moving), None
            else:
                y, rt = model(moving, out_T)
            cum += y.shape[1]
            if cum < n_steps:
                moving = torch.cat([moving[:, y.shape[1]:], y], dim=1)
            ys.append(y.permute(0, 1, 3, 4, 2))
            if rt is not None:
                rts.append(rt)
        return torch.cat(ys, 1)[:, :n_steps], (torch.cat(rts, 0) if rts else None)
    if cfg.deg:
        return roll(x)
    outs, rts = [], []
    for b in range(x.shape[0]):
        y, r = roll(x[b:b + 1])
        outs.append(y)
        rts.append(r)
    return torch.cat(outs, 0), torch.cat(rts, 0)


def _loss(y, y_ref, rts):
    l = torch.mean((y - y_ref) ** 2, dim=(-3, -2)).mean()
    if rts is None:
        return l
    avg = rts.mean()
    pen = 0.0
    if float(avg) < 1.5:
        pen = pen + 5e-3 * (1.5 - avg) ** 2
    if float(avg) > 4:
        pen = pen + 1e-1 * (avg - 4) ** 2
    return l + pen


def _train_case(name, precision):
    from gpu_util import make_model
    z, meta = load_golden(name)
    cfg = golden_cfg(meta)
    sd = O.make_state_dict(cfg, meta["seed"], meta["rt_bias"])
    model = make_model(cfg, sd, precision).train()
    x = O.make_input(cfg, meta["B"], meta["input_seed"]).cuda().requires_grad_(True)
    g = torch.Generator().manual_seed(meta["target_seed"])
    y_ref = torch.randn(meta["B"], meta["n_steps"], cfg.H, cfg.W, cfg.n_fields, generator=g).cuda()
    y, rts = _rollout_train(model, cfg, x, meta["n_steps"], 1.5)
    loss = _loss(y, y_ref, rts)
    loss.backward()
    return z, meta, cfg, model, x, y, loss


def _report(model, z, meta, tol):
    bad, worst = [], 0.0
    for name_, gn in zip(meta["param_names"], z["grad_norms"]):
        gp = dict(model.named_parameters())[name_].grad
        got = 0.0 if gp is None else float(gp.norm())
        nerr = abs(got - gn) / max(gn, 1e-12)
        err = nerr
        key = "grad::" + name_
        s = meta["stride"]
        if gn > 0 and gp is not None:
            if key in z:
                err = max(err, rel_l2(gp.cpu().numpy(), z[key]))
            elif "gradsub::" + name_ in z:
                err = max(err, rel_l2(gp.cpu().reshape(-1)[::s].numpy(), z["gradsub::" + name_]))
        worst = max(worst, err)
        if not err <= tol:      # (NaN must fail)
            bad.append(f"{name_}: rel {err:.3e} (norm got {got:.4e} ref {gn:.4e})")
    return bad, worst


@pytest.mark.parametrize("name", ["train_deg_k1", "train_adp_k2", "train_deg_k1_mlp4", "train_adp_k2_lya", "train_adp_k2_p16",
                                  "train_deg_k1_p32", "train_deg_k1_fno_p8", "train_adp_k2_fno_p4",
                                  "train_deg_k1_c512", "train_deg_k1_fno_p32", "train_deg_k1_axes_c",
                                  "train_deg_k1_ov50_p8", "train_adp_k1_ov40_p16", "train_deg_k1_fno_ov30_p16"])
def test_training_step_fp32_matches_reference_golden(name):
    z, meta, cfg, model, x, y, loss = _train_case(name, "fp32")
    assert abs(float(loss) - float(z["loss"])) < 2e-6 * max(1.0, abs(float(z["loss"])))
    s = meta["stride"]
    assert rel_l2(y.detach().cpu().reshape(-1)[::s].numpy(), z["y_pred"]) < 1e-5
    bad, worst = _report(model, z, meta, FP32_GRAD_TOL)
    assert not bad, "parameter gradients differ from the reference:\n" + "\n".join(bad)
    assert rel_l2(x.grad.cpu().reshape(-1)[::s].numpy(), z["grad_input"]) < FP32_GRAD_TOL
    assert abs(float(x.grad.norm()) - float(z["grad_input_norm"])) < FP32_GRAD_TOL * float(z["grad_input_norm"])


@pytest.mark.parametrize("name", ["train_deg_k1", "train_adp_k2", "train_deg_k1_mlp4", "train_adp_k2_lya", "train_adp_k2_p16",
                                  "train_deg_k1_p32", "train_deg_k1_fno_p8", "train_adp_k2_fno_p4",
                                  "train_deg_k1_c512", "train_deg_k1_fno_p32", "train_deg_k1_axes_c",
                                  "train_deg_k1_ov50_p8", "train_adp_k1_ov40_p16", "train_deg_k1_fno_ov30_p16"])
def test_training_step_bf16_close_to_reference_golden(name):
    z, meta, cfg, model, x, y, loss = _train_case(name, "bf16")
    assert abs(float(loss) - float(z["loss"])) < 2e-2 * max(1.0, abs(float(z["loss"])))
    bad, worst = _report(model, z, meta, BF16_GRAD_TOL)
    assert not bad, "parameter gradients differ from the reference:\n" + "\n".join(bad)
    s = meta["stride"]
    assert rel_l2(x.grad.cpu().reshape(-1)[::s].numpy(), z["grad_input"]) < BF16_GRAD_TOL


def test_bf16_training_step_at_benchmarked_shape_vs_oracle():
    """BASELINE configs[1] as bench.py runs it -- Active Matter (11 fields, 256x256), fixed step, K = 1 THWTHWTHW, four
    chained model calls with BPTT, MSE -- in bf16 (batch 2) against fp32 autograd over the CPU oracle: loss, predictions and
    every parameter gradient, the latter against 6e-2 or 3x what the reference's own bf16 autocast deviates by."""
    from gpu_util import make_model
    from tante_b200.trainer import mse_loss_frames, _roll_frames
    cfg = O.OracleConfig(n_fields=11, H=256, W=256, taylor_order=1, attn_axes="THWTHWTHW", deg=True)
    sd = O.make_state_dict(cfg, 211)
    B, n_steps = 2, 4
    x = O.make_input(cfg, B, 212)
    g = torch.Generator().manual_seed(213)
    y_ref = torch.randn(B, n_steps, cfg.H, cfg.W, cfg.n_fields, generator=g)

    def oracle(autocast):
        sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
        with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
            y, _, _ = O.rollout_eval(sdg, cfg, x, n_steps)
        loss = O.train_loss(y.float(), y_ref, None)
        loss.backward()
        return float(loss), y.detach().float(), sdg
    loss_ref, yp_ref, sdg = oracle(False)
    _, _, amp = oracle(True)

    model = make_model(cfg, sd, "bf16").train()
    frames = _roll_frames(model, x.cuda(), n_steps)
    loss = mse_loss_frames(frames, y_ref.cuda(), n_steps)
    loss.backward()
    assert abs(float(loss) - loss_ref) < 2e-2 * abs(loss_ref)
    yp = torch.cat([f.detach().permute(0, 1, 3, 4, 2) for f in frames], dim=1).cpu()
    assert rel_l2(yp.numpy(), yp_ref.numpy()) < 2e-2
    bad = []
    for n, p in model.named_parameters():
        ref = sdg[n].grad
        e = rel_l2(p.grad.cpu().numpy(), ref.numpy())
        lim = max(BF16_GRAD_TOL, 3.0 * rel_l2(amp[n].grad.numpy(), ref.numpy()))
        if not e <= lim:
            bad.append(f"{n}: rel {e:.3e} > {lim:.3e}")
    assert not bad, "bf16 gradients at the benchmarked shape differ from the oracle:\n" + "\n".join(bad)


def test_bf16_training_on_cta_pairs_equals_single_cta_calls():
    """At the benchmarked shape a call of 2 samples (8192 tokens) runs the block tail, the MLP backward and the fp32-epilogue
    GEMMs on single CTAs; a call of 6 samples (24576 >= 256 * 74 tokens on a B200) runs them on CTA pairs.  Both see the same
    rows, so the predictions and the gradient of a summed loss must agree up to the order of the weight-gradient reductions."""
    from gpu_util import make_model
    cfg = O.OracleConfig(n_fields=11, H=256, W=256, taylor_order=1, attn_axes="THWTHWTHW", deg=True)
    sd = O.make_state_dict(cfg, 211)
    x = O.make_input(cfg, 6, 214).cuda()
    model = make_model(cfg, sd, "bf16").train()
    assert 6 * cfg.in_T * cfg.Hp * cfg.Wp >= 256 * (torch.cuda.get_device_properties(0).multi_processor_count // 2)
    assert 2 * cfg.in_T * cfg.Hp * cfg.Wp < 256 * (torch.cuda.get_device_properties(0).multi_processor_count // 2)

    def run(chunks):
        model.zero_grad(set_to_none=True)
        ys = []
        for xb in chunks:
            y = model(xb)
            y.float().square().sum().backward()
            ys.append(y.detach().float())
        return torch.cat(ys), {n: p.grad.detach().clone() for n, p in model.named_parameters()}
    y6, g6 = run([x])
    y2, g2 = run(x.split(2))
    assert rel_l2(y6.cpu().numpy(), y2.cpu().numpy()) < 1e-6
    flat6 = torch.cat([g.flatten() for g in g6.values()]).cpu().numpy()
    flat2 = torch.cat([g.flatten() for g in g2.values()]).cpu().numpy()
    assert rel_l2(flat6, flat2) < 1e-4
    for n in g6:
        if ".mlp." in n:      # downstream of the fused MLP backward
            assert rel_l2(g6[n].cpu().numpy(), g2[n].cpu().numpy()) < 1e-3, n


def _oracle_grads(cfg, sd, x, gy, grt, out_T, autocast=False):
    """autocast=True: the oracle under torch.autocast(bf16) -- the reference's own amp mode (r_trainer.py:71-74,145);
    its deviation from fp32 is the yardstick for the bf16 tensor mode on cancellation-dominated gradients."""
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    xg = x.clone().requires_grad_(True)
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
        if cfg.deg:
            y = O.forward(sdg, cfg, xg)
            rt = None
        else:
            y, rt = O.forward(sdg, cfg, xg, out_T)
    if y.shape != gy.shape:
        return None, None, None
    if rt is None:
        (y.float() * gy).sum().backward()
    else:
        ((y.float() * gy).sum() + (rt.float() * grt).sum()).backward()
    return y.detach(), sdg, xg.grad


@pytest.mark.parametrize("prec,tol", [("fp32", FP32_GRAD_TOL), ("bf16", BF16_GRAD_TOL)])
@pytest.mark.parametrize("case", ["adp_k2_n3", "deg_k1_p4", "adp_k3_p2", "deg_k1_axes32", "adp_k1_axes48", "adp_k2_lya", "deg_k1_w96", "adp_k1_p64", "deg_k2_p16", "adp_k1_fno_p16", "adp_k2_axes_c", "deg_k1_axes_c256", "adp_k1_ov70_p32", "deg_k2_ov30_p4", "deg_k1_ov50_p64"])
def test_single_step_backward_vs_oracle_autograd(case, prec, tol):
    """One model call with a random cotangent on the frames AND on R_t, multi-frame emit (n = 3) included:
    every parameter gradient and the input gradient against torch autograd over the CPU oracle."""
    from gpu_util import make_model
    if case == "adp_k2_n3":
        cfg = O.OracleConfig(n_fields=3, H=32, W=64, taylor_order=2, attn_axes="THW-WHT", deg=False)
        rt_bias, out_T = 2.7, 8
    elif case == "deg_k1_p4":
        cfg = O.OracleConfig(n_fields=5, H=32, W=48, taylor_order=1, attn_axes="HWT", deg=True, patch_scale=4,
                             output_length=2, frame_interval=0.5)
        rt_bias, out_T = 0.0, 1
    elif case == "deg_k1_axes32":
        # axis lengths 32 / 16 and 11 fields (the Active Matter geometry): tensor-core propagator backward, K1 = 44
        cfg = O.OracleConfig(n_fields=11, H=256, W=128, taylor_order=1, attn_axes="HWT", deg=True)
        rt_bias, out_T = 0.0, 1
    elif case == "adp_k2_lya":
        # composite axes (attn_backbone.py:164-182): L = 96, Y = 32, A = 384 tokens -- tiled recompute backward for S > 64
        cfg = O.OracleConfig(n_fields=2, H=64, W=96, taylor_order=2, attn_axes="LTY-AW", deg=False)
        rt_bias, out_T = 2.7, 8
    elif case == "deg_k1_w96":
        # a plain axis of 96 tokens (W_p = 384 / 4)
        cfg = O.OracleConfig(n_fields=2, H=32, W=384, taylor_order=1, attn_axes="WHT", deg=True, patch_scale=4)
        rt_bias, out_T = 0.0, 1
    elif case == "adp_k1_p64":
        # patch_scale 64: three shifted 4x4 stages each way (wide_patch.cuh), multi-frame emit through the field-level head
        cfg = O.OracleConfig(n_fields=2, H=256, W=128, taylor_order=1, attn_axes="HWT", deg=False, patch_scale=64)
        rt_bias, out_T = 2.7, 8
    elif case == "deg_k2_p16":
        # patch_scale 16 (kernels 4, 2, 2), 11 fields (K1 = 176 -> padded to 192), two orders
        cfg = O.OracleConfig(n_fields=11, H=64, W=64, taylor_order=2, attn_axes="TW-H", deg=True, patch_scale=16, output_length=2)
        rt_bias, out_T = 0.0, 1
    elif case == "adp_k1_fno_p16":
        # enc_dec_type='fno' at patch_scale 16: 4x4 patch stages (shifted windows / bilinear resize) between the spectral layers
        cfg = O.OracleConfig(n_fields=4, H=64, W=128, taylor_order=1, attn_axes="WT", deg=False, enc_dec_type="fno", patch_scale=16,
                             modes1=12, modes2=20)
        rt_bias, out_T = 2.7, 8
    elif case == "adp_k2_axes_c":
        # channel attention (axis C): the block recomputed chunk by chunk in the backward; E = 256 / head_dim 32 in the first order's
        # layer is covered by the golden, here E = 128 / head_dim 16 with a C layer first, last and next to the fused tail
        cfg = O.OracleConfig(n_fields=2, H=32, W=48, taylor_order=2, attn_axes="CTW-HC", deg=False)
        rt_bias, out_T = 2.7, 8
    elif case == "deg_k1_axes_c256":
        # channel attention at expanded_channel 256: head_dim 32 -> tiled online-softmax forward, mma.sync recompute backward (bf16)
        cfg = O.OracleConfig(n_fields=2, H=32, W=32, taylor_order=1, attn_axes="TC", deg=True, expanded_channel=256)
        rt_bias, out_T = 0.0, 1
    elif case == "adp_k1_ov70_p32":
        # overlap_ratio 0.7 at patch_scale 32: strides (1, 1, 1) under kernels (4, 4, 2) -- every stage pools / overlap-adds
        cfg = O.OracleConfig(n_fields=4, H=64, W=96, taylor_order=1, attn_axes="WT", deg=False, patch_scale=32, overlap_ratio=0.7)
        rt_bias, out_T = 2.7, 8
    elif case == "deg_k1_ov50_p64":
        # overlap 0.5 at patch_scale 64: strides (2, 2, 2) under kernels (4, 4, 4); the last encoder conv has K = 2048 (split-K in the
        # tensor mode) in front of its pooling
        cfg = O.OracleConfig(n_fields=2, H=256, W=128, taylor_order=1, attn_axes="HW", deg=True, patch_scale=64, overlap_ratio=0.5)
        rt_bias, out_T = 0.0, 1
    elif case == "deg_k2_ov30_p4":
        # overlap_ratio 0.3 at patch_scale 4: kernels (2, 2, 1), strides (1, 1, 1): non-divisible pooling windows (H - 1 -> H / 2)
        cfg = O.OracleConfig(n_fields=3, H=32, W=48, taylor_order=2, attn_axes="TH-W", deg=True, patch_scale=4, overlap_ratio=0.3,
                             output_length=2)
        rt_bias, out_T = 0.0, 1
    elif case == "adp_k1_axes48":
        # TRL geometry: axis length 48 (padded to 64 in the tensor-core propagator kernels)
        cfg = O.OracleConfig(n_fields=4, H=128, W=384, taylor_order=1, attn_axes="WHT", deg=False)
        rt_bias, out_T = 1.3, 4
    else:
        cfg = O.OracleConfig(n_fields=2, H=16, W=24, taylor_order=3, attn_axes="T-H-W", deg=False, patch_scale=2)
        rt_bias, out_T = 1.3, 4
    sd = O.make_state_dict(cfg, 311, rt_bias)
    B = 2 if ("axes" in case or case in ("adp_k2_lya", "deg_k1_w96", "adp_k1_p64", "deg_k2_p16", "adp_k1_fno_p16", "adp_k2_axes_c", "deg_k1_axes_c256", "adp_k1_ov70_p32", "deg_k2_ov30_p4", "deg_k1_ov50_p64")) else 3
    x = O.make_input(cfg, B, 312)
    with torch.no_grad():
        y0 = O.forward(sd, cfg, x, out_T)
        y0 = y0 if cfg.deg else y0[0]
    g = torch.Generator().manual_seed(313)
    gy = torch.randn(y0.shape, generator=g)
    grt = torch.randn(B, generator=g)
    y_ref, sdg, gx_ref = _oracle_grads(cfg, sd, x, gy, grt, out_T)
    amp = None
    if prec == "bf16":
        _, amp, _ = _oracle_grads(cfg, sd, x, gy, grt, out_T, autocast=True)

    model = make_model(cfg, sd, prec).train()
    xc = x.cuda().requires_grad_(True)
    if cfg.deg:
        y = model(xc)
        (y * gy.cuda()).sum().backward()
    else:
        y, rt = model(xc, out_T)
        ((y * gy.cuda()).sum() + (rt * grt.cuda()).sum()).backward()
    assert y.shape == y_ref.shape
    assert rel_l2(y.detach().cpu().numpy(), y_ref.numpy()) < (1e-5 if prec == "fp32" else 2e-2)
    bad = []
    for n, p in model.named_parameters():
        ref = sdg[n].grad
        refn = 0.0 if ref is None else float(ref.norm())
        if p.grad is None:
            if refn > 0:
                bad.append(f"{n}: no gradient (ref norm {refn:.3e})")
            continue
        if refn == 0.0:
            if float(p.grad.norm()) > 1e-6:
                bad.append(f"{n}: got {float(p.grad.norm()):.3e}, reference gradient is zero")
            continue
        e = rel_l2(p.grad.cpu().numpy(), ref.numpy())
        lim = tol
        if amp is not None and amp[n].grad is not None:
            # bf16 mode: allow what the reference's own bf16 autocast deviates by on this tensor (sums with heavy
            # cancellation -- bias / LayerNorm gradients, the tiny interprator -- amplify rounding noise)
            lim = max(tol, 3.0 * rel_l2(amp[n].grad.numpy(), ref.numpy()))
        if not e <= lim:
            bad.append(f"{n}: rel {e:.3e} > {lim:.3e} (norm got {float(p.grad.norm()):.4e} ref {refn:.4e})")
    assert not bad, "gradients differ from oracle autograd:\n" + "\n".join(bad)
    assert rel_l2(xc.grad.cpu().numpy(), gx_ref.numpy()) < tol


@pytest.mark.parametrize("shape", [(4096, 256, 256), (8192 + 64, 768, 256), (5000, 256, 512), (3000, 128, 256),
                                   (2048, 512, 256), (1024, 256, 128), (777, 256, 64), (4100, 64, 44), (999, 64, 64)])
def test_wgrad_tcgen05_matches_torch(shape):
    """dW[N,K] += A[M,N]^T B[M,K] on tcgen05 with MN-major operands + TMA reduce-add, accumulating into C."""
    import ctypes
    from tante_b200 import _abi
    lib = _abi.load()
    M, N, K = shape
    g = torch.Generator(device="cuda").manual_seed(5)
    A = torch.randn(M, N, device="cuda", generator=g).to(torch.bfloat16)
    Bm = torch.randn(M, K, device="cuda", generator=g).to(torch.bfloat16)
    C0 = torch.randn(N, K, device="cuda", generator=g)
    C = C0.clone()
    Bp = Bm
    if K % 64:      # the producer zero-pads B to a multiple of 64 columns; only the first K columns of dW are kept
        Bp = torch.zeros(M, (K + 63) // 64 * 64, device="cuda", dtype=torch.bfloat16)
        Bp[:, :K] = Bm
    bias0 = torch.randn(N, device="cuda", generator=g)
    bias = bias0.clone()
    _abi.check(lib.tante_test_wgrad(1, A.data_ptr(), Bp.data_ptr(), C.data_ptr(), bias.data_ptr(), M, N, K, 1,
                                    torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = C0.double() + A.double().t() @ Bm.double()
    assert rel_l2(C.cpu().numpy(), ref.cpu().numpy()) < 2e-5
    # fused bias gradient: column sums of A ride along as an N = 16 MMA against a tile of ones
    bref = bias0.double() + A.double().sum(0)
    assert rel_l2(bias.cpu().numpy(), bref.cpu().numpy()) < 2e-5


@pytest.mark.parametrize("mode", [0, 2])
def test_wgrad_simt_matches_torch(mode):
    from tante_b200 import _abi
    lib = _abi.load()
    M, N, K = 3001, 64, 44
    g = torch.Generator(device="cuda").manual_seed(6)
    dt = torch.float32 if mode == 0 else torch.bfloat16
    A = torch.randn(M, N, device="cuda", generator=g).to(dt)
    Bm = torch.randn(M, K, device="cuda", generator=g).to(dt)
    C = torch.zeros(N, K, device="cuda")
    _abi.check(lib.tante_test_wgrad(mode, A.data_ptr(), Bm.data_ptr(), C.data_ptr(), None, M, N, K, 1,
                                    torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = A.double().t() @ Bm.double()
    assert rel_l2(C.cpu().numpy(), ref.cpu().numpy()) < 2e-5


def test_grad_accumulation_and_slot_reuse():
    """Two backward passes accumulate into .grad like the reference module; tape slots are recycled."""
    from gpu_util import make_model
    cfg = O.OracleConfig(n_fields=2, H=16, W=16, taylor_order=1, attn_axes="TH", deg=True)
    sd = O.make_state_dict(cfg, 11)
    model = make_model(cfg, sd, "fp32").train()
    x = O.make_input(cfg, 2, 12).cuda()
    model(x).square().mean().backward()
    g1 = {n: p.grad.clone() for n, p in model.named_parameters()}
    model(x).square().mean().backward()
    for n, p in model.named_parameters():
        assert rel_l2(p.grad.cpu().numpy(), (2 * g1[n]).cpu().numpy()) < 1e-4, n
    for _ in range(5):
        model.zero_grad()
        model(x).square().mean().backward()
    eng = next(iter(model._engines.values()))
    assert eng.n_slots <= 2


@pytest.mark.parametrize("kind", ["cnn", "fno"])
def test_grad_bucket_direct_accumulation_matches_autograd_path(kind):
    """GradBucket lays `p.grad` out like the library's flat gradient, so the backward accumulates with one add per
    model call and returns no per-parameter gradients: the result must equal the plain autograd path, also when the
    same parameters are used by several chained calls (BPTT) and after the bucket is zeroed."""
    from gpu_util import make_model
    from tante_b200.trainer import GradBucket, rollout_train
    cfg = O.OracleConfig(n_fields=3, H=32, W=48, taylor_order=1, attn_axes="THW", deg=True)
    if kind == "fno":      # complex spectral weights: (re, im) pairs in the flat buffer, p.grad a complex view of it
        cfg = O.OracleConfig(n_fields=3, H=32, W=48, taylor_order=1, attn_axes="TW", deg=True, enc_dec_type="fno", patch_scale=4,
                             modes1=8, modes2=8)
    sd = O.make_state_dict(cfg, 411, 0.0)
    x = O.make_input(cfg, 2, 412).cuda()
    ref = make_model(cfg, sd, "fp32").train()
    y, _ = rollout_train(ref, x, 3)
    y.square().mean().backward()
    want = {n: p.grad.clone() for n, p in ref.named_parameters()}

    model = make_model(cfg, sd, "fp32").train()
    bucket = GradBucket(model)
    eng = next(iter(model._engines.values()))
    assert model._flat_grad_view(eng) is not None, "GradBucket layout is not the library's flat layout"
    for rep in range(2):
        bucket.zero()
        y, _ = rollout_train(model, x, 3)
        y.square().mean().backward()
        for n, p in model.named_parameters():
            assert p.grad.data_ptr() >= bucket.flat.data_ptr(), n
            assert rel_l2(p.grad.cpu().numpy(), want[n].cpu().numpy()) < 1e-5, (rep, n)


@pytest.mark.parametrize("n_steps", [3, 4])
def test_fused_mse_matches_reference_loss_and_gradient(n_steps):
    """tante_mse_cl (loss of the per-call channels-first frames vs channels-last targets) == the reference's
    MSE.eval(...).mean() on the permuted, concatenated, truncated predictions -- value and gradients."""
    from tante_b200.trainer import mse_loss, mse_loss_frames
    g = torch.Generator().manual_seed(5)
    B, D, H, W = 3, 5, 16, 24
    frames = [torch.randn(B, n, D, H, W, generator=g).cuda().requires_grad_(True) for n in (1, 2, 1)]
    y_ref = torch.randn(B, 4, H, W, D, generator=g).cuda()
    y_cat = torch.cat([f.permute(0, 1, 3, 4, 2) for f in frames], dim=1)[:, :n_steps]
    want = mse_loss(y_cat, y_ref[:, :n_steps])
    gw = torch.autograd.grad(want * 1.7, frames)
    got = mse_loss_frames(frames, y_ref, n_steps)
    gg = torch.autograd.grad(got * 1.7, frames)
    assert abs(float(got) - float(want)) < 1e-5 * abs(float(want))
    for a, b in zip(gg, gw):
        assert rel_l2(a.cpu().numpy(), b.cpu().numpy()) < 1e-5


@pytest.mark.parametrize("prec,tol", [("fp32", 2e-5), ("bf16", 2e-2)])
@pytest.mark.parametrize("n_steps", [2, 5])
def test_windowed_bptt_rollout_equals_chained_calls(prec, tol, n_steps):
    """`TANTE.rollout_train` (one autograd node, every sample's window read at its device cursor over the input window and the
    prediction buffer: tante_train_forward_hist / tante_backward_hist, no torch.cat) against the reference-style chain `y = model(win); win = cat(win[:, 1:], y)` (trainer/trainer.py:144-159) on the same
    module: identical predictions, equal parameter gradients and input gradient.  n_steps = 5 > in_T: the last window holds
    predictions only."""
    from gpu_util import make_model
    cfg = O.OracleConfig(n_fields=3, H=32, W=64, taylor_order=1, attn_axes="THW", deg=True)
    sd = O.make_state_dict(cfg, 4)
    model = make_model(cfg, sd, precision=prec).train()
    x = O.make_input(cfg, 3, 8).cuda()
    g = torch.randn(3, n_steps, 3, 32, 64, generator=torch.Generator().manual_seed(1)).cuda()

    def run(windowed):
        model.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        if windowed:
            pred = model.rollout_train(xi, n_steps)
        else:
            moving, ys = xi, []
            for _ in range(n_steps):
                y = model(moving)
                moving = torch.cat([moving[:, 1:], y], dim=1)
                ys.append(y)
            pred = torch.cat(ys, dim=1)
        (pred * g).sum().backward()
        return pred.detach(), xi.grad.detach(), {n: p.grad.detach().clone() for n, p in model.named_parameters()}

    p0, gx0, gp0 = run(False)
    p1, gx1, gp1 = run(True)
    assert torch.equal(p0, p1)
    assert rel_l2(gx1.cpu().numpy(), gx0.cpu().numpy()) < tol
    for n in gp0:
        assert rel_l2(gp1[n].cpu().numpy(), gp0[n].cpu().numpy()) < max(tol, 5e-5), n


def test_train_step_uses_windowed_bptt_and_matches_chained_path(monkeypatch):
    """tante_b200.trainer.train_step (fused loss over the per-call frames) takes the windowed path for the fixed-step model:
    same loss and gradient bucket as with TANTE_BPTT_WINDOWS=0."""
    from gpu_util import make_model
    from tante_b200.trainer import GradBucket, _roll_frames, mse_loss_frames
    cfg = O.OracleConfig(n_fields=3, H=32, W=64, taylor_order=1, attn_axes="THW", deg=True)
    model = make_model(cfg, O.make_state_dict(cfg, 4), precision="fp32").train()
    bucket = GradBucket(model)
    x = O.make_input(cfg, 2, 8).cuda()
    y = torch.randn(2, 4, 32, 64, 3, generator=torch.Generator().manual_seed(2)).cuda()
    out = []
    for flag in ("0", "1"):
        monkeypatch.setenv("TANTE_BPTT_WINDOWS", flag)
        bucket.zero()
        frames = _roll_frames(model, x, 4)
        assert len(frames) == (1 if flag == "1" else 4)
        loss = mse_loss_frames(frames, y, 4)
        loss.backward()
        out.append((float(loss), bucket.flat.clone()))
    assert abs(out[0][0] - out[1][0]) < 1e-6 * max(1.0, abs(out[0][0]))
    assert rel_l2(out[1][1].cpu().numpy(), out[0][1].cpu().numpy()) < 2e-5


def test_channel_axis_chunking_is_invisible(monkeypatch):
    """The axis-C pass runs in chunks of latent tokens (forward: 2048, backward: 512): with a chunk size that does not divide the
    token count (TANTE_CHAN_CHUNK=80 over 192 tokens) outputs and gradients must equal the single-chunk run bitwise."""
    from gpu_util import make_model
    cfg = O.OracleConfig(n_fields=2, H=32, W=48, taylor_order=1, attn_axes="TCW", deg=True)
    sd = O.make_state_dict(cfg, 611, 0.0)
    x = O.make_input(cfg, 2, 612).cuda()

    def run():
        model = make_model(cfg, sd, "fp32").train()
        xg = x.clone().requires_grad_(True)
        y = model(xg)
        y.square().sum().backward()
        return y.detach().clone(), xg.grad.clone(), {n: p.grad.clone() for n, p in model.named_parameters()}
    y0, gx0, g0 = run()
    monkeypatch.setenv("TANTE_CHAN_CHUNK", "80")
    y1, gx1, g1 = run()
    assert torch.equal(y0, y1)
    assert rel_l2(gx1.cpu().numpy(), gx0.cpu().numpy()) < 1e-6      # (weight gradients accumulate per chunk: summation order differs)
    for n in g0:
        assert rel_l2(g1[n].cpu().numpy(), g0[n].cpu().numpy()) < 1e-5, n
