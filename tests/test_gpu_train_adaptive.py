"""The batched adaptive BPTT rollout (`TANTE.rollout_train` for deg=False: tante_train_forward_hist / tante_backward_hist, one
device cursor per sample) against what R_Trainer computes with its per-sample B=1 loops (trainer/r_trainer.py:117-133): the
reference goldens through the drop-in trainer, the module's own per-sample loop at out_T = 1.5 and, with out_T >= 2, samples
that take different step sequences, finish early and overshoot."""
import pytest
import torch

from conftest import golden_cfg, load_golden, rel_l2
from oracle import tante_oracle as O
from test_gpu_train import BF16_GRAD_TOL, FP32_GRAD_TOL, _report

pytestmark = pytest.mark.gpu

# in_T 3 < n_steps, two Taylor orders (R_t is the mean over both interprators)
CFG = O.OracleConfig(in_T=3, n_fields=3, H=32, W=64, taylor_order=2, attn_axes="THW-TW", deg=False)


def _counting(model):
    """Counts the calls of model.rollout_train (so that a test can assert the batched path was taken)."""
    calls = []
    inner = model.rollout_train

    def wrapped(*a, **k):
        calls.append(1)
        return inner(*a, **k)
    model.rollout_train = wrapped
    return calls


def _per_sample_loop(model, x, n_steps, out_T):
    """r_trainer.py:117-133 at B = 1 per sample: channels-first frames (B, n_steps, D, H, W), sample-major flat Rts, and the
    frames each call of each sample emitted."""
    outs, rts, seqs = [], [], []
    for b in range(x.shape[0]):
        moving, ys, cum, seq = x[b:b + 1], [], 0, []
        while cum < n_steps:
            y, rt = model(moving, out_T)
            cum += y.shape[1]
            if cum < n_steps:
                moving = torch.cat([moving[:, y.shape[1]:], y], dim=1)
            ys.append(y)
            rts.append(rt)
            seq.append(y.shape[1])
        outs.append(torch.cat(ys, dim=1)[:, :n_steps])
        seqs.append(seq)
    return torch.cat(outs, dim=0), torch.cat(rts, dim=0), seqs


def _grads(model, x):
    return x.grad.detach().clone(), {n: p.grad.detach().clone() for n, p in model.named_parameters()}


def _assert_grads_close(got, want, tol):
    (gx1, gp1), (gx0, gp0) = got, want
    assert rel_l2(gx1.cpu().numpy(), gx0.cpu().numpy()) < tol
    for n in gp0:
        assert rel_l2(gp1[n].cpu().numpy(), gp0[n].cpu().numpy()) < tol, n


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("name", ["train_adp_k2", "train_adp_k2_lya"])
def test_r_trainer_rollout_matches_reference_golden(name, prec):
    """One R_Trainer training step (rollout_model in train mode -> MSE + rt penalty -> backward) through the drop-in trainer,
    which takes the batched rollout, against the reference's own loss, predictions, Rts and gradients."""
    from gpu_util import make_model
    from tante_b200 import R_Trainer
    from tante_b200.trainer import mse_loss
    z, meta = load_golden(name)
    cfg = golden_cfg(meta)
    model = make_model(cfg, O.make_state_dict(cfg, meta["seed"], meta["rt_bias"]), prec).train()
    assert model.bptt_windows_ok
    calls = _counting(model)
    tr = R_Trainer(model=model, device="cuda", n_steps_output=meta["n_steps"])
    x = O.make_input(cfg, meta["B"], meta["input_seed"]).cuda()
    xl = x.permute(0, 1, 3, 4, 2).contiguous().requires_grad_(True)       # the loader's channels-last batch
    g = torch.Generator().manual_seed(meta["target_seed"])
    y_ref = torch.randn(meta["B"], meta["n_steps"], cfg.H, cfg.W, cfg.n_fields, generator=g)
    y, y_ref, rts = tr.rollout_model(model, {"input": xl, "output": y_ref}, tr.formatter, "train")
    assert calls == [1], "R_Trainer.rollout_model did not take the batched rollout"
    loss = mse_loss(y, y_ref, rts, 0.5, 2)
    loss.backward()
    s = meta["stride"]
    grad_input = xl.grad.permute(0, 1, 4, 2, 3)
    if prec == "fp32":
        assert abs(float(loss) - float(z["loss"])) < 2e-6 * max(1.0, abs(float(z["loss"])))
        assert rel_l2(y.detach().cpu().reshape(-1)[::s].numpy(), z["y_pred"]) < 1e-5
        assert rel_l2(rts.detach().cpu().numpy(), z["Rts"]) < 1e-5
        tol = FP32_GRAD_TOL
    else:
        assert abs(float(loss) - float(z["loss"])) < 2e-2 * max(1.0, abs(float(z["loss"])))
        tol = BF16_GRAD_TOL
    bad, _ = _report(model, z, meta, tol)
    assert not bad, "parameter gradients differ from the reference:\n" + "\n".join(bad)
    assert rel_l2(grad_input.cpu().reshape(-1)[::s].numpy(), z["grad_input"]) < tol


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("n_steps", [4, 6])
def test_batched_rollout_equals_per_sample_loop(monkeypatch, prec, n_steps):
    """out_T = 1.5 (R_Trainer): every call emits one frame per sample.  tante_b200.trainer.rollout_train on the batched path vs
    the per-sample loop of the same module (TANTE_BPTT_WINDOWS=0), B = 5: predictions and Rts, gradients of the input and of
    every parameter under a loss on both."""
    from gpu_util import make_model
    from tante_b200.trainer import rollout_train
    model = make_model(CFG, O.make_state_dict(CFG, 21), prec).train()
    x = O.make_input(CFG, 5, 22).cuda()
    gen = torch.Generator().manual_seed(23)
    gy = torch.randn(5, n_steps, CFG.H, CFG.W, CFG.n_fields, generator=gen).cuda()
    gr = torch.randn(5 * n_steps, generator=gen).cuda()

    def run(flag):
        monkeypatch.setenv("TANTE_BPTT_WINDOWS", flag)
        model.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(True)
        y, rts = rollout_train(model, xi, n_steps, 1.5)
        ((y * gy).sum() + (rts * gr).sum()).backward()
        return y.detach(), rts.detach(), _grads(model, xi)

    y0, r0, g0 = run("0")
    calls = _counting(model)
    y1, r1, g1 = run("1")
    assert calls == [1]
    if prec == "fp32":
        assert torch.equal(y1, y0)
        assert torch.equal(r1, r0)
        _assert_grads_close(g1, g0, FP32_GRAD_TOL)
    else:
        assert rel_l2(y1.cpu().numpy(), y0.cpu().numpy()) < 2e-2
        assert rel_l2(r1.cpu().numpy(), r0.cpu().numpy()) < 2e-2


def test_per_sample_step_sequences():
    """out_T = 3: R_t straddles 2, so samples take different step sequences, one finishes while others still run and last calls
    overshoot n_steps.  ns, steps, predictions, Rts and gradients against chained B = 1 `model(window, out_T)` calls."""
    from gpu_util import make_model
    from tante_b200.trainer import flat_rts
    n_steps, out_T, B = 5, 3.0, 4
    model = make_model(CFG, O.make_state_dict(CFG, 31, 0.9035), "fp32").train()
    x = (O.make_input(CFG, B, 32) * torch.tensor([0.2, 1.0, 3.0, 6.0]).view(B, 1, 1, 1, 1)).cuda()
    gen = torch.Generator().manual_seed(33)
    gy = torch.randn(B, n_steps, CFG.n_fields, CFG.H, CFG.W, generator=gen).cuda()

    xi = x.clone().requires_grad_(True)
    y0, r0, seqs = _per_sample_loop(model, xi, n_steps, out_T)
    gr = torch.randn(r0.shape[0], generator=gen).cuda()
    ((y0 * gy).sum() + (r0 * gr).sum()).backward()
    g0 = _grads(model, xi)

    # the case is not vacuous
    assert len({tuple(s) for s in seqs}) >= 2
    assert min(len(s) for s in seqs) < max(len(s) for s in seqs)
    assert any(sum(s) > n_steps for s in seqs)
    assert all(abs(r - round(r)) >= 1e-4 for r in r0.tolist())

    model.zero_grad(set_to_none=True)
    xi = x.clone().requires_grad_(True)
    y1, rts, ns, steps = model.rollout_train(xi, n_steps, out_T=out_T)
    assert ns.shape == rts.shape == (max(len(s) for s in seqs), B)
    assert steps.tolist() == [len(s) for s in seqs]
    for b, s in enumerate(seqs):
        assert ns[:, b].tolist() == s + [0] * (ns.shape[0] - len(s)), b
        assert (rts[len(s):, b] == 0).all()
    r1 = flat_rts(rts, ns)
    assert torch.equal(y1.detach(), y0.detach())
    assert torch.equal(r1.detach(), r0.detach())
    ((y1 * gy).sum() + (r1 * gr).sum()).backward()
    _assert_grads_close(_grads(model, xi), g0, FP32_GRAD_TOL)


def test_grad_bucket_slots_and_dropout_determinism():
    """GradBucket (one add per call into the flat gradient) == the plain autograd path; every tape slot is returned by the
    backward; with dropout 0.1 two runs under the same torch.manual_seed give the same loss and gradients."""
    from gpu_util import make_model
    from tante_b200.trainer import GradBucket, mse_loss, rollout_train
    sd = O.make_state_dict(CFG, 41)
    x = O.make_input(CFG, 3, 42).cuda()
    y_ref = torch.randn(3, 4, CFG.H, CFG.W, CFG.n_fields, generator=torch.Generator().manual_seed(43)).cuda()

    def step(model):
        y, rts = rollout_train(model, x, 4, 1.5)
        loss = mse_loss(y, y_ref, rts)
        loss.backward()
        return float(loss)

    plain = make_model(CFG, sd, "fp32").train()
    step(plain)
    want = {n: p.grad.clone() for n, p in plain.named_parameters()}
    model = make_model(CFG, sd, "fp32").train()
    bucket = GradBucket(model)
    eng = next(iter(model._engines.values()))
    assert model._flat_grad_view(eng) is not None
    for rep in range(2):
        bucket.zero()
        step(model)
        for n, p in model.named_parameters():
            # (the weight-gradient kernels reduce over rows with fp32 atomics: the order of those adds is not fixed)
            assert rel_l2(p.grad.cpu().numpy(), want[n].cpu().numpy()) < 1e-5, (rep, n)
    assert eng.n_slots >= 4 and sorted(eng.free_slots) == list(range(eng.n_slots))

    model.dropout = 0.1
    runs = []
    for _ in range(2):
        bucket.zero()
        torch.manual_seed(7)
        loss = step(model)
        runs.append((loss, bucket.flat.clone()))
    assert runs[0][0] == runs[1][0]
    assert rel_l2(runs[1][1].cpu().numpy(), runs[0][1].cpu().numpy()) < 1e-5
    model.dropout = 0.0
    bucket.zero()
    assert step(model) != runs[0][0]          # (the dropout was applied)
