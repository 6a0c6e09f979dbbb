"""The batched adaptive rollout returns R_t per call and sample, (n_calls, B), with the frames each call emitted; R_Trainer's
rt penalty and rt_analyse expect the flat Rts of its per-sample loops (r_trainer.py:118-133).  `flat_rts` must give that order,
and its gradient must land on the (call, sample) entries it came from."""
import torch

from tante_b200.trainer import flat_rts


def _reference_order(rts, ns):
    """torch.cat over the per-sample loops: sample 0's calls in order, then sample 1's, ..."""
    n_calls, B = rts.shape
    return torch.stack([rts[k, b] for b in range(B) for k in range(n_calls) if int(ns[k, b]) > 0])


def test_flat_rts_order_and_gradient_scatter():
    g = torch.Generator().manual_seed(0)
    # four samples: 5 calls of 1 frame, 3 calls (1, 2, 2), 2 calls (2, 3), 5 calls (1, 1, 1, 1, 1)
    ns = torch.tensor([[1, 1, 2, 1], [1, 2, 3, 1], [1, 2, 0, 1], [1, 0, 0, 1], [1, 0, 0, 1]], dtype=torch.int32)
    base = torch.randn(5, 4, generator=g) + 2.0
    w = torch.randn(int((ns > 0).sum()), generator=g)

    a = base.clone().requires_grad_(True)
    want = _reference_order(a, ns)
    (want * w).sum().backward()
    b = base.clone().requires_grad_(True)
    got = flat_rts(b, ns)
    (got * w).sum().backward()
    assert torch.equal(got.detach(), want.detach())
    assert torch.equal(b.grad, a.grad)
    assert (b.grad[ns == 0] == 0).all()


def test_flat_rts_every_call():
    """One frame per call (out_T = 1.5): every sample takes part in every call; the unmasked form gives the same order."""
    rts = torch.arange(12.0).view(3, 4)
    ns = torch.ones(3, 4, dtype=torch.int32)
    assert torch.equal(flat_rts(rts, ns, every_call=True), _reference_order(rts, ns))
    assert torch.equal(flat_rts(rts, ns), _reference_order(rts, ns))
