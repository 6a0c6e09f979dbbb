"""Oracle restatement vs the upstream module: against its outputs stored in tests/golden/ref_live_*.npz (always), and
against the LIVE module where TANTE_REFERENCE_ROOT names an upstream checkout (`python -m oracle.make_golden --live`
rewrites the stored outputs from it)."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_l2
from oracle import ref_shim, tante_oracle as O
from oracle.make_golden import LIVE_CASES

live = pytest.mark.skipif(not ref_shim.reference_available(), reason=ref_shim.SKIP_REASON)


@pytest.mark.parametrize("name", sorted(LIVE_CASES))
def test_oracle_equals_stored_reference(name):
    cfg, B, out_T, bias = LIVE_CASES[name]
    z, meta = load_golden(name)
    sd = O.make_state_dict(cfg, meta["seed"], bias)
    assert sorted(sd.keys()) == meta["keys"]
    x = O.make_input(cfg, B, meta["input_seed"])
    with torch.inference_mode():
        o = O.forward(sd, cfg, x, out_T)
    y = o if cfg.deg else o[0]
    if not cfg.deg:
        np.testing.assert_allclose(o[1].numpy(), z["R_t"], rtol=0, atol=5e-6)
    assert list(y.shape) == meta["frames_shape"]
    assert rel_l2(y.reshape(-1)[::meta["stride"]].numpy(), z["frames"]) < 2e-6


@live
@pytest.mark.parametrize("cfg,B,out_T,bias", [
    (O.OracleConfig(n_fields=4, H=64, W=64, taylor_order=1, deg=True), 2, 1, 0.0),
    (O.OracleConfig(n_fields=3, H=32, W=32, taylor_order=2, attn_axes="THWLA-TYW", deg=False, patch_scale=4,
                    frame_interval=0.5), 2, 8, 5.2),
    (O.OracleConfig(n_fields=2, H=64, W=128, taylor_order=1, attn_axes="THW", deg=False, patch_scale=16), 1, 8, 1.3),
])
def test_oracle_equals_live_reference(cfg, B, out_T, bias):
    from oracle.make_golden import build_ref
    ns = ref_shim.load_reference()
    sd = O.make_state_dict(cfg, 7, bias)
    m = build_ref(ns, cfg, sd).eval()
    assert set(m.state_dict().keys()) == set(sd.keys())
    x = O.make_input(cfg, B, 8)
    with torch.inference_mode():
        out = m(x, out_T)
        o = O.forward(sd, cfg, x, out_T)
    if cfg.deg:
        y, yo = out, o
    else:
        (y, rt), (yo, rto) = out, o
        assert torch.allclose(rt, rto, atol=5e-6)
    assert y.shape == yo.shape
    assert rel_l2(yo.numpy(), y.numpy()) < 2e-6


@live
def test_unrepaired_adaptive_branch_crashes_as_published():
    """SURVEY.md F5: documents why the oracle is 'reference + minimal repair'."""
    from oracle.make_golden import build_ref
    ns = ref_shim.load_reference()
    cfg = O.OracleConfig(n_fields=2, H=32, W=32, taylor_order=1, attn_axes="T", deg=False)
    m = build_ref(ns, cfg, O.make_state_dict(cfg, 1)).eval()
    with pytest.raises(Exception):
        ns.TANTE._unrepaired_forward(m, O.make_input(cfg, 1, 2), 4)
