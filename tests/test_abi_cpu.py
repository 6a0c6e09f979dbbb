"""Host-side checks that need no GPU: the C-ABI library loads, exports every symbol the header
declares, validates configs like the reference constructor, and the module's parameter tree /
default init equal the reference's."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden
from tante_b200 import TANTE, TanteMetadata, _abi


def header_functions():
    src = open(os.path.join(ROOT, "include", "tante_b200.h")).read()
    return sorted(set(re.findall(r"TANTE_API[^;(]*?\b(tante_\w+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _abi.load()
    names = header_functions()
    assert len(names) >= 15
    assert sorted(_abi.SIGNATURES) == names, "ctypes table and header disagree"
    out = subprocess.run(["nm", "-D", "--defined-only", _abi.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (tante_\w+)", out))
    assert set(names) <= exported
    assert lib.tante_version() >= 1


def test_library_is_sm100a_and_torch_free():
    out = subprocess.run(["ldd", _abi.LIB_PATH], capture_output=True, text=True).stdout
    assert "torch" not in out and "libc10" not in out
    cu = subprocess.run(["cuobjdump", "-lelf", _abi.LIB_PATH], capture_output=True, text=True)
    if cu.returncode == 0:
        assert "sm_100a" in cu.stdout


def _cfg(**kw):
    c = _abi.TanteConfig()
    base = dict(in_T=4, n_fields=4, H=128, W=384, taylor_order=1, n_head=8, embed_dim=256, patch_scale=8, deg=1,
                output_length=1, frame_interval=1.0, precision=0)
    base.update(kw)
    axes = base.pop("axes", ["THWTHWTHW"])
    for k, v in base.items():
        setattr(c, k, v)
    for i, seg in enumerate(axes):
        c.n_layers[i] = len(seg)
        c.axes[i].value = seg.encode()
    return c


def test_create_validates_like_the_reference_ctor():
    lib = _abi.load()
    h = ctypes.c_void_p()
    assert lib.tante_create(ctypes.byref(_cfg()), 0, ctypes.byref(h)) == 0
    n = lib.tante_param_count(h)
    names = {lib.tante_param_name(h, i).decode(): lib.tante_param_numel(h, i) for i in range(n)}
    assert names["blocks.0.blocks.8.attn.in_proj_weight"] == 768 * 256
    assert names["s_emb"] == 16 * 48 * 256
    assert lib.tante_destroy(h) == 0
    # unknown patch scale -> KeyError in the reference (enc_dec_cnn.py:199)
    assert lib.tante_create(ctypes.byref(_cfg(patch_scale=7)), 0, ctypes.byref(h)) == 1
    assert b"patch_scale" in lib.tante_last_error()
    # empty segment -> ValueError (attn_backbone.py:105-106)
    assert lib.tante_create(ctypes.byref(_cfg(taylor_order=2, axes=["THW", ""])), 0, ctypes.byref(h)) == 1
    # calls before binding fail with a state error, not a crash
    assert lib.tante_create(ctypes.byref(_cfg()), 0, ctypes.byref(h)) == 0
    assert lib.tante_pack_params(h, None) != 0
    lib.tante_destroy(h)


@pytest.mark.parametrize("kw", [
    dict(taylor_order=1, attn_axes="THWTHWTHW", deg=True),
    dict(taylor_order=2, attn_axes="THW-HWT", deg=False),
    dict(taylor_order=2, attn_axes="TCW-CHC", deg=False),      # channel attention: channel_blocks + blocks of width expanded_channel
])
def test_param_table_matches_module_state_dict(kw):
    m = TANTE(4, TanteMetadata(spatial_resolution=(64, 96), n_fields=3), patch_scale=8, **kw)
    lib = _abi.load()
    cfg = _cfg(n_fields=3, H=64, W=96, taylor_order=kw["taylor_order"], deg=int(kw["deg"]),
               axes=kw["attn_axes"].split("-"))
    h = ctypes.c_void_p()
    assert lib.tante_create(ctypes.byref(cfg), 0, ctypes.byref(h)) == 0
    table = {lib.tante_param_name(h, i).decode(): lib.tante_param_numel(h, i) for i in range(lib.tante_param_count(h))}
    sd = {k: v.numel() for k, v in m.state_dict().items()}
    assert table == sd
    lib.tante_destroy(h)


def test_ctor_errors_match_reference():
    md = TanteMetadata(spatial_resolution=(64, 64), n_fields=2)
    with pytest.raises(ValueError):
        TANTE(4, md, taylor_order=2, attn_axes="THW", patch_scale=8)
    with pytest.raises(ValueError):
        TANTE(4, md, attn_axes="THQ", patch_scale=8)
    with pytest.raises(KeyError):
        TANTE(4, md, patch_scale=7)
    m = TANTE(4, md, patch_scale=8)
    with pytest.raises(RuntimeError, match="no CPU path"):
        with torch.inference_mode():
            m(torch.zeros(1, 4, 2, 64, 64))


def test_default_init_and_state_dict_equal_the_stored_reference():
    """Parameter order and seeded default init against the reference module's, as stored in tests/golden/ref_init.npz
    (`python -m oracle.make_golden --live`): every key in order, shapes, a strided sample of each tensor bitwise, and
    the float64 sum and sum of squares over all of its elements."""
    from oracle.make_golden import INIT_CASES, init_summary
    z, meta = load_golden("ref_init")
    assert len(meta["init"]) == len(INIT_CASES)
    for i, (kw, case) in enumerate(zip(INIT_CASES, meta["init"])):
        assert case["kw"] == kw
        torch.manual_seed(211)
        sd = TANTE(4, TanteMetadata(spatial_resolution=(64, 96), n_fields=3), patch_scale=8, dropout=0.1, **kw).state_dict()
        assert list(sd.keys()) == case["keys"]
        for j, (k, v) in enumerate(sd.items()):
            sample, s, s2 = init_summary(v)
            shape, ref_s, ref_s2 = case["sums"][k]
            assert list(v.shape) == shape, k
            np.testing.assert_array_equal(sample, z[f"c{i}_{j}"], err_msg=k)
            assert s == pytest.approx(ref_s, rel=1e-12, abs=1e-12) and s2 == pytest.approx(ref_s2, rel=1e-12), k


def test_default_init_and_state_dict_equal_the_reference():
    from oracle import ref_shim
    if not ref_shim.reference_available():
        pytest.skip(ref_shim.SKIP_REASON)
    ns = ref_shim.load_reference()
    md = ref_shim.make_metadata(3, 64, 96)
    for kw in (dict(taylor_order=1, attn_axes="THWTHW", deg=True), dict(taylor_order=2, attn_axes="THW-HW", deg=False),
               dict(taylor_order=2, attn_axes="TH-W", deg=False, enc_dec_type="fno", modes1=16, modes2=16),
               dict(taylor_order=2, attn_axes="TCW-CH", deg=False, expanded_channel=256, mlp_ratio=2.0)):
        torch.manual_seed(211)
        ref = ns.TANTE(in_T=4, dset_metadata=md, patch_scale=8, dropout=0.1, **kw)
        torch.manual_seed(211)
        mine = TANTE(4, TanteMetadata(spatial_resolution=(64, 96), n_fields=3), patch_scale=8, dropout=0.1, **kw)
        rs, ms = ref.state_dict(), mine.state_dict()
        assert list(rs.keys()) == list(ms.keys())
        for k in rs:
            assert torch.equal(rs[k], ms[k]), k
