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


def test_axial_test_hooks_reject_out_of_range_arguments():
    """tante_test_attention / tante_test_propagator check their arguments before any device call (so this runs without
    a GPU).  Every call below breaks exactly one rule of an otherwise valid call; the pointers are never dereferenced."""
    lib = _abi.load()
    P = 0x10000          # 16-byte aligned stand-in for a device buffer
    kid = ctypes.c_int32(-1)

    def att(**kw):
        a = dict(dir=1, prec=_abi.PREC_BF16, qkv=P, dout=P, out=P, stats=P, nseq=8, S=80, inner=1, nh=8, C=256, causal=0,
                 p=0.0)
        a.update(kw)
        return lib.tante_test_attention(a["dir"], a["prec"], a["qkv"], a["dout"], a["out"], a["stats"], a["nseq"], a["S"],
                                        a["inner"], a["nh"], a["C"], a["causal"], a["p"], 1, 0, ctypes.byref(kid), None)

    def prop(**kw):
        a = dict(dir=1, prec=_abi.PREC_BF16, xin=P, x=P, W1=P, b1=P, W2=P, b2=P, gW1=P, gb1=P, gW2=P, gb2=P, S=32, IC=256,
                 outer=4)
        a.update(kw)
        return lib.tante_test_propagator(a["dir"], a["prec"], a["xin"], a["x"], a["W1"], a["b1"], a["W2"], a["b2"], a["gW1"],
                                         a["gb1"], a["gW2"], a["gb2"], a["S"], a["IC"], a["outer"], ctypes.byref(kid), None)

    bad = [
        (att, dict(qkv=None), "null argument"), (att, dict(out=None), "null argument"), (att, dict(dout=None), "null argument"),
        (att, dict(stats=None), "null argument"), (att, dict(qkv=P + 2), "16-byte aligned"),
        (att, dict(S=0), "must be >= 1"), (att, dict(nseq=0), "must be >= 1"), (att, dict(inner=0), "must be >= 1"),
        (att, dict(nseq=1 << 31), "must be >= 1"),
        (att, dict(C=256, nh=2), "head_dim must be 16, 32 or 64"), (att, dict(C=256, nh=32), "head_dim must be 16, 32 or 64"),
        (att, dict(C=250, nh=8), "C must be n_head * head_dim"), (att, dict(nh=0), "C must be n_head * head_dim"),
        (att, dict(p=1.0), "drop_p must be in [0, 1)"), (att, dict(p=-0.1), "drop_p must be in [0, 1)"),
        (att, dict(p=float("nan")), "drop_p must be in [0, 1)"), (att, dict(causal=2), "causal must be 0 or 1"),
        (att, dict(dir=2), "dir"), (att, dict(prec=7), "precision"),
        (prop, dict(xin=None), "null argument"), (prop, dict(W2=None), "null argument"), (prop, dict(gW1=None), "null argument"),
        (prop, dict(gb2=None), "null argument"), (prop, dict(dir=0, b2=None), "null argument"),
        (prop, dict(x=P + 4), "16-byte aligned"),
        (prop, dict(S=0), "S must be in 1 .. 96"), (prop, dict(S=97), "S must be in 1 .. 96"),
        (prop, dict(IC=0), "IC must be a positive multiple of 4"), (prop, dict(IC=258), "IC must be a positive multiple of 4"),
        (prop, dict(outer=0), "outer must be"), (prop, dict(dir=-1), "dir"), (prop, dict(prec=2), "precision"),
    ]
    for fn, kw, msg in bad:
        assert fn(**kw) == 1, (fn.__name__, kw)
        assert msg in lib.tante_last_error().decode(), (fn.__name__, kw, lib.tante_last_error())
    assert kid.value == -1


def test_gemm_plan_hook_rejects_bad_arguments():
    """tante_test_gemm_plan checks its arguments before any device call."""
    lib = _abi.load()
    n = ctypes.c_int32(-1)
    for args, msg in (((256, 256, 256, 0, None), "null argument"), ((0, 256, 256, 0, ctypes.byref(n)), "must be >= 1"),
                      ((256, 256, -64, 1, ctypes.byref(n)), "must be >= 1")):
        assert lib.tante_test_gemm_plan(*args) == 1, args
        assert msg in lib.tante_last_error().decode(), (args, lib.tante_last_error())
    assert n.value == -1


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
