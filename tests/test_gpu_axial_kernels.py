"""The axial attention and propagator kernels stand-alone, through the model's own dispatch (tante_test_attention /
tante_test_propagator), against fp64 restatements of the same operations at the shapes where each kernel changes behaviour:
packing and padding of short sequences, tail blocks, partial key blocks, head quads, causal masks, dropout, one slab and
many slabs per persistent CTA.  The error is bounded per block -- each (sequence, head) of the attention, each
(outer, 128-column) slab of the propagators -- so that an error confined to one block cannot hide inside a global norm;
a whole-tensor rel-L2 is checked on top.  Every write-only output starts as NaN and every buffer carries a sentinel guard
band, so an element never written and a write out of bounds both fail."""
import ctypes
import math

import numpy as np
import pytest
import torch

from conftest import rel_l2
from dropout_ref import multipliers

pytestmark = pytest.mark.gpu

FP32, BF16 = 0, 1
# kernel ids of include/tante_b200.h (TANTE_AXK_*)
FLASH, MMA, SIMT, LONG_MMA, LONG_FFMA, SMALL, WIDE, GENERIC = range(1, 9)
NAMES = {FLASH: "flash", MMA: "mma", SIMT: "simt", LONG_MMA: "long-mma", LONG_FFMA: "long-ffma", SMALL: "small", WIDE: "wide",
         GENERIC: "generic"}

GUARD = 512                 # sentinel elements on each side of every buffer (keeps 16-byte alignment in f32 and bf16)
SENTINEL = -1536.0          # exact in bf16, far from every value the kernels produce here
F64 = torch.float64


def _lib():
    from tante_b200 import _abi
    return _abi, _abi.load()


def _dt(prec):
    return torch.bfloat16 if prec == BF16 else torch.float32


class Guarded:
    """A device buffer with a sentinel band before and after the `n` elements the kernel may touch."""

    def __init__(self, n, dtype, init=None):
        self.buf = torch.full((n + 2 * GUARD,), SENTINEL, dtype=dtype, device="cuda")
        self.t = self.buf[GUARD:GUARD + n]
        if init is None:
            self.t.fill_(float("nan"))
        else:
            self.t.copy_(init.reshape(-1))

    def ptr(self):
        return self.t.data_ptr()

    def check_guard(self, what):
        band = torch.cat([self.buf[:GUARD], self.buf[-GUARD:]]).float()
        assert bool((band == SENTINEL).all()), f"{what}: write outside the buffer"


def _block_err(out, ref, block_dims):
    """max over blocks of (max |out - ref| in the block) / (max |ref| in the block); NaN anywhere fails."""
    out, ref = out.to(F64), ref.to(F64)
    assert not bool(torch.isnan(out).any()), "element never written (NaN left in the output)"
    err = (out - ref).abs().amax(dim=block_dims)
    mag = ref.abs().amax(dim=block_dims)
    floor = 1e-6 * float(ref.abs().max()) + 1e-30
    return float((err / mag.clamp_min(floor)).max())


def _gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _gelu_grad(x):
    return 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def _bf(t):
    return t.to(torch.bfloat16).to(F64)


# ---------------------------------------------------------------------------------------------------------------------------
# attention


HEADS = [(256, 16), (256, 8), (256, 4), (512, 16), (512, 8)]       # (C, n_head): head_dim 16 / 32 / 64, one or several quads


INNERS = [1, 3, 37, 257]      # inner_sz: contiguous sequences, odd strides, and a stride of the size of the T axis's L


def _att_cases():
    cases = []
    short = [1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64]
    for i, S in enumerate(short):
        for prec in (FP32, BF16):
            cases.append((prec, S, *HEADS[(i + prec) % 5], INNERS[(i + prec) % 4], False, 0.0))
            if prec == BF16 and HEADS[(i + prec) % 5][0] // HEADS[(i + prec) % 5][1] != 32:
                cases.append((prec, S, 256, 8, INNERS[i % 4], False, 0.0))       # every short S on the mma kernels too
    for i, S in enumerate([1, 3, 4, 5, 16, 33, 64]):
        for prec in (FP32, BF16):
            heads = HEADS[i % 5] if prec == FP32 else ((256, 8), (512, 8))[i % 2]       # bf16: the mma kernels and SIMT
            cases.append((prec, S, *heads, INNERS[i % 4], True, 0.0))
    # dropout: the mask of a probability is keyed by the query's token, (outer * S + pos) * inner_sz + inner
    for S, p, causal, inner in [(3, 0.1, False, 1), (3, 0.1, False, 37), (5, 0.1, True, 3), (16, 0.5, False, 3),
                                (33, 0.1, False, 37), (64, 0.5, True, 3), (80, 0.1, False, 1), (96, 0.5, False, 3)]:
        for prec in (FP32, BF16):
            cases.append((prec, S, 256, 8, inner, causal, p))
    for i, S in enumerate([65, 80, 96, 127, 128, 129, 384]):
        inner = 3 if S == 384 else INNERS[i % 4]
        for prec in (FP32, BF16):
            cases.append((prec, S, *HEADS[(i + prec) % 5], inner, False, 0.0))
        cases.append((BF16, S, 256, 8, INNERS[(i + 1) % 4] if S != 384 else 1, False, 0.0))   # the flash / long-mma kernels
    cases.append((BF16, 96, 256, 8, 3, True, 0.0))                               # causal S > 64: SIMT forward, long FFMA backward
    cases.append((FP32, 96, 256, 16, 1, True, 0.0))
    return sorted(set(cases))


def _n_outer(S, inner):
    """Outer groups of a case: two or more whenever inner_sz > 1, so that token = (outer * S + pos) * inner_sz + inner runs
    with outer > 0 at every stride; and nseq = n_outer * inner_sz leaving a tail block of the packed kernels
    (nseq % G != 0) wherever a packing factor allows one."""
    packs = [16 // S if S <= 16 else 1, max(1, 64 // S)]        # sequences per block: mma kernels, SIMT backward
    for k in ((5, 7, 3) if inner == 1 else (2, 3, 5, 7)):
        if all(G == 1 or (k * inner) % G for G in packs):
            return k
    return 5 if inner == 1 else 2


def _att_id(c):
    prec, S, C, nh, inner, causal, p = c
    return f"{'bf16' if prec else 'fp32'}-S{S}-hd{C // nh}-nh{nh}-in{inner}{'-causal' if causal else ''}{f'-p{p}' if p else ''}"


ATT_CASES = _att_cases()


def _att_layout(x, n_outer, S, inner, nh, hd):
    """[tokens][parts * C] with token = (outer * S + pos) * inner + i  ->  [parts][seq = outer * inner + i][head][pos][d]"""
    parts = x.shape[1] // (nh * hd)
    return x.view(n_outer, S, inner, parts, nh, hd).permute(3, 0, 2, 4, 1, 5).reshape(parts, n_outer * inner, nh, S, hd)


def _drop_mult(seed, site, p, n_outer, S, inner, nh):
    """Z[seq][head][qpos][kpos] of tests/dropout_ref: grp = ((tok_q * n_head + head) << 13) | (kpos >> 3), lane = kpos & 7."""
    o = np.arange(n_outer, dtype=np.uint64)[:, None, None]
    i = np.arange(inner, dtype=np.uint64)[None, :, None]
    pos = np.arange(S, dtype=np.uint64)[None, None, :]
    tok = ((o * np.uint64(S) + pos) * np.uint64(inner) + i).reshape(n_outer * inner, S)          # [seq][qpos]
    head = np.arange(nh, dtype=np.uint64)
    kpos = np.arange(S, dtype=np.uint64)
    grp = ((tok[:, None, :, None] * np.uint64(nh) + head[None, :, None, None]) << np.uint64(13)) | (kpos >> np.uint64(3))
    lane = np.broadcast_to((kpos & np.uint64(7)).astype(np.int64), grp.shape)
    return torch.from_numpy(multipliers(seed, site, grp, lane, p)).to("cuda", F64)


def _att_reference(qkv, dout, n_outer, S, inner, nh, hd, causal, Z):
    q, k, v = _att_layout(qkv.to(F64), n_outer, S, inner, nh, hd)
    s = q @ k.transpose(-1, -2) / math.sqrt(hd)
    if causal:
        s = s.masked_fill(torch.ones(S, S, dtype=torch.bool, device="cuda").triu(1), float("-inf"))
    P = torch.softmax(s, dim=-1)
    PZ = P if Z is None else P * Z
    out = PZ @ v
    if dout is None:
        return out
    dO = _att_layout(dout.to(F64), n_outer, S, inner, nh, hd)[0]
    dV = PZ.transpose(-1, -2) @ dO
    dP = dO @ v.transpose(-1, -2)
    if Z is not None:
        dP = dP * Z
    dS = P * (dP - (P * dP).sum(-1, keepdim=True))
    dQ = dS @ k / math.sqrt(hd)
    dK = dS.transpose(-1, -2) @ q / math.sqrt(hd)
    return torch.stack([dQ, dK, dV])


def _att_forward_model(qkv, n_outer, S, inner, nh, hd, causal, Z, kernel):
    """The bf16 forward with the roundings of `kernel` (fp64 elsewhere): the mma and flash kernels round the (dropped-out)
    unnormalised probabilities exp(s - m) to bf16 before the PV product and normalise by the sum of the unrounded ones; the
    flash kernel takes m as the running maximum over the 64-key blocks seen so far and rescales exactly.  Returns the
    model output and two per-element magnitudes: A = sum_k |p_k v_k| / l and M = max_k p_k / l * max_k |v_k|."""
    q, k, v = _att_layout(qkv.to(F64), n_outer, S, inner, nh, hd)
    s = q @ k.transpose(-1, -2) / math.sqrt(hd)
    if causal:
        s = s.masked_fill(torch.ones(S, S, dtype=torch.bool, device="cuda").triu(1), float("-inf"))
    m = s.amax(-1, keepdim=True)
    if kernel == FLASH:
        nb = (S + 63) // 64
        bm = torch.nn.functional.pad(s, (0, nb * 64 - S), value=float("-inf")).view(*s.shape[:-1], nb, 64).amax(-1)
        run = torch.cummax(bm, dim=-1).values.repeat_interleave(64, dim=-1)[..., :S]      # running max at each key
        p = _bf(torch.exp(s - run)) * torch.exp(run - m)
    else:
        p = torch.exp(s - m)
        if Z is not None:
            p = p * Z
        if kernel == MMA:
            p = _bf(p)
    l = torch.exp(s - m).sum(-1, keepdim=True)
    out = p @ v / l
    A = p.abs() @ v.abs() / l
    M = p.amax(-1, keepdim=True) / l * v.abs().amax(-2, keepdim=True)
    return out, A, M


def _bf16_ulp(x):
    """distance between adjacent bf16 values at |x| (8 significant bits)"""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.pow(2.0, e - 7)


# Bounds.  fp32 kernels: the exact mode (fp32 accumulation, expf), ~1e-6 of the block maximum; 2e-5 in the backward,
# where dQ and dK come out of sums over S keys that cancel, so their block maxima are small next to the terms.
# bf16 forward: the reference rounds the probabilities where the kernel does (_att_forward_model), so the output must be
# that value rounded to bf16: within half an ulp of it, plus what fp32 arithmetic inside the kernel can move (2^-16 of
# sum_k |p_k v_k| / l), plus one probability whose bf16 rounding an fp32 exp may flip (one ulp, <= 2^-7 of p_k |v_k| / l).
# That is checked per element; per block it leaves half an ulp, <= 2^-8 of the block maximum, with 2^-10 for the rest.
# bf16 backward: the kernels recompute P in fp32 and round to bf16 three times on the way to an output -- P (before dV)
# or dP (before dS), dS (before dQ, dK), and the output -- each up to 2^-8 relative: 3 * 2^-8 of the block maximum.  Each
# of dQ, dK and dV is checked per (sequence, head) block against its own maximum.
# Measured on a B200, largest over the cases of this file (per block / rel-L2): fp32 2.0e-6 / 5.9e-7 forward, 8.9e-6 /
# 5.4e-7 backward; bf16 forward 3.9e-3 / 1.7e-3 (every kernel); bf16 backward 8.2e-3 / 2.4e-3 (mma), 8.0e-3 / 2.4e-3
# (long-mma), 3.9e-3 / 1.7e-3 (SIMT, long-ffma).
ATT_BOUND = {(FP32, 0): 1e-5, (FP32, 1): 2e-5, (BF16, 0): 2.0 ** -8 + 2.0 ** -10, (BF16, 1): 3 * 2.0 ** -8}
# rel-L2: a bf16 rounding alone leaves up to 2^-7 / sqrt(12) ~ 2.3e-3 RMS.
ATT_L2 = {(FP32, 0): 2e-6, (FP32, 1): 2e-6, (BF16, 0): 3e-3, (BF16, 1): 4e-3}


def _run_attention(direction, prec, S, C, nh, inner, causal, p, n_outer=None, seed=0x5EED5EED1234, site=37):
    _abi, lib = _lib()
    hd = C // nh
    n_outer = n_outer or _n_outer(S, inner)
    nseq = n_outer * inner
    tokens = nseq * S
    g = torch.Generator(device="cuda").manual_seed(1000 * S + 10 * C + nh + inner)
    dt = _dt(prec)
    qkv = (torch.randn(tokens, 3 * C, device="cuda", generator=g) * 1.25).to(dt)
    dout = torch.randn(tokens, C, device="cuda", generator=g).to(dt) if direction else None
    gq = Guarded(tokens * 3 * C, dt, qkv)
    gd = Guarded(tokens * C, dt, dout) if direction else None
    go = Guarded(tokens * (3 * C if direction else C), dt)
    gs = Guarded(2 * nseq * nh * S, torch.float32, torch.zeros(2 * nseq * nh * S, device="cuda")) if direction else None
    kid = ctypes.c_int32(-1)
    _abi.check(lib.tante_test_attention(direction, prec, gq.ptr(), gd.ptr() if gd else None, go.ptr(), gs.ptr() if gs else None,
                                        nseq, S, inner, nh, C, int(causal), p, seed, site, ctypes.byref(kid),
                                        torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    for b, what in ((gq, "qkv"), (gd, "dout"), (go, "out"), (gs, "stats")):
        if b is not None:
            b.check_guard(what)
    assert torch.equal(gq.t.view(tokens, 3 * C), qkv), "qkv modified"
    Z = _drop_mult(seed, site, p, n_outer, S, inner, nh) if p > 0 else None
    out = _att_layout(go.t.view(tokens, -1), n_outer, S, inner, nh, hd).to(F64)
    if direction == 0 and prec == BF16:
        ref, A, M = _att_forward_model(qkv, n_outer, S, inner, nh, hd, causal, Z, kid.value)
        slack = 0.5 * _bf16_ulp(ref) + 2.0 ** -16 * A + (2.0 ** -7 * M if kid.value in (MMA, FLASH) else 0.0)
        excess = float(((out[0] - ref).abs() - slack).max())
        assert excess <= 0.0, f"{NAMES.get(kid.value)}: an element is {excess:.3g} further from the bf16 model than rounding allows"
    else:
        ref = _att_reference(qkv, dout, n_outer, S, inner, nh, hd, causal, Z)
    if not direction:
        ref = ref[None]
    # blocks: (sequence, head, part) over (pos, d) -- the backward's dQ, dK and dV each against their own maximum
    blk = _block_err(out.permute(1, 2, 0, 3, 4), ref.permute(1, 2, 0, 3, 4), (3, 4))
    l2 = rel_l2(out.cpu().numpy(), ref.cpu().numpy())
    return kid.value, blk, l2


@pytest.mark.parametrize("case", ATT_CASES, ids=_att_id)
@pytest.mark.parametrize("direction", [0, 1], ids=["fwd", "bwd"])
def test_attention_matches_fp64(direction, case):
    prec, S, C, nh, inner, causal, p = case
    kid, blk, l2 = _run_attention(direction, prec, S, C, nh, inner, causal, p)
    tag = f"{NAMES.get(kid, kid)}: per-block {blk:.3g}, rel-L2 {l2:.3g}"
    assert blk <= ATT_BOUND[(prec, direction)], tag
    assert l2 <= ATT_L2[(prec, direction)], tag


@pytest.mark.parametrize("direction", [0, 1], ids=["fwd", "bwd"])
def test_attention_at_the_benchmarked_geometry(direction):
    """Axis W of the benchmark: S = 32, inner 1, nseq = 16 * 4 * 32 (B = 16, T = 4, H_p = 32), bf16, C 256, 8 heads."""
    kid, blk, l2 = _run_attention(direction, BF16, 32, 256, 8, 1, False, 0.0, n_outer=16 * 4 * 32)
    assert kid == MMA
    assert blk <= ATT_BOUND[(BF16, direction)] and l2 <= ATT_L2[(BF16, direction)], (blk, l2)


# ---------------------------------------------------------------------------------------------------------------------------
# propagators


def _prop_cases():
    cases = []
    Ss = [1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 48, 49, 64, 65, 96]
    ICs = [256, 512, 768]
    for i, S in enumerate(Ss):
        for prec in (FP32, BF16):
            cases.append((prec, S, ICs[(i + prec) % 3], 3, (i + prec) % 2 == 0))
    # many slabs per persistent CTA: nslab = outer * IC / 128 far above 4 * num_sms (2 * num_sms at MB = 4)
    for S, outer in [(3, 4096), (8, 2048), (16, 4096), (32, 2048), (64, 1536), (96, 768)]:
        for prec in (FP32, BF16):
            cases.append((prec, S, 256, outer, False))
    return cases


PROP_CASES = _prop_cases()


def _prop_id(c):
    prec, S, IC, outer, inplace = c
    return f"{'bf16' if prec else 'fp32'}-S{S}-IC{IC}-outer{outer}{'-inplace' if inplace else ''}"


def _prop_weights(S, g):
    W1 = torch.randn(S, S, device="cuda", generator=g) / math.sqrt(S)
    W2 = torch.randn(S, S, device="cuda", generator=g) / math.sqrt(S)
    b1 = torch.randn(S, device="cuda", generator=g) * 0.3
    b2 = torch.randn(S, device="cuda", generator=g) * 0.3
    return W1, b1, W2, b2


def _tc(prec, S):
    """The bf16 tensor-core propagators (9 <= S <= 64) round x, dy, the weights and the hidden activations to bf16."""
    return prec == BF16 and 9 <= S <= 64


def _prop_fwd_ref(x, W1, b1, W2, b2, tc):
    x64 = x.to(F64)
    xr, W1r, W2r = (_bf(x), _bf(W1), _bf(W2)) if tc else (x64, W1.to(F64), W2.to(F64))
    h = _gelu(torch.einsum("ji,oic->ojc", W1r, xr) + b1.to(F64)[None, :, None])
    if tc:
        h = _bf(h)
    return x64 + torch.einsum("pj,ojc->opc", W2r, h) + b2.to(F64)[None, :, None]


def _prop_bwd_ref(x, dy, W1, b1, W2, tc):
    xr, dr, W1r, W2r = (_bf(x), _bf(dy), _bf(W1), _bf(W2)) if tc else (x.to(F64), dy.to(F64), W1.to(F64), W2.to(F64))
    pre = torch.einsum("ji,oic->ojc", W1r, xr) + b1.to(F64)[None, :, None]
    dh = torch.einsum("pj,opc->ojc", W2r, dr)
    h, dpre = _gelu(pre), dh * _gelu_grad(pre)
    if tc:
        h, dpre = _bf(h), _bf(dpre)
    dx = dy.to(F64) + torch.einsum("ji,ojc->oic", W1r, dpre)
    gW2 = torch.einsum("opc,ojc->pj", dr, h)
    gW1 = torch.einsum("ojc,oic->ji", dpre, xr)
    return dx, gW1, dpre.sum((0, 2)), gW2, dr.sum((0, 2))


# Bounds.  fp32 kernels: the exact mode; the weight gradients are fp32 sums over up to 10^6 columns, reduced with atomics
# in a different order from run to run.  The bf16 mode evaluates GELU and its derivative with the erf approximant of
# DESIGN §4.3 (|err| <= 3.7e-5) through tanh.approx.f32 (relative error up to 2^-11): up to ~3e-4 on an activation,
# carried through one S-term sum.  The tensor-core kernels (9 <= S <= 64) are checked against a reference that rounds x,
# dy, the weights, h and dpre to bf16 where they do; what remains is that approximant moving the bf16 rounding of some
# hidden activations by one ulp (2^-8 relative).
# Measured on a B200, largest over the cases of this file (per block / rel-L2): fp32 1.0e-6 / 7.5e-7 (gradients);
# bf16 small / generic / wide 2.2e-4 / 1.6e-4; bf16 tensor-core 4.2e-3 (dx), 3.1e-3 (y) / 6.5e-4 (gb1).
PROP_BOUND = {FP32: 1e-5, BF16: 6e-4, "tc": 1e-2}
PROP_L2 = {FP32: 5e-6, BF16: 4e-4, "tc": 1.5e-3}


def _bound(prec, S, table):
    return table["tc"] if _tc(prec, S) else table[prec]


def _run_propagator(direction, prec, S, IC, outer, inplace):
    _abi, lib = _lib()
    g = torch.Generator(device="cuda").manual_seed(77 * S + IC + outer)
    W1, b1, W2, b2 = _prop_weights(S, g)
    x = torch.randn(outer, S, IC, device="cuda", generator=g)
    n = x.numel()
    gx = Guarded(n, torch.float32, x)
    gw = [Guarded(t.numel(), torch.float32, t) for t in (W1, b1, W2, b2)]
    kid = ctypes.c_int32(-1)
    st = torch.cuda.current_stream().cuda_stream
    if direction == 0:
        gy = gx if inplace else Guarded(n, torch.float32)
        _abi.check(lib.tante_test_propagator(0, prec, gx.ptr(), gy.ptr(), *[b.ptr() for b in gw], None, None, None, None, S, IC,
                                             outer, ctypes.byref(kid), st))
        torch.cuda.synchronize()
        for b in [gx, gy] + gw:
            b.check_guard("propagator forward")
        if not inplace:
            assert torch.equal(gx.t.view_as(x), x), "xin modified by the out-of-place forward"
        ref = _prop_fwd_ref(x, W1, b1, W2, b2, _tc(prec, S))
        out = gy.t.view(outer, S, IC // 128, 128)
        blk = _block_err(out.permute(0, 2, 1, 3), ref.view(outer, S, IC // 128, 128).permute(0, 2, 1, 3), (2, 3))
        l2 = rel_l2(out.double().cpu().numpy().ravel(), ref.cpu().numpy().ravel())
        return kid.value, [("y", blk, l2)]
    dy = torch.randn(outer, S, IC, device="cuda", generator=g)
    gd = Guarded(n, torch.float32, dy)
    prefill = [torch.randn(t.numel(), device="cuda", generator=g) for t in (W1, b1, W2, b2)]
    gg = [Guarded(t.numel(), torch.float32, t) for t in prefill]
    _abi.check(lib.tante_test_propagator(1, prec, gx.ptr(), gd.ptr(), *[b.ptr() for b in gw], *[b.ptr() for b in gg], S, IC,
                                         outer, ctypes.byref(kid), st))
    torch.cuda.synchronize()
    for b in [gx, gd] + gw + gg:
        b.check_guard("propagator backward")
    assert torch.equal(gx.t.view_as(x), x), "xin modified by the backward"
    dx, rW1, rb1, rW2, rb2 = _prop_bwd_ref(x, dy, W1, b1, W2, _tc(prec, S))
    out = gd.t.view(outer, S, IC // 128, 128)
    res = [("dx", _block_err(out.permute(0, 2, 1, 3), dx.view(outer, S, IC // 128, 128).permute(0, 2, 1, 3), (2, 3)),
            rel_l2(out.double().cpu().numpy().ravel(), dx.cpu().numpy().ravel()))]
    for name, b, pre, r in zip(("gW1", "gb1", "gW2", "gb2"), gg, prefill, (rW1, rb1, rW2, rb2)):
        ref = pre.to(F64) + r.reshape(-1)        # accumulated into what the arena held
        res.append((name, _block_err(b.t[None], ref[None], (1,)), rel_l2(b.t.double().cpu().numpy(), ref.cpu().numpy())))
    return kid.value, res


def _check_prop(prec, S, kid, res):
    for name, blk, l2 in res:
        tag = f"{NAMES.get(kid, kid)} {name}: per-block {blk:.3g}, rel-L2 {l2:.3g}"
        assert blk <= _bound(prec, S, PROP_BOUND), tag
        assert l2 <= _bound(prec, S, PROP_L2), tag


@pytest.mark.parametrize("case", PROP_CASES, ids=_prop_id)
def test_propagator_forward_matches_fp64(case):
    prec, S, IC, outer, inplace = case
    kid, res = _run_propagator(0, prec, S, IC, outer, inplace)
    _check_prop(prec, S, kid, res)


@pytest.mark.parametrize("case", PROP_CASES, ids=_prop_id)
def test_propagator_backward_matches_fp64(case):
    prec, S, IC, outer, _ = case
    kid, res = _run_propagator(1, prec, S, IC, outer, False)
    _check_prop(prec, S, kid, res)


# ---------------------------------------------------------------------------------------------------------------------------
# dispatch


# (precision, S, C, n_head, causal, p) -> (forward kernel, backward kernel)
ATT_DISPATCH = [
    ((BF16, 32, 256, 8, False, 0.0), (MMA, MMA)),
    ((BF16, 3, 512, 16, True, 0.1), (MMA, MMA)),
    ((BF16, 64, 256, 8, False, 0.5), (MMA, MMA)),
    ((BF16, 65, 256, 8, False, 0.0), (FLASH, LONG_MMA)),
    ((BF16, 384, 512, 16, False, 0.0), (FLASH, LONG_MMA)),
    ((BF16, 96, 256, 8, True, 0.0), (SIMT, LONG_FFMA)),
    ((BF16, 80, 256, 8, False, 0.1), (SIMT, LONG_FFMA)),
    ((BF16, 128, 256, 16, False, 0.0), (SIMT, LONG_FFMA)),
    ((BF16, 16, 256, 16, False, 0.0), (SIMT, SIMT)),
    ((BF16, 33, 256, 4, True, 0.0), (SIMT, SIMT)),
    ((FP32, 32, 256, 8, False, 0.0), (SIMT, SIMT)),
    ((FP32, 129, 256, 8, False, 0.0), (SIMT, LONG_FFMA)),
]
# (precision, S) -> (forward kernel, backward kernel)
PROP_DISPATCH = [
    ((FP32, 1), (SMALL, SMALL)), ((BF16, 4), (SMALL, SMALL)), ((BF16, 5), (GENERIC, GENERIC)), ((BF16, 8), (GENERIC, GENERIC)),
    ((BF16, 9), (MMA, MMA)), ((BF16, 32), (MMA, MMA)), ((BF16, 64), (MMA, MMA)), ((BF16, 65), (GENERIC, WIDE)),
    ((FP32, 5), (GENERIC, GENERIC)), ((FP32, 64), (GENERIC, GENERIC)), ((FP32, 96), (GENERIC, WIDE)),
]


def test_dispatch_table_reaches_every_kernel():
    hit = set()
    for (prec, S, C, nh, causal, p), want in ATT_DISPATCH:
        got = tuple(_run_attention(d, prec, S, C, nh, 1, causal, p, n_outer=2)[0] for d in (0, 1))
        assert got == want, ((prec, S, C, nh, causal, p), got)
        hit |= {("attention-fwd", got[0]), ("attention-bwd", got[1])}
    for (prec, S), want in PROP_DISPATCH:
        got = tuple(_run_propagator(d, prec, S, 256, 2, False)[0] for d in (0, 1))
        assert got == want, ((prec, S), got)
        hit |= {("propagator-fwd", got[0]), ("propagator-bwd", got[1])}
    every = {("attention-fwd", k) for k in (FLASH, MMA, SIMT)} | {("attention-bwd", k) for k in (LONG_MMA, LONG_FFMA, MMA, SIMT)} | \
        {("propagator-fwd", k) for k in (SMALL, MMA, GENERIC)} | {("propagator-bwd", k) for k in (SMALL, MMA, WIDE, GENERIC)}
    assert hit == every, sorted(every - hit)
