"""`TANTE` -- drop-in for the reference `models.TANTE` (reference models/tante.py:37-176).

Same constructor signature, same `forward(input, out_T)` contract, same `state_dict` keys,
shapes and default initialisation stream (the parameter containers are created in the
reference's order with the same torch initialisers, so `torch.manual_seed(s); TANTE(...)`
yields the reference's weights).  All arithmetic runs in libtante_b200.so (hand-written
sm_100a CUDA) through the C ABI in include/tante_b200.h; PyTorch only owns the tensors.
There is no CPU path: calling the module on a CPU tensor raises.
"""
from __future__ import annotations

import ctypes
import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _abi

# reference models/enc_dec_cnn.py:39-46
Patch_map = {64: (4, 4, 4), 32: (4, 4, 2), 16: (4, 2, 2), 8: (2, 2, 2), 4: (2, 2, 1), 2: (2, 1, 1)}
# reference models/enc_dec_fno.py:39-46
Patch_map_fno = {64: (8, 8), 32: (8, 4), 16: (4, 4), 8: (4, 2), 4: (2, 2), 2: (2, 1)}


@dataclass
class TanteMetadata:
    """Same fields as the reference dataclass (data/dataset.py:43-63); only `n_fields` and
    `spatial_resolution` are read by the model (models/tante.py:64-66)."""
    dataset_name: str = "synthetic"
    n_spatial_dims: int = 2
    spatial_resolution: Tuple[int, ...] = (128, 384)
    field_names: Optional[Dict[int, List[str]]] = None
    boundary_condition_types: Optional[List[str]] = None
    n_files: int = 0
    n_trajectories_per_file: Optional[List[int]] = None
    n_steps_per_trajectory: Optional[List[int]] = None
    n_fields: int = 4

    @property
    def sample_shapes(self):
        return {
            "input_fields": [*self.spatial_resolution, self.n_fields],
            "output_fields": [*self.spatial_resolution, self.n_fields],
            "space_grid": [*self.spatial_resolution, self.n_spatial_dims],
        }


class _ParamsOnly(nn.Module):
    """Parameter container: keeps the reference's module tree (hence state_dict keys and the
    init RNG stream) but owns no arithmetic."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter container of tante_b200.TANTE: compute goes through libtante_b200.so")


class _PatchConv(_ParamsOnly):       # RealConv2d (enc_dec_cnn.py:49-94)
    def __init__(self, cin, cout, k):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, kernel_size=(k, k), stride=(k, k), padding=((k - 1) // 2, (k - 1) // 2))


class _PatchDeconv(_ParamsOnly):     # RealTransConv2d (enc_dec_cnn.py:113-160)
    def __init__(self, cin, cout, k):
        super().__init__()
        self.deconv = nn.ConvTranspose2d(cin, cout, kernel_size=(k, k), stride=(k, k),
                                         padding=((k - 1) // 2, (k - 1) // 2), output_padding=0)


class _EncCNN(_ParamsOnly):          # enc_CNN (enc_dec_cnn.py:187-215)
    def __init__(self, D, C, ks):
        super().__init__()
        self.enc_conv_1 = _PatchConv(D, C // 4, ks[0])
        self.enc_conv_2 = _PatchConv(C // 4, C // 2, ks[1])
        self.enc_conv_3 = _PatchConv(C // 2, C, ks[2])


class _DecCNN(_ParamsOnly):          # dec_CNN (enc_dec_cnn.py:232-261)
    def __init__(self, D, C, ks):
        super().__init__()
        self.dec_conv_1 = _PatchDeconv(C, C // 2, ks[2])
        self.dec_conv_2 = _PatchDeconv(C // 2, C // 4, ks[1])
        self.dec_conv_3 = _PatchDeconv(C // 4, D, ks[0])


class _Spectral(_ParamsOnly):        # SpectralLayer (enc_dec_fno.py:184-197)
    def __init__(self, cin, cout, m1, m2):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(cin, cout, m1, m2, dtype=torch.cfloat) * (1.0 / (cin * cout) ** 0.5))
        self.w0 = nn.Conv2d(cin, cout, kernel_size=1, bias=True)


class _EncFNO(_ParamsOnly):          # enc_FNO (enc_dec_fno.py:224-252)
    def __init__(self, D, C, ps, m1, m2):
        super().__init__()
        self.enc_spectral_1 = _Spectral(D, C // 8, m1, m2)
        self.enc_conv_1 = _PatchConv(C // 8, C // 4, ps[0])
        self.enc_spectral_2 = _Spectral(C // 4, C // 2, m1 // ps[0], m2 // ps[0])
        self.enc_conv_2 = _PatchConv(C // 2, C, ps[1])


class _DecFNO(_ParamsOnly):          # dec_FNO (enc_dec_fno.py:274-301)
    def __init__(self, D, C, ps, m1, m2):
        super().__init__()
        self.dec_conv_1 = _PatchDeconv(C, C // 2, ps[1])
        self.dec_spectral_1 = _Spectral(C // 2, C // 4, m1 // ps[0], m2 // ps[0])
        self.dec_conv_2 = _PatchDeconv(C // 4, C // 8, ps[0])
        self.dec_spectral_2 = _Spectral(C // 8, D, m1, m2)


class _Block(_ParamsOnly):           # TransformerBlock (attn_backbone.py:38-57)
    def __init__(self, C, n_head, mlp_ratio, dropout):
        super().__init__()
        self.ln1 = nn.LayerNorm(C)
        self.attn = nn.MultiheadAttention(C, n_head, batch_first=True, dropout=dropout, bias=True)
        self.ln2 = nn.LayerNorm(C)
        hidden = int(C * mlp_ratio)
        self.mlp = nn.Sequential(nn.Linear(C, hidden), nn.GELU(approximate="tanh"), nn.Linear(hidden, C))
        self.drop = nn.Dropout(dropout)


class _Backbone(_ParamsOnly):        # Attn_Backbone (attn_backbone.py:88-132)
    def __init__(self, T, Hp, Wp, C, axes, n_head, mlp_ratio, dropout, expanded_channel=128):
        super().__init__()
        if axes == "":
            raise ValueError("Invalid block: empty segment.")
        self.blocks = nn.ModuleList()
        self.vertical_propagator = nn.Sequential(nn.Linear(Hp, Hp), nn.GELU(), nn.Linear(Hp, Hp))
        self.horizontal_propagator = nn.Sequential(nn.Linear(Wp, Wp), nn.GELU(), nn.Linear(Wp, Wp))
        self.temporal_propagator = nn.Sequential(nn.Linear(T, T), nn.GELU(), nn.Linear(T, T))
        self.channel_blocks = nn.ModuleList()
        for axis in axes:
            width = C
            if axis == "C":       # channel attention: 1 -> expanded_channel lift, block of that width (attn_backbone.py:124-132)
                width = expanded_channel
                self.channel_blocks.append(nn.Sequential(nn.Linear(1, width // 4), nn.GELU(), nn.Linear(width // 4, width)))
            self.blocks.append(_Block(width, n_head, mlp_ratio, dropout))


class _Film(_ParamsOnly):            # film (tante.py:203-216)
    def __init__(self, C):
        super().__init__()
        self.condition_to_scale = nn.Sequential(nn.Linear(1, C // 2), nn.ReLU(), nn.Linear(C // 2, C))
        self.condition_to_shift = nn.Sequential(nn.Linear(1, C // 2), nn.ReLU(), nn.Linear(C // 2, C))


class _Interprator(_ParamsOnly):     # interprator (tante.py:178-189)
    def __init__(self, C):
        super().__init__()
        self.interprete = nn.Sequential(nn.Linear(C, C // 2), nn.ReLU(), nn.Linear(C // 2, C // 4), nn.ReLU(),
                                        nn.Linear(C // 4, 1))


def _sincos_1d(embed_dim, pos):       # tante.py:232-242
    omega = torch.arange(embed_dim // 2, dtype=torch.float32)
    omega /= embed_dim / 2.0
    omega = 1.0 / 10000 ** omega
    out = torch.einsum("m,d->md", pos.reshape(-1), omega)
    return torch.cat([torch.sin(out), torch.cos(out)], dim=1)


def _t_emb_init(C, T):                # tante.py:243-249
    return _sincos_1d(C, torch.arange(T, dtype=torch.float32)).unsqueeze(0)


def _s_emb_init(C, Hp, Wp):           # tante.py:251-276 ("w goes first" meshgrid + raw reshape)
    gw, gh = torch.meshgrid(torch.arange(Wp, dtype=torch.float32), torch.arange(Hp, dtype=torch.float32),
                            indexing="ij")
    grid = torch.stack([gh, gw], dim=0).reshape(2, 1, Hp, Wp)
    emb = torch.cat([_sincos_1d(C // 2, grid[0]), _sincos_1d(C // 2, grid[1])], dim=1)
    return emb.view(Hp, Wp, C).unsqueeze(0)


class _Engine:
    """One libtante_b200 handle = (config, precision, device) + bound parameters."""

    def __init__(self, model: "TANTE", precision: int, device: torch.device):
        self.lib = _abi.load()
        cfg = _abi.TanteConfig()
        cfg.in_T = model.T
        cfg.n_fields = model.n_channel
        cfg.H, cfg.W = model.shape
        cfg.taylor_order = model.taylor_order
        cfg.n_head = model.n_head
        cfg.embed_dim = model.C
        cfg.patch_scale = model.patch_scale
        cfg.deg = 1 if model.deg else 0
        cfg.output_length = int(model.output_length)
        cfg.frame_interval = float(model.frame_interval)
        cfg.precision = precision
        cfg.enc_dec_fno = 1 if model.enc_dec_type == "fno" else 0
        cfg.modes1, cfg.modes2 = int(model.modes1), int(model.modes2)
        cfg.mlp_hidden = int(model.C * model.mlp_ratio)
        for i, k in enumerate(model.patch_kernels[:3]):      # (cnn: three stages; fno: two)
            # enc_dec_cnn.py:64-66 / 130-132: Python's round() (half to even) -- computed here so that both sides agree
            cfg.stride[i] = max(1, int(round(k * (1.0 - model.overlap_ratio))))
        cfg.expanded_channel = int(model.expanded_channel)
        cfg.mlp_hidden_c = int(model.expanded_channel * model.mlp_ratio)
        for k, seg in enumerate(model.blocks_axes):
            if len(seg) > _abi.TANTE_MAX_LAYERS:
                raise ValueError("too many layers in one attn_axes segment")
            cfg.n_layers[k] = len(seg)
            cfg.axes[k].value = seg.encode()
        self.handle = ctypes.c_void_p()
        self.device = device
        _abi.check(self.lib.tante_create(ctypes.byref(cfg), device.index or 0, ctypes.byref(self.handle)))
        self.names = [self.lib.tante_param_name(self.handle, i).decode()
                      for i in range(self.lib.tante_param_count(self.handle))]
        self.bound_sig = None
        self.max_batch = 0
        self.max_roll = 0
        # training: tape slots (one per live autograd node) and the flat gradient layout
        self.grad_numel = int(self.lib.tante_grad_numel(self.handle))
        self.grad_offsets = [int(self.lib.tante_param_grad_offset(self.handle, i)) for i in range(len(self.names))]
        self.n_slots = 0
        self.free_slots: List[int] = []

    def close(self):
        if self.handle:
            self.lib.tante_destroy(self.handle)
            self.handle = ctypes.c_void_p()

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    def _signature(self, model: "TANTE"):
        params = dict(model.named_parameters())
        def version(p):
            try:
                return p._version
            except RuntimeError:      # inference tensors carry no version counter (immutable outside inference mode)
                return -1
        return tuple((n, params[n].data_ptr(), version(params[n])) for n in self.names)

    def mark_synced(self, model: "TANTE"):
        """The packed weights were refreshed by the library itself (tante_optimizer_step + tante_pack_params)."""
        self.bound_sig = self._signature(model)

    def sync_params(self, model: "TANTE", stream: int):
        """(Re)bind + repack when any parameter storage or version changed (optimizer step,
        load_state_dict, .to())."""
        params = dict(model.named_parameters())
        sig = self._signature(model)
        if sig == self.bound_sig:
            return
        for n in self.names:
            p = params[n]
            ok_dtype = p.dtype == torch.float32 or p.dtype == torch.complex64     # SpectralLayer.weight is cfloat: bound as float pairs
            if p.device != self.device or not ok_dtype or not p.is_contiguous():
                raise RuntimeError(f"parameter {n} must be a contiguous float32 (or complex64) tensor on {self.device}")
            numel = p.numel() * (2 if p.dtype == torch.complex64 else 1)
            _abi.check(self.lib.tante_bind_param(self.handle, n.encode(), p.data_ptr(), None, numel))
        _abi.check(self.lib.tante_pack_params(self.handle, stream))
        self.bound_sig = sig

    def reserve(self, B: int, n_roll: int = 0):
        if B > self.max_batch or n_roll > self.max_roll:
            self.max_batch = max(B, self.max_batch)
            self.max_roll = max(n_roll, self.max_roll)
            _abi.check(self.lib.tante_reserve(self.handle, self.max_batch, self.max_roll, self.n_slots))

    def acquire_slot(self) -> int:
        """Tape slot for one model call in grad mode; released by its backward (or when the autograd node dies).
        The pool grows with the number of live model calls (R_Trainer's per-sample BPTT keeps batch_size x n_steps
        tapes alive until loss.backward(), r_trainer.py:118-133); the only limit is device memory."""
        if not self.free_slots:
            self.n_slots += 1
            try:
                _abi.check(self.lib.tante_reserve(self.handle, max(self.max_batch, 1), self.max_roll, self.n_slots))
            except _abi.TanteError as e:
                self.n_slots -= 1
                raise RuntimeError(
                    f"tante_b200: cannot grow the activation-tape pool beyond {self.n_slots} live model calls ({e.msg}); "
                    "every model call made in grad mode keeps its tape until its backward runs -- call loss.backward() "
                    "(or run evaluation under torch.no_grad()/inference_mode(), r_trainer.py:181)") from e
            self.max_batch = max(self.max_batch, 1)
            self.free_slots.append(self.n_slots - 1)
        return self.free_slots.pop()

    def release_slot(self, slot: int):
        if slot not in self.free_slots:
            self.free_slots.append(slot)


class _SlotGuard:
    """Returns a tape slot to its engine when the autograd node that owns it is freed without a backward."""

    def __init__(self, eng: _Engine, slot: int):
        self.eng, self.slot, self.released = eng, slot, False

    def release(self):
        if not self.released:
            self.released = True
            self.eng.release_slot(self.slot)

    def __del__(self):  # pragma: no cover
        try:
            self.release()
        except Exception:
            pass


class _TanteStep(torch.autograd.Function):
    """One differentiable model call: tante_train_forward / tante_backward on a tape slot.  The parameters are
    passed as inputs so that autograd routes their gradients into `.grad` exactly as for the reference module
    (accumulation over the chained BPTT rollout of r_trainer.py:122-126 included)."""

    @staticmethod
    def forward(ctx, model, x, out_T, n_cap, *params):
        eng = model._engine(x.device)
        B = x.shape[0]
        eng.reserve(B)
        slot = eng.acquire_slot()
        frames = torch.empty((B, n_cap, model.n_channel, *model.shape), device=x.device, dtype=torch.float32)
        R_t = torch.zeros((B,), device=x.device, dtype=torch.float32)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        n_host = ctypes.c_int32(n_cap)
        try:
            _abi.check(eng.lib.tante_train_forward(eng.handle, slot, x.data_ptr(), B, float(out_T), n_cap,
                                                   frames.data_ptr(), R_t.data_ptr(),
                                                   None if model.deg else ctypes.byref(n_host), stream))
        except Exception:
            eng.release_slot(slot)
            raise
        n = n_host.value
        ctx.eng, ctx.slot, ctx.n, ctx.model = eng, slot, n, model
        ctx.guard = _SlotGuard(eng, slot)
        ctx.save_for_backward(x)
        out = frames if n == n_cap else frames[:, :n].contiguous()
        if model.deg:
            ctx.mark_non_differentiable(R_t)
        return out, R_t

    @staticmethod
    def backward(ctx, g_frames, g_rt):
        (x,) = ctx.saved_tensors
        eng, model = ctx.eng, ctx.model
        dev = x.device
        g_frames = g_frames.to(torch.float32).contiguous()
        g_rt_ptr = None
        if not model.deg and g_rt is not None:
            g_rt = g_rt.to(torch.float32).contiguous()
            g_rt_ptr = g_rt.data_ptr()
        flat = torch.empty((eng.grad_numel,), device=dev, dtype=torch.float32)
        g_in = torch.empty_like(x) if ctx.needs_input_grad[1] else None
        stream = torch.cuda.current_stream(dev).cuda_stream
        _abi.check(eng.lib.tante_backward(eng.handle, ctx.slot, x.data_ptr(), g_frames.data_ptr(), int(g_frames.shape[1]),
                                          g_rt_ptr, None if g_in is None else g_in.data_ptr(), flat.data_ptr(), stream))
        ctx.guard.release()
        # Fast path: every `p.grad` already is a view into ONE flat buffer laid out like the library's gradient
        # (tante_b200.trainer.GradBucket): accumulate with a single add instead of one AccumulateGrad launch per
        # parameter and model call (142 x 4 tiny kernels per BPTT step at tante.yaml).
        if all(ctx.needs_input_grad[4:]):
            acc = model._flat_grad_view(eng)
            if acc is not None:
                acc.add_(flat)
                return (None, g_in, None, None, *([None] * len(eng.names)))
        return (None, g_in, None, None, *ctx.model._grad_views(eng, flat))


class _TanteBPTT(torch.autograd.Function):
    """The chained BPTT rollout of both training drivers as ONE autograd node: the fixed-step model (trainer/trainer.py:144-159:
    `window = cat(window[:, 1:], y)`) and the per-sample adaptive loops of R_Trainer (r_trainer.py:117-133: each sample its own
    while-loop of `y, rt = model(window_b, out_T)`, the window sliding by floor(R_t) frames over its own predictions), NOT
    detached in either.  Every call is one batched tante_train_forward_hist: the library keeps a device cursor per sample
    (frames emitted so far), reads each sample's window at its cursor and writes its frames behind it, so no window is ever
    concatenated; a sample that has its n_steps frames emits nothing.  The backward walks the calls in reverse
    (tante_backward_hist), ACCUMULATING each call's window gradient into the gradient of the earlier predictions in place --
    what autograd does with a cat / slice / add chain per call.  Returns pred for the fixed-step model, (pred, rts, ns, steps)
    for the adaptive one."""

    @staticmethod
    def forward(ctx, model, x, n_steps, out_T, *params):
        eng = model._engine(x.device)
        B = x.shape[0]
        D, (H, W) = model.n_channel, model.shape
        DHW = D * H * W
        # the fixed-step model emits output_length frames per call and sample, and has no R_t
        n_cap = int(model.output_length) if model.deg else max(1, int(math.floor(out_T + 0.001)))
        n_hist = n_steps + n_cap - 1          # an overshooting last call writes past n_steps, into this slack
        eng.reserve(B)
        dev = x.device
        pred = torch.empty((B, n_hist, D, H, W), device=dev, dtype=torch.float32)
        cursor = torch.zeros((B,), device=dev, dtype=torch.int32)
        steps = torch.zeros((B,), device=dev, dtype=torch.int32)
        rts = None if model.deg else torch.zeros((n_steps, B), device=dev, dtype=torch.float32)
        ns = torch.zeros((n_steps, B), device=dev, dtype=torch.int32)
        # one frame per call (the fixed-step model, R_Trainer's out_T = 1.5): every sample makes exactly n_steps calls, no need
        # to ask the device
        n_active = torch.zeros((1,), device=dev, dtype=torch.int32) if n_cap > 1 else None
        stream = torch.cuda.current_stream(dev).cuda_stream
        p_drop = float(model.dropout) if model.training else 0.0
        slots = []
        try:
            for k in range(n_steps):
                slot = eng.acquire_slot()
                slots.append(slot)
                seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if p_drop > 0 else 0
                _abi.check(eng.lib.tante_set_dropout(eng.handle, p_drop, seed))
                _abi.check(eng.lib.tante_train_forward_hist(
                    eng.handle, slot, x.data_ptr(), pred.data_ptr(), n_hist * DHW, cursor.data_ptr(), B, float(out_T), n_cap,
                    n_steps, None if rts is None else rts[k].data_ptr(), ns[k].data_ptr(), steps.data_ptr(),
                    None if n_active is None else n_active.data_ptr(), stream))
                if n_active is not None and int(n_active.item()) == 0:
                    break
        except Exception:
            for sl in slots:
                eng.release_slot(sl)
            raise
        n_calls = len(slots)
        ctx.eng, ctx.model, ctx.slots, ctx.n_steps, ctx.n_hist = eng, model, slots, n_steps, n_hist
        ctx.guards = [_SlotGuard(eng, sl) for sl in slots]
        ctx.x_shape = tuple(x.shape)
        out = pred if n_hist == n_steps else pred[:, :n_steps].contiguous()
        if model.deg:
            return out
        ns = ns[:n_calls].clone()
        ctx.save_for_backward(ns)
        ctx.mark_non_differentiable(ns, steps)
        return out, rts[:n_calls].clone(), ns, steps

    @staticmethod
    def backward(ctx, g_pred, g_rts=None, *_):
        eng, model, n_steps, n_hist = ctx.eng, ctx.model, ctx.n_steps, ctx.n_hist
        B, T, D, H, W = ctx.x_shape
        DHW = D * H * W
        dev = eng.device
        # gradient of the whole prediction buffer: accumulated in place below (never autograd's own tensor); the slack past
        # n_steps stays zero
        g_acc = torch.empty((B, n_hist, D, H, W), device=dev, dtype=torch.float32)
        g_acc[:, :n_steps] = 0.0 if g_pred is None else g_pred
        g_acc[:, n_steps:] = 0.0
        g_r = None
        if g_rts is not None:      # R_t of a call a sample did not take part in is unused
            (ns,) = ctx.saved_tensors
            g_r = torch.where(ns > 0, g_rts.to(torch.float32), 0.0).contiguous()
        g_x = torch.zeros(ctx.x_shape, device=dev, dtype=torch.float32) if ctx.needs_input_grad[1] else None
        acc = model._flat_grad_view(eng) if all(ctx.needs_input_grad[4:]) else None
        flat_sum = None
        stream = torch.cuda.current_stream(dev).cuda_stream
        for k in range(len(ctx.slots) - 1, -1, -1):
            flat = torch.empty((eng.grad_numel,), device=dev, dtype=torch.float32)
            _abi.check(eng.lib.tante_backward_hist(eng.handle, ctx.slots[k], g_acc.data_ptr(), n_hist * DHW,
                                                   None if g_r is None else g_r[k].data_ptr(),
                                                   None if g_x is None else g_x.data_ptr(), flat.data_ptr(), stream))
            ctx.guards[k].release()
            if acc is not None:
                acc.add_(flat)
            else:
                flat_sum = flat if flat_sum is None else flat_sum.add_(flat)
        if acc is not None:
            return (None, g_x, None, None, *([None] * len(eng.names)))
        return (None, g_x, None, None, *model._grad_views(eng, flat_sum))


import weakref

_LIVE_MODELS: "weakref.WeakSet" = weakref.WeakSet()


def live_models():
    """The TANTE modules alive in this process (FusedAdamW finds the module its parameters belong to)."""
    return list(_LIVE_MODELS)


class TANTE(nn.Module):
    """B200-native TANTE.  Constructor mirrors reference models/tante.py:38-60."""

    def __init__(
        self,
        in_T,
        dset_metadata=None,
        taylor_order: int = 1,
        frame_interval: float = 1.0,
        output_length=1,
        attn_axes: str = "THWTHWTHW",
        expanded_channel: int = 128,
        n_head: int = 8,
        mlp_ratio: float = 1.0,
        dropout: float = 0.0,
        enc_dec_type: str = "cnn",
        embed_dim: int = 256,
        modes1: int = 32,
        modes2: int = 32,
        patch_scale: int = 32,
        overlap_ratio: float = 0.0,
        deg: bool = True,
        precision: str = "fp32",
    ):
        super().__init__()
        self.n_channel = dset_metadata.n_fields if dset_metadata else 4
        self.T = in_T
        self.shape = tuple(dset_metadata.spatial_resolution) if dset_metadata else (128, 384)
        self.patch_scale = patch_scale
        self.H_p = self.shape[0] // patch_scale
        self.W_p = self.shape[1] // patch_scale
        self.C = embed_dim
        self.n_head = n_head
        self.taylor_order = taylor_order
        self.frame_interval = frame_interval
        self.output_length = output_length
        self.deg = deg
        self.dropout = dropout
        self.precision = precision

        # validation identical to tante.py:75-83 (including the unreachable 'X,' entry)
        self.attn_axes = attn_axes.replace(" ", "")
        if set(self.attn_axes) - {'T', 'H', 'W', 'L', 'A', 'C', 'X,', 'Y', '-'}:
            raise ValueError("There are invalid letters")
        self.blocks_axes = [p.strip() for p in self.attn_axes.split("-")]
        if len(self.blocks_axes) != taylor_order:
            raise ValueError(
                f"Block allocation doesn't match expansion order: expected {taylor_order} parts, "
                f"got {len(self.blocks_axes)} (input='{self.attn_axes}').")
        if enc_dec_type not in ("cnn", "fno"):
            raise ValueError(f"unknown enc_dec_type {enc_dec_type!r}")
        self.enc_dec_type, self.modes1, self.modes2 = enc_dec_type, modes1, modes2
        if not 0.0 <= overlap_ratio < 1.0:
            raise AssertionError("overlap_ratio must be in [0, 1).")      # enc_dec_cnn.py:63
        self.overlap_ratio = float(overlap_ratio)
        hidden = int(embed_dim * float(mlp_ratio))
        if hidden < 64 or hidden > 1024 or hidden % 64:
            raise NotImplementedError("int(embed_dim * mlp_ratio) must be a multiple of 64 in 64..1024 (mlp_ratio 0.25 .. 4 at embed_dim 256)")
        self.mlp_ratio = float(mlp_ratio)
        ks = Patch_map[patch_scale]   # KeyError for unknown patch scales, as in enc_dec_cnn.py:199
        self.patch_kernels = ks
        if enc_dec_type == "fno":
            ps = Patch_map_fno[patch_scale]
            self.patch_kernels = ps
            H1, W1 = self.shape[0] // ps[0], self.shape[1] // ps[0]
            if (min(modes1, modes2) < ps[0] or 2 * modes1 > self.shape[0] or modes2 > self.shape[1] // 2
                    or 2 * (modes1 // ps[0]) > H1 or modes2 // ps[0] > W1 // 2):
                raise NotImplementedError("enc_dec_type='fno': the kept modes must fit the grid at both resolutions "
                                          "(ps[0] <= modes, 2*modes1 <= H, modes2 <= W/2)")
        # what the CUDA library does not cover is refused HERE, not at the first forward
        self.expanded_channel = int(expanded_channel)
        if "C" in self.attn_axes:      # channel attention (attn_backbone.py:124-130,184-189)
            E = self.expanded_channel
            hc = int(E * float(mlp_ratio))
            if E % 64 or not 64 <= E <= 256 or n_head <= 0 or E % n_head or E // n_head not in (16, 32, 64):
                raise NotImplementedError("attention axis 'C': expanded_channel must be a multiple of 64 in 64..256 with "
                                          "expanded_channel / n_head in (16, 32, 64)")
            if hc < 64 or hc > 1024 or hc % 64:
                raise NotImplementedError("attention axis 'C': int(expanded_channel * mlp_ratio) must be a multiple of 64 in 64..1024")
        if embed_dim not in (256, 512):
            raise NotImplementedError("embed_dim must be 256 (configs/tante.yaml:31; the fused block kernels) or 512 (plain GEMM path): "
                                      "C/4 and the interprator widths must stay multiples of 64")
        if n_head <= 0 or embed_dim % n_head or embed_dim // n_head not in (16, 32, 64):
            raise NotImplementedError("head_dim = embed_dim / n_head must be 16, 32 or 64")
        if not 1 <= self.n_channel <= 16:
            raise NotImplementedError("1..16 fields are supported")
        if self.shape[0] % patch_scale or self.shape[1] % patch_scale:
            raise ValueError("the spatial resolution must be divisible by patch_scale")
        if self.H_p > 96 or self.W_p > 96 or in_T > 64:
            raise NotImplementedError("latent axes longer than 96 (H_p, W_p) / 64 (in_T) are not supported")
        if not 1 <= taylor_order <= 4:
            raise NotImplementedError("taylor_order must be in 1..4")

        # parameter containers, created in the reference's order (tante.py:85-123)
        self.decoders = nn.ModuleList()
        if enc_dec_type == "fno":             # enc_dec_fno.py:224-301
            self.encoder = _EncFNO(self.n_channel, embed_dim, self.patch_kernels, modes1, modes2)
            for _ in range(taylor_order):
                self.decoders.append(_DecFNO(self.n_channel, embed_dim, self.patch_kernels, modes1, modes2))
        else:
            self.encoder = _EncCNN(self.n_channel, embed_dim, ks)
            for _ in range(taylor_order):
                self.decoders.append(_DecCNN(self.n_channel, embed_dim, ks))
        self.blocks = nn.ModuleList()
        for seg in self.blocks_axes:
            self.blocks.append(_Backbone(self.T, self.H_p, self.W_p, self.C, seg, n_head, mlp_ratio, dropout, expanded_channel))
        self.t_emb = nn.Parameter(_t_emb_init(self.C, self.T))
        self.s_emb = nn.Parameter(_s_emb_init(self.C, self.H_p, self.W_p))
        self.t_encode = _Film(self.C)
        if not self.deg:
            self.interprators = nn.ModuleList([_Interprator(self.C) for _ in range(taylor_order)])
            self.modifiers = nn.ModuleList([_Film(self.C) for _ in range(taylor_order)])
        self._engines: Dict[Tuple[int, str], _Engine] = {}
        _LIVE_MODELS.add(self)

    def __getstate__(self):
        st = self.__dict__.copy()
        st["_engines"] = {}          # native handles are per-process, rebuilt lazily
        return st

    # ------------------------------------------------------------------ engine plumbing
    def _precision_code(self) -> int:
        if torch.is_autocast_enabled() and torch.get_autocast_dtype("cuda") == torch.bfloat16:
            return _abi.PREC_BF16
        return _abi.PREC_BF16 if self.precision == "bf16" else _abi.PREC_FP32

    def _engine(self, device: torch.device) -> _Engine:
        if device.type != "cuda":
            raise RuntimeError("tante_b200.TANTE runs only on CUDA (sm_100a) tensors; there is no CPU path")
        prec = self._precision_code()
        key = (prec, str(device))
        eng = self._engines.get(key)
        if eng is None:
            eng = _Engine(self, prec, device)
            self._engines[key] = eng
        eng.sync_params(self, torch.cuda.current_stream(device).cuda_stream)
        return eng

    def grad_layout(self, device):
        """(parameter names, element offsets, total elements) of the library's flat gradient on `device`."""
        eng = self._engine(torch.device(device))
        return list(eng.names), list(eng.grad_offsets), int(eng.grad_numel)

    def _flat_grad_view(self, eng: _Engine):
        """The flat fp32 tensor all `p.grad` are views of, if they are laid out like the library's gradient
        (same storage, element offset = base + grad_offsets[i]); else None."""
        params = dict(self.named_parameters())
        g0 = params[eng.names[0]].grad
        if g0 is None or g0.dtype != torch.float32 or not g0.is_contiguous():
            return None
        base = g0.data_ptr() - 4 * eng.grad_offsets[0]
        for n, off in zip(eng.names, eng.grad_offsets):
            g = params[n].grad
            if (g is None or g.dtype not in (torch.float32, torch.complex64) or not g.is_contiguous()
                    or g.data_ptr() != base + 4 * off):
                return None
        st = g0.untyped_storage()
        first = g0.storage_offset() - eng.grad_offsets[0]
        if first < 0 or (first + eng.grad_numel) * 4 > st.nbytes():
            return None
        return torch.as_strided(g0, (eng.grad_numel,), (1,), first)

    def _grad_views(self, eng: _Engine, flat: torch.Tensor):
        """Per-parameter views of the library's flat fp32 gradient (tante_param order); complex parameters (SpectralLayer.weight)
        are stored as (re, im) float pairs."""
        params = dict(self.named_parameters())
        out = []
        for n, off in zip(eng.names, eng.grad_offsets):
            p = params[n]
            if p.dtype == torch.complex64:
                out.append(torch.view_as_complex(flat[off:off + 2 * p.numel()].view(*p.shape, 2)))
            else:
                out.append(flat[off:off + p.numel()].view(p.shape))
        return out

    def _param_shapes(self, eng: _Engine):
        params = dict(self.named_parameters())
        return [(n, tuple(params[n].shape)) for n in eng.names]

    def _needs_grad(self, input) -> bool:
        return torch.is_grad_enabled() and (input.requires_grad or any(p.requires_grad for p in self.parameters()))

    def _forward_train(self, x, out_T, n_cap):
        eng = self._engine(x.device)
        # nn.Dropout / MultiheadAttention(dropout=p) act in train() mode only (attn_backbone.py:47-57,81-83).  Every model
        # call draws a fresh 64-bit key for the counter-based mask generator from torch's CPU generator (reproducible
        # under torch.manual_seed); the tape keeps it so that the backward regenerates the same masks.
        p = float(self.dropout) if self.training else 0.0
        seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if p > 0 else 0
        _abi.check(eng.lib.tante_set_dropout(eng.handle, p, seed))
        params = dict(self.named_parameters())
        return _TanteStep.apply(self, x, float(out_T), int(n_cap), *[params[n] for n in eng.names])

    def _prep_input(self, input: torch.Tensor) -> torch.Tensor:
        if input.dim() != 5:
            raise ValueError("input must be (B, T, D, H, W)")
        if input.shape[1] != self.T:
            input = input[:, -self.T:, ...]           # tante.py:127-128
        B, T, D, H, W = input.shape
        if T != self.T or D != self.n_channel or (H, W) != tuple(self.shape):
            raise ValueError(f"input shape {tuple(input.shape)} does not match the model "
                             f"(T={self.T}, D={self.n_channel}, HxW={self.shape})")
        return input.to(torch.float32).contiguous()

    # ------------------------------------------------------------------ reference API
    def forward(self, input, out_T=1):
        """(B,>=T,D,H,W) -> frames (B,n,D,H,W) [and R_t (B,) when deg=False] (tante.py:125-176)."""
        x = self._prep_input(input)
        if not self.deg and out_T < 1:
            raise ValueError("out_T must be >= 1")
        n_cap = int(self.output_length) if self.deg else max(1, int(math.floor(out_T + 0.001)))
        if self._needs_grad(x) or (self.training and self.dropout > 0):
            # (train() mode with dropout under no_grad still drops, like the reference module: same taped path, the tape
            #  slot is returned as soon as the unused autograd context dies)
            frames, R_t = self._forward_train(x, out_T, n_cap)
            return frames if self.deg else (frames, R_t)
        eng = self._engine(x.device)
        B = x.shape[0]
        eng.reserve(B)
        frames = torch.empty((B, n_cap, self.n_channel, *self.shape), device=x.device, dtype=torch.float32)
        R_t = None if self.deg else torch.empty((B,), device=x.device, dtype=torch.float32)
        n_host = ctypes.c_int32(0)
        stream = torch.cuda.current_stream(x.device).cuda_stream
        _abi.check(eng.lib.tante_forward(eng.handle, x.data_ptr(), B, float(out_T), n_cap, 0, frames.data_ptr(),
                                         None if R_t is None else R_t.data_ptr(), None, ctypes.byref(n_host),
                                         stream))
        n = n_host.value
        out = frames if n == n_cap else frames[:, :n].contiguous()
        if self.deg:
            return out
        return out, R_t

    @property
    def bptt_windows_ok(self) -> bool:
        """The windowed BPTT entry points (per-sample cursors) exist for the nested-order patch stages (patch_scale <= 8, cnn) without axis-C layers."""
        return self.patch_scale <= 8 and self.enc_dec_type == "cnn" and "C" not in self.attn_axes and self.overlap_ratio == 0.0

    def rollout_train(self, window, n_steps: int, out_T: float = 1.5):
        """BPTT rollout of the training drivers as one autograd node, no window concatenation.

        Fixed-step model (`deg=True`, `output_length=1`; trainer/trainer.py:144-159): (B, T, D, H, W) -> predictions
        (B, n_steps, D, H, W), the arithmetic of n_steps chained `forward` calls on `cat(window[:, 1:], y)`.  out_T is unused.

        Adaptive model (`deg=False`; r_trainer.py:117-133): what the per-sample B=1 loops `y, rt = model(window_b, out_T)`
        compute, each sample with its own step sequence -> pred (B, n_steps, D, H, W), rts (n_calls, B) R_t of every call,
        ns (n_calls, B) frames each call emitted per sample (0 once the sample had its n_steps frames; its rts entry is then
        unused), steps (B,) calls per sample.  With floor(out_T + 0.001) == 1 (R_Trainer's out_T = 1.5) every sample makes
        n_steps calls and nothing is synchronised; otherwise one 4-byte count is read after each call."""
        if self.deg and int(self.output_length) != 1:
            raise ValueError("rollout_train covers the fixed-step model with output_length=1 and the adaptive model")
        if not self.deg:
            if not self.bptt_windows_ok:
                raise ValueError("rollout_train for deg=False covers patch_scale <= 8 with the cnn encoder, no overlap and no axis C")
            if out_T < 1:
                raise ValueError("out_T must be >= 1")
        x = self._prep_input(window)
        eng = self._engine(x.device)
        params = dict(self.named_parameters())
        return _TanteBPTT.apply(self, x, int(n_steps), float(out_T), *[params[n] for n in eng.names])

    @torch.no_grad()
    def rollout(self, window, n_steps_rollout: int, out_T=None, per_sample: bool = False, sync: bool = True):
        """Device-resident adaptive rollout (R_Evaler.rollout_model, r_evaler.py:87-105).

        window (B,>=T,D,H,W) channels-first -> y (B,n_roll,H,W,D) channels-last, Rts (max_steps,B),
        ns (max_steps,B) frames per model call, steps (B,) model calls per sample.  `per_sample=False`
        reproduces the reference (sample 0's R_t governs the batch); `per_sample=True` gives each
        trajectory its own step sequence (the reference's B=1 behaviour, applied per trajectory)."""
        x = self._prep_input(window)
        eng = self._engine(x.device)
        B = x.shape[0]
        out_T = float(n_steps_rollout if out_T is None else out_T)
        eng.reserve(B, n_steps_rollout)
        dev = x.device
        y = torch.empty((B, n_steps_rollout, *self.shape, self.n_channel), device=dev, dtype=torch.float32)
        rts = torch.zeros((n_steps_rollout, B), device=dev, dtype=torch.float32)
        ns = torch.zeros((n_steps_rollout, B), device=dev, dtype=torch.int32)
        steps = torch.zeros((B,), device=dev, dtype=torch.int32)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _abi.check(eng.lib.tante_rollout(eng.handle, x.data_ptr(), B, int(n_steps_rollout), out_T,
                                         1 if per_sample else 0, y.data_ptr(), rts.data_ptr(), ns.data_ptr(),
                                         steps.data_ptr(), 1 if sync else 0, stream))
        return y, rts, ns, steps

    # ------------------------------------------------------------------ test / profiling hooks
    def debug_stage(self, stage: str, numel: int) -> torch.Tensor:
        dev = next(self.parameters()).device
        eng = self._engine(dev)
        out = torch.empty((max(numel, 1),), device=dev, dtype=torch.float32)
        got = ctypes.c_int64(0)
        _abi.check(eng.lib.tante_debug_stage(eng.handle, stage.encode(), out.data_ptr(), out.numel(), ctypes.byref(got),
                                             torch.cuda.current_stream(dev).cuda_stream))
        return out[:got.value]

    @torch.no_grad()
    def bench_head(self, window: torch.Tensor, n_frames: int, iters: int = 20) -> float:
        """Average device time (ms) of one stand-alone fused-head launch emitting `n_frames` frames per sample."""
        x = self._prep_input(window)
        eng = self._engine(x.device)
        B = x.shape[0]
        eng.reserve(B)
        frames = torch.empty((B, n_frames, self.n_channel, *self.shape), device=x.device, dtype=torch.float32)
        ms = ctypes.c_float(0)
        _abi.check(eng.lib.tante_bench_head(eng.handle, x.data_ptr(), frames.data_ptr(), B, int(n_frames), int(iters),
                                            ctypes.byref(ms), torch.cuda.current_stream(x.device).cuda_stream))
        return float(ms.value)

    def profile_gemms(self, enable: bool):
        for e in self._engines.values():
            _abi.check(e.lib.tante_profile(e.handle, 1 if enable else 0))

    def profile_read_classes(self):
        """{class: (ms, flops, bytes, launches)} of the bracketed GEMM launches since profile_gemms(True); call before
        profile_read().  0 = plain-epilogue GEMMs, 1 = fp32 residual/LayerNorm/embedding epilogues, 2 = weight gradients,
        3 = fused block tail (out-proj + LN2 + MLP + LN1' in one kernel)."""
        out = {}
        for cls in (0, 1, 2, 3, 4):
            ms = fl = by = 0.0
            n = 0
            for e in self._engines.values():
                a, b, c, d = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_double(0), ctypes.c_int64(0)
                _abi.check(e.lib.tante_profile_read_class(e.handle, cls, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c),
                                                          ctypes.byref(d)))
                ms += a.value; fl += b.value; by += c.value; n += d.value
            out[cls] = (ms, fl, by, n)
        return out

    def profile_read(self):
        """(gemm_ms, gemm_flops, gemm_launches) accumulated since profile_gemms(True)."""
        ms = fl = 0.0
        n = 0
        for e in self._engines.values():
            a, b, c = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_int64(0)
            _abi.check(e.lib.tante_profile_read(e.handle, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
            ms += a.value
            fl += b.value
            n += c.value
        return ms, fl, n

    def launch_count(self) -> int:
        return sum(int(e.lib.tante_launch_count(e.handle)) for e in self._engines.values())
