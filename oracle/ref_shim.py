"""Import shim for the upstream TANTE reference (TEST INFRASTRUCTURE ONLY).

The reference is an upstream TANTE checkout that is not part of this repository;
point TANTE_REFERENCE_ROOT at it.  It cannot be imported as published without
`torchinfo`, `h5py`, `matplotlib`, `hydra`, `timm`, `neuralop` (SURVEY.md F9).
This module registers stub modules for the three that the hot-path files
import but never use, bypasses `models/__init__.py` (which
pulls in the baselines), and applies the *minimal repair* of the adaptive
(`deg=False`) branch of `TANTE.forward` (reference models/tante.py:147-153,
SURVEY.md F5 / §8(c)) as a monkey-patch -- the reference tree is never edited.

It is used only by `oracle/make_golden.py` (to generate tests/golden/*) and by
the tests that compare with the live reference (skipped when TANTE_REFERENCE_ROOT
is unset).  Nothing in the product path imports it.
"""
from __future__ import annotations

import importlib
import math
import os
import sys
import types

REF_ROOT = os.environ.get("TANTE_REFERENCE_ROOT", "")
SKIP_REASON = "upstream reference not found: set TANTE_REFERENCE_ROOT to an upstream TANTE checkout"


def reference_available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "models", "tante.py"))


def _stub(name: str, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


_loaded = None


def load_reference():
    """Return a namespace with the reference's TANTE, Attn_Backbone, enc/dec, metrics."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not reference_available():
        raise RuntimeError(SKIP_REASON)
    _stub("torchinfo", summary=lambda *a, **k: None)
    _stub("h5py")
    mpl = _stub("matplotlib")
    mpl.pyplot = _stub("matplotlib.pyplot")
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    # `models` as an empty namespace package so models/__init__.py is skipped
    if "models" not in sys.modules or not hasattr(sys.modules["models"], "__path__"):
        pkg = types.ModuleType("models")
        pkg.__path__ = [os.path.join(REF_ROOT, "models")]
        sys.modules["models"] = pkg
    tante = importlib.import_module("models.tante")
    backbone = importlib.import_module("models.attn_backbone")
    encdec = importlib.import_module("models.enc_dec_cnn")
    if "trainer" not in sys.modules or not hasattr(sys.modules["trainer"], "__path__"):
        tpkg = types.ModuleType("trainer")
        tpkg.__path__ = [os.path.join(REF_ROOT, "trainer")]
        sys.modules["trainer"] = tpkg
    metrics = importlib.import_module("trainer.metrics")
    dataset = importlib.import_module("data.dataset")

    _apply_deg_false_repair(tante)

    ns = types.SimpleNamespace(
        TANTE=tante.TANTE, tante=tante, Attn_Backbone=backbone.Attn_Backbone,
        backbone=backbone, encdec=encdec, metrics=metrics,
        TanteMetadata=dataset.TanteMetadata,
    )
    _loaded = ns
    return ns


def _apply_deg_false_repair(tante_mod):
    """Flatten the last-frame latent to (B, L, C) *before* interprator+modifier.

    Upstream (models/tante.py:147-153) feeds the 5-D tensor to the FiLM modifier
    and then applies a 3-D rearrange to the 5-D result, which raises EinopsError.
    The repaired order is the unique reading consistent with the in-code shape
    comment `# (B, L, C)` and the 3-D branch of `film.forward` (:222-224).
    Everything else in forward (:125-146, :156-176) is executed unchanged by
    re-stating only the loop body here.
    """
    import torch
    from einops import rearrange

    def forward(self, input, out_T=1):
        if input.shape[1] != self.T:
            input = input[:, -self.T:, ...]
        B, T, D, H, W = input.shape
        x = self.encoder(input)
        _, _, H_p, W_p, C = x.shape
        x = self.t_encode(x, self.t_seq)
        x = x + self.s_emb
        x = rearrange(x, 'b t h w c -> (b h w) t c')
        x = x + self.t_emb
        x = rearrange(x, '(b h w) t c -> b t h w c', b=B, h=H_p, w=W_p)
        derivatives, r_t = [], []
        for i in range(self.taylor_order):
            x = self.blocks[i](x)
            derivative = x[:, -1:, ...]
            if not self.deg:
                d = rearrange(derivative, 'b 1 h w c -> b (h w) c')
                rt = self.interprators[i](d, out_T)
                r_t.append(rt)
                d = self.modifiers[i](d, rt)
                derivative = rearrange(d, 'b (h w) c -> b 1 h w c', h=H_p, w=W_p)
            derivative = self.decoders[i](derivative)
            derivatives.append(derivative)
        outputs = []
        if not self.deg:
            r_t = torch.stack(r_t, dim=1)
            R_t = torch.mean(r_t, dim=1)
        output_length = self.output_length if self.deg else math.floor(R_t[0])
        for i in range(1, output_length + 1):
            output = 0
            for order in range(1, self.taylor_order + 1):
                output += derivatives[order - 1] * (i * self.frame_interval) ** order / math.factorial(order)
            outputs.append(output + input[:, -1:, ...])
        outputs = torch.cat(outputs, dim=1)
        if not self.deg:
            return outputs, R_t
        return outputs

    tante_mod.TANTE._unrepaired_forward = tante_mod.TANTE.forward
    tante_mod.TANTE.forward = forward


def make_metadata(n_fields: int, H: int, W: int):
    ns = load_reference()
    return ns.TanteMetadata(
        dataset_name="synthetic", n_spatial_dims=2, spatial_resolution=(H, W),
        field_names={0: [f"f{i}" for i in range(n_fields)]}, boundary_condition_types=["periodic"],
        n_files=0, n_trajectories_per_file=[], n_steps_per_trajectory=[], n_fields=n_fields,
    )
