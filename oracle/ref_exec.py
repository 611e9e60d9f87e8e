"""ORACLE (test infrastructure only - never imported by the product path).

Executes the REFERENCE's own `models/Compression/MCM.py` (class MCM: `__init__` topology, `forward_encoder`,
`random_masking`, `get_ids_shuffle`, `forward` incl. the slice loop, `forward_decoder`, `unpatchify`,
`forward_loss`) verbatim from the reference checkout (oracle.REFERENCE_ROOT), with only the absent
third-party leaf classes supplied by oracle/ref_stubs.py (timm / compressai / pytorch_msssim restated from
their published definitions) and the pretrained-VGG feature loss replaced by zero (it needs a download).
This is the strongest pin of the in-repo oracle (oracle/ref_model.py): every line of MCM.py on the path runs as written.  Used by the
`-m "not gpu"` tests that skip without the checkout and by tests/golden/make_refexec_golden.py, whose
outputs (tests/golden/refexec_*) let every other machine compare against the reference.
"""
from __future__ import annotations

import contextlib
import sys
import types

import numpy as np
import torch

from . import REFERENCE_ROOT, SKIP_REASON, ref_stubs, reference_has

_STUBBED = ("compressai", "compressai.ans", "compressai.entropy_models", "compressai.layers", "compressai.models",
            "compressai.ops", "pytorch_msssim", "timm", "timm.models", "timm.models.vision_transformer",
            "models.Compression.loss.vgg")
_cached_cls = None


def reference_available() -> bool:
    return reference_has("models/Compression/MCM.py")


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    return m


def load_reference_mcm_class():
    """Import the reference's models/Compression/MCM.py as written and return its `MCM` class."""
    global _cached_cls
    if _cached_cls is not None:
        return _cached_cls
    if not reference_available():
        raise RuntimeError(SKIP_REASON)
    S = ref_stubs
    stubs = {
        "compressai": _mod("compressai"),
        "compressai.ans": _mod("compressai.ans", BufferedRansEncoder=S.BufferedRansEncoder, RansDecoder=S.RansDecoder),
        "compressai.entropy_models": _mod("compressai.entropy_models", EntropyBottleneck=S.EntropyBottleneck,
                                          GaussianConditional=S.GaussianConditional),
        "compressai.layers": _mod("compressai.layers", conv3x3=S.conv3x3, subpel_conv3x3=S.subpel_conv3x3),
        "compressai.models": _mod("compressai.models", CompressionModel=S.CompressionModel),
        "compressai.ops": _mod("compressai.ops", quantize_ste=S.quantize_ste),
        "pytorch_msssim": _mod("pytorch_msssim", SSIM=S.SSIM),
        "timm": _mod("timm"),
        "timm.models": _mod("timm.models"),
        "timm.models.vision_transformer": _mod("timm.models.vision_transformer", PatchEmbed=S.PatchEmbed, Block=S.Block),
        # loss/vgg.py:99 downloads VGG16 weights and moves them .cuda(): replaced by a zero feature loss
        "models.Compression.loss.vgg": _mod("models.Compression.loss.vgg",
                                            cal_features_loss=lambda preds, imgs: torch.zeros((), dtype=preds.dtype)),
    }
    saved = {k: sys.modules.get(k) for k in list(stubs) + ["models", "models.Compression", "models.Compression.MCM",
                                                            "models.Compression.common", "models.Compression.loss",
                                                            "models.Compression.common.pos_embed"]}
    had_float_ = hasattr(np, "float_")
    try:
        sys.modules.update(stubs)
        for k in ("models", "models.Compression", "models.Compression.MCM", "models.Compression.common",
                  "models.Compression.loss", "models.Compression.common.pos_embed"):
            sys.modules.pop(k, None)
        sys.path.insert(0, str(REFERENCE_ROOT))
        if not had_float_:
            np.float_ = np.float64                     # pos_embed.py:83 (alias removed in NumPy 2)
        import importlib
        mod = importlib.import_module("models.Compression.MCM")
        _cached_cls = mod.MCM
    finally:
        if str(REFERENCE_ROOT) in sys.path:
            sys.path.remove(str(REFERENCE_ROOT))
        for k, v in saved.items():
            if k in stubs:
                if v is None:
                    sys.modules.pop(k, None)
                else:
                    sys.modules[k] = v
    return _cached_cls


@contextlib.contextmanager
def _np_float_shim():
    had = hasattr(np, "float_")
    if not had:
        np.float_ = np.float64
    try:
        yield
    finally:
        if not had and hasattr(np, "float_"):
            del np.float_


def build_reference_model(cfg, state_dict, extra_state=None):
    """Reference `MCM(**ctor kwargs)` in eval mode with `state_dict` (reference names) loaded.  The synthetic
    checkpoint only carries the tensors of the compression forward path; `extra_state` may add decoder-side tensors
    (g_s, decoder_*, mask_token).  Returns (model, missing_keys, unexpected_keys)."""
    MCM = load_reference_mcm_class()
    with _np_float_shim():
        m = MCM(img_size=cfg.img_size, patch_size=cfg.patch_size, in_chans=cfg.in_chans,
                encoder_embed_dim=cfg.encoder_embed_dim, encoder_depth=cfg.encoder_depth,
                encoder_num_heads=cfg.encoder_num_heads, decoder_embed_dim=cfg.decoder_embed_dim,
                decoder_depth=cfg.decoder_depth, decoder_num_heads=cfg.decoder_num_heads, mlp_ratio=cfg.mlp_ratio,
                latent_depth=cfg.latent_depth, hyperprior_depth=cfg.hyperprior_depth, num_slices=cfg.num_slices,
                num_keep_patches=cfg.num_keep_patches)
    sd = dict(state_dict)
    if extra_state:
        sd.update(extra_state)
    res = torch.nn.Module.load_state_dict(m, sd, strict=False)
    m.eval()
    return m, list(res.missing_keys), list(res.unexpected_keys)


@torch.no_grad()
def reference_forward(model, imgs, total_scores):
    """`MCM.forward(imgs, total_scores)` of the reference, as written (MCM.py:714-803)."""
    return model(imgs, total_scores)
