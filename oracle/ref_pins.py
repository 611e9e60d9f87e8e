"""ORACLE (test infrastructure only - never imported by the product path).

Pins of the model-half oracle against the two reference files on the compression forward path that have no
third-party dependency beyond numpy / torch; they are executed where they lie, unmodified:

  models/Compression/loss/rd_loss.py:7-28      RateDistortionLoss (bpp_loss, rd_loss.py:19-20)
  models/Compression/common/pos_embed.py:23-94  get_2d_sincos_pos_embed (MCM.py:457-464)

`pos_embed.py:83` uses `np.float_`, removed in NumPy 2: the module is executed with a numpy
namespace proxy that maps `float_` to `float64` (what `np.float_` was); the reference source is not
edited.  Everything here needs the reference checkout (oracle.REFERENCE_ROOT), so it is only used by
`-m "not gpu"` tests that skip without it and by tests/golden/make_refexec_golden.py, which freezes the
outputs into tests/golden/refexec_small.pt for the checks that run everywhere.
"""
from __future__ import annotations

import importlib.util
import types

import numpy as np
import torch

from . import REFERENCE_ROOT, reference_has

RD_LOSS = REFERENCE_ROOT / "models/Compression/loss/rd_loss.py"
POS_EMBED = REFERENCE_ROOT / "models/Compression/common/pos_embed.py"
ENGINE = REFERENCE_ROOT / "utils/engine.py"


def reference_available() -> bool:
    return reference_has("models/Compression/loss/rd_loss.py", "models/Compression/common/pos_embed.py")


def load_rate_distortion_loss():
    """The reference's own `RateDistortionLoss` class (rd_loss.py:7-28), loaded by path."""
    spec = importlib.util.spec_from_file_location("_ref_rd_loss", str(RD_LOSS))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.RateDistortionLoss


class _NumpyCompat(types.ModuleType):
    """numpy with the removed NumPy-1 alias `float_` (== float64) restored, for pos_embed.py:83."""

    def __init__(self):
        super().__init__("numpy")

    def __getattr__(self, name):
        if name == "float_":
            return np.float64
        return getattr(np, name)


def load_get_2d_sincos_pos_embed():
    """The reference's own `get_2d_sincos_pos_embed(embed_dim, grid_size, cls_token)` (pos_embed.py:23-94)."""
    src = POS_EMBED.read_text()
    ns = {"__name__": "_ref_pos_embed"}
    code = compile(src, str(POS_EMBED), "exec")
    # the file does `import numpy as np` itself: run it, then rebind its `np` to the compat proxy
    exec(code, ns)
    ns["np"] = _NumpyCompat()
    return ns["get_2d_sincos_pos_embed"]


def reference_pos_embed_parameter(embed_dim: int, grid_size: int) -> torch.Tensor:
    """What MCM.initialize_weights copies into `encoder_pos_embed` (MCM.py:457-464): fp32 [1, 1+L, C]."""
    fn = load_get_2d_sincos_pos_embed()
    table = fn(embed_dim, grid_size, cls_token=True)
    return torch.from_numpy(table).float().unsqueeze(0)


def reference_bpp_loss(y_lik: torch.Tensor, z_lik: torch.Tensor, img_size: int) -> torch.Tensor:
    """bpp_loss of the reference's RateDistortionLoss on a likelihoods dict shaped like MCM.forward's
    (MCM.py:801); the distortion terms are irrelevant to it and passed as zeros."""
    crit = load_rate_distortion_loss()(lmbda=1e-2)
    n = y_lik.shape[0]
    zero = torch.zeros(())
    output = {"likelihoods": {"y": y_lik, "z": z_lik}, "loss": (zero, zero, zero)}
    target = torch.empty(n, 3, img_size, img_size)
    return crit(output, target)["bpp_loss"]
