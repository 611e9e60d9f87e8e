"""ORACLE (test infrastructure only - never imported by the product path).

The decoder side of the reference's MCM.decompress (MCM.py:896-968) in plain torch fp32, with the range decoder replaced by
given symbols, built from the restated layers of oracle/ref_model.py.  compressai 1.2.4 GaussianConditional.build_indexes is
restated here as well (the scale-table bucket of every sigma: the list decode_stream receives).
"""
from __future__ import annotations

import torch

from .ref_model import SCALE_BOUND, _seq_convs, _w, h_s


def build_indexes(scales, table):
    """compressai 1.2.4 GaussianConditional.build_indexes (MCM.py:839, 867): scales lower-bounded (0.11), then
    indexes = len(table) - 1 - sum(scales <= s for s in table[:-1])."""
    scales = torch.clamp_min(scales, SCALE_BOUND)
    idx = scales.new_full(scales.size(), len(table) - 1).int()
    for s in table[:-1]:
        idx -= (scales <= s).int()
    return idx


def decode_from_symbols(sd, cfg, z_sym, y_sym, table=None, dtype=torch.float32):
    """The slice loop of MCM.decompress (MCM.py:896-968) with the range decoder replaced by the given symbols.
    z_sym [N,Cz,s/4,s/4], y_sym [N,Cy,s,s] (or [N, Cy*s*s] in the coder's order, which is the same memory order).
    Returns z_hat, mu, sigma, y_hat [N,*,h,w] and - with a scale table - the indexes the range decoder would have been
    handed, [N,Cy,s,s]: the same arithmetic as rate_from_latent, so fed its symbols it reproduces its latents exactly."""
    s = cfg.side
    N = z_sym.shape[0]
    y_sym = y_sym.reshape(N, cfg.latent_depth, s, s)
    med = _w(sd, "entropy_bottleneck.quantiles", dtype)[:, :, 1:2]      # [C,1,1]
    z_hat = z_sym.to(dtype) + med                                       # quantize(z, "dequantize", medians)
    latent_scales = h_s(sd, cfg, "h_s_scale", z_hat, dtype)
    latent_means = h_s(sd, cfg, "h_s_mean", z_hat, dtype)
    y_hat_slices, mus, sigmas, idxs = [], [], [], []
    for i, sym in enumerate(y_sym.chunk(cfg.num_slices, 1)):
        support = y_hat_slices[: cfg.max_support_slices]
        mean_support = torch.cat([latent_means] + support, dim=1)
        mu = _seq_convs(sd, f"cc_transform_mean.{i}", mean_support, dtype)[:, :, :s, :s]
        scale_support = torch.cat([latent_scales] + support, dim=1)
        sigma = _seq_convs(sd, f"cc_transform_scale.{i}", scale_support, dtype)[:, :, :s, :s]
        if table is not None:
            idxs.append(build_indexes(sigma, table))                    # -> decode_stream(indexes, ...)
        y_hat_slice = sym.to(dtype) + mu                                # dequantize(rv, mu)
        lrp_support = torch.cat([mean_support, y_hat_slice], dim=1)
        lrp = _seq_convs(sd, f"lrp_transform.{i}", lrp_support, dtype)
        y_hat_slice = y_hat_slice + 0.5 * torch.tanh(lrp)
        y_hat_slices.append(y_hat_slice)
        mus.append(mu); sigmas.append(sigma)
    out = dict(z_hat=z_hat, mu=torch.cat(mus, 1), sigma=torch.cat(sigmas, 1), y_hat=torch.cat(y_hat_slices, 1))
    if table is not None:
        out["indexes"] = torch.cat(idxs, 1)
    return out
