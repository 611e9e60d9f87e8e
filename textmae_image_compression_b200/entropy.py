"""Quantised CDF tables and torch front ends of the library's rANS coder (compressai 1.2.4's bitstream format).

The tables are built as compressai's `update(force=True)` builds them - in fp32 torch on the CPU, then
`pmf_to_quantized_cdf` (here the library's host-only `tmae_pmf_to_quantized_cdf`) - and come out under compressai's buffer
names: `_quantized_cdf` int32 [n, max_length + 2] (padded), `_cdf_length` int32 [n], `_offset` int32 [n].
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Tuple

import torch
import torch.nn.functional as F

from . import _native

TAIL_MASS = 1e-9


def quantized_cdf(pmf: torch.Tensor) -> torch.Tensor:
    """compressai's pmf_to_quantized_cdf(pmf, 16): float32 [n] -> int32 [n + 1]."""
    p = pmf.detach().float().cpu().contiguous()
    out = torch.empty(p.numel() + 1, dtype=torch.int32)
    _native.check(_native.load().tmae_pmf_to_quantized_cdf(C.c_void_p(p.data_ptr()), p.numel(), C.c_void_p(out.data_ptr())))
    return out


def _pmf_to_cdf(pmf, tail, pmf_length, max_length) -> torch.Tensor:
    cdf = torch.zeros((len(pmf_length), max_length + 2), dtype=torch.int32)
    for i, p in enumerate(pmf):
        q = quantized_cdf(torch.cat((p[: int(pmf_length[i])], tail[i]), dim=0))
        cdf[i, : q.numel()] = q
    return cdf


def _gaussian_multiplier() -> float:
    """-Phi^-1(tail_mass / 2), computed with scipy as compressai's _standardized_quantile does."""
    from scipy.stats import norm
    return -float(norm.ppf(TAIL_MASS / 2))


def gaussian_tables(scale_table: torch.Tensor) -> Dict[str, torch.Tensor]:
    """GaussianConditional.update(): one table per scale-table entry s, centre ceil(s * m), length 2 * centre + 1 + tail."""
    scale_table = torch.tensor([float(s) for s in scale_table], dtype=torch.float32)
    pmf_center = torch.ceil(scale_table * _gaussian_multiplier()).int()
    pmf_length = 2 * pmf_center + 1
    max_length = int(torch.max(pmf_length).item())
    samples = torch.abs(torch.arange(max_length).int() - pmf_center[:, None]).float()
    scales = scale_table.unsqueeze(1)
    upper = 0.5 * torch.erfc(float(-(2 ** -0.5)) * ((0.5 - samples) / scales))
    lower = 0.5 * torch.erfc(float(-(2 ** -0.5)) * ((-0.5 - samples) / scales))
    pmf = upper - lower
    tail = 2 * lower[:, :1]
    return {"_quantized_cdf": _pmf_to_cdf(pmf, tail, pmf_length, max_length), "_cdf_length": (pmf_length + 2).int(),
            "_offset": (-pmf_center).int()}


def bottleneck_tables(weights: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """EntropyBottleneck.update(force=True) from the module's `entropy_bottleneck.*` parameters: one table per channel over
    [median - minima, median + maxima]; the tail is sigmoid(lower[:, 0, :1]) + sigmoid(-upper[:, 0, -1:]) of the padded row."""
    w = {k[len("entropy_bottleneck."):]: v.detach().float().cpu() for k, v in weights.items()
         if k.startswith("entropy_bottleneck.")}
    q = w["quantiles"]
    medians = q[:, 0, 1]
    minima = torch.clamp(torch.ceil(medians - q[:, 0, 0]).int(), min=0)
    maxima = torch.clamp(torch.ceil(q[:, 0, 2] - medians).int(), min=0)
    pmf_start = medians - minima
    pmf_length = maxima + minima + 1
    max_length = int(pmf_length.max().item())
    samples = torch.arange(max_length)[None, :] + pmf_start[:, None, None]

    def logits_cumulative(x):
        for i in range(5):
            x = torch.matmul(F.softplus(w[f"_matrix{i}"]), x) + w[f"_bias{i}"]
            if i < 4:
                x = x + torch.tanh(w[f"_factor{i}"]) * torch.tanh(x)
        return x

    lower = logits_cumulative(samples - 0.5)
    upper = logits_cumulative(samples + 0.5)
    sign = -torch.sign(lower + upper)
    pmf = torch.abs(torch.sigmoid(sign * upper) - torch.sigmoid(sign * lower))[:, 0, :]
    tail = torch.sigmoid(lower[:, 0, :1]) + torch.sigmoid(-upper[:, 0, -1:])
    return {"_quantized_cdf": _pmf_to_cdf(pmf, tail, pmf_length, max_length), "_cdf_length": (pmf_length + 2).int(),
            "_offset": (-minima).int()}


def set_tables(handle, model: int, tables: Dict[str, torch.Tensor]):
    cdf = tables["_quantized_cdf"].int().contiguous()
    ln = tables["_cdf_length"].int().contiguous()
    off = tables["_offset"].int().contiguous()
    _native.check(_native.load().tmae_set_cdf_tables(handle, model, C.c_void_p(cdf.data_ptr()), cdf.shape[0], cdf.shape[1],
                                                     C.c_void_p(ln.data_ptr()), C.c_void_p(off.data_ptr())), handle)


def rans_bound(n_symbols: int) -> int:
    return int(_native.load().tmae_rans_bound(n_symbols))


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def encode(handle, model: int, symbols: torch.Tensor, indexes: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """encode_with_indexes + flush of every row of symbols / indexes (int32 [n_streams, n] on the handle's device), enqueued on
    the current stream -> (packed bytes uint8 [capacity], offsets int64 [n_streams + 1], status int32 [n_streams])."""
    n_streams, n = symbols.shape
    sym = symbols.to(torch.int32).contiguous()
    idx = indexes.to(torch.int32).contiguous()
    cap = n_streams * rans_bound(n)
    out = torch.empty(cap, dtype=torch.uint8, device=sym.device)
    offsets = torch.empty(n_streams + 1, dtype=torch.int64, device=sym.device)
    status = torch.empty(n_streams, dtype=torch.int32, device=sym.device)
    _native.check(_native.load().tmae_rans_encode(handle, model, C.c_void_p(sym.data_ptr()), C.c_void_p(idx.data_ptr()), n_streams, n,
                                                  C.c_void_p(out.data_ptr()), cap, C.c_void_p(offsets.data_ptr()),
                                                  C.c_void_p(status.data_ptr()), _stream()), handle)
    return out, offsets, status


def decode(handle, model: int, data: torch.Tensor, offsets: torch.Tensor, indexes: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """decode_with_indexes of every stream (bytes [offsets[i], offsets[i + 1]) of data) -> (symbols int32 [n_streams, n],
    status int32 [n_streams])."""
    n_streams, n = indexes.shape
    idx = indexes.to(torch.int32).contiguous()
    data = data.contiguous()
    offsets = offsets.to(torch.int64).contiguous()
    if data.numel() == 0:
        data = torch.zeros(4, dtype=torch.uint8, device=idx.device)
    sym = torch.empty((n_streams, n), dtype=torch.int32, device=idx.device)
    status = torch.empty(n_streams, dtype=torch.int32, device=idx.device)
    _native.check(_native.load().tmae_rans_decode(handle, model, C.c_void_p(data.data_ptr()), C.c_void_p(offsets.data_ptr()), n_streams,
                                                  C.c_void_p(idx.data_ptr()), n, C.c_void_p(sym.data_ptr()),
                                                  C.c_void_p(status.data_ptr()), _stream()), handle)
    return sym, status


def rans_bound_lanes(n_symbols: int, lanes: int) -> int:
    return int(_native.load().tmae_rans_bound_lanes(n_symbols, lanes))


def encode_lanes(handle, model: int, symbols: torch.Tensor, indexes: torch.Tensor, lanes: int
                 ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """`encode` in the laned format: every row becomes {lanes, lane byte lengths, lanes}, lane l being the compressai stream of the
    row's symbols l, l + lanes, ... (DESIGN.md section 7)."""
    n_streams, n = symbols.shape
    sym = symbols.to(torch.int32).contiguous()
    idx = indexes.to(torch.int32).contiguous()
    cap = n_streams * max(rans_bound_lanes(n, lanes), 0)
    out = torch.empty(max(cap, 4), dtype=torch.uint8, device=sym.device)
    offsets = torch.empty(n_streams + 1, dtype=torch.int64, device=sym.device)
    status = torch.empty(n_streams, dtype=torch.int32, device=sym.device)
    _native.check(_native.load().tmae_rans_encode_lanes(handle, model, C.c_void_p(sym.data_ptr()), C.c_void_p(idx.data_ptr()),
                                                        n_streams, n, lanes, C.c_void_p(out.data_ptr()), cap,
                                                        C.c_void_p(offsets.data_ptr()), C.c_void_p(status.data_ptr()), _stream()),
                  handle)
    return out, offsets, status


def decode_lanes(handle, model: int, data: torch.Tensor, offsets: torch.Tensor, indexes: torch.Tensor, lanes: int
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
    """`decode` of laned streams."""
    n_streams, n = indexes.shape
    idx = indexes.to(torch.int32).contiguous()
    data = data.contiguous()
    offsets = offsets.to(torch.int64).contiguous()
    if data.numel() == 0:
        data = torch.zeros(4, dtype=torch.uint8, device=idx.device)
    sym = torch.empty((n_streams, n), dtype=torch.int32, device=idx.device)
    status = torch.empty(n_streams, dtype=torch.int32, device=idx.device)
    _native.check(_native.load().tmae_rans_decode_lanes(handle, model, C.c_void_p(data.data_ptr()), C.c_void_p(offsets.data_ptr()),
                                                        n_streams, C.c_void_p(idx.data_ptr()), n, lanes, C.c_void_p(sym.data_ptr()),
                                                        C.c_void_p(status.data_ptr()), _stream()), handle)
    return sym, status


def pack_strings(strings) -> Tuple[torch.Tensor, torch.Tensor]:
    """list of bytes -> (uint8 [total] host tensor, int64 [n + 1] byte offsets)."""
    lens = [len(s) for s in strings]
    offsets = torch.zeros(len(strings) + 1, dtype=torch.int64)
    offsets[1:] = torch.cumsum(torch.tensor(lens, dtype=torch.int64), 0)
    data = torch.frombuffer(bytearray(b"".join(strings)), dtype=torch.uint8) if sum(lens) else torch.zeros(0, dtype=torch.uint8)
    return data, offsets
