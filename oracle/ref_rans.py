"""Independent restatement of compressai 1.2.4's entropy coder, for tests of the library's GPU coder.

- `pmf_to_quantized_cdf`              cpp_exts/ops/ops.cpp (precision 16)
- `gaussian_tables` / `bottleneck_tables`   GaussianConditional.update() / EntropyBottleneck.update(force=True)
                                      (entropy_models.py), in fp32 torch on the CPU as compressai computes them
- `encode_with_indexes`              BufferedRansEncoder.encode_with_indexes + flush (cpp_exts/rans/rans_interface.cpp over
                                      third_party/ryg_rans/rans64.h)
- `decode_with_indexes`              RansDecoder.decode_with_indexes

Pure Python / numpy / torch: nothing here imports the library.  `compressai_available()` and the live check in
tests/test_rans_cpu.py compare against compressai itself where it is installed.
"""
from __future__ import annotations

import bisect
import math
import struct
from typing import Dict, List, Sequence

import numpy as np
import torch
import torch.nn.functional as F

PRECISION = 16
BYPASS_PRECISION = 4
MAX_BYPASS_VAL = (1 << BYPASS_PRECISION) - 1
RANS64_L = 1 << 31
_M32 = (1 << 32) - 1


def pmf_to_quantized_cdf(pmf: Sequence[float], precision: int = PRECISION) -> List[int]:
    pmf = np.asarray(pmf, dtype=np.float32)
    scale = np.float32(1 << precision)
    # std::round of the float product p * 2^16: halves away from zero (p >= 0)
    cdf = [0] + [int(math.floor(float(np.float32(p) * scale) + 0.5)) for p in pmf]
    total = sum(cdf)
    if total == 0:
        raise ValueError("all-zero pmf")
    cdf = [((1 << precision) * p) // total for p in cdf]
    for i in range(1, len(cdf)):
        cdf[i] += cdf[i - 1]
    cdf[-1] = 1 << precision
    for i in range(len(cdf) - 1):
        if cdf[i] == cdf[i + 1]:
            best_freq, best_steal = None, -1
            for j in range(len(cdf) - 1):
                f = cdf[j + 1] - cdf[j]
                if f > 1 and (best_freq is None or f < best_freq):
                    best_freq, best_steal = f, j
            if best_steal < 0:
                raise ValueError("cannot give every bin a count")
            if best_steal < i:
                for j in range(best_steal + 1, i + 1):
                    cdf[j] -= 1
            else:
                for j in range(i + 1, best_steal + 1):
                    cdf[j] += 1
    return cdf


def _pmf_to_cdf(pmf: torch.Tensor, tail: torch.Tensor, pmf_length: torch.Tensor, max_length: int) -> torch.Tensor:
    cdf = torch.zeros((len(pmf_length), max_length + 2), dtype=torch.int32)
    for i, p in enumerate(pmf):
        prob = torch.cat((p[: int(pmf_length[i])], tail[i]), dim=0)
        q = pmf_to_quantized_cdf(prob.tolist())
        cdf[i, : len(q)] = torch.tensor(q, dtype=torch.int32)
    return cdf


def gaussian_tables(scale_table, tail_mass: float = 1e-9) -> Dict[str, torch.Tensor]:
    """GaussianConditional.update(): one table per scale-table entry."""
    from scipy.stats import norm
    scale_table = torch.tensor([float(s) for s in scale_table], dtype=torch.float32)
    multiplier = -float(norm.ppf(tail_mass / 2))
    pmf_center = torch.ceil(scale_table * multiplier).int()
    pmf_length = 2 * pmf_center + 1
    max_length = int(torch.max(pmf_length).item())
    samples = torch.abs(torch.arange(max_length).int() - pmf_center[:, None]).float()
    scales = scale_table.unsqueeze(1).float()
    cum = lambda x: 0.5 * torch.erfc(float(-(2 ** -0.5)) * x)
    upper = cum((0.5 - samples) / scales)
    lower = cum((-0.5 - samples) / scales)
    pmf = upper - lower
    tail = 2 * lower[:, :1]
    return {"_quantized_cdf": _pmf_to_cdf(pmf, tail, pmf_length, max_length), "_offset": -pmf_center,
            "_cdf_length": pmf_length + 2}


def bottleneck_tables(sd: Dict[str, torch.Tensor], prefix: str = "entropy_bottleneck.") -> Dict[str, torch.Tensor]:
    """EntropyBottleneck.update(force=True): one table per channel, from the module's parameters."""
    p = {k[len(prefix):]: v.detach().float().cpu() for k, v in sd.items() if k.startswith(prefix)}
    q = p["quantiles"]
    medians = q[:, 0, 1]
    minima = torch.clamp(torch.ceil(medians - q[:, 0, 0]).int(), min=0)
    maxima = torch.clamp(torch.ceil(q[:, 0, 2] - medians).int(), min=0)
    pmf_start = medians - minima
    pmf_length = maxima + minima + 1
    max_length = int(pmf_length.max().item())
    samples = torch.arange(max_length)[None, :] + pmf_start[:, None, None]

    def logits_cumulative(x):
        for i in range(5):
            x = torch.matmul(F.softplus(p[f"_matrix{i}"]), x) + p[f"_bias{i}"]
            if i < 4:
                x = x + torch.tanh(p[f"_factor{i}"]) * torch.tanh(x)
        return x

    lower = logits_cumulative(samples - 0.5)
    upper = logits_cumulative(samples + 0.5)
    sign = -torch.sign(lower + upper)
    pmf = torch.abs(torch.sigmoid(sign * upper) - torch.sigmoid(sign * lower))[:, 0, :]
    tail = torch.sigmoid(lower[:, 0, :1]) + torch.sigmoid(-upper[:, 0, -1:])
    return {"_quantized_cdf": _pmf_to_cdf(pmf, tail, pmf_length, max_length), "_offset": -minima,
            "_cdf_length": pmf_length + 2}


def _as_lists(cdfs, cdf_lengths, offsets):
    cdfs = np.asarray(cdfs).tolist()
    return cdfs, [int(v) for v in np.asarray(cdf_lengths).ravel()], [int(v) for v in np.asarray(offsets).ravel()]


def encode_with_indexes(symbols, indexes, cdfs, cdf_lengths, offsets) -> bytes:
    """BufferedRansEncoder.encode_with_indexes(...) followed by flush()."""
    cdfs, cdf_lengths, offsets = _as_lists(cdfs, cdf_lengths, offsets)
    syms = []                                    # (start, freq, bypass)
    for s, t in zip(np.asarray(symbols).ravel().tolist(), np.asarray(indexes).ravel().tolist()):
        cdf = cdfs[t]
        max_value = cdf_lengths[t] - 2
        value = s - offsets[t]
        raw = 0
        if value < 0:
            raw = -2 * value - 1
            value = max_value
        elif value >= max_value:
            raw = 2 * (value - max_value)
            value = max_value
        raw &= _M32
        syms.append((cdf[value], cdf[value + 1] - cdf[value], False))
        if value == max_value:
            n_bypass = 0
            while n_bypass < 8 and (raw >> (n_bypass * BYPASS_PRECISION)) != 0:
                n_bypass += 1
            val = n_bypass
            while val >= MAX_BYPASS_VAL:
                syms.append((MAX_BYPASS_VAL, MAX_BYPASS_VAL + 1, True))
                val -= MAX_BYPASS_VAL
            syms.append((val, val + 1, True))
            for j in range(n_bypass):
                v = (raw >> (j * BYPASS_PRECISION)) & MAX_BYPASS_VAL
                syms.append((v, v + 1, True))
    x = RANS64_L
    words = []                                   # emitted back to front
    for start, freq, bypass in reversed(syms):
        if not bypass:
            x_max = ((RANS64_L >> PRECISION) << 32) * freq
            if x >= x_max:
                words.append(x & _M32)
                x >>= 32
            x = ((x // freq) << PRECISION) + x % freq + start
        else:
            x_max = ((RANS64_L >> BYPASS_PRECISION) << 32)
            if x >= x_max:
                words.append(x & _M32)
                x >>= 32
            x = (x << BYPASS_PRECISION) | start
    words.append(x >> 32)
    words.append(x & _M32)
    words.reverse()
    return struct.pack(f"<{len(words)}I", *words)


def decode_with_indexes(data: bytes, indexes, cdfs, cdf_lengths, offsets) -> List[int]:
    """RansDecoder.decode_with_indexes(...).  Raises ValueError when the stream is shorter than the decode needs."""
    cdfs, cdf_lengths, offsets = _as_lists(cdfs, cdf_lengths, offsets)
    if len(data) % 4:
        raise ValueError("stream length is not a multiple of 4")
    words = struct.unpack(f"<{len(data) // 4}I", data)
    pos = 0

    def word():
        nonlocal pos
        if pos >= len(words):
            raise ValueError("read past the end of the stream")
        pos += 1
        return words[pos - 1]

    x = word()
    x |= word() << 32
    out = []
    mask = (1 << PRECISION) - 1
    for t in np.asarray(indexes).ravel().tolist():
        cdf = cdfs[t]
        n = cdf_lengths[t]
        max_value = n - 2
        cum = x & mask
        s = bisect.bisect_right(cdf, cum, 0, n) - 1          # first entry > cum, minus one (std::find_if)
        x = (cdf[s + 1] - cdf[s]) * (x >> PRECISION) + (x & mask) - cdf[s]
        if x < RANS64_L:
            x = (x << 32) | word()
        value = s

        def get_bits():
            nonlocal x
            v = x & MAX_BYPASS_VAL
            x >>= BYPASS_PRECISION
            if x < RANS64_L:
                x = (x << 32) | word()
            return v

        if value == max_value:
            val = get_bits()
            n_bypass = val
            while val == MAX_BYPASS_VAL:
                val = get_bits()
                n_bypass += val
            raw = 0
            for j in range(n_bypass):
                raw |= get_bits() << (j * BYPASS_PRECISION)
            raw = raw - (1 << 32) if raw & (1 << 31) else raw           # int32, as the C++
            value = raw >> 1
            value = -value - 1 if raw & 1 else value + max_value
        out.append(value + offsets[t])
    return out


def compressai_available() -> bool:
    try:
        import compressai.ans  # noqa: F401
        from compressai._CXX import pmf_to_quantized_cdf as _p  # noqa: F401
        return True
    except Exception:                                                # noqa: BLE001
        return False
