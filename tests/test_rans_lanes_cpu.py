"""The laned rANS format without a GPU: the reference laned coder (tests/ref_rans_lanes.py), its relation to compressai's
format, the lane bound and the argument checks of the laned ABI calls and methods."""
import struct

import numpy as np
import pytest
import torch

from oracle import ref_rans as R
from tests import ref_rans_lanes as L
from textmae_image_compression_b200 import MCM, PathConfig, _native, make_state_dict

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16)


def _gauss():
    return R.gaussian_tables(MCM.get_scale_table())


def _tabs(tabs):
    return tabs["_quantized_cdf"], tabs["_cdf_length"], tabs["_offset"]


def _random_case(rng, tabs, n, escape_rate=0.1):
    n_tab = tabs["_cdf_length"].shape[0]
    idx = rng.integers(0, n_tab, n)
    off = tabs["_offset"].numpy()[idx]
    ln = tabs["_cdf_length"].numpy()[idx]
    sym = off + (rng.random(n) * (ln - 2)).astype(np.int64)
    esc = rng.random(n) < escape_rate
    far = rng.integers(1, 5000, n)
    sym[esc] = np.where(rng.random(esc.sum()) < 0.5, off[esc] - far[esc], off[esc] + ln[esc] - 2 + far[esc])
    return sym, idx


def _near_2_31(tabs, t=5):
    o, ln = int(tabs["_offset"][t]), int(tabs["_cdf_length"][t])
    return [o - 2 ** 30, o + ln - 2 + 2 ** 30 - 1, o - 1, o + ln - 2, o + ln - 2 + 2 ** 27]


@pytest.mark.parametrize("W", [1, 5, 32])
@pytest.mark.parametrize("n,escape_rate", [(0, 0.0), (3, 0.0), (31, 0.1), (100, 0.9), (1001, 0.05)])
def test_oracle_laned_round_trip(W, n, escape_rate):
    tabs = _gauss()
    rng = np.random.default_rng(n * 33 + W)
    sym, idx = _random_case(rng, tabs, n, escape_rate)
    if n >= 31:                                   # escapes whose raw values come near 2^31
        extra = _near_2_31(tabs)
        sym = np.concatenate([sym, extra])
        idx = np.concatenate([idx, [5] * len(extra)])
    data = L.encode_lanes(sym, idx, W, *_tabs(tabs))
    head = struct.unpack(f"<{1 + W}I", data[: 4 * (1 + W)])
    assert head[0] == W and len(data) == 4 * (1 + W) + sum(head[1:])
    assert all(h % 4 == 0 and h >= 8 for h in head[1:])
    if len(sym) < W:                              # lanes without symbols: the 8 flush bytes of state L
        for lane in L.split_lanes(data, W)[len(sym):]:
            assert lane == struct.pack("<2I", R.RANS64_L, 0)
    assert L.decode_lanes(data, idx, W, *_tabs(tabs)) == list(sym)


def test_one_lane_is_the_compressai_stream_behind_a_header():
    tabs = _gauss()
    sym, idx = _random_case(np.random.default_rng(0), tabs, 500)
    plain = R.encode_with_indexes(sym, idx, *_tabs(tabs))
    assert L.encode_lanes(sym, idx, 1, *_tabs(tabs)) == struct.pack("<2I", 1, len(plain)) + plain


@pytest.mark.parametrize("W", [5, 32])
def test_every_lane_is_a_compressai_stream(W):
    tabs = _gauss()
    sym, idx = _random_case(np.random.default_rng(W), tabs, 777, 0.2)
    lanes = L.split_lanes(L.encode_lanes(sym, idx, W, *_tabs(tabs)), W)
    for l, lane in enumerate(lanes):
        assert lane == R.encode_with_indexes(sym[l::W], idx[l::W], *_tabs(tabs))
        assert R.decode_with_indexes(lane, idx[l::W], *_tabs(tabs)) == list(sym[l::W])


def test_oracle_rejects_malformed_headers():
    tabs = _gauss()
    sym, idx = _random_case(np.random.default_rng(1), tabs, 64)
    data = L.encode_lanes(sym, idx, 4, *_tabs(tabs))
    with pytest.raises(ValueError):
        L.decode_lanes(data, idx, 5, *_tabs(tabs))                  # another W
    with pytest.raises(ValueError):
        L.decode_lanes(data[:-4], idx, 4, *_tabs(tabs))             # truncated
    bad = bytearray(data)
    bad[4:8] = struct.pack("<I", struct.unpack("<I", data[4:8])[0] + 4)
    with pytest.raises(ValueError):
        L.decode_lanes(bytes(bad), idx, 4, *_tabs(tabs))            # lengths that do not add up
    with pytest.raises(ValueError):
        L.encode_lanes(sym, idx, 33, *_tabs(tabs))


@pytest.mark.parametrize("W", [1, 7, 32])
def test_rans_bound_lanes_covers_the_worst_case(W):
    lib = _native.load()
    tabs = _gauss()
    for n in (0, 1, W - 1, W, 3 * W + 1, 200):
        # every symbol an escape of an 8-nibble raw value, in the table with the most probable escape-free symbols
        worst = [int(tabs["_offset"][0]) - 2 ** 30] * n
        data = L.encode_lanes(worst, [0] * n, W, *_tabs(tabs))
        assert len(data) <= lib.tmae_rans_bound_lanes(n, W)
    assert lib.tmae_rans_bound_lanes(10, 3) == 4 * 4 + 4 * (100 + 6)
    for n, W in ((-1, 4), (5, 0), (5, 33), (5, -1)):
        assert lib.tmae_rans_bound_lanes(n, W) == -1


def test_laned_abi_rejects_bad_arguments_without_a_gpu():
    lib = _native.load()
    E = _native.TMAE_EINVAL
    for W in (0, 33, 4):                          # null handle: EINVAL whatever the lanes
        assert lib.tmae_rans_encode_lanes(None, 0, None, None, 1, 1, W, None, 0, None, None, None) == E
        assert lib.tmae_rans_decode_lanes(None, 0, None, None, 1, None, 1, W, None, None, None) == E
        assert lib.tmae_decompress_streams_lanes(None, None, None, W, None, None, W, 1, None, None, None) == E


def _small_model():
    cfg = PathConfig(**SMALL)
    m = MCM(**SMALL)
    m.load_state_dict(make_state_dict(cfg, seed=3))
    return cfg, m


def test_laned_bitstream_methods_are_cuda_only():
    cfg, m = _small_model()
    imgs, scores = torch.rand(1, 3, 64, 64), torch.rand(1, cfg.num_patches)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.compress_bitstream(imgs, scores, lanes=(32, 4))
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.decompress_bitstream([[b"\0" * 400], [b"\0" * 64]], (1, 1), torch.zeros(1, cfg.num_patches, dtype=torch.long),
                               need_recon=False, lanes=(32, 4))


@pytest.mark.parametrize("lanes", [(0, 4), (32, 33), (4,), 4, (4.0, 4), (True, 4), "32,4"])
def test_bad_lanes_values_raise_value_error(lanes):
    cfg, m = _small_model()
    with pytest.raises(ValueError, match="lanes"):
        m.compress_bitstream(torch.rand(1, 3, 64, 64), torch.rand(1, cfg.num_patches), lanes=lanes)
    with pytest.raises(ValueError, match="lanes"):
        m.decompress_bitstream([[b"\0" * 400], [b"\0" * 64]], (1, 1), torch.zeros(1, cfg.num_patches, dtype=torch.long),
                               need_recon=False, lanes=lanes)
