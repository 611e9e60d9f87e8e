"""CPU: the rANS coder's oracle, the quantised CDF tables and the coder's C ABI argument checks (no GPU needed)."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import ref_rans as R
from textmae_image_compression_b200 import MCM, PathConfig, _native, entropy, make_state_dict, vit_base

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16)


def _gauss():
    return R.gaussian_tables(MCM.get_scale_table())


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


@pytest.mark.parametrize("seed", [0, 1])
def test_oracle_round_trip_with_escapes(seed):
    tabs = _gauss()
    rng = np.random.default_rng(seed)
    sym, idx = _random_case(rng, tabs, 3000)
    # escapes at the edges: -1 below / exactly at max_value, and raw values near 2^31
    o, L = int(tabs["_offset"][5]), int(tabs["_cdf_length"][5])
    extra = [o - 1, o + L - 2, o + L - 3, o - 2 ** 30, o + L - 2 + 2 ** 30 - 1, o + L - 2 + 2 ** 27, o - 2 ** 27]
    sym = np.concatenate([sym, extra])
    idx = np.concatenate([idx, [5] * len(extra)])
    data = R.encode_with_indexes(sym, idx, tabs["_quantized_cdf"], tabs["_cdf_length"], tabs["_offset"])
    assert len(data) % 4 == 0
    out = R.decode_with_indexes(data, idx, tabs["_quantized_cdf"], tabs["_cdf_length"], tabs["_offset"])
    assert np.array_equal(np.asarray(out), sym)
    with pytest.raises(ValueError):
        R.decode_with_indexes(data[:-4], idx, tabs["_quantized_cdf"], tabs["_cdf_length"], tabs["_offset"])


def _lib_cdf(pmf):
    p = np.ascontiguousarray(pmf, dtype=np.float32)
    out = np.zeros(p.size + 1, dtype=np.int32)
    rc = _native.load().tmae_pmf_to_quantized_cdf(p.ctypes.data, p.size, out.ctypes.data)
    return rc, out


def test_pmf_to_quantized_cdf_matches_oracle():
    rng = np.random.default_rng(0)
    cases = [np.array([1.0]), np.array([0.0, 1.0, 0.0]), np.array([1.0, 0, 0, 0, 0]), np.full(7, 1e-12) + np.eye(7)[3],
             np.array([0.5, 0.25, 0.25, 0.0]), np.array([1e-9] * 40 + [1.0])]
    for n in (2, 5, 31, 300, 3000):
        p = rng.random(n) ** 4
        p[rng.random(n) < 0.3] = 0
        p[0] = max(p[0], 1e-3)
        cases.append(p / p.sum())
        cases.append(rng.random(n) * 3e-5)                    # tiny masses: many round to 0, the rescale by the total decides
    for p in cases:
        rc, got = _lib_cdf(p)
        try:
            ref = R.pmf_to_quantized_cdf(p)
        except ValueError:                                    # every mass rounds to 0 / too few counts for the bins
            assert rc == _native.TMAE_EINVAL
            continue
        assert rc == 0
        assert got.tolist() == ref, p
        assert got[0] == 0 and got[-1] == 65536 and np.all(np.diff(got) > 0)


def test_pmf_to_quantized_cdf_rejects_bad_pmfs():
    for p in (np.zeros(4), np.array([0.5, -0.1]), np.array([np.nan, 1.0]), np.array([np.inf])):
        assert _lib_cdf(p)[0] == _native.TMAE_EINVAL
    assert _native.load().tmae_pmf_to_quantized_cdf(None, 3, None) == _native.TMAE_EINVAL


def test_rans_bound():
    lib = _native.load()
    assert lib.tmae_rans_bound(0) == 8
    assert lib.tmae_rans_bound(24576) == 4 * (10 * 24576 + 2)
    assert lib.tmae_rans_bound(-1) == -1


@pytest.mark.parametrize("scale_table", ["default", "custom"])
def test_gaussian_tables_equal_oracle(scale_table):
    st = MCM.get_scale_table() if scale_table == "default" else torch.tensor([0.11, 0.3, 1.0, 2.5, 7.0, 19.0, 60.0])
    got, ref = entropy.gaussian_tables(st), R.gaussian_tables(st)
    for k in ("_quantized_cdf", "_cdf_length", "_offset"):
        assert torch.equal(got[k].int(), ref[k].int()), k
    if scale_table == "default":
        assert got["_quantized_cdf"].shape == (64, 3133) and int(got["_cdf_length"].sum()) == 27256


@pytest.mark.parametrize("which", ["small", "vitB"])
def test_bottleneck_tables_equal_oracle(which):
    cfg = PathConfig(**SMALL) if which == "small" else vit_base(64)
    sd = make_state_dict(cfg, seed=3)
    got, ref = entropy.bottleneck_tables(sd), R.bottleneck_tables(sd)
    for k in ("_quantized_cdf", "_cdf_length", "_offset"):
        assert torch.equal(got[k].int(), ref[k].int()), k
    assert got["_quantized_cdf"].shape[0] == cfg.hyperprior_depth


def test_entropy_tables_names_and_rebuild():
    cfg = PathConfig(**SMALL)
    m = MCM(**SMALL)
    m.load_state_dict(make_state_dict(cfg, seed=3))
    t = m.entropy_tables()
    assert sorted(t) == sorted(p + k for p in ("gaussian_conditional.", "entropy_bottleneck.")
                               for k in ("_quantized_cdf", "_cdf_length", "_offset"))
    assert t["gaussian_conditional._quantized_cdf"].shape[0] == 64
    m.update(scale_table=[0.2, 1.0, 5.0])
    assert m.entropy_tables()["gaussian_conditional._quantized_cdf"].shape[0] == 3
    sd = make_state_dict(cfg, seed=4)
    m.load_state_dict(sd)
    assert torch.equal(m.entropy_tables()["entropy_bottleneck._quantized_cdf"], R.bottleneck_tables(sd)["_quantized_cdf"])


def test_coder_abi_rejects_bad_arguments_without_a_gpu():
    lib = _native.load()
    E = _native.TMAE_EINVAL
    assert lib.tmae_set_cdf_tables(None, 0, None, 1, 3, None, None) == E
    assert lib.tmae_rans_encode(None, 0, None, None, 1, 1, None, 0, None, None, None) == E
    assert lib.tmae_rans_decode(None, 0, None, None, 1, None, 1, None, None, None) == E
    assert lib.tmae_decompress_streams(None, None, None, None, None, 1, None, None, None) == E


def test_bitstream_methods_are_cuda_only():
    cfg = PathConfig(**SMALL)
    m = MCM(**SMALL)
    m.load_state_dict(make_state_dict(cfg, seed=3))
    imgs, scores = torch.rand(1, 3, 64, 64), torch.rand(1, cfg.num_patches)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.compress_bitstream(imgs, scores)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.decompress_bitstream([[b"\0" * 8], [b"\0" * 8]], (1, 1), torch.zeros(1, cfg.num_patches, dtype=torch.long),
                               need_recon=False)


@pytest.mark.skipif(not R.compressai_available(), reason="compressai is not installed: live check against compressai.ans skipped")
def test_oracle_against_compressai():
    from compressai._CXX import pmf_to_quantized_cdf as cxx_cdf
    from compressai.ans import BufferedRansEncoder, RansDecoder
    rng = np.random.default_rng(0)
    for n in (1, 3, 40, 500):
        p = (rng.random(n) ** 3).astype(np.float32)
        assert list(cxx_cdf(p.tolist(), 16)) == R.pmf_to_quantized_cdf(p)
    tabs = _gauss()
    sym, idx = _random_case(rng, tabs, 2000)
    args = (tabs["_quantized_cdf"].tolist(), tabs["_cdf_length"].tolist(), tabs["_offset"].tolist())
    enc = BufferedRansEncoder()
    enc.encode_with_indexes(sym.tolist(), idx.tolist(), *args)
    data = enc.flush()
    assert data == R.encode_with_indexes(sym, idx, *args)
    assert RansDecoder().decode_with_indexes(data, idx.tolist(), *args) == sym.tolist()
