"""CPU: the decode side (MCM.decompress without the range coder).  The oracle's decode_from_symbols against the oracle's
own forward, the host-only slice-group query of the C ABI, argument validation, the module's CUDA-only error, and - where a
checkout of the original project exists - the reference's own MCM.decompress with its range decoder replaced by given
symbols."""
import ctypes as C

import pytest
import torch

from oracle import SKIP_REASON, ref_decode, ref_model
from textmae_image_compression_b200 import MCM, PathConfig, make_state_dict

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16)
MID = dict(img_size=128, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=64)


@pytest.fixture(scope="module")
def lib():
    from textmae_image_compression_b200 import build, _native
    build.build()
    return _native.load()


def _latent(cfg, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, cfg.latent_depth, cfg.side, cfg.side, generator=g) * 3.0


@pytest.mark.parametrize("kw", [SMALL, MID], ids=["small", "mid"])
def test_oracle_decode_reproduces_forward_latents(kw):
    cfg = PathConfig(**kw)
    sd = make_state_dict(cfg, seed=11)
    fwd = ref_model.rate_from_latent(sd, cfg, _latent(cfg, 2, 5))
    table = MCM.get_scale_table()
    dec = ref_decode.decode_from_symbols(sd, cfg, fwd["z_sym"], fwd["y_sym"], table)
    for k in ("z_hat", "mu", "sigma", "y_hat"):
        assert torch.equal(dec[k], fwd[k]), k
    assert torch.equal(dec["indexes"], ref_decode.build_indexes(fwd["sigma"], table))
    # the coder's flat order [N, Cy*s*s] is the same memory order as [N, Cy, s, s]
    flat = ref_decode.decode_from_symbols(sd, cfg, fwd["z_sym"], fwd["y_sym"].reshape(2, -1))
    assert torch.equal(flat["y_hat"], fwd["y_hat"]) and "indexes" not in flat


def test_build_indexes_counts_table_entries_below_scale():
    table = MCM.get_scale_table()
    sc = torch.tensor([0.0, 0.11, 0.1100001, 1.0, 255.9, 256.0, 1e6])
    idx = ref_decode.build_indexes(sc, table)
    want = torch.tensor([int((table[:-1] < max(v, 0.11)).sum()) for v in sc.tolist()], dtype=torch.int32)
    assert torch.equal(idx, want)


def test_decode_groups(lib):
    first, cnt = (C.c_int * 12)(), (C.c_int * 12)()
    assert lib.tmae_decode_groups(12, first, cnt, 12) == 7
    assert list(zip(first[:7], cnt[:7])) == [(0, 1), (1, 1), (2, 1), (3, 1), (4, 1), (5, 1), (6, 6)]
    assert lib.tmae_decode_groups(12, None, None, 0) == 7
    assert lib.tmae_decode_groups(4, first, cnt, 12) == 3 and list(zip(first[:3], cnt[:3])) == [(0, 1), (1, 1), (2, 2)]


def test_decode_entry_points_reject_bad_arguments(lib):
    from textmae_image_compression_b200 import _native
    o = _native.TmaeOutputs()
    buf = (C.c_int32 * 16)()
    assert lib.tmae_decode_begin(None, buf, 1, C.byref(o), None) == _native.TMAE_EINVAL
    assert lib.tmae_decode_step(None, 0, buf, C.byref(o), None) == _native.TMAE_EINVAL
    first = (C.c_int * 12)()
    assert lib.tmae_decode_groups(0, None, None, 0) == -_native.TMAE_EINVAL
    assert lib.tmae_decode_groups(7, None, None, 0) == -_native.TMAE_EINVAL
    assert lib.tmae_decode_groups(12, first, None, 6) == -_native.TMAE_EINVAL       # capacity below the group count


def test_decompress_symbols_is_cuda_only():
    cfg = PathConfig(**SMALL)
    m = MCM(**SMALL)
    m.load_state_dict(make_state_dict(cfg, 0))
    s, s4 = cfg.side, cfg.side // 4
    z = torch.zeros(1, cfg.hyperprior_depth, s4, s4, dtype=torch.int32)
    y = torch.zeros(1, cfg.latent_depth * s * s, dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.decompress_symbols(z, torch.zeros(1, cfg.num_patches, dtype=torch.int64), y_symbols=y)
    with pytest.raises(ValueError):
        m.decompress_symbols(z, torch.zeros(1, cfg.num_patches, dtype=torch.int64))              # neither y_symbols nor decode_fn
    with pytest.raises(NotImplementedError):
        m.decompress(None, None)


def _reference_available():
    from oracle import ref_exec
    return ref_exec.reference_available()


@pytest.mark.skipif(not _reference_available(), reason=SKIP_REASON)
def test_oracle_decode_matches_reference_decompress():
    """The reference's MCM.decompress executed as written, its range decoders replaced by given symbols: the indexes it hands
    decode_stream and its y_hat / x_hat equal the oracle's (x_hat settles whether decompress post-processes the image)."""
    from oracle import ref_exec, ref_stubs
    from textmae_image_compression_b200 import recon
    cfg = PathConfig(**SMALL)
    sd = make_state_dict(cfg, seed=11, include_decoder=True)
    fwd = ref_model.rate_from_latent(sd, cfg, _latent(cfg, 1, 5))
    table = MCM.get_scale_table()
    model, _, _ = ref_exec.build_reference_model(cfg, sd)
    seen = []
    sym_slices = list(fwd["y_sym"].chunk(cfg.num_slices, 1))

    class GivenSymbols:
        def set_stream(self, *a, **k):
            pass

        def decode_stream(self, indexes, *a, **k):
            seen.append(torch.as_tensor(indexes).reshape(-1).clone())
            return sym_slices[len(seen) - 1].reshape(-1).tolist()

    gc, eb = model.gaussian_conditional, model.entropy_bottleneck
    gc.build_indexes = lambda scales: ref_decode.build_indexes(scales, table)
    gc.dequantize = lambda v, means=None, dtype=torch.float: (v.to(dtype) + means) if means is not None else v.to(dtype)
    gc.quantized_cdf, gc.cdf_length, gc.offset = torch.zeros(1, 1, dtype=torch.int32), torch.ones(1, dtype=torch.int32), torch.zeros(1, dtype=torch.int32)
    med = sd["entropy_bottleneck.quantiles"][:, :, 1:2]
    eb.decompress = lambda strings, size: fwd["z_sym"].float() + med
    ref_mod = __import__(type(model).__module__, fromlist=["RansDecoder"])
    saved = getattr(ref_mod, "RansDecoder", ref_stubs.RansDecoder)
    ref_mod.RansDecoder = GivenSymbols
    try:
        ids_restore = torch.argsort(torch.randperm(cfg.num_patches, generator=torch.Generator().manual_seed(2))).unsqueeze(0)
        res = model.decompress([[b""], [b""]], list(fwd["z_sym"].shape[2:]), ids_restore)
    finally:
        ref_mod.RansDecoder = saved
    dec = ref_decode.decode_from_symbols(sd, cfg, fwd["z_sym"], fwd["y_sym"], table)
    want_idx = list(dec["indexes"].chunk(cfg.num_slices, 1))
    assert len(seen) == cfg.num_slices
    for i, got in enumerate(seen):
        assert torch.equal(got.int(), want_idx[i].reshape(-1)), i
    x_hat = res["x_hat"] if isinstance(res, dict) else res
    y_tok = dec["y_hat"].permute(0, 2, 3, 1).reshape(1, cfg.num_keep_patches, cfg.latent_depth)
    assert torch.allclose(x_hat, recon.synthesize(sd, cfg, y_tok, ids_restore), atol=1e-5)
