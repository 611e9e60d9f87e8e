"""CPU: the synthesis calls of the C ABI (tmae_enable_synthesis, tmae_synthesize, tmae_attention_hd32_bf16) exist, reject a null
handle / bad arguments without touching a device, and MCM(native_synthesis=True) stays CUDA-only."""
import ctypes as C

import pytest
import torch

from textmae_image_compression_b200 import MCM, PathConfig, _native, make_state_dict

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16,
             decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=2)


def test_synthesis_calls_are_declared():
    for name in ("tmae_enable_synthesis", "tmae_synthesize", "tmae_attention_hd32_bf16"):
        assert name in _native.SIGNATURES
    header = (_native._PKG.parent / "include" / "tmae.h").read_text()
    for name in ("tmae_enable_synthesis", "tmae_synthesize", "tmae_attention_hd32_bf16"):
        assert f"TMAE_API int  {name}(" in header


def test_null_handle_is_einval():
    lib = _native.load()
    assert lib.tmae_enable_synthesis(None, 8, 16) == _native.TMAE_EINVAL
    assert lib.tmae_synthesize(None, None, None, 1, None, None) == _native.TMAE_EINVAL
    assert lib.tmae_attention_hd32_bf16(None, None, 1, 17, 16, None) == _native.TMAE_EINVAL


def test_native_synthesis_is_cuda_only():
    cfg = PathConfig(**SMALL)
    m = MCM(**SMALL, softmax_isa=16, native_synthesis=True)
    m.load_state_dict(make_state_dict(cfg, seed=3, include_decoder=True))
    g = torch.Generator().manual_seed(0)
    imgs, scores = torch.rand(1, 3, 64, 64, generator=g), torch.rand(1, cfg.num_patches, generator=g)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m(imgs, scores, need_recon=True)
