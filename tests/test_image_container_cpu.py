"""CPU: the image container (DESIGN.md section 7) through its plain-Python reference (tests/ref_image_container.py), the
canonical ids_restore the decoder rebuilds, and the container calls of the C ABI / MCM without a GPU."""
import struct

import pytest
import torch

from oracle import ref_mask
from tests import ref_image_container as R
from textmae_image_compression_b200 import MCM, PathConfig, _native, make_state_dict, recon

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16,
             decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=2)
FIELDS = dict(img_size=64, patch_size=16, mode=2, y_lanes=32, z_lanes=4, tag=0x12345678)


def test_hand_written_container_is_pinned_byte_for_byte():
    # L = 16 -> 4-bit ids; K = 3 ids {5, 0, 15}: bits 0-3 = 5, 4-7 = 0, 8-11 = 15 -> word 0x00000F05
    got = R.pack(b"\x01\x02\x03\x04" * 2, b"\xaa\xbb\xcc\xdd" * 3, [5, 0, 15], FIELDS)
    want = bytes.fromhex(
        "544d4145"      # magic "TMAE"
        "01022004"      # version 1, mode 2, W_y 32, W_z 4
        "40001000"      # img_size 64, patch_size 16, reserved 0
        "03000000"      # K = 3
        "78563412"      # tag
        "0c000000"      # z stream: 12 bytes
        "08000000"      # y stream: 8 bytes
        "050f0000"      # the ids, one word
        + "aabbccdd" * 3 + "01020304" * 2)
    assert got == want
    f = R.parse(got)
    assert f["ids_keep"] == [5, 0, 15] and f["K"] == 3 and f["tag"] == 0x12345678
    assert (f["mode"], f["y_lanes"], f["z_lanes"], f["img_size"], f["patch_size"]) == (2, 32, 4, 64, 16)
    assert f["z"] == b"\xaa\xbb\xcc\xdd" * 3 and f["y"] == b"\x01\x02\x03\x04" * 2


@pytest.mark.parametrize("L,w,K,ids_bytes", [(16, 4, 16, 8), (196, 8, 64, 64), (196, 8, 144, 144), (1024, 10, 256, 320),
                                            (1, 1, 1, 4), (4, 2, 4, 4)])
def test_id_widths_and_section_sizes(L, w, K, ids_bytes):
    assert R.id_bits(L) == w
    side = int(round(L ** 0.5))
    fields = dict(FIELDS, img_size=16 * side, patch_size=16)
    data = R.pack(b"", b"", list(range(L - K, L)), fields)
    assert len(data) == R.HEADER + ids_bytes
    assert R.parse(data)["ids_keep"] == list(range(L - K, L))


@pytest.mark.parametrize("seed", range(4))
def test_round_trips_through_the_reference(seed):
    g = torch.Generator().manual_seed(seed)
    for img_size, K in ((64, 16), (224, 64), (224, 144), (512, 256)):
        L = (img_size // 16) ** 2
        ids = torch.randperm(L, generator=g)[:K].tolist()
        y = bytes(torch.randint(0, 256, (4 * (seed + 3),), generator=g).tolist())
        z = bytes(torch.randint(0, 256, (4 * (seed + 1),), generator=g).tolist())
        fields = dict(FIELDS, img_size=img_size, tag=int(torch.randint(0, 2 ** 31, (1,), generator=g)))
        data = R.pack(y, z, ids, fields)
        assert len(data) == 28 + 4 * ((K * R.id_bits(L) + 31) // 32) + len(z) + len(y)
        f = R.parse(data)
        assert (f["ids_keep"], f["y"], f["z"], f["tag"]) == (ids, y, z, fields["tag"])


def test_reference_parse_refuses_malformed_containers():
    good = R.pack(b"\0" * 8, b"\0" * 8, [3, 1], FIELDS)
    for bad in (b"XMAE" + good[4:], good[:4] + b"\x02" + good[5:], good[:11] + b"\x01" + good[12:], good[:-4],
                R.pack(b"\0" * 8, b"\0" * 8, [3, 3], FIELDS), R.pack(b"\0" * 8, b"\0" * 8, [3, 12], dict(FIELDS, img_size=48))):
        with pytest.raises(ValueError):
            R.parse(bad)


def _small_weights():
    cfg = PathConfig(**SMALL)
    return cfg, make_state_dict(cfg, seed=3, include_decoder=True)


def test_canonical_ids_restore_gives_forwards_x_hat():
    cfg = PathConfig(**dict(SMALL, img_size=128))                       # L = 64 patches, K = 16 kept
    w = make_state_dict(cfg, seed=3, include_decoder=True)
    L, K = cfg.num_patches, cfg.num_keep_patches
    g = torch.Generator().manual_seed(0)
    score_sets = [torch.rand(3, L, generator=g), (torch.rand(2, L, generator=g) * 4).round() / 4,
                  torch.arange(L, dtype=torch.float32)[None].flip(1)]
    shuffles = [ref_mask.ids_shuffle_spec_batch(scores, K) for scores in score_sets]
    shuffles.append(torch.stack([torch.randperm(L, generator=g) for _ in range(3)]))     # unkept tails in any order
    tails_not_ascending = 0
    for shuffle in shuffles:
        ids_restore = torch.argsort(shuffle, dim=1)                    # what forward returns (MCM.py:580)
        ids_keep = shuffle[:, :K]
        canon = torch.tensor([R.canonical_ids_restore(r.tolist(), L) for r in ids_keep])
        assert torch.equal(canon.gather(1, ids_keep), ids_restore.gather(1, ids_keep))
        tails_not_ascending += sum(int(not torch.equal(r[K:], r[K:].sort().values)) for r in shuffle)
        y_hat = torch.randn(shuffle.shape[0], K, cfg.latent_depth, generator=g)
        x_ref = recon.synthesize(w, cfg, y_hat, ids_restore)
        x_can = recon.synthesize(w, cfg, y_hat, canon)
        assert torch.equal(x_can, x_ref)
    assert tails_not_ascending > 0                                       # the case where canon differs from forward's


def test_container_calls_are_declared():
    header = (_native._PKG.parent / "include" / "tmae.h").read_text()
    for name in ("tmae_model_tag", "tmae_compress_images", "tmae_decompress_images"):
        assert name in _native.SIGNATURES and f"TMAE_API int  {name}(" in header
    assert "tmae_images_bound" in _native.SIGNATURES and "TMAE_API int64_t tmae_images_bound(" in header
    assert (_native.IMG_HEADER, _native.IMG_CONFIG, _native.IMG_MODEL, _native.IMG_IDS) == (64, 128, 256, 512)


def test_images_bound_rejects_bad_arguments():
    lib = _native.load()
    for N, yl, zl in ((1, 32, 4), (0, 32, 4), (1, 33, 4), (1, -1, 0), (1, 0, 33)):
        assert lib.tmae_images_bound(None, N, yl, zl) == -1


def test_container_abi_rejects_bad_arguments_without_a_gpu():
    lib = _native.load()
    E = _native.TMAE_EINVAL
    for lanes in ((0, 0), (32, 4), (33, 4)):
        assert lib.tmae_compress_images(None, None, None, 1, *lanes, None, 0, None, None, None) == E
        assert lib.tmae_decompress_images(None, None, 0, None, 1, *lanes, None, None, None, None, None) == E
    assert lib.tmae_model_tag(None, None) == E


def test_container_methods_are_cuda_only():
    cfg, w = _small_weights()
    m = MCM(**SMALL)
    m.load_state_dict(w)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.compress_images(torch.rand(1, 3, 64, 64), torch.rand(1, cfg.num_patches))
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.decompress_images([R.pack(b"\0" * 8, b"\0" * 8, list(range(16)), FIELDS)])


@pytest.mark.parametrize("lanes", [(0, 4), (32, 33), (4,), 4, "32,4"])
def test_bad_lanes_raise_value_error(lanes):
    cfg, w = _small_weights()
    m = MCM(**SMALL)
    m.load_state_dict(w)
    with pytest.raises(ValueError, match="lanes"):
        m.compress_images(torch.rand(1, 3, 64, 64), torch.rand(1, cfg.num_patches), lanes=lanes)


def test_strings_that_cannot_be_containers_are_named():
    cfg, w = _small_weights()
    m = MCM(**SMALL)
    m.load_state_dict(w)
    good = R.pack(b"\0" * 8, b"\0" * 8, list(range(16)), FIELDS)
    with pytest.raises(ValueError, match=r"images \[1, 2\]"):
        m.decompress_images([good, good[:-1], b"\0" * 24])
    with pytest.raises(ValueError):
        m.decompress_images([])
    assert struct.unpack_from("<I", good)[0] == R.MAGIC
