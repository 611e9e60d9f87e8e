"""CPU: the picture container (DESIGN.md section 7, "The picture container") through its plain-Python reference
(tests/ref_picture_container.py), the host-only picture calls of the C ABI, their argument checks, and the picture methods of MCM
without a GPU."""
import ctypes as C
import struct

import pytest
import torch

from tests import ref_image_container as I
from tests import ref_picture_container as R
from textmae_image_compression_b200 import MCM, _native, entropy, tiling
from tests.test_image_container_cpu import FIELDS, SMALL, _small_weights


def _tile(k, img_size=64, y_lanes=32, z_lanes=4):
    return I.pack(b"\x01\x02\x03\x04" * (k + 2), b"\xaa\xbb\xcc\xdd" * (k + 1), list(range(16)),
                  dict(FIELDS, img_size=img_size, y_lanes=y_lanes, z_lanes=z_lanes))


def _picture(H, W, img_size=64, **kw):
    return R.pack([_tile(k, img_size, **kw) for k in range(R.tile_count(H, W, img_size))], H, W)


def test_hand_written_picture_is_pinned_byte_for_byte():
    a, b = _tile(0), _tile(1)
    got = R.pack([a, b], 50, 100)
    want = bytes.fromhex("544d4150" "01000000" "32006400" "02000000") + struct.pack("<2I", len(a), len(b)) + a + b
    assert got == want
    f = R.parse_all(got, 50, 100, 64)
    assert (f["H"], f["W"], f["T"], f["tiles"]) == (50, 100, 2, [a, b])
    assert f["tile_fields"][1]["y"] == b"\x01\x02\x03\x04" * 3


@pytest.mark.parametrize("H,W,S,T", [(512, 768, 224, 12), (768, 512, 224, 12), (224, 224, 224, 1), (225, 223, 224, 2),
                                     (1, 1, 224, 1), (100, 60, 224, 1), (1080, 2048, 512, 12), (448, 448, 224, 4),
                                     (896, 448, 224, 8)])
def test_tile_counts_follow_the_tiling_policy(H, W, S, T):
    rows, cols = tiling.tile_grid(H, W, S)
    assert R.tile_count(H, W, S) == rows * cols == T


@pytest.mark.parametrize("seed", range(3))
def test_round_trips_through_the_reference(seed):
    g = torch.Generator().manual_seed(seed)
    for H, W in ((64, 64), (65, 63), (1, 200), (130, 129)):
        T = R.tile_count(H, W, 64)
        tiles = [bytes(torch.randint(0, 256, (4 * int(torch.randint(7, 20, (1,), generator=g)),), generator=g).tolist())
                 for _ in range(T)]
        data = R.pack(tiles, H, W)
        assert len(data) == 4 * (4 + T) + sum(map(len, tiles))
        f = R.parse(data, H, W, 64)
        assert (f["H"], f["W"], f["T"], f["tiles"]) == (H, W, T, tiles)


def test_reference_parse_refuses_every_header_condition():
    good = _picture(100, 130)                       # 2 x 3 tiles of 64
    T = 6
    R.parse(good, 100, 130, 64)
    bad = {
        "magic": b"XMAP" + good[4:],
        "version": good[:4] + b"\x02" + good[5:],
        "reserved": good[:5] + b"\x01" + good[6:],
        "height": good[:8] + struct.pack("<I", 101 | 130 << 16) + good[12:],
        "tile count": good[:12] + struct.pack("<I", 5) + good[16:],
        "length not a multiple of 4": good[:16] + struct.pack("<I", struct.unpack_from("<I", good, 16)[0] + 1) + good[20:],
        "lengths short of the picture": good + b"\0\0\0\0",
        "lengths past the picture": good[:-4],
        "table past the picture": good[:12] + struct.pack("<I", 10 ** 6) + good[16:],
        "not words": good[:-1],
        "too short": good[:12],
    }
    for why, data in bad.items():
        with pytest.raises(ValueError, match="picture header"):
            R.parse(data, 100, 130, 64)
    with pytest.raises(ValueError, match="picture header"):
        R.parse(good, 100, 131, 64)               # the call's geometry differs
    assert T == R.parse(good)["T"]


def test_picture_calls_are_declared():
    header = (_native._PKG.parent / "include" / "tmae.h").read_text()
    for name in ("tmae_picture_tiles", "tmae_picture_untile", "tmae_picture_geometry", "tmae_compress_pictures",
                 "tmae_decompress_pictures"):
        assert name in _native.SIGNATURES and f"TMAE_API int  {name}(" in header
    assert "tmae_pictures_bound" in _native.SIGNATURES and "TMAE_API int64_t tmae_pictures_bound(" in header
    assert _native.PIC_HEADER == 1024 and "#define TMAE_PIC_HEADER         1024" in header
    assert entropy.image_status_reason(_native.PIC_HEADER | _native.IMG_HEADER) == "picture header, header"


def test_picture_geometry_reads_good_bytes():
    for H, W, lanes in ((100, 130, (32, 4)), (1, 1, (0, 0)), (64, 65, (1, 32))):
        data = _picture(H, W, y_lanes=lanes[0], z_lanes=lanes[1])
        assert entropy.picture_geometry(data) == (H, W, R.tile_count(H, W, 64), *lanes)
    vals = [C.c_int(0) for _ in range(5)]
    data = _picture(100, 130)
    assert _native.load().tmae_picture_geometry(data, len(data), *[C.byref(v) for v in vals]) == 0
    assert _native.load().tmae_picture_geometry(data, len(data), None, None, None, None, None) == 0


def test_picture_geometry_refuses_bad_bytes():
    good = _picture(100, 130)
    first = 4 * (4 + 6)
    bad = [b"", good[:12], good[:-1], b"XMAP" + good[4:], good[:4] + b"\x02" + good[5:],
           good[:8] + struct.pack("<I", 0 | 130 << 16) + good[12:],              # H = 0
           good[:8] + struct.pack("<I", 100) + good[12:],                         # W = 0
           good[:12] + struct.pack("<I", 5) + good[16:],                          # T other than the grid of the tile size
           good[:12] + struct.pack("<I", 0) + good[16:],                          # T = 0
           good[:first] + b"XMAE" + good[first + 4:],                             # first tile not an image container
           good[:first + 4],                                                      # first tile cut short
           R.pack([], 100, 130)]
    for data in bad:
        assert entropy.picture_geometry(data) is None
        assert _native.load().tmae_picture_geometry(data if data else None, len(data), None, None, None, None, None) == \
            _native.TMAE_EINVAL
    assert _native.load().tmae_picture_geometry(None, 64, None, None, None, None, None) == _native.TMAE_EINVAL


def test_pictures_bound_rejects_bad_arguments():
    lib = _native.load()
    for P, H, W, yl, zl in ((1, 64, 64, 32, 4), (0, 64, 64, 32, 4), (1, 0, 64, 0, 0), (1, 64, 65536, 0, 0),
                            (1, 64, 64, 33, 4), (1, 64, 64, 0, -1)):
        assert lib.tmae_pictures_bound(None, P, H, W, yl, zl) == -1


def test_picture_abi_rejects_bad_arguments_without_a_gpu():
    lib = _native.load()
    E = _native.TMAE_EINVAL
    p = C.c_void_p(64)                               # never dereferenced: every call below fails its checks first
    for lanes in ((0, 0), (32, 4), (33, 4)):
        assert lib.tmae_compress_pictures(None, p, None, 1, 64, 64, *lanes, p, 0, p, p, None) == E
        assert lib.tmae_decompress_pictures(None, p, 0, p, 1, 64, 64, *lanes, None, None, None, p, None) == E
    # stand-alone operators: null pointers, P < 1, H / W / tile outside 1..65535
    for args in ((None, None, 1, 64, 64, 64, p, p), (p, None, 0, 64, 64, 64, p, p), (p, None, 1, 0, 64, 64, p, p),
                 (p, None, 1, 64, 65536, 64, p, p), (p, None, 1, 64, 64, 0, p, p)):
        assert lib.tmae_picture_tiles(*args, None) == E
    for args in ((None, 1, 64, 64, 64, p), (p, 1, 64, 64, 64, None), (p, 0, 64, 64, 64, p), (p, 1, 65536, 64, 64, p),
                 (p, 1, 64, 0, 64, p), (p, 1, 64, 64, -1, p)):
        assert lib.tmae_picture_untile(*args, None) == E


def test_picture_methods_are_cuda_only():
    cfg, w = _small_weights()
    m = MCM(**SMALL)
    m.load_state_dict(w)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.compress_pictures([torch.rand(3, 70, 90)])
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.decompress_pictures([_picture(70, 90)])


def test_decompress_pictures_needs_the_decoder_weights():
    from textmae_image_compression_b200 import PathConfig, make_state_dict
    m = MCM(**SMALL)
    m.load_state_dict(make_state_dict(PathConfig(**SMALL), seed=3, include_decoder=False))
    with pytest.raises(RuntimeError, match="decoder"):
        m.decompress_pictures([_picture(70, 90)])


@pytest.mark.parametrize("lanes", [(0, 4), (32, 33), (4,), 4])
def test_bad_lanes_raise_value_error(lanes):
    cfg, w = _small_weights()
    m = MCM(**SMALL)
    m.load_state_dict(w)
    with pytest.raises(ValueError, match="lanes"):
        m.compress_pictures([torch.rand(3, 70, 90)], lanes=lanes)
