"""GPU: pictures of any size (MCM.compress_pictures / decompress_pictures, csrc/picture.cu).  The tiling kernels equal tiling.py bit
for bit; a picture container equals the reference packing of compress_images' tile containers (tiles from tiling.tile_image, scores
from the tiles' grey pixels); x_hat decodes from the bytes alone to forward's x_hat of the tiles, untiled; plans of equal tile
counts never mix; a bad picture is refused alone."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ref_mask
from tests import ref_picture_container as R
from tests.test_gpu_bitstream import _model
from textmae_image_compression_b200 import _native, entropy, tiling
from textmae_image_compression_b200.scores import generate_scores

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "kodak_gray6.npz")


def _kodak_greys():
    z = np.load(GOLDEN)
    return [torch.from_numpy(np.ascontiguousarray(z[k])) for k in sorted(z.files)]


def _grey_pictures():
    """The six Kodak greys at native size as grey RGB pictures: x = g / 255 on all three channels."""
    greys = _kodak_greys()
    return [(g.float() / 255).expand(3, -1, -1).contiguous() for g in greys], greys


def _tiles_op(x, gray, S):
    P, _, H, W = x.shape
    T = R.tile_count(H, W, S)
    tiles = torch.empty((P * T, 3, S, S), dtype=torch.float32, device=x.device)
    gt = torch.empty((P * T, S, S), dtype=torch.uint8, device=x.device)
    rc = _native.load().tmae_picture_tiles(C.c_void_p(x.data_ptr()), C.c_void_p(gray.data_ptr()) if gray is not None else None,
                                           P, H, W, S, C.c_void_p(tiles.data_ptr()), C.c_void_p(gt.data_ptr()), None)
    assert rc == 0
    return tiles, gt


def _untile_op(tiles, P, H, W):
    S = tiles.shape[-1]
    canvas = torch.empty((P, 3, H, W), dtype=torch.float32, device=tiles.device)
    assert _native.load().tmae_picture_untile(C.c_void_p(tiles.data_ptr()), P, H, W, S, C.c_void_p(canvas.data_ptr()), None) == 0
    return canvas


def _cv_gray(x):
    """cv2.cvtColor(RGB2GRAY) of the 8-bit pixels, in integer arithmetic (OpenCV's fixed-point weights)."""
    v = (x.double() * 255).float().round().clamp(0, 255).to(torch.int64)      # fp32 product, rint, saturate
    return ((9798 * v[:, 0] + 19235 * v[:, 1] + 3735 * v[:, 2] + 16384) >> 15).to(torch.uint8)


SHAPES = [(512, 768, 224), (768, 512, 224), (224, 224, 224), (225, 223, 224), (1, 1, 224), (100, 60, 224), (1080, 2048, 512)]


@pytest.mark.parametrize("P", [1, 3])
@pytest.mark.parametrize("H,W,S", SHAPES)
def test_tiles_and_untile_equal_tiling_py(cuda_dev, H, W, S, P):
    g = torch.Generator().manual_seed(H * 7 + W + P)
    x = torch.rand(P, 3, H, W, generator=g)
    x[:, :, : H // 3, : W // 4] = 1.0                 # saturated and exact-half pixels
    x[:, 1, -1, -1] = 0.5 / 255
    gray = torch.randint(0, 256, (P, H, W), generator=g, dtype=torch.uint8)
    xd, gd = x.cuda(), gray.cuda()
    tiles, gt = _tiles_op(xd, gd, S)
    assert torch.equal(tiles.cpu(), tiling.tile_image(x, S))
    assert torch.equal(gt.cpu(), tiling.tile_image(gray[:, None], S)[:, 0])
    _, gt_rgb = _tiles_op(xd, None, S)
    assert torch.equal(gt_rgb.cpu(), tiling.tile_image(_cv_gray(x)[:, None], S)[:, 0])
    canvas = _untile_op(tiles, P, H, W)
    T = R.tile_count(H, W, S)
    want = torch.stack([tiling.untile_image(tiling.tile_image(x, S)[p * T:(p + 1) * T], H, W) for p in range(P)])
    assert torch.equal(canvas.cpu(), want) and torch.equal(want, x)


def test_rgb2gray_formula_matches_opencv(cuda_dev):
    cv2 = pytest.importorskip("cv2")
    g = torch.Generator().manual_seed(5)
    x = torch.rand(1, 3, 97, 131, generator=g)
    u8 = (x * 255).round().clamp(0, 255).to(torch.uint8)[0].permute(1, 2, 0).contiguous().numpy()
    want = torch.from_numpy(cv2.cvtColor(u8, cv2.COLOR_RGB2GRAY))
    _, gt = _tiles_op(x.cuda(), None, 224)
    assert torch.equal(gt.cpu()[0, :97, :131], want)


def _reference_pictures(m, pictures, greys, lanes):
    """compress_images of tiling.tile_image(x) with the scores of tiling.tile_image(g), one call per size, packed per picture."""
    S = m.cfg.img_size
    out = [None] * len(pictures)
    groups = {}
    for i, x in enumerate(pictures):
        groups.setdefault(tuple(x.shape[1:]), []).append(i)
    for (H, W), idx in groups.items():
        T = R.tile_count(H, W, S)
        x = torch.stack([pictures[i] for i in idx]).cuda()
        g = torch.stack([greys[i] for i in idx]).cuda()
        tiles = tiling.tile_image(x, S)
        scores = generate_scores(tiling.tile_image(g[:, None], S)[:, 0].contiguous(), S)
        cont = m.compress_images(tiles, scores, lanes=lanes)
        for k, i in enumerate(idx):
            out[i] = R.pack(cont[k * T:(k + 1) * T], H, W)
    return out


@pytest.mark.parametrize("lanes", [(32, 4), None])
@pytest.mark.parametrize("precise", [None, "all"])
def test_pictures_equal_reference_packing(cuda_dev, precise, lanes):
    cfg, m = _model("vitB_K144", precise, decoder=False)
    pictures, greys = _grey_pictures()
    got = m.compress_pictures(pictures, gray=greys, lanes=lanes)
    assert got == _reference_pictures(m, pictures, greys, lanes)
    # the grey of a grey RGB picture is the grey itself: gray=None codes the same bytes
    assert m.compress_pictures(pictures, lanes=lanes) == got
    for b, x in zip(got, pictures):
        H, W = x.shape[1:]
        f = R.parse_all(b, H, W, 224)
        assert f["T"] == 12 and all(t["img_size"] == 224 and t["K"] == 144 for t in f["tile_fields"])
        assert entropy.picture_geometry(b) == (H, W, 12, *(lanes or (0, 0)))
        assert len(b) <= entropy.pictures_bound(m._handle, 1, H, W, *(lanes or (0, 0)))


def _forward_x_hat(m, pictures, greys=None):
    """untile_image of forward's x_hat of the tiles (one forward per size, as compress_pictures batches them)."""
    S = m.cfg.img_size
    out = [None] * len(pictures)
    groups = {}
    for i, x in enumerate(pictures):
        groups.setdefault(tuple(x.shape[1:]), []).append(i)
    fwds = {}
    for (H, W), idx in groups.items():
        T = R.tile_count(H, W, S)
        x = torch.stack([pictures[i] for i in idx]).cuda()
        g = torch.stack([greys[i] for i in idx]).cuda() if greys is not None else _cv_gray(x.cpu()).cuda()
        fwd = m(tiling.tile_image(x, S), generate_scores(tiling.tile_image(g[:, None], S)[:, 0].contiguous(), S), need_recon=True)
        fwds[(H, W)] = fwd
        for k, i in enumerate(idx):
            out[i] = tiling.untile_image(fwd["x_hat"][k * T:(k + 1) * T], H, W)
    return out, fwds


def _raw_decode(m, b, H, W, lanes):
    """tmae_decompress_pictures of one picture with tile_out: (status, tile y_hat [T, s, s, Cy], ids_keep [T, K])."""
    c = m.cfg
    T = R.tile_count(H, W, c.img_size)
    data, off = entropy.pack_strings([b])
    data, off = data.cuda(), off.cuda()
    y_hat = torch.empty((T, c.side, c.side, c.latent_depth), dtype=torch.float32, device="cuda")
    ids_keep = torch.empty((T, c.num_keep_patches), dtype=torch.int64, device="cuda")
    status = torch.empty(1, dtype=torch.int32, device="cuda")
    o = _native.TmaeOutputs()
    o.y_hat, o.ids_keep = y_hat.data_ptr(), ids_keep.data_ptr()
    _native.check(_native.load().tmae_decompress_pictures(m._handle, C.c_void_p(data.data_ptr()), data.numel(),
                                                          C.c_void_p(off.data_ptr()), 1, H, W, *lanes, C.byref(o), None, None,
                                                          C.c_void_p(status.data_ptr()), None), m._handle)
    torch.cuda.synchronize()
    return int(status.item()), y_hat, ids_keep


@pytest.mark.parametrize("native", [True, False])
def test_round_trip_x_hat_is_forwards(cuda_dev, native):
    cfg, m = _model("vitB_K144", None, native_synthesis=native)
    pictures, greys = _grey_pictures()
    strings = m.compress_pictures(pictures, gray=greys)
    got = m.decompress_pictures(strings)
    want, fwds = _forward_x_hat(m, pictures, greys)
    for i, (a, b) in enumerate(zip(got, want)):
        assert a.shape == pictures[i].shape and torch.equal(a, b), f"picture {i}"
    status, y_hat, ids_keep = _raw_decode(m, strings[3], 768, 512, (32, 4))      # the one 768 x 512 picture: 12 tiles
    assert status == 0
    assert torch.equal(y_hat, fwds[(768, 512)]["latents"]["y_hat"].permute(0, 2, 3, 1))
    assert torch.equal(ids_keep, fwds[(768, 512)]["ids_keep"])


@pytest.mark.parametrize("P", [24, 1])
def test_scale_288_tiles(cuda_dev, P):
    cfg, m = _model("vitB_K144", None, native_synthesis=True)
    g = torch.Generator().manual_seed(P)
    x = torch.rand(P, 3, 512, 768, generator=g)
    strings = m.compress_pictures(x)
    got = m.decompress_pictures(strings)
    want, _ = _forward_x_hat(m, list(x))
    assert all(torch.equal(a, b) for a, b in zip(got, want))


def test_flat_tile_scores_are_nan_and_mask_like_the_oracle(cuda_dev):
    cfg, m = _model("vitB_K144", None, native_synthesis=True)
    g = torch.Generator().manual_seed(9)
    x = torch.rand(1, 3, 448, 300, generator=g)
    x[:, :, :224, :224] = 1.0                         # tile 0 is flat white: every patch scores 0/0
    gray = _cv_gray(x).cuda()
    scores = generate_scores(tiling.tile_image(gray[:, None], 224)[:, 0].contiguous(), 224)
    assert torch.isnan(scores[0]).all() and not torch.isnan(scores[1:]).any()
    oracle = ref_mask.mask_oracle_c(scores.cpu(), 144, isa=16)
    assert oracle[0].tolist() == list(range(196))
    assert torch.equal(m.get_ids_shuffle(scores).cpu(), oracle)
    strings = m.compress_pictures(x)
    assert strings == _reference_pictures(m, list(x), list(gray.cpu()), (32, 4))
    status, _, ids_keep = _raw_decode(m, strings[0], 448, 300, (32, 4))
    assert status == 0
    assert torch.equal(ids_keep.cpu(), oracle[:, :144])
    got = m.decompress_pictures(strings)
    want, _ = _forward_x_hat(m, list(x))
    assert torch.equal(got[0], want[0])


def _plan_cases():
    g = torch.Generator().manual_seed(11)
    return [torch.rand(2, 3, 448, 448, generator=g), torch.rand(1, 3, 896, 448, generator=g), torch.rand(1, 3, 300, 700, generator=g)]


def test_plans_of_equal_tile_counts_never_mix(cuda_dev):
    cases = _plan_cases()
    fresh = []
    for x in cases:                                   # every shape on a handle of its own
        _, f = _model("vitB_K64", None, native_synthesis=True)
        s = f.compress_pictures(x)
        fresh.append((s, f.decompress_pictures(s)))
        del f
    _, m = _model("vitB_K64", None, native_synthesis=True)
    for _ in range(3):                                # plain launches, capture, replay; the shapes alternate
        for x, (s0, d0) in zip(cases, fresh):
            s = m.compress_pictures(x)
            assert s == s0
            d = m.decompress_pictures(s)
            assert all(torch.equal(a, b) for a, b in zip(d, d0))
    code = ("import sys, torch; from tests.test_gpu_bitstream import _model; from tests.test_gpu_pictures import _plan_cases\n"
            "_, m = _model('vitB_K64', None, native_synthesis=True)\n"
            "out = []\n"
            "for x in _plan_cases():\n"
            "    s = m.compress_pictures(x); out.append((s, [t.cpu() for t in m.decompress_pictures(s)]))\n"
            "torch.save(out, sys.argv[1])")
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"nograph_pictures_{os.getpid()}.pt")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-c", code, path], check=True, env=dict(os.environ, TMAE_NO_GRAPH="1"), cwd=root)
    ng = torch.load(path, weights_only=False)
    os.remove(path)
    for (s, d), (s0, d0) in zip(ng, fresh):
        assert s == s0 and all(torch.equal(a, b.cpu()) for a, b in zip(d, d0))


def test_defects_are_refused_one_by_one(cuda_dev):
    cfg, m = _model("small", None, native_synthesis=True)
    S = cfg.img_size
    g = torch.Generator().manual_seed(4)
    x = torch.rand(5, 3, 100, 150, generator=g)       # 2 x 3 tiles of 64
    good = m.compress_pictures(x)
    want, _ = _forward_x_hat(m, [x[0]])
    T = 6
    bad_magic = b"XMAP" + good[1][4:]
    f = R.parse(good[2])
    short = R.pack(f["tiles"], 100, 150)
    short = short[:16] + (int.from_bytes(short[16:20], "little") + 4).to_bytes(4, "little") + short[20:]
    other_hw = m.compress_pictures(torch.rand(1, 3, 100, 140, generator=g))[0]     # same tile count, other H x W
    f4 = R.parse(good[4])
    t3 = bytearray(f4["tiles"][3])
    t3[16] ^= 1                                       # word 4 of the tile container: the model tag
    flipped = R.pack(f4["tiles"][:3] + [bytes(t3)] + f4["tiles"][4:], 100, 150)
    strings = [good[0], bad_magic, short, other_hw, flipped]
    # the statuses of one call: picture header (and with it every tile's container header), the model bit of tile 3
    data, off = entropy.pack_strings(strings)
    data, off = data.cuda(), off.cuda()
    status = torch.empty(5, dtype=torch.int32, device="cuda")
    canvas = torch.empty((5, 3, 100, 150), dtype=torch.float32, device="cuda")
    _native.check(_native.load().tmae_decompress_pictures(m._handle, C.c_void_p(data.data_ptr()), data.numel(),
                                                          C.c_void_p(off.data_ptr()), 5, 100, 150, 32, 4, None, None,
                                                          C.c_void_p(canvas.data_ptr()), C.c_void_p(status.data_ptr()), None),
                  m._handle)
    # a refused tile container hands the decoders empty ranges, which they report as streams that do not decode
    empty = _native.RANS_OVERRUN | _native.RANS_UNFINISHED | _native.RANS_MALFORMED
    hdr = _native.PIC_HEADER | _native.IMG_HEADER | empty
    assert status.tolist() == [0, hdr, hdr, hdr, _native.IMG_MODEL | empty]
    assert torch.equal(canvas[0], want[0])
    with pytest.raises(ValueError) as e:
        m.decompress_pictures(strings)
    msg = str(e.value)                              # the Python call groups by each picture's own geometry: picture 3 decodes
    assert "pictures [1, 2, 4]" in msg and f"picture 4: model (status {_native.IMG_MODEL | empty}), tiles [3]" in msg
    assert "picture 1: header: not a picture container" in msg
    assert f"picture 2: picture header, header (status {hdr}), tiles all" in msg
    assert m.decompress_pictures([other_hw])[0].shape == (3, 100, 140)
    assert T == f["T"]
