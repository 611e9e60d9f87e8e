"""GPU: the laned rANS format (csrc/rans.cu) against the reference laned coder (tests/ref_rans_lanes.py), and
MCM.compress_bitstream / decompress_bitstream with lanes=(W_y, W_z) reproducing forward's latents bit for bit."""
import ctypes as C
import os
import struct
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import gpu_util as G
from tests import ref_rans_lanes as L
from tests.test_gpu_bitstream import CONFIGS, _coder_handle, _gauss_case, _inputs, _model
from textmae_image_compression_b200 import _native, entropy

pytestmark = pytest.mark.gpu

LANES = (32, 4)


def _tab_args(tabs):
    return tabs["_quantized_cdf"], tabs["_cdf_length"], tabs["_offset"]


def _check_gpu_matches_oracle(m, model, tabs, sym, idx, W):
    n_streams = sym.shape[0]
    ref = [L.encode_lanes(sym[i], idx[i], W, *_tab_args(tabs)) for i in range(n_streams)]
    out, offs, st = entropy.encode_lanes(m._handle, model, torch.from_numpy(sym).cuda(), torch.from_numpy(idx).cuda(), W)
    torch.cuda.synchronize()
    offs = offs.cpu().tolist()
    assert st.cpu().eq(0).all()
    got = out.cpu().numpy().tobytes()
    for i in range(n_streams):
        assert got[offs[i]:offs[i + 1]] == ref[i], f"stream {i}"
    data, doffs = entropy.pack_strings(ref)
    dec, dst = entropy.decode_lanes(m._handle, model, data.cuda(), doffs.cuda(), torch.from_numpy(idx).cuda(), W)
    torch.cuda.synchronize()
    assert dst.cpu().eq(0).all()
    assert torch.equal(dec.cpu(), torch.from_numpy(sym))


@pytest.mark.parametrize("n_streams,n,W,escape_rate", [(1, 1, 32, 0.0), (3, 31, 7, 0.1), (32, 33, 32, 0.05), (65, 2048, 32, 0.02),
                                                        (7, 2048, 5, 0.9), (2, 1, 1, 1.0), (4, 24576, 32, 0.02)])
def test_laned_bytes_equal_oracle_and_decoder_inverts(cuda_dev, n_streams, n, W, escape_rate):
    m = _coder_handle()
    tabs, sym, idx = _gauss_case(np.random.default_rng(n_streams * 1000 + n + W), n_streams, n, escape_rate)
    _check_gpu_matches_oracle(m, _native.MODEL_GAUSSIAN, tabs, sym, idx, W)


def test_laned_bottleneck_streams(cuda_dev):
    m = _coder_handle()
    t = m.entropy_tables()
    tabs = {k: t["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")}
    rng = np.random.default_rng(1)
    Cz, hw, N = tabs["_quantized_cdf"].shape[0], 4, 5
    idx = np.repeat(np.arange(Cz), hw)[None].repeat(N, 0).astype(np.int32)
    sym = rng.normal(0, 6, idx.shape).astype(np.int32)
    _check_gpu_matches_oracle(m, _native.MODEL_BOTTLENECK, tabs, sym, idx, 4)


def _laned_round_trip(m, imgs, scores, lanes=LANES):
    enc = m.compress_bitstream(imgs, scores, lanes=lanes)
    assert enc["lanes"] == lanes
    fwd = m(imgs, scores)
    dec = m.decompress_bitstream(enc["strings"], enc["shape"], enc["ids_restore"], lanes=lanes)
    torch.cuda.synchronize()
    assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"])
    assert torch.equal(dec["z_hat"], fwd["latents"]["z_hat"])
    assert torch.equal(dec["x_hat"], fwd["x_hat"])
    return enc


@pytest.mark.parametrize("precise", [None, "all"])
@pytest.mark.parametrize("key", list(CONFIGS))
def test_laned_bitstream_round_trip_is_bit_exact(cuda_dev, key, precise):
    cfg, m = _model(key, precise)
    imgs, scores = _inputs(cfg, CONFIGS[key][1])
    enc = _laned_round_trip(m, imgs, scores)
    sym = m.compress_symbols(imgs, scores)
    t = m.entropy_tables()
    g = [t["gaussian_conditional." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    b = [t["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    ys, yi = sym["y_symbols"].cpu().numpy(), sym["y_indexes"].cpu().numpy()
    N = ys.shape[0]
    zs, zi = sym["z_symbols"].reshape(N, -1).cpu().numpy(), sym["z_indexes"].reshape(N, -1).cpu().numpy()
    for i in range(N):
        assert enc["strings"][0][i] == L.encode_lanes(ys[i], yi[i], LANES[0], *g)
        assert enc["strings"][1][i] == L.encode_lanes(zs[i], zi[i], LANES[1], *b)


def test_laned_batch64_share_sm_encode_decodes_alone_and_in_halves(cuda_dev):
    cfg, enc_m = _model("vitB_K64", None, share_sm=True)
    _, dec_m = _model("vitB_K64", None)
    imgs, scores = _inputs(cfg, 64, seed=5)
    enc = enc_m.compress_bitstream(imgs, scores, lanes=LANES)
    fwd = enc_m(imgs, scores, need_recon=False)
    y, z = enc["strings"]
    one = dec_m.decompress_bitstream([[y[5]], [z[5]]], enc["shape"], enc["ids_restore"][5:6], need_recon=False, lanes=LANES)
    assert torch.equal(one["y_hat"], fwd["latents"]["y_hat"][5:6])
    for a, b in ((0, 32), (32, 64)):
        d = dec_m.decompress_bitstream([y[a:b], z[a:b]], enc["shape"], enc["ids_restore"][a:b], need_recon=False, lanes=LANES)
        assert torch.equal(d["y_hat"], fwd["latents"]["y_hat"][a:b])
        assert torch.equal(d["z_hat"], fwd["latents"]["z_hat"][a:b])


def _set_lane_len(s, lane, delta):
    b = bytearray(s)
    old = struct.unpack_from("<I", b, 4 * (1 + lane))[0]
    struct.pack_into("<I", b, 4 * (1 + lane), old + delta)
    return bytes(b)


def test_malformed_laned_streams_name_the_image_and_the_rest_decodes(cuda_dev):
    cfg, m = _model("vitB_K64", None)
    imgs, scores = _inputs(cfg, 4, seed=7)
    enc = m.compress_bitstream(imgs, scores, lanes=LANES)
    fwd = m(imgs, scores, need_recon=False)
    y0, z0 = [list(v) for v in enc["strings"]]
    W = LANES[0]
    truncated = _set_lane_len(y0[1][:-4], W - 1, -4)                  # the last lane one word short, the header consistent
    other_w = struct.pack("<I", 16) + y0[1][4:]                           # a header with another W
    not_sum = _set_lane_len(y0[1], 3, 4)                              # lane lengths that do not add up
    ref = fwd["latents"]["y_hat"].permute(0, 2, 3, 1)
    for bad in (truncated, other_w, not_sum):
        y = list(y0)
        y[1] = bad
        with pytest.raises(ValueError, match=r"\[1\]"):
            m.decompress_bitstream([y, z0], enc["shape"], enc["ids_restore"], need_recon=False, lanes=LANES)
        # through the ABI status the other images of the batch still decode bit-exactly
        data, offs = entropy.pack_strings(y)
        zdata, zoffs = entropy.pack_strings(z0)
        N, c = 4, m.cfg
        y_hat = torch.empty((N, c.side, c.side, c.latent_depth), device="cuda")
        z_hat = torch.empty((N, c.side // 4, c.side // 4, c.hyperprior_depth), device="cuda")
        st = torch.empty(N, dtype=torch.int32, device="cuda")
        o = _native.TmaeOutputs()
        o.y_hat, o.z_hat = y_hat.data_ptr(), z_hat.data_ptr()
        d, dz, oy, oz = data.cuda(), zdata.cuda(), offs.cuda(), zoffs.cuda()
        _native.check(_native.load().tmae_decompress_streams_lanes(m._handle, G.ptr(d), G.ptr(oy), LANES[0], G.ptr(dz), G.ptr(oz),
                                                                   LANES[1], N, C.byref(o), G.ptr(st), G.stream()), m._handle)
        torch.cuda.synchronize()
        s = st.cpu().tolist()
        assert s[1] != 0 and [v for i, v in enumerate(s) if i != 1] == [0, 0, 0]
        for i in (0, 2, 3):
            assert torch.equal(y_hat[i], ref[i])
    # a string shorter than the format's minimum for that W
    with pytest.raises(ValueError, match=">= 388"):
        m.decompress_bitstream([[b"\0" * 384], z0[:1]], enc["shape"], enc["ids_restore"][:1], need_recon=False, lanes=LANES)


def test_laned_graph_replays_no_graph_and_plan_keys_agree(cuda_dev):
    cfg, m = _model("small", None)
    imgs, scores = _inputs(cfg, 3, seed=9)
    enc = m.compress_bitstream(imgs, scores, lanes=LANES)
    outs = [m.decompress_bitstream(enc["strings"], enc["shape"], enc["ids_restore"], lanes=LANES) for _ in range(3)]
    for o in outs[1:]:
        for k in ("y_hat", "z_hat", "x_hat"):
            assert torch.equal(o[k], outs[0][k])
    # one handle, one N: compressai-format and laned decodes alternate, each replaying its own plan
    plain = m.compress_bitstream(imgs, scores)
    other = m.compress_bitstream(imgs, scores, lanes=(5, 1))
    for _ in range(2):
        for e, lanes in ((plain, None), (enc, LANES), (other, (5, 1))):
            d = m.decompress_bitstream(e["strings"], e["shape"], e["ids_restore"], lanes=lanes)
            for k in ("y_hat", "z_hat", "x_hat"):
                assert torch.equal(d[k], outs[0][k]), (lanes, k)
    code = ("import sys, torch; sys.path.insert(0, '.'); from tests.test_gpu_bitstream import _model, _inputs;"
            "cfg, m = _model('small', None); i, s = _inputs(cfg, 3, seed=9); e = m.compress_bitstream(i, s, lanes=(32, 4));"
            "d = m.decompress_bitstream(e['strings'], e['shape'], e['ids_restore'], lanes=(32, 4));"
            "torch.save({k: v.cpu() for k, v in d.items()}, sys.argv[1])")
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"nograph_lanes_{os.getpid()}.pt")
    env = dict(os.environ, TMAE_NO_GRAPH="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-c", code, path], check=True, env=env, cwd=root)
    ng = torch.load(path)
    os.remove(path)
    for k in ("y_hat", "z_hat", "x_hat"):
        assert torch.equal(ng[k], outs[0][k].cpu())


def test_laned_large_table_set_decodes_from_global_memory(cuda_dev):
    # 4 tables of 20,001 bins (320 KB): more than the decoder stages in shared memory, so it reads them from global memory
    cfg, m = _model("small", None, decoder=False)
    m._install_scale_table()
    rng = np.random.default_rng(11)
    n_tab, bins = 4, 20001
    cdf = np.zeros((n_tab, bins + 2), dtype=np.int32)
    for t in range(n_tab):
        freq = 1 + rng.multinomial(65536 - (bins + 1), np.full(bins + 1, 1.0 / (bins + 1)))
        cdf[t, 1:] = np.cumsum(freq)
    tabs = {"_quantized_cdf": torch.from_numpy(cdf), "_cdf_length": torch.full((n_tab,), bins + 2, dtype=torch.int32),
            "_offset": torch.tensor([-10000, -5, 0, 7], dtype=torch.int32)}
    entropy.set_tables(m._handle, _native.MODEL_GAUSSIAN, tabs)
    idx = rng.integers(0, n_tab, (5, 3000)).astype(np.int32)
    sym = (tabs["_offset"].numpy()[idx] + rng.integers(0, bins, idx.shape)).astype(np.int32)
    sym[:, ::97] += 30000
    _check_gpu_matches_oracle(m, _native.MODEL_GAUSSIAN, tabs, sym, idx, 32)


def test_laned_calls_need_tables(cuda_dev):
    _, fresh = _model("small", None, decoder=False)
    fresh._install_scale_table()
    lib = _native.load()
    buf = torch.zeros(64, dtype=torch.int64, device="cuda")
    p = G.ptr(buf)
    out = _native.TmaeOutputs()
    E = _native.TMAE_ESTATE
    assert lib.tmae_rans_encode_lanes(fresh._handle, 0, p, p, 1, 1, 4, p, 512, p, p, G.stream()) == E
    assert lib.tmae_rans_decode_lanes(fresh._handle, 0, p, p, 1, p, 1, 4, p, p, G.stream()) == E
    assert lib.tmae_decompress_streams_lanes(fresh._handle, p, p, 32, p, p, 4, 1, C.byref(out), p, G.stream()) == E
    # bad lanes on a live handle: EINVAL before the table check
    assert lib.tmae_rans_decode_lanes(fresh._handle, 0, p, p, 1, p, 1, 33, p, p, G.stream()) == _native.TMAE_EINVAL
