"""GPU: the rANS coder (csrc/rans.cu) against the oracle's byte format, and MCM.compress_bitstream / decompress_bitstream
round trips that reproduce forward's latents bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import ref_rans as R
from tests import gpu_util as G
from textmae_image_compression_b200 import MCM, PathConfig, _native, entropy, make_state_dict, vit_base

pytestmark = pytest.mark.gpu

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16)
CONFIGS = {"small": (SMALL, 3), "vitB_K64": (dict(num_keep_patches=64), 2), "vitB_K144": (dict(num_keep_patches=144), 2)}
_SD = {}


def _model(key, precise=None, decoder=True, **flags):
    kw, _ = CONFIGS[key]
    cfg = vit_base(kw["num_keep_patches"]) if key.startswith("vitB") else PathConfig(**kw)
    if (key, decoder) not in _SD:
        _SD[(key, decoder)] = make_state_dict(cfg, seed=3, include_decoder=decoder)
    m = MCM(**kw, softmax_isa=16, precise=precise, **flags)
    m.load_state_dict(_SD[(key, decoder)])
    return cfg, m.cuda().eval()


def _inputs(cfg, n, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, 3, cfg.img_size, cfg.img_size, generator=g).cuda(),
            torch.rand(n, cfg.num_patches, generator=g).cuda())


def _coder_handle():
    cfg, m = _model("small", decoder=False)
    m._install_coder_tables()
    return m


def _gauss_case(rng, n_streams, n, escape_rate):
    tabs = R.gaussian_tables(MCM.get_scale_table())
    idx = rng.integers(0, 64, (n_streams, n))
    off, ln = tabs["_offset"].numpy()[idx], tabs["_cdf_length"].numpy()[idx]
    sym = off + (rng.random(idx.shape) * (ln - 2)).astype(np.int64)
    esc = rng.random(idx.shape) < escape_rate
    far = rng.integers(1, 1 << 20, idx.shape)
    sym = np.where(esc, np.where(rng.random(idx.shape) < 0.5, off - far, off + ln - 2 + far - 1), sym)
    if n >= 4:                                          # raw values near 2^31 in every stream
        sym[:, 1] = off[:, 1] - 2 ** 30
        sym[:, 2] = off[:, 2] + ln[:, 2] - 2 + 2 ** 30 - 1
    return tabs, sym.astype(np.int32), idx.astype(np.int32)


@pytest.mark.parametrize("n_streams,n,escape_rate", [(1, 1, 0.0), (3, 31, 0.1), (32, 33, 0.05), (65, 2048, 0.02),
                                                      (7, 2048, 0.9), (2, 1, 1.0)])
def test_encoder_bytes_equal_oracle_and_decoder_inverts(cuda_dev, n_streams, n, escape_rate):
    m = _coder_handle()
    rng = np.random.default_rng(n_streams * 1000 + n)
    tabs, sym, idx = _gauss_case(rng, n_streams, n, escape_rate)
    ref = [R.encode_with_indexes(sym[i], idx[i], tabs["_quantized_cdf"], tabs["_cdf_length"], tabs["_offset"]) for i in range(n_streams)]
    out, offs, st = entropy.encode(m._handle, _native.MODEL_GAUSSIAN, torch.from_numpy(sym).cuda(), torch.from_numpy(idx).cuda())
    torch.cuda.synchronize()
    offs = offs.cpu().tolist()
    assert st.cpu().eq(0).all()
    got = out.cpu().numpy().tobytes()
    for i in range(n_streams):
        assert got[offs[i]:offs[i + 1]] == ref[i], f"stream {i}"
    # the GPU decoder inverts the oracle's streams
    data, doffs = entropy.pack_strings(ref)
    dec, dst = entropy.decode(m._handle, _native.MODEL_GAUSSIAN, data.cuda(), doffs.cuda(), torch.from_numpy(idx).cuda())
    torch.cuda.synchronize()
    assert dst.cpu().eq(0).all()
    assert torch.equal(dec.cpu(), torch.from_numpy(sym))


def test_bottleneck_streams(cuda_dev):
    m = _coder_handle()
    tabs = m.entropy_tables()
    cdf, ln, off = (tabs["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset"))
    rng = np.random.default_rng(1)
    Cz, hw, N = cdf.shape[0], 4, 5
    idx = np.repeat(np.arange(Cz), hw)[None].repeat(N, 0).astype(np.int32)
    sym = (rng.normal(0, 6, idx.shape)).astype(np.int32)
    ref = [R.encode_with_indexes(sym[i], idx[i], cdf, ln, off) for i in range(N)]
    out, offs, st = entropy.encode(m._handle, _native.MODEL_BOTTLENECK, torch.from_numpy(sym).cuda(), torch.from_numpy(idx).cuda())
    offs = offs.cpu().tolist()
    got = out.cpu().numpy().tobytes()
    assert st.cpu().eq(0).all() and all(got[offs[i]:offs[i + 1]] == ref[i] for i in range(N))


def _check_round_trip(m, cfg, imgs, scores):
    enc = m.compress_bitstream(imgs, scores)
    fwd = m(imgs, scores)
    dec = m.decompress_bitstream(enc["strings"], enc["shape"], enc["ids_restore"])
    torch.cuda.synchronize()
    assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"])
    assert torch.equal(dec["z_hat"], fwd["latents"]["z_hat"])
    assert torch.equal(dec["x_hat"], fwd["x_hat"])
    return enc


@pytest.mark.parametrize("precise", [None, "all"])
@pytest.mark.parametrize("key", list(CONFIGS))
def test_bitstream_round_trip_is_bit_exact(cuda_dev, key, precise):
    cfg, m = _model(key, precise)
    imgs, scores = _inputs(cfg, CONFIGS[key][1])
    enc = _check_round_trip(m, cfg, imgs, scores)
    # the strings are the oracle's encoding of compress_symbols' output
    sym = m.compress_symbols(imgs, scores)
    t = m.entropy_tables()
    g = [t["gaussian_conditional." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    b = [t["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    ys, yi = sym["y_symbols"].cpu().numpy(), sym["y_indexes"].cpu().numpy()
    N = ys.shape[0]
    zs, zi = sym["z_symbols"].reshape(N, -1).cpu().numpy(), sym["z_indexes"].reshape(N, -1).cpu().numpy()
    for i in range(N):
        assert enc["strings"][0][i] == R.encode_with_indexes(ys[i], yi[i], *g)
        assert enc["strings"][1][i] == R.encode_with_indexes(zs[i], zi[i], *b)


def test_batch64_share_sm_encode_decodes_alone_and_in_halves(cuda_dev):
    cfg, enc_m = _model("vitB_K64", None, share_sm=True)
    _, dec_m = _model("vitB_K64", None)
    imgs, scores = _inputs(cfg, 64, seed=5)
    enc = enc_m.compress_bitstream(imgs, scores)
    fwd = enc_m(imgs, scores, need_recon=False)
    y, z = enc["strings"]
    one = dec_m.decompress_bitstream([[y[5]], [z[5]]], enc["shape"], enc["ids_restore"][5:6], need_recon=False)
    assert torch.equal(one["y_hat"], fwd["latents"]["y_hat"][5:6])
    for a, b in ((0, 32), (32, 64)):
        d = dec_m.decompress_bitstream([y[a:b], z[a:b]], enc["shape"], enc["ids_restore"][a:b], need_recon=False)
        assert torch.equal(d["y_hat"], fwd["latents"]["y_hat"][a:b])
        assert torch.equal(d["z_hat"], fwd["latents"]["z_hat"][a:b])


def test_oracle_decoder_through_decode_fn_agrees(cuda_dev):
    cfg, m = _model("small", None)
    imgs, scores = _inputs(cfg, 2, seed=2)
    enc = m.compress_bitstream(imgs, scores)
    t = m.entropy_tables()
    g = [t["gaussian_conditional." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    b = [t["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    N, s4 = 2, cfg.side // 4
    zi = np.repeat(np.arange(cfg.hyperprior_depth), s4 * s4)
    z_sym = torch.tensor([R.decode_with_indexes(enc["strings"][1][i], zi, *b) for i in range(N)], dtype=torch.int32)
    z_sym = z_sym.view(N, cfg.hyperprior_depth, s4, s4).cuda()
    decoded = [[] for _ in range(N)]          # the oracle decoder reads each y string group by group, as decode_stream would

    def decode_fn(first, indexes):
        ix = indexes.cpu().numpy().reshape(N, -1)
        out = []
        for i in range(N):
            decoded[i].extend(ix[i].tolist())
            full = R.decode_with_indexes(enc["strings"][0][i], np.asarray(decoded[i]), *g)
            out.append(full[-ix.shape[1]:])
        return torch.tensor(out, dtype=torch.int32).view(indexes.shape)

    a = m.decompress_symbols(z_sym, enc["ids_restore"], decode_fn=decode_fn)
    bb = m.decompress_bitstream(enc["strings"], enc["shape"], enc["ids_restore"])
    assert torch.equal(a["y_hat"], bb["y_hat"]) and torch.equal(a["x_hat"], bb["x_hat"])


def test_truncated_stream_names_the_image_and_the_rest_decodes(cuda_dev):
    cfg, m = _model("vitB_K64", None)
    imgs, scores = _inputs(cfg, 4, seed=7)
    enc = m.compress_bitstream(imgs, scores)
    fwd = m(imgs, scores, need_recon=False)
    y, z = [list(v) for v in enc["strings"]]
    y[2] = y[2][:-4]
    with pytest.raises(ValueError, match=r"\[2\]"):
        m.decompress_bitstream([y, z], enc["shape"], enc["ids_restore"], need_recon=False)
    # the status path does not disturb the other images: decode them with the bad one still in the batch, read y_hat directly
    data, offs = entropy.pack_strings(y)
    zdata, zoffs = entropy.pack_strings(z)
    N, c = 4, m.cfg
    y_hat = torch.empty((N, c.side, c.side, c.latent_depth), device="cuda")
    z_hat = torch.empty((N, c.side // 4, c.side // 4, c.hyperprior_depth), device="cuda")
    st = torch.empty(N, dtype=torch.int32, device="cuda")
    o = _native.TmaeOutputs()
    o.y_hat, o.z_hat = y_hat.data_ptr(), z_hat.data_ptr()
    d, dz, oy, oz = data.cuda(), zdata.cuda(), offs.cuda(), zoffs.cuda()
    _native.check(_native.load().tmae_decompress_streams(m._handle, G.ptr(d), G.ptr(oy), G.ptr(dz), G.ptr(oz), N, C.byref(o), G.ptr(st),
                                                         G.stream()), m._handle)
    torch.cuda.synchronize()
    assert st.cpu().tolist()[2] != 0 and [v for i, v in enumerate(st.cpu().tolist()) if i != 2] == [0, 0, 0]
    ref = fwd["latents"]["y_hat"].permute(0, 2, 3, 1)
    for i in (0, 1, 3):
        assert torch.equal(y_hat[i], ref[i])
    # malformed arguments
    with pytest.raises(ValueError):
        m.decompress_bitstream([y[:1], z[:1]], enc["shape"], enc["ids_restore"][:2], need_recon=False)
    with pytest.raises(ValueError):
        m.decompress_bitstream([[y[0][:6]], z[:1]], enc["shape"], enc["ids_restore"][:1], need_recon=False)
    with pytest.raises(ValueError):
        m.decompress_bitstream([y[:1], z[:1]], (3, 3), enc["ids_restore"][:1], need_recon=False)
    with pytest.raises(ValueError):
        m.decompress_bitstream([y[:2], z[:1]], enc["shape"], enc["ids_restore"][:2], need_recon=False)


def test_graph_replays_and_no_graph_agree(cuda_dev):
    cfg, m = _model("small", None)
    imgs, scores = _inputs(cfg, 3, seed=9)
    enc = m.compress_bitstream(imgs, scores)
    outs = [m.decompress_bitstream(enc["strings"], enc["shape"], enc["ids_restore"]) for _ in range(3)]   # plain, capture, replay
    for o in outs[1:]:
        for k in ("y_hat", "z_hat", "x_hat"):
            assert torch.equal(o[k], outs[0][k])
    code = ("import sys, torch; sys.path.insert(0, '.'); from tests.test_gpu_bitstream import _model, _inputs;"
            "cfg, m = _model('small', None); i, s = _inputs(cfg, 3, seed=9); e = m.compress_bitstream(i, s);"
            "d = m.decompress_bitstream(e['strings'], e['shape'], e['ids_restore']); torch.save({k: v.cpu() for k, v in d.items()}, sys.argv[1])")
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"nograph_{os.getpid()}.pt")
    env = dict(os.environ, TMAE_NO_GRAPH="1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-c", code, path], check=True, env=env, cwd=root)
    ng = torch.load(path)
    os.remove(path)
    for k in ("y_hat", "z_hat", "x_hat"):
        assert torch.equal(ng[k], outs[0][k].cpu())


def test_missing_or_mismatched_tables(cuda_dev):
    cfg, m = _model("small", None, decoder=False)
    imgs, scores = _inputs(cfg, 1)
    enc = m.compress_bitstream(imgs, scores)
    lib = _native.load()
    # a fresh handle without cdf tables
    _, fresh = _model("small", None, decoder=False)
    fresh._install_scale_table()
    data, offs = entropy.pack_strings(enc["strings"][0])
    d, o = data.cuda(), offs.cuda()
    st = torch.empty(1, dtype=torch.int32, device="cuda")
    out = _native.TmaeOutputs()
    assert lib.tmae_decompress_streams(fresh._handle, G.ptr(d), G.ptr(o), G.ptr(d), G.ptr(o), 1, C.byref(out), G.ptr(st), G.stream()) == _native.TMAE_ESTATE
    assert lib.tmae_rans_decode(fresh._handle, 0, G.ptr(d), G.ptr(o), 1, G.ptr(st), 1, G.ptr(st), G.ptr(st), G.stream()) == _native.TMAE_ESTATE
    # Gaussian set of another size than the scale table
    t = m.entropy_tables()
    small = {k: t["gaussian_conditional." + k][:10] for k in ("_quantized_cdf", "_cdf_length", "_offset")}
    entropy.set_tables(fresh._handle, _native.MODEL_GAUSSIAN, small)
    entropy.set_tables(fresh._handle, _native.MODEL_BOTTLENECK, {k: t["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")})
    assert lib.tmae_decompress_streams(fresh._handle, G.ptr(d), G.ptr(o), G.ptr(d), G.ptr(o), 1, C.byref(out), G.ptr(st), G.stream()) == _native.TMAE_ESTATE
    # invalid tables
    bad = {k: v.clone() for k, v in small.items()}
    bad["_quantized_cdf"][0, 2] = bad["_quantized_cdf"][0, 1]              # not strictly increasing
    with pytest.raises(ValueError):
        entropy.set_tables(fresh._handle, _native.MODEL_GAUSSIAN, bad)
    bad = {k: v.clone() for k, v in small.items()}
    bad["_cdf_length"][3] = 2
    with pytest.raises(ValueError):
        entropy.set_tables(fresh._handle, _native.MODEL_GAUSSIAN, bad)
    eb = {k: t["entropy_bottleneck." + k][:5] for k in ("_quantized_cdf", "_cdf_length", "_offset")}
    with pytest.raises(ValueError):                                           # one table per channel
        entropy.set_tables(fresh._handle, _native.MODEL_BOTTLENECK, eb)


def test_large_table_set_decodes_from_global_memory(cuda_dev):
    # 4 tables of 20,001 bins (320 KB): more than the decoder stages in shared memory, so it reads them from global memory
    cfg, m = _model("small", None, decoder=False)
    m._install_scale_table()                                       # creates the handle
    rng = np.random.default_rng(11)
    n_tab, bins = 4, 20001
    cdf = np.zeros((n_tab, bins + 2), dtype=np.int32)
    for t in range(n_tab):
        freq = 1 + rng.multinomial(65536 - (bins + 1), np.full(bins + 1, 1.0 / (bins + 1)))
        cdf[t, 1:] = np.cumsum(freq)
    tabs = {"_quantized_cdf": torch.from_numpy(cdf), "_cdf_length": torch.full((n_tab,), bins + 2, dtype=torch.int32),
            "_offset": torch.tensor([-10000, -5, 0, 7], dtype=torch.int32)}
    entropy.set_tables(m._handle, _native.MODEL_GAUSSIAN, tabs)
    n_streams, n = 5, 3000
    idx = rng.integers(0, n_tab, (n_streams, n)).astype(np.int32)
    off = tabs["_offset"].numpy()[idx]
    sym = (off + rng.integers(0, bins, idx.shape)).astype(np.int32)
    sym[:, ::97] += 30000                                          # a few escapes as well
    ref = [R.encode_with_indexes(sym[i], idx[i], *tabs.values()) for i in range(n_streams)]
    out, offs, st = entropy.encode(m._handle, _native.MODEL_GAUSSIAN, torch.from_numpy(sym).cuda(), torch.from_numpy(idx).cuda())
    offs = offs.cpu().tolist()
    got = out.cpu().numpy().tobytes()
    assert st.cpu().eq(0).all() and all(got[offs[i]:offs[i + 1]] == ref[i] for i in range(n_streams))
    data, doffs = entropy.pack_strings(ref)
    dec, dst = entropy.decode(m._handle, _native.MODEL_GAUSSIAN, data.cuda(), doffs.cuda(), torch.from_numpy(idx).cuda())
    torch.cuda.synchronize()
    assert dst.cpu().eq(0).all()
    assert torch.equal(dec.cpu(), torch.from_numpy(sym))
