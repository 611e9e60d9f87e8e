"""GPU: synthesis on the engine (tmae_synthesize: g_s, the MAE decoder and unpatchify; MCM(native_synthesis=True)) against
recon.synthesize in fp32 torch, its head-dim-32 attention, batch invariance, graph replay, the end-to-end decodes and the
error paths.  Synthesis runs bf16 operands with fp32 accumulation; a CPU emulation of that arithmetic lands at a relative L2
of about 5e-3 against fp32 (ViT-B/16, K = 64 and 144), so 1.5e-2 leaves room for accumulation order and nothing more."""
import ctypes as C

import pytest
import torch

from tests import gpu_util as G
from textmae_image_compression_b200 import MCM, PathConfig, _native, make_state_dict, recon

pytestmark = pytest.mark.gpu

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16,
             decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=2)
# the refexec "mid" geometry; its golden decoder has head dim 64, so synthesis (head dim 32 only) runs it with 4 heads
MID4 = dict(img_size=128, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=64,
            decoder_embed_dim=128, decoder_depth=2, decoder_num_heads=4)
VITL = dict(img_size=512, encoder_embed_dim=1024, encoder_depth=24, encoder_num_heads=16, num_keep_patches=256)
CONFIGS = {"small": (SMALL, 3), "mid": (MID4, 2), "vitB_K64": (dict(num_keep_patches=64), 4),
           "vitB_K144": (dict(num_keep_patches=144), 4), "vitL_512_K256": (VITL, 2)}
_SD = {}


def _model(kw, seed=3, native=True, decoder=True, **flags):
    cfg = PathConfig(**kw)
    key = (tuple(sorted(kw.items())), seed, decoder)
    if key not in _SD:
        _SD[key] = make_state_dict(cfg, seed=seed, include_decoder=decoder)
    m = MCM(**kw, softmax_isa=16, native_synthesis=native, **flags)
    m.load_state_dict(_SD[key])
    return cfg, m.cuda().eval()


def _inputs(cfg, n, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, 3, cfg.img_size, cfg.img_size, generator=g).cuda(),
            torch.rand(n, cfg.num_patches, generator=g).cuda())


def _latents(m, cfg, n, seed=0):
    """y_hat (channels-last) and ids_restore of a forward with random scores."""
    fwd = m(*_inputs(cfg, n, seed), need_recon=False)
    return fwd["latents"]["y_hat"].permute(0, 2, 3, 1).contiguous(), fwd["ids_restore"]


def _synth(m, y_nhwc, ids):
    """tmae_synthesize on m's handle into a fresh x_hat."""
    m._ensure_handle()
    cfg = m.cfg
    N = y_nhwc.shape[0]
    x_hat = torch.full((N, 3, cfg.img_size, cfg.img_size), float("nan"), device=y_nhwc.device)
    rc = _native.load().tmae_synthesize(m._handle, G.ptr(y_nhwc), G.ptr(ids.contiguous()), N, G.ptr(x_hat), G.stream())
    _native.check(rc, m._handle, RuntimeError)
    torch.cuda.synchronize()
    return x_hat


def _reference(m, y_nhwc, ids):
    cfg = m.cfg
    return recon.synthesize(m._weights, cfg, y_nhwc.reshape(y_nhwc.shape[0], cfg.num_keep_patches, cfg.latent_depth), ids)


def _close(got, want):
    rel = G.rel_err(got, want)
    mx = (got - want).abs().max().item()
    assert torch.isfinite(got).all()
    assert rel <= 1.5e-2 and mx <= 0.1, f"rel L2 {rel:.3e}, max abs {mx:.3e}"
    return rel, mx


@pytest.mark.parametrize("key", list(CONFIGS))
def test_synthesis_matches_fp32_torch(cuda_dev, key):
    kw, n = CONFIGS[key]
    cfg, m = _model(kw)
    y, ids = _latents(m, cfg, n, seed=1)
    rel, mx = _close(_synth(m, y, ids), _reference(m, y, ids))
    print(f"{key}: rel L2 {rel:.3e}, max abs {mx:.3e}")


def test_synthesis_in_precise_mode_is_bf16(cuda_dev):
    """The precise flags govern the rate path; a precise="all" handle synthesizes with the same bf16 arithmetic."""
    cfg, m = _model(SMALL, precise="all")
    y, ids = _latents(m, cfg, 3, seed=2)
    x = _synth(m, y, ids)
    _close(x, _reference(m, y, ids))
    _, plain = _model(SMALL)
    assert torch.equal(x, _synth(plain, y, ids))


@pytest.mark.parametrize("T", [17, 65, 197, 1025])
def test_attention_hd32_matches_torch(cuda_dev, T):
    H, N = 16, 2
    g = torch.Generator().manual_seed(T)
    qkv = (torch.randn(N * T, 3 * H * 32, generator=g) * 1.5).to(cuda_dev).bfloat16()
    q, k, v = qkv.float().reshape(N, T, 3, H, 32).permute(2, 0, 3, 1, 4)
    ref = (((q @ k.transpose(-2, -1)) * 32 ** -0.5).softmax(-1) @ v).transpose(1, 2).reshape(N * T, H * 32)
    out = torch.zeros(N * T, H * 32, dtype=torch.bfloat16, device=cuda_dev)
    _native.check(_native.load().tmae_attention_hd32_bf16(G.ptr(qkv), G.ptr(out), N, T, H, G.stream()), None, RuntimeError)
    out = out.float()
    assert torch.isfinite(out).all()
    assert G.rel_err(out, ref) < 6e-3, G.rel_err(out, ref)


def test_batch_invariance(cuda_dev):
    """An image's x_hat does not depend on what it is batched with, nor on the share_sm launch shapes."""
    kw = dict(num_keep_patches=64)
    cfg, m = _model(kw)
    _, shared = _model(kw, share_sm=True)
    y, ids = _latents(m, cfg, 64, seed=3)
    full = _synth(m, y, ids)
    assert torch.equal(_synth(shared, y, ids), full)
    halves = torch.cat([_synth(m, y[:32], ids[:32]), _synth(m, y[32:], ids[32:])])
    assert torch.equal(halves, full)
    for i in (0, 17, 63):
        assert torch.equal(_synth(m, y[i:i + 1], ids[i:i + 1]), full[i:i + 1])
        assert torch.equal(_synth(shared, y[i:i + 1], ids[i:i + 1]), full[i:i + 1])


def test_graph_replay_equals_plain_launches(cuda_dev, monkeypatch):
    cfg, m = _model(SMALL)
    monkeypatch.setenv("TMAE_NO_GRAPH", "1")
    _, plain = _model(SMALL)
    plain._ensure_handle()                         # the handle reads TMAE_NO_GRAPH when it is created
    monkeypatch.delenv("TMAE_NO_GRAPH")
    y, ids = _latents(m, cfg, 4, seed=4)
    y2, ids2 = _latents(m, cfg, 4, seed=5)
    want, want2 = _synth(plain, y, ids), _synth(plain, y2, ids2)
    for _ in range(3):                             # plain launches, then capture + replay, then replay
        assert torch.equal(_synth(m, y, ids), want)
    assert torch.equal(_synth(m, y2.clone(), ids2.clone()), want2)          # fresh buffers through the IoBlock
    _close(want2, _reference(m, y2, ids2))
    m.profile(True)
    _synth(m, y, ids)
    names = [s["name"] for s in m.profile_read_steps()]
    m.profile(False)
    assert names[0] == "synth_input" and names[-1] == "unpatchify" and "unshuffle" in names and "dec_blk1.fc2" in names


def test_other_plans_unchanged(cuda_dev):
    cfg, native = _model(SMALL)
    _, torch_path = _model(SMALL, native=False)
    assert native.launch_count(4) == torch_path.launch_count(4)
    imgs, scores = _inputs(cfg, 3, seed=6)
    a, b = native(imgs, scores, need_recon=False), torch_path(imgs, scores, need_recon=False)
    assert torch.equal(a["latents"]["y_hat"], b["latents"]["y_hat"]) and torch.equal(a["bpp"], b["bpp"])
    # native_synthesis=False keeps recon.synthesize: the torch path's x_hat, bit for bit
    y, ids = a["latents"]["y_hat"].permute(0, 2, 3, 1).contiguous(), a["ids_restore"]
    assert torch.equal(torch_path(imgs, scores)["x_hat"], _reference(torch_path, y, ids))


@pytest.mark.parametrize("key", ["small", "vitB_K64"])
def test_decodes_return_forward_x_hat(cuda_dev, key):
    kw, n = CONFIGS[key]
    cfg, m = _model(kw)
    imgs, scores = _inputs(cfg, n, seed=7)
    fwd = m(imgs, scores, need_recon=True)
    x = fwd["x_hat"]
    _close(x, _reference(m, fwd["latents"]["y_hat"].permute(0, 2, 3, 1).contiguous(), fwd["ids_restore"]))
    sym = m.compress_symbols(imgs, scores)
    dec = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    assert torch.equal(dec["x_hat"], x)
    for lanes in (None, (32, 4)):
        bs = m.compress_bitstream(imgs, scores, lanes=lanes)
        out = m.decompress_bitstream(bs["strings"], bs["shape"], bs["ids_restore"], lanes=lanes)
        assert torch.equal(out["x_hat"], x), lanes


def test_refexec_goldens_in_bf16(cuda_dev, golden_dir):
    """The native forward under the reference's loss, against the reference MCM's own outputs (refexec_small.pt, "small"; the
    "mid" golden has a decoder head dim of 64): the bf16 tolerance of tests/test_gpu_recon.py."""
    from tests.test_gpu_recon import rd_loss_restated
    blob = torch.load(golden_dir / "refexec_small.pt")["small"]
    cfg = PathConfig(**blob["kwargs"])
    m = MCM(**blob["kwargs"], softmax_isa=16, native_synthesis=True)
    m.load_state_dict(make_state_dict(cfg, seed=blob["seed"], include_decoder=True))
    m.cuda().eval()
    out = m(blob["imgs"].cuda(), blob["scores"].cuda())
    assert m._syn_on
    rd, want = rd_loss_restated(out, blob["imgs"].cuda()), blob["rd_loss"]
    assert abs(rd["L1_loss"].item() - want["L1_loss"]) < 2e-2 and abs(rd["ssim_loss"].item() - want["ssim_loss"]) < 2e-2


def test_errors(cuda_dev):
    cfg, m = _model(SMALL)
    imgs, scores = _inputs(cfg, 2, seed=8)
    sym = m.compress_symbols(imgs, scores)
    bad = sym["ids_restore"].clone()
    bad[1, 0] = bad[1, 1]
    with pytest.raises(ValueError, match="permutation"):
        m.decompress_symbols(sym["z_symbols"], bad, y_symbols=sym["y_symbols"])
    bs = m.compress_bitstream(imgs, scores)
    with pytest.raises(ValueError, match="permutation"):
        m.decompress_bitstream(bs["strings"], bs["shape"], bad)
    # out-of-range ids are clamped: no fault, finite pixels
    wild = sym["ids_restore"].clone()
    wild[0, :3] = torch.tensor([-5, 1 << 40, cfg.num_patches], device=wild.device)
    y, _ = _latents(m, cfg, 2, seed=8)
    assert torch.isfinite(_synth(m, y, wild)).all()
    # need_recon without decoder weights: the existing error
    _, bare = _model(SMALL, decoder=False)
    with pytest.raises(RuntimeError, match="no g_s / decoder tensors"):
        bare(imgs, scores, need_recon=True)
    # head dim other than 32
    with pytest.raises(ValueError, match="head dim of 32"):
        _model(dict(MID4, decoder_num_heads=2))[1](*_inputs(PathConfig(**MID4), 1), need_recon=True)
    # a missing decoder tensor is named at finalize
    sd = dict(make_state_dict(cfg, seed=3, include_decoder=True))
    del sd["decoder_blocks.1.mlp.fc2.bias"]
    m2 = MCM(**SMALL, softmax_isa=16, native_synthesis=True)
    m2.load_state_dict(sd)
    m2.cuda().eval()
    with pytest.raises(RuntimeError, match="decoder_blocks.1.mlp.fc2.bias"):
        m2(imgs, scores, need_recon=True)
    # enabling synthesis after finalize unfinalizes the weights: tmae_synthesize is then TMAE_ESTATE
    lib = _native.load()
    assert lib.tmae_enable_synthesis(m._handle, cfg.decoder_depth, cfg.decoder_num_heads) == _native.TMAE_OK
    x_hat = torch.empty(2, 3, cfg.img_size, cfg.img_size, device=cuda_dev)
    rc = lib.tmae_synthesize(m._handle, G.ptr(y), G.ptr(sym["ids_restore"]), 2, G.ptr(x_hat), G.stream())
    assert rc == _native.TMAE_ESTATE
    # and a handle without synthesis enabled reports TMAE_ESTATE as well
    _, off = _model(SMALL, native=False)
    off._ensure_handle()
    assert lib.tmae_synthesize(off._handle, G.ptr(y), G.ptr(sym["ids_restore"]), 2, G.ptr(x_hat), G.stream()) == _native.TMAE_ESTATE
    assert lib.tmae_enable_synthesis(off._handle, 0, 16) == _native.TMAE_EINVAL
    assert lib.tmae_enable_synthesis(off._handle, 2, 3) == _native.TMAE_EINVAL
