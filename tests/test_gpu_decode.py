"""GPU: the decode side (MCM.decompress_symbols: the rate half with y replaced by the range coder's symbols).  A handle of
the same configuration must rebuild the encoder's latents and hand the range decoder the encoder's indexes bit for bit -
otherwise a real rANS stream desynchronises at the first index that differs."""
import ctypes as C

import pytest
import torch

from oracle import ref_decode
from tests import gpu_util as G
from textmae_image_compression_b200 import MCM, PathConfig, _native, make_state_dict, vit_base

pytestmark = pytest.mark.gpu

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16)
CONFIGS = {"small": (SMALL, 3), "vitB_K64": (dict(num_keep_patches=64), 2), "vitB_K144": (dict(num_keep_patches=144), 2)}
PRECISE = [None, "all"]
_SD = {}


def _cfg_sd(key, decoder=False):
    kw, _ = CONFIGS[key]
    cfg = vit_base(kw["num_keep_patches"]) if key.startswith("vitB") else PathConfig(**kw)
    if (key, decoder) not in _SD:
        _SD[(key, decoder)] = make_state_dict(cfg, seed=3, include_decoder=decoder)
    return cfg, _SD[(key, decoder)]


def _model(key, precise, decoder=False, **flags):
    kw, _ = CONFIGS[key]
    cfg, sd = _cfg_sd(key, decoder)
    m = MCM(**kw, softmax_isa=16, precise=precise, **flags)
    m.load_state_dict(sd)
    return cfg, sd, m.cuda().eval()


def _inputs(cfg, n, seed=0):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(n, 3, cfg.img_size, cfg.img_size, generator=g).cuda(),
            torch.rand(n, cfg.num_patches, generator=g).cuda())


def _encode(m, imgs, scores):
    sym = m.compress_symbols(imgs, scores)
    fwd = m(imgs, scores, need_recon=False)
    return sym, fwd


def _by_slice(t, cfg):
    return t.view(t.shape[0], cfg.num_slices, cfg.slice_ch, cfg.side, cfg.side)


@pytest.mark.parametrize("precise", PRECISE)
@pytest.mark.parametrize("key", list(CONFIGS))
def test_round_trip_is_bit_exact(cuda_dev, key, precise):
    cfg, _, m = _model(key, precise)
    imgs, scores = _inputs(cfg, CONFIGS[key][1])
    sym, fwd = _encode(m, imgs, scores)
    dec = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    torch.cuda.synchronize()
    assert "x_hat" not in dec
    assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"])
    assert torch.equal(dec["z_hat"], fwd["latents"]["z_hat"])
    assert torch.equal(dec["y_indexes"], sym["y_indexes"])


@pytest.mark.parametrize("precise", PRECISE)
def test_decode_across_batch_sizes_and_launch_shapes(cuda_dev, precise):
    """Encoded at batch 64 on a handle tuned for sharing the GPU, decoded one image and half batches at a time on a
    default handle: every launch shape on the way (tile counts, CTA pairs, persistent kernels, stage counts) must keep
    the k order, so each row comes out bit for bit."""
    cfg, sd, enc = _model("vitB_K64", precise, share_sm=True)
    imgs, scores = _inputs(cfg, 64, seed=4)
    sym, fwd = _encode(enc, imgs, scores)
    _, _, dec_m = _model("vitB_K64", precise)
    parts = [(5, 6), (0, 32), (32, 64)]
    for a, b in parts:
        dec = dec_m.decompress_symbols(sym["z_symbols"][a:b].contiguous(), sym["ids_restore"][a:b],
                                       y_symbols=sym["y_symbols"][a:b].contiguous())
        torch.cuda.synchronize()
        assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"][a:b]), (a, b)
        assert torch.equal(dec["z_hat"], fwd["latents"]["z_hat"][a:b]), (a, b)
        assert torch.equal(dec["y_indexes"], sym["y_indexes"][a:b]), (a, b)


@pytest.mark.parametrize("precise", PRECISE)
@pytest.mark.parametrize("key", list(CONFIGS))
def test_stepwise_decode_sees_the_encoders_indexes(cuda_dev, key, precise):
    cfg, _, m = _model(key, precise)
    n = CONFIGS[key][1]
    imgs, scores = _inputs(cfg, n, seed=1)
    sym, fwd = _encode(m, imgs, scores)
    one = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    want_idx, want_sym = _by_slice(sym["y_indexes"], cfg), _by_slice(sym["y_symbols"], cfg).cpu()
    calls = []

    def decode_fn(first, indexes):
        cnt = indexes.shape[1]
        assert indexes.dtype == torch.int32 and tuple(indexes.shape) == (n, cnt, cfg.slice_ch, cfg.side, cfg.side)
        assert torch.equal(indexes, want_idx[:, first:first + cnt]), first
        calls.append((first, cnt))
        return want_sym[:, first:first + cnt].clone()              # host tensor, as a range decoder returns it

    step = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], decode_fn=decode_fn)
    torch.cuda.synchronize()
    assert calls == [(0, 1), (1, 1), (2, 1), (3, 1), (4, 1), (5, 1), (6, 6)]
    for k in ("y_hat", "z_hat", "y_indexes"):
        assert torch.equal(step[k], one[k]), k
    assert torch.equal(step["y_hat"], fwd["latents"]["y_hat"])


@pytest.mark.parametrize("precise", PRECISE)
@pytest.mark.parametrize("key", list(CONFIGS))
def test_decode_against_oracle_with_forced_symbols(cuda_dev, key, precise):
    """Both sides decode the same symbols, so no rounding decision is taken and nothing can cascade: the GPU decode is
    the fp32 decode within the accuracy of its arithmetic, and indexes differ only where sigma sits on a bucket edge."""
    cfg, sd, m = _model(key, precise)
    imgs, scores = _inputs(cfg, CONFIGS[key][1], seed=2)
    sym, _ = _encode(m, imgs, scores)
    dec = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    torch.cuda.synchronize()
    table = MCM.get_scale_table()
    ref = ref_decode.decode_from_symbols(sd, cfg, sym["z_symbols"].cpu(), sym["y_symbols"].cpu(), table)
    assert torch.equal(dec["z_hat"].cpu(), ref["z_hat"])
    y_rel = G.rel_err(dec["y_hat"].cpu(), ref["y_hat"])
    assert y_rel < (1e-4 if precise else 2e-2), y_rel
    got_idx, ref_idx = dec["y_indexes"].cpu(), ref["indexes"].reshape(dec["y_indexes"].shape)
    diff = got_idx != ref_idx
    if precise:
        # bf16 operands move sigma by up to a few percent, across one or more 13 % wide buckets: only reported below
        assert (got_idx - ref_idx).abs().max().item() <= 1                 # a neighbouring bucket, never further
        assert diff.float().mean().item() < 2e-3, diff.float().mean().item()
        # every mismatch is a scale within rounding distance of a table entry
        sig = ref["sigma"].reshape(diff.shape)[diff].clamp_min(0.11)
        near = ((sig[:, None] - table[None, :]).abs() / table[None, :]).min(1)[0]
        assert (near < 1e-3).all(), near.max().item()
    print(f"{key} precise={precise}: y_hat rel {y_rel:.2e}, index mismatches {int(diff.sum())} of {diff.numel()}")


@pytest.mark.parametrize("precise", PRECISE)
def test_changed_symbol_affects_only_its_slice_and_later(cuda_dev, precise):
    cfg, _, m = _model("small", precise)
    imgs, scores = _inputs(cfg, 3, seed=5)
    sym, _ = _encode(m, imgs, scores)
    base = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    ys = sym["y_symbols"].clone()
    _by_slice(ys, cfg)[0, 2, 0, 0, 0] += 1
    alt = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=ys)
    torch.cuda.synchronize()
    sc = cfg.slice_ch
    a, b = base["y_hat"], alt["y_hat"]
    assert torch.equal(a[:, :2 * sc], b[:, :2 * sc])                          # slices 0-1 do not read slice 2
    assert torch.equal(a[1:], b[1:])                                          # other images untouched
    for j in range(2, cfg.num_slices):
        assert not torch.equal(a[0, j * sc:(j + 1) * sc], b[0, j * sc:(j + 1) * sc]), j
    assert torch.equal(base["y_indexes"][:, :3 * sc * cfg.side ** 2], alt["y_indexes"][:, :3 * sc * cfg.side ** 2])


@pytest.mark.parametrize("precise", PRECISE)
def test_reconstruction_equals_forward(cuda_dev, precise):
    cfg, _, m = _model("small", precise, decoder=True)
    imgs, scores = _inputs(cfg, 2, seed=6)
    sym = m.compress_symbols(imgs, scores)
    fwd = m(imgs, scores)
    dec = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    torch.cuda.synchronize()
    assert torch.equal(dec["x_hat"], fwd["x_hat"])
    assert "x_hat" not in m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"], need_recon=False)


def _raw_out(cfg, n, dev):
    s, s4 = cfg.side, cfg.side // 4
    t = {"y_hat": torch.empty(n, s, s, cfg.latent_depth, device=dev), "z_hat": torch.empty(n, s4, s4, cfg.hyperprior_depth, device=dev),
         "y_indexes": torch.empty(n, cfg.latent_depth * s * s, dtype=torch.int32, device=dev)}
    o = _native.TmaeOutputs()
    for k, v in t.items():
        setattr(o, k, v.data_ptr())
    return t, o


def test_decode_state_and_errors(cuda_dev):
    cfg, _, m = _model("small", None)
    lib = _native.load()
    imgs, scores = _inputs(cfg, 2, seed=7)
    # no update() on this module: decompress_symbols installs the default table itself, like compress_symbols
    fresh_cfg, _, fresh = _model("small", None)
    fresh._ensure_handle()
    t, o = _raw_out(cfg, 2, cuda_dev)
    z0 = torch.zeros(2, cfg.hyperprior_depth, cfg.side // 4, cfg.side // 4, dtype=torch.int32, device=cuda_dev)
    assert lib.tmae_decode_begin(fresh._handle, G.ptr(z0), 2, C.byref(o), G.stream()) == _native.TMAE_ESTATE   # no scale table
    sym, fwd = _encode(m, imgs, scores)
    dec = fresh.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
    assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"])
    # steps out of order, and a forward in the middle of a decode, end it with TMAE_ESTATE
    h, st = m._handle, G.stream()
    zs, ys = sym["z_symbols"].contiguous(), sym["y_symbols"].contiguous()
    assert lib.tmae_decode_step(h, 0, G.ptr(ys), C.byref(o), st) == _native.TMAE_ESTATE            # no begin yet
    assert lib.tmae_decode_begin(h, G.ptr(zs), 2, C.byref(o), st) == 0
    assert lib.tmae_decode_step(h, 2, G.ptr(ys), C.byref(o), st) == _native.TMAE_ESTATE
    assert "out of order" in _native.last_error(h)
    assert lib.tmae_decode_step(h, 0, G.ptr(ys), C.byref(o), st) == _native.TMAE_ESTATE            # the bad step ended it
    assert lib.tmae_decode_begin(h, G.ptr(zs), 2, C.byref(o), st) == 0
    assert lib.tmae_decode_step(h, 0, G.ptr(ys), C.byref(o), st) == 0
    m(imgs, scores, need_recon=False)
    assert lib.tmae_decode_step(h, 1, G.ptr(ys), C.byref(o), st) == _native.TMAE_ESTATE
    assert lib.tmae_decode_begin(h, G.ptr(zs), 2, None, st) == _native.TMAE_EINVAL
    # a complete raw decode through the ABI
    assert lib.tmae_decode_begin(h, G.ptr(zs), 2, C.byref(o), st) == 0
    for g in range(7):
        assert lib.tmae_decode_step(h, g, G.ptr(ys), C.byref(o), st) == 0, _native.last_error(h)
    assert lib.tmae_decode_step(h, 7, G.ptr(ys), C.byref(o), st) == _native.TMAE_ESTATE
    torch.cuda.synchronize()
    assert torch.equal(t["y_hat"], fwd["latents"]["y_hat"].permute(0, 2, 3, 1))
    assert torch.equal(t["y_indexes"], sym["y_indexes"])
    # wrong shapes / dtypes
    with pytest.raises(ValueError):
        m.decompress_symbols(sym["z_symbols"].long(), sym["ids_restore"], y_symbols=sym["y_symbols"])
    with pytest.raises(ValueError):
        m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"][:, 1:])
    with pytest.raises(ValueError):
        m.decompress_symbols(sym["z_symbols"], sym["ids_restore"][:1], y_symbols=sym["y_symbols"])
    with pytest.raises(ValueError):
        m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"], decode_fn=lambda f, i: i)
    with pytest.raises(ValueError):
        m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], decode_fn=lambda f, i: i[:, :, :1])


def test_graph_replays_honour_per_call_pointers(cuda_dev, monkeypatch):
    """From the second decode of a batch size every stage replays a captured graph: fresh symbols and fresh output buffers
    must be read and written on every call.  TMAE_NO_GRAPH=1 (plain launches throughout) gives the same results."""
    cfg, sd, m = _model("small", None)
    batches = [_inputs(cfg, 4, seed=10 + k) for k in range(2)]
    enc = [_encode(m, i, s) for i, s in batches]
    for rep in range(3):
        for sym, fwd in enc:
            dec = m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
            torch.cuda.synchronize()
            assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"]), rep
            assert torch.equal(dec["y_indexes"], sym["y_indexes"]), rep
    assert not torch.equal(enc[0][1]["latents"]["y_hat"], enc[1][1]["latents"]["y_hat"])
    monkeypatch.setenv("TMAE_NO_GRAPH", "1")
    _, _, plain = _model("small", None)
    plain._ensure_handle()                       # the environment is read when the handle is created
    monkeypatch.delenv("TMAE_NO_GRAPH")
    for rep in range(2):
        for sym, fwd in enc:
            dec = plain.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"])
            torch.cuda.synchronize()
            assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"]), rep
