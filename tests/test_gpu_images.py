"""GPU: MCM.compress_images / decompress_images.  The containers equal the plain-Python reference's packing of compress_bitstream's
streams and forward's ids_keep, and they decode from the bytes alone to forward's y_hat / z_hat / x_hat bit for bit; malformed
containers are refused one by one while the rest of the batch decodes."""
import ctypes as C
import os
import struct
import subprocess
import sys

import pytest
import torch

from tests import ref_image_container as R
from tests.test_gpu_bitstream import CONFIGS, _inputs, _model
from textmae_image_compression_b200 import MCM, _native, entropy

pytestmark = pytest.mark.gpu

MODES = {None: 0, "all": 2}


def _fields(m, lanes):
    c = m.cfg
    tag = R.model_tag(m.entropy_tables(), m._scale_table.tolist())
    yl, zl = lanes if lanes is not None else (0, 0)
    return dict(img_size=c.img_size, patch_size=c.patch_size, mode=MODES[m.precise], y_lanes=yl, z_lanes=zl, tag=tag)


def _check_decode(m, containers, fwd, dec=None):
    dec = dec if dec is not None else m.decompress_images(containers)
    assert torch.equal(dec["y_hat"], fwd["latents"]["y_hat"])
    assert torch.equal(dec["z_hat"], fwd["latents"]["z_hat"])
    assert torch.equal(dec["ids_keep"], fwd["ids_keep"])
    assert torch.equal(dec["ids_restore"].gather(1, fwd["ids_keep"]), fwd["ids_restore"].gather(1, fwd["ids_keep"]))
    L = fwd["ids_restore"].shape[1]             # every position: the canonical ids_restore, unkept positions ascending K .. L-1
    canon = torch.tensor([R.canonical_ids_restore(r, L) for r in fwd["ids_keep"].tolist()], dtype=torch.int64)
    assert torch.equal(dec["ids_restore"].cpu(), canon)
    if "x_hat" in fwd:
        assert torch.equal(dec["x_hat"], fwd["x_hat"])
    return dec


@pytest.mark.parametrize("lanes", [None, (32, 4)])
@pytest.mark.parametrize("precise", [None, "all"])
@pytest.mark.parametrize("key", list(CONFIGS))
def test_containers_equal_reference_and_decode_bit_exact(cuda_dev, key, precise, lanes):
    cfg, m = _model(key, precise)
    imgs, scores = _inputs(cfg, CONFIGS[key][1])
    containers = m.compress_images(imgs, scores, lanes=lanes)
    enc = m.compress_bitstream(imgs, scores, lanes=lanes)
    fwd = m(imgs, scores)
    f = _fields(m, lanes)
    tag = C.c_uint32(0)
    assert _native.load().tmae_model_tag(m._handle, C.byref(tag)) == 0 and tag.value == f["tag"]
    N = imgs.shape[0]
    for i in range(N):
        assert containers[i] == R.pack(enc["strings"][0][i], enc["strings"][1][i], fwd["ids_keep"][i].tolist(), f), f"image {i}"
        assert R.parse(containers[i])["tag"] == f["tag"]
    yl, zl = f["y_lanes"], f["z_lanes"]
    assert sum(map(len, containers)) <= entropy.images_bound(m._handle, N, yl, zl)
    dec = _check_decode(m, containers, fwd)
    ref = m.decompress_bitstream(enc["strings"], enc["shape"], enc["ids_restore"], need_recon=False, lanes=lanes)
    assert torch.equal(dec["y_hat"], ref["y_hat"]) and torch.equal(dec["z_hat"], ref["z_hat"])


@pytest.mark.parametrize("key", list(CONFIGS))
def test_native_synthesis_x_hat_is_forwards(cuda_dev, key):
    cfg, m = _model(key, None, native_synthesis=True)
    imgs, scores = _inputs(cfg, CONFIGS[key][1], seed=1)
    for lanes in ((32, 4), None):
        containers = m.compress_images(imgs, scores, lanes=lanes)
        fwd = m(imgs, scores)
        _check_decode(m, containers, fwd)


def test_images_bound_formula(cuda_dev):
    cfg, m = _model("vitB_K64", None, decoder=False)
    m._install_coder_tables()
    lib = _native.load()
    ny, nz = 384 * 64, 192 * 4
    for yl, zl in ((0, 0), (32, 4), (7, 1)):
        per = 28 + 64 + (lib.tmae_rans_bound_lanes(ny, yl) if yl else lib.tmae_rans_bound(ny)) + \
            (lib.tmae_rans_bound_lanes(nz, zl) if zl else lib.tmae_rans_bound(nz))
        assert lib.tmae_images_bound(m._handle, 3, yl, zl) == 3 * per


def test_batch64_and_single_images(cuda_dev):
    cfg, m = _model("vitB_K64", None)
    imgs, scores = _inputs(cfg, 64, seed=5)
    containers = m.compress_images(imgs, scores)
    fwd = m(imgs, scores, need_recon=False)
    _check_decode(m, containers, fwd, m.decompress_images(containers, need_recon=False))
    one = m.decompress_images(containers[7:8], need_recon=False)
    assert torch.equal(one["y_hat"], fwd["latents"]["y_hat"][7:8]) and torch.equal(one["ids_keep"], fwd["ids_keep"][7:8])


def test_graph_replay_equals_no_graph_and_plan_keys(cuda_dev):
    cfg, m = _model("small", None)
    imgs, scores = _inputs(cfg, 3, seed=9)
    fwd = m(imgs, scores)
    per_lanes = {lanes: m.compress_images(imgs, scores, lanes=lanes) for lanes in (None, (32, 4), (5, 1))}
    for _ in range(3):                          # plain launches, capture, replay; the keys (N, W_y, W_z) alternate
        for lanes, containers in per_lanes.items():
            _check_decode(m, containers, fwd)
    code = ("import sys, torch; sys.path.insert(0, '.'); from tests.test_gpu_bitstream import _model, _inputs;"
            "cfg, m = _model('small', None); i, s = _inputs(cfg, 3, seed=9); c = m.compress_images(i, s);"
            "d = m.decompress_images(c); torch.save({'c': c, **{k: v.cpu() for k, v in d.items()}}, sys.argv[1])")
    path = os.path.join(os.environ.get("TMPDIR", "/tmp"), f"nograph_images_{os.getpid()}.pt")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run([sys.executable, "-c", code, path], check=True, env=dict(os.environ, TMAE_NO_GRAPH="1"), cwd=root)
    ng = torch.load(path, weights_only=False)
    os.remove(path)
    assert ng["c"] == per_lanes[(32, 4)]
    d = m.decompress_images(per_lanes[(32, 4)])
    for k in ("y_hat", "z_hat", "x_hat", "ids_restore", "ids_keep"):
        assert torch.equal(ng[k], d[k].cpu()), k


def test_new_tables_and_grown_workspace_drop_the_plans(cuda_dev):
    cfg, m = _model("small", None)
    imgs, scores = _inputs(cfg, 8, seed=2)
    fwd = m(imgs[:2], scores[:2])
    old = m.compress_images(imgs[:2], scores[:2])
    for _ in range(2):
        _check_decode(m, old, fwd)
    m.compress_bitstream(imgs, scores)           # grows the coder workspace past N = 2
    bs = m.compress_bitstream(imgs, scores)
    m.decompress_bitstream(bs["strings"], bs["shape"], bs["ids_restore"])
    _check_decode(m, old, fwd)
    # new CDF tables (another scale table): the old containers carry the old tag and are refused; new ones decode
    m.update(scale_table=MCM.get_scale_table(0.2, 128.0, 48))
    with pytest.raises(ValueError, match=r"image 0: model.*image 1: model"):
        m.decompress_images(old)
    new = m.compress_images(imgs[:2], scores[:2])
    fwd_new = m(imgs[:2], scores[:2])
    for _ in range(2):
        _check_decode(m, new, fwd_new)
    # a module with the same weights and mode decodes the bytes alone; one with other tables refuses them
    _, fresh = _model("small", None)
    fresh.update(scale_table=MCM.get_scale_table(0.2, 128.0, 48))
    _check_decode(fresh, new, fwd_new)
    _, other = _model("small", None)
    with pytest.raises(ValueError, match="model"):
        other.decompress_images(new)


def _word(b, i, v):
    b = bytearray(b)
    struct.pack_into("<I", b, 4 * i, v)
    return bytes(b)


def _get(b, i):
    return struct.unpack_from("<I", b, 4 * i)[0]


def test_mixed_batch_refuses_exactly_the_bad_containers(cuda_dev):
    cfg, m = _model("vitB_K64", None)
    imgs, scores = _inputs(cfg, 4, seed=7)
    good = m.compress_images(imgs, scores)
    fwd = m(imgs, scores, need_recon=False)
    g = good[1]
    f = R.parse(g)
    ids = f["ids_keep"]
    fields = dict(_fields(m, (32, 4)))
    H, CFG, MOD, IDS = _native.IMG_HEADER, _native.IMG_CONFIG, _native.IMG_MODEL, _native.IMG_IDS
    defects = [
        ("magic", _word(g, 0, 0x45414D55), H),
        ("version", _word(g, 1, (_get(g, 1) & ~0xFF) | 2), H),
        ("reserved word 2", _word(g, 2, _get(g, 2) | 1 << 24), H),
        ("reserved word 3", _word(g, 3, _get(g, 3) | 1 << 20), H),
        ("another K", R.pack(f["y"], f["z"], ids[:-1], fields), CFG),
        ("another mode", _word(g, 1, _get(g, 1) ^ (2 << 8)), CFG),
        ("another lane count", _word(g, 1, (_get(g, 1) & 0x00FFFFFF) | 5 << 24), CFG),
        ("flipped tag", _word(g, 4, _get(g, 4) ^ 1), MOD),
        ("duplicate id", R.pack(f["y"], f["z"], ids[:-1] + ids[:1], fields), IDS),
        ("id >= L", R.pack(f["y"], f["z"], ids[:-1] + [200], fields), IDS),
        ("lengths overrun", _word(g, 6, _get(g, 6) + 4), H),
        ("truncated", g[:-4], H),
    ]
    batch, expect = [], []
    for k, (_, bad, bit) in enumerate(defects):
        batch.append(good[k % 4])
        expect.append(0)
        batch.append(bad)
        expect.append(bit)
    N = len(batch)
    # through the ABI: every status, and the good images bit-exact
    data, offs = entropy.pack_strings(batch)
    d, o_dev = data.cuda(), offs.cuda()
    c = m.cfg
    y_hat = torch.empty((N, c.side, c.side, c.latent_depth), device="cuda")
    z_hat = torch.empty((N, c.side // 4, c.side // 4, c.hyperprior_depth), device="cuda")
    ids_restore = torch.empty((N, c.num_patches), dtype=torch.int64, device="cuda")
    st = torch.empty(N, dtype=torch.int32, device="cuda")
    o = _native.TmaeOutputs()
    o.y_hat, o.z_hat = y_hat.data_ptr(), z_hat.data_ptr()
    lib = _native.load()
    _native.check(lib.tmae_decompress_images(m._handle, C.c_void_p(d.data_ptr()), d.numel(), C.c_void_p(o_dev.data_ptr()), N, 32, 4,
                                             C.byref(o), C.c_void_p(ids_restore.data_ptr()), None, C.c_void_p(st.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)), m._handle)
    s = st.cpu().tolist()
    img_bits = H | CFG | MOD | IDS
    for k, (name, _, bit) in enumerate(defects):
        assert s[2 * k] == 0, name
        assert s[2 * k + 1] & img_bits == bit, (name, s[2 * k + 1])
        assert torch.equal(y_hat[2 * k], fwd["latents"]["y_hat"][k % 4].permute(1, 2, 0)), name
        assert torch.equal(z_hat[2 * k], fwd["latents"]["z_hat"][k % 4].permute(1, 2, 0)), name
    # through MCM: the error names exactly the bad images
    bad_ids = [i for i in range(N) if expect[i]]
    with pytest.raises(ValueError) as e:
        m.decompress_images(batch, need_recon=False)
    assert f"images {bad_ids} do not decode" in str(e.value)
    for i in bad_ids:
        assert f"image {i}: " in str(e.value)
    # a corrupt stream inside a well-formed container: the stream's reason
    bad_stream = bytearray(good[2])
    bad_stream[-8:] = b"\xff" * 8
    with pytest.raises(ValueError, match=r"images \[1\] do not decode - image 1: a stream that does not decode"):
        m.decompress_images([good[0], bytes(bad_stream)], need_recon=False)
    # a blob range the offsets put outside n_bytes
    offs_bad = offs.clone()
    offs_bad[-1] = d.numel() + 4
    _native.check(lib.tmae_decompress_images(m._handle, C.c_void_p(d.data_ptr()), d.numel(), C.c_void_p(offs_bad.cuda().data_ptr()), N,
                                             32, 4, C.byref(o), C.c_void_p(ids_restore.data_ptr()), None, C.c_void_p(st.data_ptr()),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)), m._handle)
    assert st.cpu().tolist()[-1] & img_bits == H


def test_container_calls_need_tables_and_synthesis(cuda_dev):
    _, fresh = _model("small", None, decoder=False)
    fresh._install_scale_table()
    lib = _native.load()
    buf = torch.zeros(64, dtype=torch.int64, device="cuda")
    p = C.c_void_p(buf.data_ptr())
    out = _native.TmaeOutputs()
    out.y_hat = out.z_hat = buf.data_ptr()
    E, S = _native.TMAE_EINVAL, _native.TMAE_ESTATE
    tag = C.c_uint32(0)
    assert lib.tmae_model_tag(fresh._handle, C.byref(tag)) == S
    assert lib.tmae_compress_images(fresh._handle, p, p, 1, 32, 4, p, 512, p, p, None) == S
    assert lib.tmae_decompress_images(fresh._handle, p, 512, p, 1, 32, 4, C.byref(out), p, None, p, None) == S
    fresh._install_coder_tables()
    assert lib.tmae_model_tag(fresh._handle, C.byref(tag)) == 0
    # x_hat without synthesis enabled, bad lanes, misaligned data
    assert lib.tmae_decompress_images(fresh._handle, p, 512, p, 1, 32, 4, C.byref(out), p, p, p, None) == S
    assert lib.tmae_decompress_images(fresh._handle, p, 512, p, 1, 33, 4, C.byref(out), p, None, p, None) == E
    assert lib.tmae_decompress_images(fresh._handle, C.c_void_p(buf.data_ptr() + 2), 8, p, 1, 32, 4, C.byref(out), p, None, p, None) == E
    assert lib.tmae_compress_images(fresh._handle, p, p, 0, 32, 4, p, 512, p, p, None) == E
    # int64 arrays off their 8-byte alignment: offsets, ids_restore, out->ids_keep
    q = C.c_void_p(buf.data_ptr() + 4)
    assert lib.tmae_compress_images(fresh._handle, p, p, 1, 32, 4, p, 512, q, p, None) == E
    assert lib.tmae_decompress_images(fresh._handle, p, 8, q, 1, 32, 4, C.byref(out), p, None, p, None) == E
    assert lib.tmae_decompress_images(fresh._handle, p, 8, p, 1, 32, 4, C.byref(out), q, None, p, None) == E
    out.ids_keep = buf.data_ptr() + 4
    assert lib.tmae_decompress_images(fresh._handle, p, 8, p, 1, 32, 4, C.byref(out), p, None, p, None) == E
