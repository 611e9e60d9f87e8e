"""CPU: the GEMM engine's launch policy (tmae_gemm_launch_plan) - no device needed, the resolver only computes the launch."""
import ctypes as C
import os

import pytest

from textmae_image_compression_b200 import _native

ONE_CTA, PERSISTENT, PAIR, PAIR_PERSISTENT, SIMT = range(5)
OTHER, BF16, F32_RESID = range(3)
ACT_NONE, ACT_GELU, ACT_HALF_TANH = range(3)
EPI_BF16_TMA, EPI_F32_SAME_RESID = 3, 2
KEYS = ("form", "act", "epi", "block_n", "m_tiles", "n_tiles", "gx", "gy", "gz", "block", "smem", "stages", "kgroup",
        "two_producers", "conv_reuse_stage")


def _conv_rows(side, n_img):
    g = (C.c_int * 6)()
    assert _native.load().tmae_conv_geometry(side, n_img, g) == 0
    return g[3] * 128


def _plan(groups=1, M=0, N=0, conv=None, out=OTHER, act=ACT_NONE, gauss=0, ln_in=False, ln_out=False, shuffle=False,
          tma=True, share=False, simt=False, force_bn=0, force_form=-1):
    side, n_img = conv if conv else (0, 0)
    if conv:
        M = _conv_rows(side, n_img)
    shape = (C.c_int * 17)(groups, M, N, 1 if conv else 0, side, n_img, out, act, gauss, int(ln_in), int(ln_out), int(shuffle),
                           int(tma), int(share), int(simt), force_bn, force_form)
    res = (C.c_int * 15)()
    assert _native.load().tmae_gemm_launch_plan(shape, res) == 0, _native.last_error()
    return dict(zip(KEYS, list(res)))


def _shapes():
    """Step shapes of the plans: the encoder (ViT-B at K = 64 / 144, ViT-L at K = 256, batch 1..64), the conv nets (g_a, h_s
    PixelShuffle, cc / lrp slice groups) and the fused Gaussian layer."""
    for n in (1, 8, 64):
        for T, C_, mlp in ((65, 768, 3072), (145, 768, 3072), (257, 1024, 4096)):
            rows = n * T
            yield dict(M=rows, N=3 * C_, out=BF16, ln_in=True)                     # QKV (LayerNorm folded)
            yield dict(M=rows, N=C_, out=F32_RESID, ln_out=True)                   # proj
            yield dict(M=rows, N=mlp, out=BF16, act=ACT_GELU, ln_in=True)          # fc1
            yield dict(M=rows, N=C_, out=F32_RESID, ln_out=True)                   # fc2
            yield dict(M=n * (T - 1), N=C_, out=OTHER)                             # patch embed (gathered rows)
        for side in (8, 12, 16):
            for cout, act in ((224, ACT_GELU), (176, ACT_GELU), (128, ACT_GELU), (80, ACT_GELU), (320, ACT_NONE)):
                yield dict(conv=(side, n), N=cout, out=BF16, act=act)
            yield dict(conv=(side, n), N=64, out=F32_RESID, act=ACT_HALF_TANH)     # lrp last layer (y_hat += 0.5 tanh)
            for groups in (2, 6, 12):
                yield dict(groups=groups, conv=(side, n), N=224, out=BF16, act=ACT_GELU)
                yield dict(groups=groups, conv=(side, n), N=32, out=OTHER)         # cc last layers: mu / sigma
                yield dict(groups=groups, conv=(side, n), N=64, gauss=1)           # fused Gaussian (encoder)
                yield dict(groups=groups, conv=(side, n), N=64, gauss=2)           # fused Gaussian (decoder)
            yield dict(groups=2, conv=(side // 4 if side >= 8 else 1, n), N=4 * 192, out=OTHER, act=ACT_GELU, shuffle=True)


def _covered_once(p, groups):
    """Every 128 x block_n tile of the largest member is computed by exactly one CTA (or one CTA pair)."""
    m, n = p["m_tiles"], p["n_tiles"]
    if p["form"] == ONE_CTA:
        return (p["gx"], p["gy"], p["gz"]) == (m, n, groups)
    if p["form"] == PAIR:
        return (p["gx"], p["gy"], p["gz"]) == ((m + 1) // 2 * 2, n, groups)
    count = {}
    if p["form"] == PERSISTENT:
        for cta in range(p["gx"]):
            for t in range(cta, m * n, p["gx"]):
                count[(t // n, t % n)] = count.get((t // n, t % n), 0) + 1
    elif p["form"] == PAIR_PERSISTENT:
        pairs, m_pairs = p["gx"] // 2, (m + 1) // 2
        for pair in range(pairs):
            for t in range(pair, m_pairs * n, pairs):
                for rank in (0, 1):
                    key = (2 * (t // n) + rank, t % n)
                    if key[0] < m:
                        count[key] = count.get(key, 0) + 1
    return groups == 1 and sorted(count) == [(i, j) for i in range(m) for j in range(n)] and set(count.values()) == {1}


@pytest.mark.parametrize("share", [False, True], ids=["one_batch", "share_sm"])
def test_gemm_launch_plan_invariants(share):
    default_env = not any(k in os.environ for k in ("TMAE_PP_SHARE", "TMAE_NO_TMA_STORE", "TMAE_NO_LN_FOLD"))
    forms = set()
    for kw in _shapes():
        groups = kw.get("groups", 1)
        p = _plan(share=share, **kw)
        forms.add(p["form"])
        assert p["form"] != SIMT
        assert p["smem"] <= 227 * 1024 and p["stages"] >= 2, (kw, p)
        assert p["block_n"] % 16 == 0 and 16 <= p["block_n"] <= 256, (kw, p)
        if p["form"] in (PAIR, PAIR_PERSISTENT):
            assert p["block_n"] % 16 == 0 and p["m_tiles"] >= 8, (kw, p)
        if share and default_env:
            assert p["form"] not in (PERSISTENT, PAIR_PERSISTENT), (kw, p)
        if kw.get("gauss"):
            assert p["form"] == ONE_CTA and p["block_n"] == 32, (kw, p)
        if kw.get("shuffle") or kw.get("ln_out"):
            assert p["block_n"] % 32 == 0, (kw, p)
        if kw.get("ln_in") and default_env:
            assert p["epi"] == EPI_BF16_TMA, (kw, p)
        if kw.get("ln_out"):
            assert p["epi"] == EPI_F32_SAME_RESID, (kw, p)
        assert _covered_once(p, groups), (kw, p)
    assert {ONE_CTA, PAIR} <= forms
    if not share:
        assert {PERSISTENT, PAIR_PERSISTENT} & forms


def test_gemm_launch_plan_forced_forms():
    """The engine self-tests' forced forms: CTA pairs need block_n % 16 == 0; persistent pairs only take bf16 same-row outputs."""
    p = _plan(M=4160, N=768, out=BF16, force_bn=192, force_form=PAIR_PERSISTENT)
    assert p["form"] == PAIR_PERSISTENT and p["block_n"] == 192 and _covered_once(p, 1)
    assert _plan(M=300, N=512, out=F32_RESID, force_bn=128, force_form=PAIR)["form"] == PAIR
    s = _plan(M=300, N=512, out=F32_RESID, force_form=SIMT)
    assert (s["form"], s["gx"], s["block"]) == (SIMT, 300, 128)
    lib = _native.load()
    res = (C.c_int * 15)()
    bad_pair = (C.c_int * 17)(1, 300, 512, 0, 0, 0, F32_RESID, 0, 0, 0, 0, 0, 1, 0, 0, 40, PAIR)
    assert lib.tmae_gemm_launch_plan(bad_pair, res) == _native.TMAE_EINVAL
    bad_pp = (C.c_int * 17)(1, 4160, 768, 0, 0, 0, F32_RESID, 0, 0, 0, 0, 0, 1, 0, 0, 192, PAIR_PERSISTENT)
    assert lib.tmae_gemm_launch_plan(bad_pp, res) == _native.TMAE_EINVAL
