"""CPU: pins of the in-repo oracle and of this package's host side against the original project.

Every test runs everywhere against reference outputs frozen under tests/golden/ (refexec_small.pt, refexec_extra.pt,
refexec_params.json; see tests/golden/make_refexec_golden.py).  Where a checkout of the original project exists
(oracle.REFERENCE_ROOT), the tests also run the REFERENCE CODE WHERE IT LIES: its own `MCM` class - `__init__` topology,
`forward_encoder`, `random_masking`, `get_ids_shuffle`, the whole `forward` incl. the slice loop - verbatim from
models/Compression/MCM.py with only the absent third-party leaf classes (timm / compressai / pytorch_msssim) supplied by
oracle/ref_stubs.py (oracle/ref_exec.py).  What is pinned:
 * the oracle's forward (oracle/ref_model.py) and the synthetic checkpoint's names and shapes against `MCM`;
 * `synthetic.sincos_pos_embed` against `common/pos_embed.py:get_2d_sincos_pos_embed`, bit for bit;
 * the per-image / batch rate (`bpp`, `rate_sums`) against `loss/rd_loss.py:RateDistortionLoss`;
 * the reconstruction half of this package (recon.py, stock PyTorch) against the reference forward's `x_hat` / `loss`;
 * this package's `MCM` module under the reference's `RateDistortionLoss` (and, live, `utils/engine.py:val_one_epoch`)
   (host contract: dict keys, `aux_loss()`, `parameters()`, `eval()`); the native forward is replaced by a test double
   built from the oracle so that it runs without a GPU - the GPU twin of this test is tests/test_gpu_recon.py.
"""
import hashlib
import importlib.util
import json
import sys

import pytest
import torch

from oracle import ref_exec, ref_mask, ref_model, ref_pins
from tests.test_gpu_recon import rd_loss_restated
from textmae_image_compression_b200 import MCM, PathConfig, make_state_dict, recon
from textmae_image_compression_b200.config import vit_base
from textmae_image_compression_b200.synthetic import sincos_pos_embed

LIVE = ref_exec.reference_available()
# The goldens were written with AVX512 ATen kernels: on such a host the oracle runs the same torch ops in the same order
# and reproduces them bit for bit.  Elsewhere the comparisons hold to float32 rounding.
EXACT = ref_mask.torch_softmax_isa() == 16

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16,
             decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=2)
MID = dict(img_size=128, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=64,
           decoder_embed_dim=128, decoder_depth=2, decoder_num_heads=2)
REFEXEC = {"small": SMALL, "mid": MID}           # configurations frozen in tests/golden/refexec_small.pt


def _same(got, want, rtol=1e-4, atol=1e-6):
    if EXACT:
        return torch.equal(got, want)
    return got.shape == want.shape and torch.allclose(got.double(), want.double(), rtol=rtol, atol=atol)


@pytest.fixture(scope="module")
def params(golden_dir):
    """Names and shapes of the reference module's state dict, per configuration."""
    return json.loads((golden_dir / "refexec_params.json").read_text())


@pytest.fixture(scope="module")
def refexec(golden_dir):
    blobs = torch.load(golden_dir / "refexec_small.pt")
    for key, kw in REFEXEC.items():
        assert blobs[key]["kwargs"] == kw, key
    return blobs


@pytest.fixture(scope="module")
def extra(golden_dir):
    return torch.load(golden_dir / "refexec_extra.pt")


def _inputs(cfg, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 3, cfg.img_size, cfg.img_size, generator=g), torch.rand(n, cfg.num_patches, generator=g)


def _missing_unexpected(sd, names):
    """What load_state_dict(strict=False) of `sd` into the reference module would report, plus shape mismatches."""
    assert all(list(sd[k].shape) == names[k] for k in sd if k in names)
    return [k for k in names if k not in sd], [k for k in sd if k not in names]


# ---------------------------------------------------------------------------------------------- oracle vs reference MCM
@pytest.mark.parametrize("kw,n", [(SMALL, 3), (MID, 2)])
def test_oracle_equals_reference_mcm_forward(refexec, params, kw, n):
    key = next(k for k, v in REFEXEC.items() if v == kw)
    blob = refexec[key]
    cfg = PathConfig(**kw)
    sd = make_state_dict(cfg, seed=blob["seed"], include_decoder=True)
    imgs, scores = blob["imgs"], blob["scores"]
    assert imgs.shape[0] == n
    # every synthetic tensor name exists in the reference module and every reference tensor is provided (names AND shapes)
    assert _missing_unexpected(sd, params[key]) == ([], [])
    ref = ref_model.forward_rate(sd, cfg, imgs, scores)
    assert _same(ref["y_lik"], blob["y_lik"]) and _same(ref["z_lik"], blob["z_lik"])   # same torch ops in the same order
    assert _same(ref["x_remain"], blob["x_remain"]) and _same(ref["ids_restore"], blob["ids_restore"])
    if LIVE:
        model, missing, unexpected = ref_exec.build_reference_model(cfg, sd)
        assert (missing, unexpected) == ([], [])
        out = ref_exec.reference_forward(model, imgs, scores)
        assert torch.equal(out["likelihoods"]["y"], ref["y_lik"]) and torch.equal(out["likelihoods"]["z"], ref["z_lik"])
        x_remain, ids_restore = model.forward_encoder(imgs, scores)
        assert torch.equal(x_remain, ref["x_remain"]) and torch.equal(ids_restore, ref["ids_restore"])


def test_oracle_equals_reference_mcm_forward_vit_base(extra, params):
    """The production geometry (ViT-B/16, K=64, default decoder in the reference module)."""
    cfg = vit_base(64)
    frozen = extra["vit_base"]
    sd = make_state_dict(cfg, seed=frozen["seed"])
    imgs, scores = _inputs(cfg, 1, frozen["input_seed"])
    ref = ref_model.forward_rate(sd, cfg, imgs, scores)
    if LIVE:
        model, missing, unexpected = ref_exec.build_reference_model(cfg, sd)
        out = ref_exec.reference_forward(model, imgs, scores)
        y_lik, z_lik = out["likelihoods"]["y"], out["likelihoods"]["z"]
        assert torch.equal(y_lik, ref["y_lik"]) and torch.equal(z_lik, ref["z_lik"])
    else:
        missing, unexpected = _missing_unexpected(sd, params["vit_base"])
        y_lik, z_lik = frozen["y_lik"], frozen["z_lik"]
    assert unexpected == [] and missing and all(k.startswith(recon.DECODER_PREFIXES) for k in missing), (unexpected, missing[:5])
    assert _same(ref["y_lik"], y_lik) and _same(ref["z_lik"], z_lik)


def test_reference_rejects_what_the_config_rejects():
    """K with sqrt(K) % 4 != 0 fails inside the reference forward (torch.cat size mismatch, MCM.py:761); the config
    rejects it up front."""
    cfg = PathConfig(img_size=128, encoder_embed_dim=128, encoder_depth=1, encoder_num_heads=2, num_keep_patches=64)
    bad = PathConfig(img_size=128, encoder_embed_dim=128, encoder_depth=1, encoder_num_heads=2, num_keep_patches=36)
    with pytest.raises(RuntimeError):
        bad.validate()
    cfg.validate()
    if not LIVE:
        return
    MCMref = ref_exec.load_reference_mcm_class()
    with ref_exec._np_float_shim():
        m = MCMref(img_size=128, encoder_embed_dim=128, encoder_depth=1, encoder_num_heads=2, num_keep_patches=36,
                   decoder_embed_dim=64, decoder_depth=1, decoder_num_heads=2).eval()
    imgs, scores = _inputs(cfg, 1, 2)
    with pytest.raises(RuntimeError):
        with torch.no_grad():
            m(imgs, scores)


# ---------------------------------------------------------------------------------------------- pos-embed / rd_loss pins
@pytest.mark.parametrize("dim,grid", [(768, 14), (1024, 32), (128, 4), (512, 14)])
def test_sincos_pos_embed_is_bit_equal_to_reference(extra, dim, grid):
    table = sincos_pos_embed(dim, grid)
    if LIVE:
        assert torch.equal(table, ref_pins.reference_pos_embed_parameter(dim, grid))
    name = f"{dim}x{grid}"
    if EXACT:
        assert hashlib.sha256(table.numpy().tobytes()).hexdigest() == extra["pos_embed_sha256"][name]
    idx = torch.randperm(table.numel(), generator=torch.Generator().manual_seed(0))[:2048]
    assert torch.allclose(table.reshape(-1)[idx], extra["pos_embed_sample"][name], rtol=0, atol=1e-7)


def test_bpp_equals_reference_rate_distortion_loss(refexec):
    """bpp_loss of the reference's RateDistortionLoss on the reference forward's likelihoods (frozen with them)."""
    for blob in refexec.values():
        img_size, n = blob["kwargs"]["img_size"], blob["imgs"].shape[0]
        y_lik, z_lik = blob["y_lik"], blob["z_lik"]
        bpp_loss = torch.tensor(blob["rd_loss"]["bpp_loss"], dtype=torch.float32)
        if LIVE:
            assert torch.equal(ref_pins.reference_bpp_loss(y_lik, z_lik, img_size), bpp_loss)
        assert _same(ref_model.bpp_batch(y_lik, z_lik, img_size), bpp_loss, rtol=1e-6)     # oracle restatement == reference class
        assert torch.allclose(ref_model.bpp_per_image(y_lik, z_lik, img_size).mean(), bpp_loss, rtol=2e-6)  # per-image form averages to it
        # the library's rate_sums pair {sum log2 lik, pixels} is the same quantity: bpp_loss == -sums[0] / sums[1]
        sum_log2 = (torch.log2(y_lik.double()).sum() + torch.log2(z_lik.double()).sum()).item()
        assert abs(-sum_log2 / (n * img_size ** 2) - bpp_loss.item()) < 2e-6 * bpp_loss.item()


# ---------------------------------------------------------------------------------------------- reconstruction half
def test_recon_matches_reference_forward(refexec):
    blob = refexec["small"]
    cfg = PathConfig(**SMALL)
    sd = make_state_dict(cfg, seed=blob["seed"], include_decoder=True)
    imgs, scores = blob["imgs"], blob["scores"]
    ref = ref_model.forward_rate(sd, cfg, imgs, scores)
    tokens = ref["y_hat"].permute(0, 2, 3, 1).reshape(3, cfg.num_keep_patches, cfg.latent_depth)
    loss, x_hat = recon.reconstruct(sd, cfg, tokens, ref["ids_restore"], imgs)
    assert torch.allclose(x_hat, blob["x_hat"], rtol=1e-5, atol=1e-6)
    assert torch.allclose(loss[0], blob["loss"][0], rtol=1e-5, atol=1e-6)       # 1 - SSIM
    assert torch.allclose(loss[1], blob["loss"][1], rtol=1e-6)                  # L1
    assert float(loss[2]) == 0.0 and float(blob["loss"][2]) == 0.0


# ---------------------------------------------------------------------------------------------- the reference's callers
class _OracleBackedMCM(MCM):
    """Test double for a machine without a GPU: the C-ABI call is replaced by the fp32 oracle; everything around it -
    argument checks, result dict, reconstruction half, aux_loss, parameters - is the product code."""

    def _ensure_handle(self):
        self._handle_device = torch.device("cpu")

    def _native_forward(self, imgs, total_scores, indexes=False):
        ref = ref_model.forward_rate(self._weights, self.cfg, imgs, total_scores)
        nhwc = lambda t: t.permute(0, 2, 3, 1).contiguous()
        return {"y_likelihoods": nhwc(ref["y_lik"]), "z_likelihoods": nhwc(ref["z_lik"]), "y_symbols": nhwc(ref["y_sym"]),
                "z_symbols": nhwc(ref["z_sym"]), "y_hat": nhwc(ref["y_hat"]), "z_hat": nhwc(ref["z_hat"]), "bpp": ref["bpp"],
                "rate_sums": torch.zeros(2, dtype=torch.float64), "ids_restore": ref["ids_restore"], "ids_keep": ref["ids_keep"],
                "ids_shuffle": ref["ids_restore"]}


def _load_reference_engine():
    """utils/engine.py imports `models.Compression.common.{distributed, logger}` (plain torch): import as written."""
    sys.path.insert(0, str(ref_exec.REFERENCE_ROOT))
    try:
        for k in [k for k in sys.modules if k == "models" or k.startswith("models.") or k == "utils" or k.startswith("utils.")]:
            del sys.modules[k]
        spec = importlib.util.spec_from_file_location("_ref_engine", str(ref_pins.ENGINE))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    finally:
        sys.path.remove(str(ref_exec.REFERENCE_ROOT))


def test_reference_val_one_epoch_and_rd_loss_run_against_this_module(refexec, capsys):
    cfg = PathConfig(**SMALL)
    blob = refexec["small"]
    sd = make_state_dict(cfg, seed=blob["seed"], include_decoder=True)
    ours = _OracleBackedMCM(**SMALL)
    ours.load_state_dict(sd)
    assert ours.eval() is ours and len(list(ours.parameters())) > 0
    # the criterion on one forward (rd_loss.py:14-28) and aux_loss (engine.py:194), against the reference's values on the
    # same inputs, frozen with its forward
    a = rd_loss_restated(ours(blob["imgs"], blob["scores"]), blob["imgs"])
    for k in ("bpp_loss", "ssim_loss", "L1_loss", "vgg_loss", "loss"):
        assert abs(float(a[k]) - blob["rd_loss"][k]) <= 1e-4 * abs(blob["rd_loss"][k]) + 1e-6, (k, float(a[k]), blob["rd_loss"][k])
    assert abs(ours.aux_loss().item() - blob["aux_loss"]) <= 1e-5 * blob["aux_loss"]
    if not LIVE:
        return
    ref_model_, _, _ = ref_exec.build_reference_model(cfg, sd)
    criterion = ref_pins.load_rate_distortion_loss()(lmbda=1e-2)
    engine = _load_reference_engine()
    batches = [(*_inputs(cfg, 2, s)[:1], torch.tensor([[64, 64]] * 2), _inputs(cfg, 2, s)[1]) for s in (1, 2)]   # (img, size, scores)
    stats_ours = engine.val_one_epoch(0, batches, ours, criterion)
    stats_ref = engine.val_one_epoch(0, batches, ref_model_, criterion)
    capsys.readouterr()
    assert stats_ours.keys() == stats_ref.keys() and "bpp_loss" in stats_ours
    for k in stats_ref:
        assert abs(stats_ours[k] - stats_ref[k]) <= 0.011 * max(1.0, abs(stats_ref[k])), (k, stats_ours[k], stats_ref[k])
    # and the reference's own criterion class directly on one forward
    imgs, scores = _inputs(cfg, 2, 7)
    a = criterion(ours(imgs, scores), imgs)
    b = criterion(ref_model_(imgs, scores), imgs)
    for k in ("bpp_loss", "ssim_loss", "L1_loss", "vgg_loss", "loss"):
        assert torch.allclose(a[k].float(), b[k].float(), rtol=1e-4, atol=1e-6), k
