"""Freezes outputs of the REFERENCE's own `MCM.forward` (models/Compression/MCM.py executed verbatim from a checkout of the
original project, oracle.REFERENCE_ROOT; third-party leaf classes from oracle/ref_stubs.py - see oracle/ref_exec.py) into
tests/golden/refexec_small.pt, the names and shapes of its state dict into tests/golden/refexec_params.json, and its
ViT-B/16 K=64 likelihoods and `get_2d_sincos_pos_embed` tables (sha256 of the fp32 bytes + a seeded sample) into
tests/golden/refexec_extra.pt, so that machines without that checkout can check the oracle, the CUDA path and the
reconstruction half against reference outputs.  Run where the checkout exists:

    python tests/golden/make_refexec_golden.py

The committed refexec_small.pt was written by this script.  refexec_params.json and refexec_extra.pt were recorded later,
without a checkout, from the in-repo synthetic checkpoint, oracle forward and `sincos_pos_embed`, unchanged since this
script and the live tests of tests/test_reference_exec.py found them equal to the reference (DESIGN.md section 4): no
missing or unexpected state-dict key for small / mid (asserted by `one` below) and with the default decoder
(decoder_embed_dim 512, depth 8, 16 heads), no unexpected key at ViT-B/16, bit-equal likelihoods for this ViT-B/16
configuration and inputs, bit-equal tables.  Running this script replaces them
with values taken from the reference itself.
"""
from __future__ import annotations

import hashlib
import json
import sys
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))

from oracle import SKIP_REASON, ref_exec, ref_pins  # noqa: E402
from textmae_image_compression_b200 import PathConfig, make_state_dict  # noqa: E402
from textmae_image_compression_b200.config import vit_base  # noqa: E402

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16,
             decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=2)
MID = dict(img_size=128, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=64,
           decoder_embed_dim=128, decoder_depth=2, decoder_num_heads=2)


def one(kw, seed, n):
    cfg = PathConfig(**kw)
    sd = make_state_dict(cfg, seed=seed, include_decoder=True)
    model, missing, unexpected = ref_exec.build_reference_model(cfg, sd)
    assert not missing and not unexpected, (missing, unexpected)
    g = torch.Generator().manual_seed(100 + seed)
    imgs = torch.rand(n, 3, cfg.img_size, cfg.img_size, generator=g)
    scores = torch.rand(n, cfg.num_patches, generator=g)
    out = ref_exec.reference_forward(model, imgs, scores)
    x_remain, ids_restore = model.forward_encoder(imgs, scores)
    crit = ref_pins.load_rate_distortion_loss()(lmbda=1e-2)
    rd = crit(out, imgs)
    params = {k: list(v.shape) for k, v in model.state_dict().items()}
    return params, {"kwargs": kw, "seed": seed, "imgs": imgs, "scores": scores,
            "y_lik": out["likelihoods"]["y"], "z_lik": out["likelihoods"]["z"], "x_hat": out["x_hat"],
            "loss": torch.stack([l.float() for l in out["loss"]]), "x_remain": x_remain, "ids_restore": ids_restore,
            "rd_loss": {k: float(v) for k, v in rd.items()}, "aux_loss": float(model.aux_loss())}


def extra():
    """ViT-B/16 K=64 (seed 0, one image from input seed 5) and the pos-embed tables tests/test_reference_exec.py checks."""
    cfg = vit_base(64)
    model, _, _ = ref_exec.build_reference_model(cfg, make_state_dict(cfg, seed=0))
    g = torch.Generator().manual_seed(5)
    imgs = torch.rand(1, 3, cfg.img_size, cfg.img_size, generator=g)
    scores = torch.rand(1, cfg.num_patches, generator=g)
    out = ref_exec.reference_forward(model, imgs, scores)
    blob = {"vit_base": {"K": 64, "seed": 0, "input_seed": 5, "y_lik": out["likelihoods"]["y"], "z_lik": out["likelihoods"]["z"]},
            "pos_embed_sha256": {}, "pos_embed_sample": {}}
    for dim, grid in ((768, 14), (1024, 32), (128, 4), (512, 14)):
        table = ref_pins.reference_pos_embed_parameter(dim, grid)
        idx = torch.randperm(table.numel(), generator=torch.Generator().manual_seed(0))[:2048]
        blob["pos_embed_sha256"][f"{dim}x{grid}"] = hashlib.sha256(table.numpy().tobytes()).hexdigest()
        blob["pos_embed_sample"][f"{dim}x{grid}"] = table.reshape(-1)[idx].clone()
    params = {k: list(v.shape) for k, v in model.state_dict().items()}
    return params, blob


def main():
    assert ref_exec.reference_available(), SKIP_REASON
    runs = {"small": one(SMALL, 3, 3), "mid": one(MID, 5, 2), "vit_base": extra()}
    blob = {k: runs[k][1] for k in ("small", "mid")}
    torch.save(blob, HERE / "refexec_small.pt")
    torch.save(runs["vit_base"][1], HERE / "refexec_extra.pt")
    with open(HERE / "refexec_params.json", "w") as f:
        json.dump({k: v[0] for k, v in runs.items()}, f, sort_keys=True, separators=(",", ":"))
        f.write("\n")
    print({k: {kk: (tuple(vv.shape) if torch.is_tensor(vv) else vv) for kk, vv in v.items() if kk not in ("kwargs",)} for k, v in blob.items()})


if __name__ == "__main__":
    main()
