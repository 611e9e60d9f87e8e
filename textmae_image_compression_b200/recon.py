"""Reconstruction half of `MCM.forward` (SURVEY 8f-2), stock PyTorch on the module's device.

The compression forward path (everything up to the rate) runs in libtmae_b200.so; what follows it in the
reference - `g_s`, the MAE decoder, `unpatchify` and the distortion terms
(/root/reference/models/Compression/MCM.py:96-112, 636-688, 524-546, 690-712, 789-797) - is outside that path
(BASELINE north_star) and is provided here with plain torch ops on the library's `y_hat`, so that the
reference's callers (`utils/engine.py:189-199`, `loss/rd_loss.py:21-23`, `testing.py:106-109`) find the
`"loss"` / `"x_hat"` entries they read.  Functional, keyed by the reference's state-dict names.

Not reproduced: the pretrained-VGG16 feature term (`loss/vgg.py:99` downloads ImageNet weights and builds the
network on every call); `feature_loss` is a hook (callable(preds, imgs) -> scalar) and 0 when unset.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Tuple

import torch
import torch.nn.functional as F

DECODER_PREFIXES = ("g_s.", "decoder_embed.", "mask_token", "decoder_pos_embed", "decoder_blocks.", "decoder_norm.",
                    "decoder_pred.")


def has_decoder_weights(w: Dict[str, torch.Tensor]) -> bool:
    return "decoder_pred.weight" in w and "g_s.0.weight" in w and "mask_token" in w


def g_s(w, y_hat_tokens: torch.Tensor) -> torch.Tensor:
    """MCM.py:96-112, 790-792.  ConvTranspose2d(cin, cout, k=1) on NCHW == per-token linear with weight[cin, cout]^T;
    `y_hat_tokens` [N, K, Cy] is the library's channels-last y_hat, i.e. already the token matrix the reference forms
    with permute(0,2,3,1).view(-1, K, C)."""
    x = y_hat_tokens
    for li, idx in enumerate((0, 2, 4, 6)):
        wt = w[f"g_s.{idx}.weight"][:, :, 0, 0]                 # [cin, cout]
        x = F.linear(x, wt.t(), w[f"g_s.{idx}.bias"])
        if li < 3:
            x = F.gelu(x)
    return x


def _block(w, pre: str, x: torch.Tensor, heads: int, eps: float) -> torch.Tensor:
    """timm 0.4.5 Block.forward (eval): pre-norm attention + MLP with erf GELU."""
    B, T, C = x.shape
    hd = C // heads
    h = F.layer_norm(x, (C,), w[pre + ".norm1.weight"], w[pre + ".norm1.bias"], eps)
    qkv = F.linear(h, w[pre + ".attn.qkv.weight"], w[pre + ".attn.qkv.bias"]).reshape(B, T, 3, heads, hd).permute(2, 0, 3, 1, 4)
    attn = ((qkv[0] @ qkv[1].transpose(-2, -1)) * (hd ** -0.5)).softmax(dim=-1)
    a = (attn @ qkv[2]).transpose(1, 2).reshape(B, T, C)
    x = x + F.linear(a, w[pre + ".attn.proj.weight"], w[pre + ".attn.proj.bias"])
    h = F.layer_norm(x, (C,), w[pre + ".norm2.weight"], w[pre + ".norm2.bias"], eps)
    h = F.gelu(F.linear(h, w[pre + ".mlp.fc1.weight"], w[pre + ".mlp.fc1.bias"]))
    return x + F.linear(h, w[pre + ".mlp.fc2.weight"], w[pre + ".mlp.fc2.bias"])


def forward_decoder(w, x_remain: torch.Tensor, ids_restore: torch.Tensor, depth: int, heads: int, eps: float) -> torch.Tensor:
    """MCM.forward_decoder (MCM.py:636-688) as written - including its treatment of the FIRST kept token as the cls
    token (the tokens g_s returns carry no cls token, yet `x_decode[:, 1:, :]` drops one and `x_decode[:, :1, :]` is
    re-attached in front): reproduced, not corrected, because x_hat must match the reference."""
    ids_restore = ids_restore.to(x_remain.device)
    x_decode = F.linear(x_remain, w["decoder_embed.weight"], w["decoder_embed.bias"])
    mask_tokens = w["mask_token"].repeat(x_decode.shape[0], ids_restore.shape[1] + 1 - x_decode.shape[1], 1)
    x_ = torch.cat([x_decode[:, 1:, :], mask_tokens], dim=1)
    x_ = torch.gather(x_, dim=1, index=ids_restore.unsqueeze(-1).repeat(1, 1, x_decode.shape[2]))
    x = torch.cat([x_decode[:, :1, :], x_], dim=1)
    x = x + w["decoder_pos_embed"]
    for i in range(depth):
        x = _block(w, f"decoder_blocks.{i}", x, heads, eps)
    C = x.shape[-1]
    x = F.layer_norm(x, (C,), w["decoder_norm.weight"], w["decoder_norm.bias"], eps)
    x = F.linear(x, w["decoder_pred.weight"], w["decoder_pred.bias"])
    return x[:, 1:, :]


def unpatchify(preds: torch.Tensor, patch: int) -> torch.Tensor:
    """MCM.unpatchify (MCM.py:524-546): [N, L, p*p*3] in (p, q, c) order -> [N, 3, H, W]."""
    h = int(preds.shape[1] ** 0.5)
    assert h * h == preds.shape[1]
    x = preds.reshape(preds.shape[0], h, h, patch, patch, 3)
    x = torch.einsum("nhwpqc->nchpwq", x)
    return x.reshape(x.shape[0], 3, h * patch, h * patch)


def _gauss_win(size: int, sigma: float, channels: int, like: torch.Tensor) -> torch.Tensor:
    coords = torch.arange(size, dtype=torch.float) - size // 2
    g = torch.exp(-(coords ** 2) / (2 * sigma ** 2))
    g = (g / g.sum()).to(like.device, like.dtype)
    return g.reshape(1, 1, 1, size).repeat(channels, 1, 1, 1)


def _gauss_filter(x: torch.Tensor, win: torch.Tensor) -> torch.Tensor:
    C = x.shape[1]
    out = x
    if x.shape[2] >= win.shape[-1]:
        out = F.conv2d(out, win.transpose(2, 3), groups=C)
    if x.shape[3] >= win.shape[-1]:
        out = F.conv2d(out, win, groups=C)
    return out


def ssim(X: torch.Tensor, Y: torch.Tensor, data_range: float = 1.0, win_size: int = 11, win_sigma: float = 1.5) -> torch.Tensor:
    """pytorch_msssim.SSIM(win_size=11, win_sigma=1.5, data_range=1, size_average=True, channel=3) as the reference
    builds it (MCM.py:705-708): separable Gaussian window, valid convolution, K = (0.01, 0.03)."""
    win = _gauss_win(win_size, win_sigma, X.shape[1], X)
    C1, C2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    mu1, mu2 = _gauss_filter(X, win), _gauss_filter(Y, win)
    mu1_sq, mu2_sq, mu12 = mu1 * mu1, mu2 * mu2, mu1 * mu2
    s1 = _gauss_filter(X * X, win) - mu1_sq
    s2 = _gauss_filter(Y * Y, win) - mu2_sq
    s12 = _gauss_filter(X * Y, win) - mu12
    cs = (2 * s12 + C2) / (s1 + s2 + C2)
    ssim_map = ((2 * mu12 + C1) / (mu1_sq + mu2_sq + C1)) * cs
    return torch.flatten(ssim_map, 2).mean(-1).mean()


def forward_loss(imgs: torch.Tensor, x_hat: torch.Tensor,
                 feature_loss: Optional[Callable[[torch.Tensor, torch.Tensor], torch.Tensor]] = None
                 ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """MCM.forward_loss (MCM.py:690-712): (1 - SSIM, L1, feature loss)."""
    ssim_loss = 1 - ssim(x_hat, imgs)
    l1 = (x_hat - imgs).abs().mean()
    feat = feature_loss(x_hat, imgs) if feature_loss is not None else torch.zeros((), device=imgs.device, dtype=imgs.dtype)
    return ssim_loss, l1, feat


@torch.no_grad()
def synthesize(w: Dict[str, torch.Tensor], cfg, y_hat_tokens: torch.Tensor, ids_restore: torch.Tensor) -> torch.Tensor:
    """MCM.py:789-792 (and the decoder side of MCM.decompress): g_s -> forward_decoder -> unpatchify.  Returns x_hat."""
    tok = g_s(w, y_hat_tokens)
    preds = forward_decoder(w, tok, ids_restore, cfg.decoder_depth, cfg.decoder_num_heads, cfg.ln_eps).float()
    return unpatchify(preds, cfg.patch_size)


@torch.no_grad()
def reconstruct(w: Dict[str, torch.Tensor], cfg, y_hat_tokens: torch.Tensor, ids_restore: torch.Tensor, imgs: torch.Tensor,
                feature_loss=None):
    """MCM.py:789-797: synthesize -> forward_loss.  Returns (loss 3-tuple, x_hat)."""
    x_hat = synthesize(w, cfg, y_hat_tokens, ids_restore)
    return forward_loss(imgs, x_hat, feature_loss), x_hat
