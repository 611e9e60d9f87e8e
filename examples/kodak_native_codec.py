"""The Kodak fixtures at their native size (five 512 x 768, one 768 x 512) through the picture codec: grey RGB picture ->
MCM.compress_pictures (GPU tiling into 224 x 224 tiles, tile scores, one self-contained byte string per picture) ->
MCM.decompress_pictures from those bytes alone -> x_hat at the picture's own size.  No resize to 224 x 224: the decoded picture
is the one that was coded.  Prints the bytes, the actual bpp over the original pixels (8 * len(bytes) / (H * W)) and the PSNR.

    python examples/kodak_native_codec.py [--keep 144] [--precise all] [--lanes 32 4 | --compressai]

The pictures are the committed greys as RGB (x = g / 255 on all three channels; cvtColor of (g, g, g) is g, so the tile scores
are the reference's).  Weights are the seeded synthetic checkpoint, so the PSNR is meaningless."""
import argparse
import math
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from textmae_image_compression_b200 import MCM, make_state_dict, vit_base  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keep", type=int, default=144)
    ap.add_argument("--precise", default=None)
    ap.add_argument("--lanes", type=int, nargs=2, default=[32, 4])
    ap.add_argument("--compressai", action="store_true", help="compressai-format streams inside the tile containers")
    args = ap.parse_args()
    lanes = None if args.compressai else tuple(args.lanes)
    gray = np.load(ROOT / "tests" / "golden" / "kodak_gray6.npz")
    names = sorted(gray.files)
    greys = [torch.from_numpy(np.ascontiguousarray(gray[n])) for n in names]
    pictures = [(g.float() / 255).expand(3, -1, -1).contiguous() for g in greys]

    cfg = vit_base(args.keep)
    state = make_state_dict(cfg, seed=0, include_decoder=True)
    encoder = MCM(num_keep_patches=args.keep, precise=args.precise)
    encoder.load_state_dict(state)
    encoder = encoder.cuda().eval()
    decoder = MCM(num_keep_patches=args.keep, precise=args.precise, native_synthesis=True)   # same weights and mode
    decoder.load_state_dict(state)
    decoder = decoder.cuda().eval()

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    strings = encoder.compress_pictures(pictures, gray=greys, lanes=lanes)
    t1 = time.perf_counter()
    x_hat = decoder.decompress_pictures(strings)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    for name, x, data, xh in zip(names, pictures, strings, x_hat):
        H, W = x.shape[1:]
        mse = torch.mean((x.cuda() - xh.clamp(0, 1)) ** 2).item()
        print(f"{name}: {H} x {W}, {len(data)} bytes, bpp {8 * len(data) / (H * W):.4f} actual, "
              f"psnr {10 * math.log10(1.0 / max(mse, 1e-12)):.2f} dB (synthetic weights)")
    print(f"{len(strings)} pictures: compress {(t1 - t0) * 1e3:.1f} ms, decompress {(t2 - t1) * 1e3:.1f} ms (first calls, plans built)")


if __name__ == "__main__":
    main()
