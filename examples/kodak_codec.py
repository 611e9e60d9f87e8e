"""testing.py's default (non-estimation) flow (testing.py:58-97) on the committed Kodak fixtures, with real bytes: grey image ->
GPU patch scores -> MCM.compress_images (one self-contained byte string per image: header, patch selection, rANS streams) ->
MCM.decompress_images from those bytes alone -> x_hat.  Prints the actual bpp, 8 * len(bytes) / pixels - side information
included - beside the likelihood estimate and the PSNR.

    python examples/kodak_codec.py [--keep 144] [--precise all] [--lanes 32 4 | --compressai]

Weights are the seeded synthetic checkpoint (no trained checkpoint ships with the reference), so the PSNR is meaningless; the
point is that an image goes to bytes and back through nothing but the bytes."""
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
from textmae_image_compression_b200.scores import generate_scores  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keep", type=int, default=144)
    ap.add_argument("--precise", default=None)
    ap.add_argument("--lanes", type=int, nargs=2, default=[32, 4])
    ap.add_argument("--compressai", action="store_true", help="compressai-format streams inside the containers")
    args = ap.parse_args()
    lanes = None if args.compressai else tuple(args.lanes)
    golden = ROOT / "tests" / "golden"
    gray = np.load(golden / "kodak_gray6.npz")
    names = sorted(gray.files)
    rgb = torch.from_numpy(np.load(golden / "kodak_224.npz")["imgs"][:len(names)]).permute(0, 3, 1, 2).float() / 255.0

    cfg = vit_base(args.keep)
    state = make_state_dict(cfg, seed=0, include_decoder=True)
    encoder = MCM(num_keep_patches=args.keep, precise=args.precise)
    encoder.load_state_dict(state)
    encoder = encoder.cuda().eval()
    decoder = MCM(num_keep_patches=args.keep, precise=args.precise)        # another module with the same weights and mode
    decoder.load_state_dict(state)
    decoder = decoder.cuda().eval()

    for i, name in enumerate(names):
        x = rgb[i:i + 1].cuda()
        total_score = generate_scores(torch.from_numpy(gray[name]).cuda())[None]   # generate_scores_file.py:19-31
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        data = encoder.compress_images(x, total_score, lanes=lanes)[0]
        t1 = time.perf_counter()
        out = decoder.decompress_images([data])
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        num_pixels = x.size(2) * x.size(3)
        estimate = encoder(x, total_score, need_recon=False)["bpp"].item()
        mse = torch.mean((x - out["x_hat"].clamp(0, 1)) ** 2).item()
        print(f"{name}: {len(data)} bytes, bpp {8 * len(data) / num_pixels:.4f} actual (estimate {estimate:.4f}), "
              f"psnr {10 * math.log10(1.0 / max(mse, 1e-12)):.2f} dB (synthetic weights), "
              f"compress {(t1 - t0) * 1e3:.2f} ms, decompress {(t2 - t1) * 1e3:.2f} ms")


if __name__ == "__main__":
    main()
