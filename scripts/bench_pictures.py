"""Picture containers against the hand-made flow they replace, timed alternately in the same run (native synthesis, bf16 operands).

    pictures:   MCM.compress_pictures / decompress_pictures (tiling, scores, forward, encodes, pack / parse, decode, synthesis and
                untiling enqueued by the library, one call per size)
    hand-made:  tiling.tile_image + generate_scores + compress_images, then decompress_images + tiling.untile_image per picture
Workloads: 24 Kodak-sized pictures (the five 512 x 768 Kodak greys of tests/golden/kodak_gray6.npz cycled, as grey RGB) at ViT-B/16
K = 144 with lanes (32, 4) = 288 tiles of 224 (bench.py's TILES288 shape); the same at P = 1 (latency); one seeded 2048 x 1080
picture at ViT-L/16 512^2 K = 256 (12 tiles).  Pictures/s and latency are host-clock medians over --rounds rounds of --steps calls;
the device time of the tile and untile kernels comes from CUDA events over --kernel-steps launches.  Every timed output is checked:
compress byte for byte, x_hat bit for bit, between the two flows.  The card name and power limit are read (nvidia-smi
--query-gpu, read-only) in the same run.

    python scripts/bench_pictures.py [--steps 10] [--warmup 2] [--rounds 3] [--out profiles/r08_pictures_B200.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import sys
from pathlib import Path

sys.dont_write_bytecode = True
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from bench_bitstream import host_time  # noqa: E402
from bench_decode import gpu_info, time_device  # noqa: E402
from tests import ref_picture_container as R  # noqa: E402
from textmae_image_compression_b200 import MCM, _native, make_state_dict, tiling, vit_base, vit_large  # noqa: E402
from textmae_image_compression_b200.scores import generate_scores  # noqa: E402


def _cv_gray(x):
    v = (x.double() * 255).float().round().clamp(0, 255).to(torch.int64)
    return ((9798 * v[:, 0] + 19235 * v[:, 1] + 3735 * v[:, 2] + 16384) >> 15).to(torch.uint8)


def run_workload(name, cfg, kw, x, steps, warmup, rounds, kernel_steps):
    m = MCM(**kw, native_synthesis=True)
    m.load_state_dict(make_state_dict(cfg, seed=0, include_decoder=True))
    m.cuda().eval()
    S = cfg.img_size
    P, _, H, W = x.shape
    T = R.tile_count(H, W, S)
    xd = x.cuda()
    gd = _cv_gray(x).cuda()

    def pictures_c():
        return m.compress_pictures(xd)

    def hand_c():
        cont = m.compress_images(tiling.tile_image(xd, S), generate_scores(tiling.tile_image(gd[:, None], S)[:, 0].contiguous(), S))
        return [R.pack(cont[p * T:(p + 1) * T], H, W) for p in range(P)]

    strings = pictures_c()
    assert strings == hand_c(), f"{name}: picture bytes differ from the hand-made flow"
    tiles_of = [R.parse(b)["tiles"] for b in strings]

    def pictures_d():
        return m.decompress_pictures(strings)

    def hand_d():
        x_t = m.decompress_images([t for ts in tiles_of for t in ts])["x_hat"]
        return [tiling.untile_image(x_t[p * T:(p + 1) * T], H, W) for p in range(P)]

    t = {"pictures_compress": [], "hand_compress": [], "pictures_decompress": [], "hand_decompress": []}
    for _ in range(rounds):
        for key, fn, check in (("pictures_compress", pictures_c, None), ("hand_compress", hand_c, None),
                               ("pictures_decompress", pictures_d, True), ("hand_decompress", hand_d, True)):
            ms, out = host_time(fn, steps, warmup)
            if check:
                ref = hand_d() if key == "pictures_decompress" else pictures_d()
                assert all(torch.equal(a, b) for a, b in zip(out, ref)), f"{name}: {key} x_hat differs"
            else:
                assert out == strings, f"{name}: {key} bytes differ"
            t[key].append(ms)
    med = {k: statistics.median(v) for k, v in t.items()}
    # device time of the two tiling kernels alone
    lib = _native.load()
    tiles = torch.empty((P * T, 3, S, S), device="cuda")
    gt = torch.empty((P * T, S, S), dtype=torch.uint8, device="cuda")
    canvas = torch.empty((P, 3, H, W), device="cuda")
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)
    tile_ms = time_device(lambda: lib.tmae_picture_tiles(C.c_void_p(xd.data_ptr()), None, P, H, W, S, C.c_void_p(tiles.data_ptr()),
                                                          C.c_void_p(gt.data_ptr()), st()), kernel_steps, 10)
    untile_ms = time_device(lambda: lib.tmae_picture_untile(C.c_void_p(tiles.data_ptr()), P, H, W, S, C.c_void_p(canvas.data_ptr()),
                                                            st()), kernel_steps, 10)
    n_bytes = sum(map(len, strings))
    res = {
        "workload": name, "pictures": P, "H": H, "W": W, "tiles": P * T, "img_size": S, "K": cfg.num_keep_patches, "lanes": [32, 4],
        "compress_pictures_per_s": {"pictures": P * 1e3 / med["pictures_compress"], "hand_made": P * 1e3 / med["hand_compress"]},
        "decompress_pictures_per_s": {"pictures": P * 1e3 / med["pictures_decompress"], "hand_made": P * 1e3 / med["hand_decompress"]},
        "ms_per_call": med,
        "tile_kernel_ms": tile_ms, "untile_kernel_ms": untile_ms,
        "bytes": n_bytes, "bytes_per_picture": n_bytes / P, "bpp": 8 * n_bytes / (P * H * W),
        "checked": "compress byte for byte, x_hat bit for bit, every timed call",
    }
    del m
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--kernel-steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pictures.py measures the GPU codec: no CUDA device")
    z = np.load(ROOT / "tests" / "golden" / "kodak_gray6.npz")
    greys = [torch.from_numpy(np.ascontiguousarray(z[k])) for k in sorted(z.files)]
    land = [g for g in greys if g.shape == (512, 768)]            # the five 512 x 768 greys: one size per library call
    kodak = torch.stack([(land[i % len(land)].float() / 255).expand(3, -1, -1) for i in range(24)])
    g = torch.Generator().manual_seed(0)
    div2k = torch.rand(1, 3, 1080, 2048, generator=g)
    out = {"info": gpu_info(), "results": []}
    b = vit_base(144)
    out["results"].append(run_workload("kodak24_vitB_K144", b, dict(num_keep_patches=144), kodak, a.steps, a.warmup, a.rounds,
                                       a.kernel_steps))
    out["results"].append(run_workload("kodak1_vitB_K144", b, dict(num_keep_patches=144), kodak[:1], a.steps, a.warmup, a.rounds,
                                       a.kernel_steps))
    lcfg = vit_large(256, 512)
    out["results"].append(run_workload("div2k1_vitL512_K256", lcfg, dict(img_size=512, encoder_embed_dim=1024, encoder_depth=24,
                                                                           encoder_num_heads=16, num_keep_patches=256),
                                       div2k, a.steps, a.warmup, a.rounds, a.kernel_steps))
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")


if __name__ == "__main__":
    main()
