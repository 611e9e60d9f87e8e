"""The laned rANS format against compressai's format, timed in the same run (ViT-B/16, K=64, throughput mode, batch 64).

For both formats - compressai's (one chain per stream) and the laned one with (W_y, W_z) lanes - reports, as one JSON document
(stdout, and --out if given):
  - compress_bitstream images/s (host clock around synchronised calls) and the encode kernels' device time;
  - decompress_bitstream images/s at batch 64 and batch-1 latency (host clock);
  - the coder's per-stage device time (per-launch profile of one batch-64 decode) and its total at batch 1;
  - mean y / z bytes per image and the stream bpp;
then the laned / compressai ratios.  The two formats alternate over --rounds rounds of every measurement; each figure is the
median over the rounds.  Every timed result is checked bit-exact (decoded y_hat / z_hat equal the forward's; the first two
images' strings equal the oracle's).  The card name and power limit are read (nvidia-smi --query-gpu, read-only) in the same run.

    python scripts/bench_bitstream_lanes.py [--lanes 32 4] [--steps 20] [--warmup 3] [--rounds 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import functools
import json
import statistics
import sys
from pathlib import Path

sys.dont_write_bytecode = True
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

import torch  # noqa: E402

from bench_bitstream import host_time  # noqa: E402
from bench_decode import gpu_info, time_device  # noqa: E402
from oracle import ref_rans  # noqa: E402
from tests import ref_rans_lanes  # noqa: E402
from textmae_image_compression_b200 import MCM, _native, entropy, make_state_dict, vit_base  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lanes", type=int, nargs=2, default=[32, 4])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bitstream_lanes.py measures the GPU coder: no CUDA device")
    K, N, lanes = 64, a.batch, tuple(a.lanes)
    cfg = vit_base(K)
    m = MCM(num_keep_patches=K)
    m.load_state_dict(make_state_dict(cfg, seed=0, include_decoder=False))
    m.cuda().eval()
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(N, 3, 224, 224, generator=g).cuda()
    scores = torch.rand(N, cfg.num_patches, generator=g).cuda()
    m.update()
    fwd = m(imgs, scores, need_recon=False)
    want_y, want_z = fwd["latents"]["y_hat"], fwd["latents"]["z_hat"]
    sym = m.compress_symbols(imgs, scores)
    tabs = m.entropy_tables()
    gt = [tabs["gaussian_conditional." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    bt = [tabs["entropy_bottleneck." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    ys, yi = sym["y_symbols"].cpu().numpy(), sym["y_indexes"].cpu().numpy()
    zs, zi = sym["z_symbols"].reshape(N, -1).contiguous(), sym["z_indexes"].reshape(N, -1).contiguous()
    zsn, zin = zs.cpu().numpy(), zi.cpu().numpy()
    h = m._handle
    formats = {"compressai": None, "laned": lanes}

    @functools.lru_cache(maxsize=None)
    def oracle(fmt, i):
        if fmt is None:
            return ref_rans.encode_with_indexes(ys[i], yi[i], *gt), ref_rans.encode_with_indexes(zsn[i], zin[i], *bt)
        return ref_rans_lanes.encode_lanes(ys[i], yi[i], fmt[0], *gt), ref_rans_lanes.encode_lanes(zsn[i], zin[i], fmt[1], *bt)

    def encode_only(fmt):
        if fmt is None:
            entropy.encode(h, _native.MODEL_GAUSSIAN, sym["y_symbols"], sym["y_indexes"])
            entropy.encode(h, _native.MODEL_BOTTLENECK, zs, zi)
        else:
            entropy.encode_lanes(h, _native.MODEL_GAUSSIAN, sym["y_symbols"], sym["y_indexes"], fmt[0])
            entropy.encode_lanes(h, _native.MODEL_BOTTLENECK, zs, zi, fmt[1])

    def coder_profile(dec, lo, hi):
        m.profile(True)
        dec(lo, hi)
        torch.cuda.synchronize()
        steps = m.profile_read_steps()
        m.profile(False)
        return {s["name"]: s["ms"] for s in steps if s["name"].startswith("rans_decode")}

    samples = {k: [] for k in formats}
    exact = {}
    for _ in range(a.rounds):
        for name, fmt in formats.items():          # the two formats alternate within every round
            r = {}
            r["compress_ms"], enc = host_time(lambda: m.compress_bitstream(imgs, scores, lanes=fmt), a.steps, a.warmup)
            r["encode_kernels_device_ms"] = time_device(lambda: encode_only(fmt), a.steps, a.warmup)

            def dec(lo, hi):
                return m.decompress_bitstream([enc["strings"][0][lo:hi], enc["strings"][1][lo:hi]], enc["shape"],
                                              enc["ids_restore"][lo:hi], need_recon=False, lanes=fmt)
            r["decompress_ms"], out = host_time(lambda: dec(0, N), a.steps, a.warmup)
            r["decompress_batch1_ms"], out1 = host_time(lambda: dec(0, 1), a.steps, a.warmup)
            stages = coder_profile(dec, 0, N)
            r["coder_stages_ms"] = stages
            r["coder_device_ms"] = sum(stages.values())
            r["coder_device_batch1_ms"] = sum(coder_profile(dec, 0, 1).values())
            ok = (torch.equal(out["y_hat"], want_y) and torch.equal(out["z_hat"], want_z) and torch.equal(out1["y_hat"], want_y[:1])
                  and all(tuple(enc["strings"][k][i] for k in (0, 1)) == oracle(fmt, i) for i in range(2)))
            exact[name] = exact.get(name, True) and ok
            r["y_bytes_mean"] = sum(len(s) for s in enc["strings"][0]) / N
            r["z_bytes_mean"] = sum(len(s) for s in enc["strings"][1]) / N
            samples[name].append(r)

    def med(name, key):
        return statistics.median(r[key] for r in samples[name])

    res = {"config": f"ViT-B/16 K={K}, throughput mode (bf16 operands), synthetic checkpoint seed 0, batch {N}", **gpu_info(),
           "lanes": list(lanes), "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
           "note": "host clock for compress / decompress (synchronised calls); device events for the encode kernels; per-launch "
                   "profile for the coder stages; medians over the rounds, the two formats alternating within each round"}
    pixels = 224 * 224
    for name in formats:
        last = samples[name][-1]
        res[name] = {
            "compress_images_per_s": N * 1e3 / med(name, "compress_ms"), "compress_ms": med(name, "compress_ms"),
            "encode_kernels_device_ms": med(name, "encode_kernels_device_ms"),
            "decompress_images_per_s": N * 1e3 / med(name, "decompress_ms"), "decompress_ms": med(name, "decompress_ms"),
            "decompress_batch1_ms": med(name, "decompress_batch1_ms"),
            "coder_device_ms": med(name, "coder_device_ms"), "coder_device_batch1_ms": med(name, "coder_device_batch1_ms"),
            "coder_stages_ms_last_round": last["coder_stages_ms"],
            "y_bytes_mean": last["y_bytes_mean"], "z_bytes_mean": last["z_bytes_mean"],
            "stream_bpp_mean": 8 * (last["y_bytes_mean"] + last["z_bytes_mean"]) / pixels,
            "bit_exact": exact[name]}
    c, l = res["compressai"], res["laned"]
    res["laned_over_compressai"] = {
        "coder_device_ms": l["coder_device_ms"] / c["coder_device_ms"],
        "encode_kernels_device_ms": l["encode_kernels_device_ms"] / c["encode_kernels_device_ms"],
        "decompress_images_per_s": l["decompress_images_per_s"] / c["decompress_images_per_s"],
        "decompress_batch1_ms": l["decompress_batch1_ms"] / c["decompress_batch1_ms"],
        "stream_bytes": (l["y_bytes_mean"] + l["z_bytes_mean"]) / (c["y_bytes_mean"] + c["z_bytes_mean"])}
    r = res["laned_over_compressai"]
    res["acceptance"] = {"coder_device_ms <= 1/4": r["coder_device_ms"] <= 0.25,
                         "encode_kernels_device_ms <= 1/4": r["encode_kernels_device_ms"] <= 0.25,
                         "decompress_images_per_s >= 3x": r["decompress_images_per_s"] >= 3.0,
                         "decompress_batch1_ms <= 1/2": r["decompress_batch1_ms"] <= 0.5,
                         "stream_bytes <= 1.03": r["stream_bytes"] <= 1.03}
    res["all_bit_exact"] = all(exact.values())
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")
    if not res["all_bit_exact"]:
        raise SystemExit("a timed result is not bit-exact")


if __name__ == "__main__":
    main()
