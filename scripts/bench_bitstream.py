"""Bitstream timings of MCM.compress_bitstream / decompress_bitstream (ViT-B/16, K=64, throughput mode) on the current GPU.

Reports, as one JSON document (stdout, and --out if given):
  - compress_bitstream images/s at batch 64 (host clock around synchronised calls: forward + encode + read back), and the
    encode kernels' own device time (device events around the two encode calls on the same symbols);
  - decompress_bitstream images/s at batch 64 and batch-1 latency, next to decompress_symbols one-shot (symbols given), so the
    coder's added cost shows;
  - the coder's per-stage device time (per-launch profile of one decode);
  - stream bits per image next to the likelihood-estimated bpp.
Every timed result is checked bit-exact (decoded y_hat / z_hat equal the forward's; GPU strings equal the oracle's).  The card
name and power limit are read (nvidia-smi --query-gpu, read-only) in the same run.

    python scripts/bench_bitstream.py [--steps 20] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import sys
import time
from pathlib import Path

sys.dont_write_bytecode = True
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

import torch  # noqa: E402

from bench_decode import gpu_info, time_device  # noqa: E402
from oracle import ref_rans  # noqa: E402
from textmae_image_compression_b200 import MCM, _native, entropy, make_state_dict, vit_base  # noqa: E402


def host_time(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(steps):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) * 1e3 / steps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bitstream.py measures the GPU coder: no CUDA device")
    K, N = 64, a.batch
    cfg = vit_base(K)
    sd = make_state_dict(cfg, seed=0, include_decoder=False)
    m = MCM(num_keep_patches=K)
    m.load_state_dict(sd)
    m.cuda().eval()
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(N, 3, 224, 224, generator=g).cuda()
    scores = torch.rand(N, cfg.num_patches, generator=g).cuda()
    m.update()
    res = {"config": f"ViT-B/16 K={K}, throughput mode (bf16 operands), synthetic checkpoint seed 0", **gpu_info(),
           "steps": a.steps, "warmup": a.warmup}
    fwd = m(imgs, scores, need_recon=False)
    want_y, want_z = fwd["latents"]["y_hat"], fwd["latents"]["z_hat"]
    sym = m.compress_symbols(imgs, scores)
    tabs = m.entropy_tables()

    # --- compress
    ms_c, enc = host_time(lambda: m.compress_bitstream(imgs, scores), a.steps, a.warmup)
    ys, yi = sym["y_symbols"].cpu().numpy(), sym["y_indexes"].cpu().numpy()
    gt = [tabs["gaussian_conditional." + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")]
    t0 = time.perf_counter()
    oracle_strings = [ref_rans.encode_with_indexes(ys[i], yi[i], *gt) for i in range(2)]
    oracle_ms = (time.perf_counter() - t0) * 1e3 / 2
    strings_exact = all(enc["strings"][0][i] == oracle_strings[i] for i in range(2))
    zs, zi = sym["z_symbols"].reshape(N, -1), sym["z_indexes"].reshape(N, -1).contiguous()
    h = m._handle

    def encode_only():
        entropy.encode(h, _native.MODEL_GAUSSIAN, sym["y_symbols"], sym["y_indexes"])
        entropy.encode(h, _native.MODEL_BOTTLENECK, zs, zi)
    enc_ms = time_device(encode_only, a.steps, a.warmup)
    res["compress_bitstream"] = {"batch": N, "ms": ms_c, "images_per_s": N * 1e3 / ms_c, "encode_kernels_device_ms": enc_ms,
                                 "y_strings_equal_oracle_first_2": strings_exact,
                                 "note": "host clock: forward + indexes + encode + offsets / bytes read back"}

    # --- decompress
    def dec(lo, hi):
        return m.decompress_bitstream([enc["strings"][0][lo:hi], enc["strings"][1][lo:hi]], enc["shape"], enc["ids_restore"][lo:hi],
                                      need_recon=False)
    ms_d, out = host_time(lambda: dec(0, N), a.steps, a.warmup)
    exact_d = torch.equal(out["y_hat"], want_y) and torch.equal(out["z_hat"], want_z)
    ms_d1, out1 = host_time(lambda: dec(0, 1), a.steps, a.warmup)
    exact_d1 = torch.equal(out1["y_hat"], want_y[:1])

    def sym_dec(lo, hi):
        return m.decompress_symbols(sym["z_symbols"][lo:hi], sym["ids_restore"][lo:hi], y_symbols=sym["y_symbols"][lo:hi], need_recon=False)
    ms_s = time_device(lambda: sym_dec(0, N), a.steps, a.warmup)
    ms_s1 = time_device(lambda: sym_dec(0, 1), a.steps, a.warmup)
    exact_s = torch.equal(sym_dec(0, N)["y_hat"], want_y)
    res["decompress_bitstream"] = {"batch": N, "ms": ms_d, "images_per_s": N * 1e3 / ms_d, "bit_exact": exact_d,
                                   "batch1_ms": ms_d1, "batch1_bit_exact": exact_d1,
                                   "note": "host clock: H2D of the bytes, coder + network in one enqueued decode, status read back"}
    res["decompress_symbols_one_shot"] = {"batch": N, "ms": ms_s, "images_per_s": N * 1e3 / ms_s, "batch1_ms": ms_s1,
                                          "bit_exact": exact_s, "note": "device events; symbols given, no coder"}

    # --- per-stage device time of the coder (one profiled decode, per launch)
    m.profile(True)
    dec(0, N)
    torch.cuda.synchronize()
    steps = m.profile_read_steps()
    m.profile(False)
    coder = [s for s in steps if s["name"].startswith("rans_decode")]
    res["coder_stages_batch64_ms"] = {s["name"]: s["ms"] for s in coder}
    res["coder_total_batch64_ms"] = sum(s["ms"] for s in coder)
    res["decode_total_profiled_batch64_ms"] = sum(s["ms"] for s in steps)
    m.profile(True)
    dec(0, 1)
    torch.cuda.synchronize()
    steps1 = m.profile_read_steps()
    m.profile(False)
    res["coder_total_batch1_ms"] = sum(s["ms"] for s in steps1 if s["name"].startswith("rans_decode"))

    # --- rate
    pixels = 224 * 224
    bits = [8 * (len(enc["strings"][0][i]) + len(enc["strings"][1][i])) for i in range(N)]
    res["rate"] = {"stream_bpp_mean": sum(bits) / N / pixels, "likelihood_bpp_mean": float(enc["bpp"].mean()),
                   "y_bytes_mean": sum(len(s) for s in enc["strings"][0]) / N, "z_bytes_mean": sum(len(s) for s in enc["strings"][1]) / N,
                   "note": "synthetic checkpoint: many y symbols escape their table; an escape costs its tail frequency plus "
                           "nibbles while the likelihood floor is 1e-9 (~30 bits), so stream bits can fall below the estimate"}
    res["oracle_python_encode_ms_per_image"] = oracle_ms
    res["all_bit_exact"] = bool(strings_exact and exact_d and exact_d1 and exact_s)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")
    if not res["all_bit_exact"]:
        raise SystemExit("a timed result is not bit-exact")


if __name__ == "__main__":
    main()
