"""Decode-side timings of MCM.decompress_symbols (ViT-B/16, K=64, throughput mode) on the current GPU.

Reports, as one JSON document (stdout, and --out if given):
  - one-shot decode images/s at batch 64 (all symbols given up front; device events around the whole call);
  - batch-1 one-shot latency;
  - batch-1 stepwise latency: after each of the 7 slice-group stages the indexes go device -> host and the group's symbols
    host -> device, standing in for the range decoder.  The range decoder's own time is NOT included;
  - the fp32 oracle's decode of one image on one host thread (the reference's eval CLI decodes image by image on the CPU).
Every timed decode is checked to reproduce the forward's y_hat bit for bit.  The card name and power limit are read
(nvidia-smi --query-gpu, read-only) in the same run.

    python scripts/bench_decode.py [--steps 20] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

sys.dont_write_bytecode = True
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from oracle import ref_decode  # noqa: E402
from textmae_image_compression_b200 import MCM, make_state_dict, vit_base  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        name, power = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:                                   # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def time_device(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decode.py measures the GPU decode: no CUDA device")
    K, N = 64, a.batch
    cfg = vit_base(K)
    sd = make_state_dict(cfg, seed=0)
    m = MCM(num_keep_patches=K)
    m.load_state_dict(sd)
    m.cuda().eval()
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(N, 3, 224, 224, generator=g).cuda()
    scores = torch.rand(N, cfg.num_patches, generator=g).cuda()
    m.update()
    sym = m.compress_symbols(imgs, scores)
    fwd = m(imgs, scores, need_recon=False)
    want = fwd["latents"]["y_hat"]
    res = {"config": f"ViT-B/16 K={K}, throughput mode (bf16 operands)", **gpu_info(), "steps": a.steps, "warmup": a.warmup}

    def one_shot(lo, hi):
        return m.decompress_symbols(sym["z_symbols"][lo:hi], sym["ids_restore"][lo:hi], y_symbols=sym["y_symbols"][lo:hi])

    ms = time_device(lambda: one_shot(0, N), a.steps, a.warmup)
    exact = torch.equal(one_shot(0, N)["y_hat"], want)
    res["one_shot_batch"] = {"batch": N, "ms": ms, "images_per_s": N * 1e3 / ms, "y_hat_bit_exact": exact}
    ms1 = time_device(lambda: one_shot(0, 1), a.steps, a.warmup)
    exact1 = torch.equal(one_shot(0, 1)["y_hat"], want[:1])
    res["one_shot_batch1"] = {"ms": ms1, "y_hat_bit_exact": exact1}

    host_sym = sym["y_symbols"][:1].view(1, cfg.num_slices, cfg.slice_ch, cfg.side, cfg.side).cpu()

    def decode_fn(first, indexes):
        indexes.cpu()                                       # D2H of the group's indexes (the range decoder's input)
        return host_sym[:, first:first + indexes.shape[1]]   # host symbols, copied H2D by decompress_symbols

    def stepwise():
        return m.decompress_symbols(sym["z_symbols"][:1], sym["ids_restore"][:1], decode_fn=decode_fn)

    for _ in range(a.warmup):
        stepwise()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(a.steps):
        out = stepwise()
    torch.cuda.synchronize()
    res["stepwise_batch1"] = {"ms": (time.perf_counter() - t) * 1e3 / a.steps, "y_hat_bit_exact": torch.equal(out["y_hat"], want[:1]),
                              "note": "host clock; includes 7 index D2H + symbol H2D round trips; range-decoder time excluded"}

    torch.set_num_threads(1)
    z1, y1 = sym["z_symbols"][:1].cpu(), sym["y_symbols"][:1].cpu()
    table = MCM.get_scale_table()
    ref_decode.decode_from_symbols(sd, cfg, z1, y1, table)
    t = time.perf_counter()
    reps = 3
    for _ in range(reps):
        ref_decode.decode_from_symbols(sd, cfg, z1, y1, table)
    res["oracle_fp32_cpu_1thread"] = {"ms": (time.perf_counter() - t) * 1e3 / reps,
                                      "note": "fp32 torch decode_from_symbols of one image, one host thread, same slice loop"}
    res["all_bit_exact"] = bool(exact and exact1 and res["stepwise_batch1"]["y_hat_bit_exact"])
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")
    if not res["all_bit_exact"]:
        raise SystemExit("decoded y_hat differs from the forward's")


if __name__ == "__main__":
    main()
