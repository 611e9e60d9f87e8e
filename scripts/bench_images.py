"""Image containers against the flow they replace, timed in the same run (ViT-B/16, K=64, throughput mode (bf16 operands)).

    compress:   MCM.compress_images  vs  compress_bitstream + the host HuffmanCoding of every image's ids_restore (testing.py:73-76,
                the reference's flow, whose side information is not decodable on its own)
    decompress: MCM.decompress_images  vs  decompress_bitstream given ids_restore
in images/s at batch 64 and latency at batch 1 (host clock around synchronised calls; the two paths alternate over --rounds rounds,
medians reported), then image_parse_kernel's device time from a per-launch profile taken in a run of its own (after the timed
ones), and the bytes per image split into header, patch selection, z and y, with the actual bpp (8 * bytes / pixels) beside the
likelihood estimate.  Every timed result is checked bit-exact against the forward, and the containers byte for byte against
the reference packing (tests/ref_image_container.py) of compress_bitstream's streams and forward's ids_keep.  The card name and
power limit are read (nvidia-smi --query-gpu, read-only) in the same run.

    python scripts/bench_images.py [--lanes 32 4] [--steps 20] [--warmup 3] [--rounds 3] [--out profiles/r07_images_B200.json]
"""
from __future__ import annotations

import argparse
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
from bench_decode import gpu_info  # noqa: E402
from tests import ref_image_container as R  # noqa: E402
from textmae_image_compression_b200 import MCM, make_state_dict, vit_base  # noqa: E402
from textmae_image_compression_b200.huffman import HuffmanCoding  # noqa: E402


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
        raise SystemExit("bench_images.py measures the GPU codec: no CUDA device")
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

    def reference_compress(lo, hi):
        enc = m.compress_bitstream(imgs[lo:hi], scores[lo:hi], lanes=lanes)
        ids = enc["ids_restore"].cpu()
        enc["side_info"] = [HuffmanCoding().compress(ids[i])[0] for i in range(hi - lo)]
        return enc

    def reference_decompress(enc, lo, hi):
        return m.decompress_bitstream([enc["strings"][0][lo:hi], enc["strings"][1][lo:hi]], enc["shape"], enc["ids_restore"][lo:hi],
                                      need_recon=False, lanes=lanes)

    paths = ("images", "reference")
    samples = {p: [] for p in paths}
    exact = True
    for _ in range(a.rounds):
        for p in paths:                                # the two paths alternate within every round
            r = {}
            if p == "images":
                r["compress_ms"], cont = host_time(lambda: m.compress_images(imgs, scores, lanes=lanes), a.steps, a.warmup)
                r["compress_batch1_ms"], _ = host_time(lambda: m.compress_images(imgs[:1], scores[:1], lanes=lanes), a.steps, a.warmup)
                r["decompress_ms"], out = host_time(lambda: m.decompress_images(cont, need_recon=False), a.steps, a.warmup)
                r["decompress_batch1_ms"], out1 = host_time(lambda: m.decompress_images(cont[:1], need_recon=False), a.steps, a.warmup)
            else:
                r["compress_ms"], enc = host_time(lambda: reference_compress(0, N), a.steps, a.warmup)
                r["compress_batch1_ms"], _ = host_time(lambda: reference_compress(0, 1), a.steps, a.warmup)
                r["decompress_ms"], out = host_time(lambda: reference_decompress(enc, 0, N), a.steps, a.warmup)
                r["decompress_batch1_ms"], out1 = host_time(lambda: reference_decompress(enc, 0, 1), a.steps, a.warmup)
            exact = exact and torch.equal(out["y_hat"], want_y) and torch.equal(out["z_hat"], want_z) and \
                torch.equal(out1["y_hat"], want_y[:1])
            samples[p].append(r)

    # the timed containers are the reference packing of compress_bitstream's streams and forward's ids_keep
    fields = dict(img_size=224, patch_size=16, mode=0, y_lanes=lanes[0], z_lanes=lanes[1],
                  tag=R.model_tag(m.entropy_tables(), m._scale_table.tolist()))
    exact = exact and all(cont[j] == R.pack(enc["strings"][0][j], enc["strings"][1][j], fwd["ids_keep"][j].tolist(), fields)
                          for j in range(N))

    # image_parse_kernel alone: a per-launch profile of one batch-64 decode, kept apart from the timed runs
    m.profile(True)
    m.decompress_images(cont, need_recon=False)
    torch.cuda.synchronize()
    steps = m.profile_read_steps()
    m.profile(False)
    parse_ms = sum(s["ms"] for s in steps if s["name"] == "image_parse")
    coder_ms = sum(s["ms"] for s in steps if s["name"].startswith("rans_decode"))

    def med(p, key):
        return statistics.median(r[key] for r in samples[p])

    pixels = 224 * 224
    parsed = [R.parse(c) for c in cont]
    ids_bytes = len(cont[0]) - R.HEADER - len(parsed[0]["z"]) - len(parsed[0]["y"])
    z_mean = sum(len(f["z"]) for f in parsed) / N
    y_mean = sum(len(f["y"]) for f in parsed) / N
    total_mean = sum(len(c) for c in cont) / N
    huff_bits = sum(len(s) for s in enc["side_info"]) / N
    res = {"config": f"ViT-B/16 K={K}, throughput mode (bf16 operands), synthetic checkpoint seed 0, batch {N}", **gpu_info(),
           "lanes": list(lanes), "steps": a.steps, "warmup": a.warmup, "rounds": a.rounds,
           "note": "host clock around synchronised calls, medians over the rounds, the two paths alternating within each round; "
                   "image_parse_kernel from a per-launch profile of one batch-64 decode run apart from the timed calls"}
    for p in paths:
        res[p] = {"compress_images_per_s": N * 1e3 / med(p, "compress_ms"), "compress_batch1_ms": med(p, "compress_batch1_ms"),
                  "decompress_images_per_s": N * 1e3 / med(p, "decompress_ms"), "decompress_batch1_ms": med(p, "decompress_batch1_ms")}
    i, rf = res["images"], res["reference"]
    res["images_over_reference"] = {
        "compress_images_per_s": i["compress_images_per_s"] / rf["compress_images_per_s"],
        "compress_batch1_ms": i["compress_batch1_ms"] / rf["compress_batch1_ms"],
        "decompress_images_per_s": i["decompress_images_per_s"] / rf["decompress_images_per_s"],
        "decompress_batch1_ms": i["decompress_batch1_ms"] / rf["decompress_batch1_ms"]}
    res["image_parse_kernel_device_ms_batch64"] = parse_ms
    res["rans_decode_device_ms_batch64"] = coder_ms
    res["bytes_per_image"] = {"header": R.HEADER, "patch_selection": ids_bytes, "z_mean": z_mean, "y_mean": y_mean,
                              "container_mean": total_mean}
    res["bpp"] = {"actual_container": 8 * total_mean / pixels, "actual_streams_only": 8 * (z_mean + y_mean) / pixels,
                  "patch_selection_and_header": 8 * (R.HEADER + ids_bytes) / pixels,
                  "likelihood_estimate": float(fwd["bpp"].mean()),
                  "reference_huffman_side_info": huff_bits / pixels}
    res["all_bit_exact"] = exact
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")
    if not exact:
        raise SystemExit("a timed result is not bit-exact")


if __name__ == "__main__":
    main()
