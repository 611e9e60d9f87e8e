"""Synthesis (x_hat from y_hat: g_s, the MAE decoder, unpatchify) on the engine against recon.synthesize in fp32 torch, timed in
the same run (ViT-B/16, K=64, throughput mode).

Reports, as one JSON document (stdout, and --out if given):
  - synthesis alone at batch 64 and at batch 1 (device events around --steps back-to-back calls), torch and native;
  - images/s of decompress_bitstream(lanes=(32, 4), need_recon=True) and of forward(need_recon=True) (host clock around
    synchronised calls), torch and native;
  - the native plan's device time per step family (per-launch profile of one batch-64 call) and its achieved TFLOP/s against
    the 10.9 GFLOP per image the synthesis needs (counted from shapes: g_s 0.19, decoder_embed 0.05, block linears 9.91,
    attention 0.64, decoder_pred 0.155);
  - the native x_hat against the torch one (relative L2, max abs; the tests require <= 1.5e-2 and <= 0.1).
Torch and native alternate over --rounds rounds of every measurement; each figure is the median over the rounds.  --vitl adds a
ViT-L/16 512^2 K=256 line (synthesis alone at batch 8).  The card name and power limit are read (nvidia-smi --query-gpu,
read-only) in the same run.

    python scripts/bench_synthesis.py [--steps 20] [--warmup 3] [--rounds 3] [--vitl] [--out result.json]
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
from bench_decode import gpu_info, time_device  # noqa: E402
from textmae_image_compression_b200 import MCM, make_state_dict, recon, vit_base, vit_large  # noqa: E402


def synth_gflop(cfg) -> float:
    """GFLOP per image of recon.synthesize, counted from shapes."""
    K, L, E, Dd, Cy = cfg.num_keep_patches, cfg.num_patches, cfg.encoder_embed_dim, cfg.decoder_embed_dim, cfg.latent_depth
    T, mlp = L + 1, int(cfg.decoder_embed_dim * cfg.mlp_ratio)
    ch = [Cy] + cfg.g_a_channels()[::-1][1:]
    gs = sum(2 * K * ch[i] * ch[i + 1] for i in range(4))
    blocks = cfg.decoder_depth * (2 * T * Dd * (3 * Dd + Dd + 2 * mlp) + 4 * T * T * Dd)
    return (gs + 2 * K * E * Dd + blocks + 2 * T * Dd * cfg.patch_size ** 2 * 3) / 1e9


def models(cfg, kw, share_sm=False):
    sd = make_state_dict(cfg, seed=0, include_decoder=True)
    out = {}
    for name, native in (("torch", False), ("native", True)):
        m = MCM(**kw, native_synthesis=native, share_sm=share_sm)
        m.load_state_dict(sd)
        out[name] = m.cuda().eval()
    return out


def synth_fn(m, y, ids):
    """One synthesis call of either path on the current stream."""
    c = m.cfg
    if m._syn_on:
        cur = torch.cuda.current_stream()
        return lambda: m._synthesize(y, ids, cur)
    return lambda: recon.synthesize(m._weights, c, y.reshape(y.shape[0], c.num_keep_patches, c.latent_depth), ids)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--vitl", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_synthesis.py measures the GPU synthesis: no CUDA device")
    res = {"workload": f"ViT-B/16 224^2 K=64, bf16, batch {a.batch} (and 1)", **gpu_info(), "gflop_per_image": None}
    K, N = 64, a.batch
    cfg = vit_base(K)
    res["gflop_per_image"] = round(synth_gflop(cfg), 3)
    ms = models(cfg, dict(num_keep_patches=K))
    ms["native"]._ensure_handle()
    assert ms["native"]._syn_on
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(N, 3, 224, 224, generator=g).cuda()
    scores = torch.rand(N, cfg.num_patches, generator=g).cuda()
    fwd = ms["native"](imgs, scores, need_recon=False)
    y, ids = fwd["latents"]["y_hat"].permute(0, 2, 3, 1).contiguous(), fwd["ids_restore"]
    # accuracy of the timed native output
    x_t, x_n = synth_fn(ms["torch"], y, ids)(), synth_fn(ms["native"], y, ids)()
    torch.cuda.synchronize()
    d = (x_n.double() - x_t.double())
    res["native_vs_torch"] = {"rel_l2": d.norm().item() / x_t.double().norm().item(), "max_abs": d.abs().max().item(),
                              "psnr_db": (10 * torch.log10(1.0 / d.pow(2).mean())).item()}
    bs = ms["native"].compress_bitstream(imgs, scores, lanes=(32, 4))
    times = {k: [] for k in ("synth_ms_b%d" % N, "synth_ms_b1", "decompress_bitstream_ips", "forward_recon_ips")}
    out = {"torch": {k: [] for k in times}, "native": {k: [] for k in times}}
    for _ in range(a.rounds):
        for name in ("torch", "native"):
            m = ms[name]
            out[name]["synth_ms_b%d" % N].append(time_device(synth_fn(m, y, ids), a.steps, a.warmup))
            out[name]["synth_ms_b1"].append(time_device(synth_fn(m, y[:1].contiguous(), ids[:1].contiguous()), a.steps, a.warmup))
            t, _ = host_time(lambda: m.decompress_bitstream(bs["strings"], bs["shape"], bs["ids_restore"], lanes=(32, 4), need_recon=True),
                             a.steps, a.warmup)
            out[name]["decompress_bitstream_ips"].append(N / (t * 1e-3))
            t, _ = host_time(lambda: m(imgs, scores, need_recon=True), a.steps, a.warmup)
            out[name]["forward_recon_ips"].append(N / (t * 1e-3))
    for name in out:
        res[name] = {k: round(statistics.median(v), 4 if "ms" in k else 1) for k, v in out[name].items()}
    nat = ms["native"]
    res["native"]["tflops_b%d" % N] = round(res["gflop_per_image"] * N / (res["native"]["synth_ms_b%d" % N] * 1e-3) / 1e3, 1)
    res["speedup"] = {k: round(res["torch"][k] / res["native"][k] if "ms" in k else res["native"][k] / res["torch"][k], 2)
                      for k in times}
    # per step family of one profiled batch-64 call (plain launches with events: slower than the graph replay)
    nat.profile(True)
    synth_fn(nat, y, ids)()
    torch.cuda.synchronize()
    fam = {}
    for s in nat.profile_read_steps():
        n = s["name"]
        key = ("attention" if n.endswith(".attn") else "block_gemms" if n.startswith("dec_blk") else n.split(".")[0])
        f = fam.setdefault(key, {"ms": 0.0, "gflop": 0.0})
        f["ms"] += s["ms"]
        f["gflop"] += s["flops"] / 1e9
    nat.profile(False)
    res["native_profile_b%d" % N] = {k: {"ms": round(v["ms"], 4), "gflop": round(v["gflop"], 2),
                                          "tflops": round(v["gflop"] / v["ms"], 1) if v["ms"] > 0 and v["gflop"] > 0 else None}
                                      for k, v in fam.items()}
    if a.vitl:
        cl = vit_large(256, 512)
        kw = dict(img_size=512, encoder_embed_dim=1024, encoder_depth=24, encoder_num_heads=16, num_keep_patches=256)
        del ms, nat
        ml = models(cl, kw)
        nl = 8
        gl = torch.Generator().manual_seed(1)
        fl = ml["native"](torch.rand(nl, 3, 512, 512, generator=gl).cuda(), torch.rand(nl, cl.num_patches, generator=gl).cuda(),
                          need_recon=False)
        yl, il = fl["latents"]["y_hat"].permute(0, 2, 3, 1).contiguous(), fl["ids_restore"]
        xt, xn = synth_fn(ml["torch"], yl, il)(), synth_fn(ml["native"], yl, il)()
        torch.cuda.synchronize()
        dl = xn.double() - xt.double()
        line = {"workload": f"ViT-L/16 512^2 K=256, bf16, batch {nl}", "gflop_per_image": round(synth_gflop(cl), 2),
                "rel_l2": dl.norm().item() / xt.double().norm().item(), "max_abs": dl.abs().max().item()}
        tt, tn = [], []
        for _ in range(a.rounds):
            tt.append(time_device(synth_fn(ml["torch"], yl, il), max(a.steps // 4, 3), 1))
            tn.append(time_device(synth_fn(ml["native"], yl, il), max(a.steps // 4, 3), 1))
        line["torch_synth_ms"], line["native_synth_ms"] = round(statistics.median(tt), 3), round(statistics.median(tn), 3)
        line["native_tflops"] = round(line["gflop_per_image"] * nl / (line["native_synth_ms"] * 1e-3) / 1e3, 1)
        res["vitl_512_K256"] = line
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")


if __name__ == "__main__":
    main()
