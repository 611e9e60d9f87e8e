#!/usr/bin/env python
"""Benchmark of the compression forward path (encode + rate), BASELINE.json metric:
images/s masked-ViT encode+rate.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--precise all|rate]
                    [--scaling weak|strong] [--dump-outputs DIR]

One "step" = one pass of the path (mask-select -> gather -> ViT encoder -> g_a/h_a/h_s/slice nets -> quantise ->
likelihoods -> bpp) over one batch of images.  Default workload = BASELINE.json configs[1]: synthetic 224x224, batch 64
per GPU, ViT-B/16, K=64 kept patches (nearest valid value to mask ratio 0.75; the reference needs sqrt(K) % 4 == 0,
SURVEY 0.2 #4), bf16 tensor-core operands, fp32 accumulate.  The other BASELINE configs are `--workload` names:
  KODAK24 / KODAK24_K64   the 24 bundled Kodak images through the reference's test transform (224x224) + reference-generated
                          scores (tests/golden), ViT-B/16, K=144 (shipped) / K=64; also reports the batch-1 latency (config 1)
  TILES288                config 3 native-resolution extension: 24 images x 12 tiles of 224x224 = 288 tiles (synthetic pixels
                          and Kodak-like heavy-tie scores: the native PNGs and the score generator do not travel)
  L256                    config 4: synthetic 512x512, ViT-L/16, K=256, 32 images per GPU (256 over 8 GPUs)
  DIV2K_L400/_L256/_L144  config 5: one 2048x1080 image = 12 tiles of 512x512, ViT-L/16, K = 400 / 256 / 144
Images are sharded across ranks, weights replicated; the only collective is the 16-byte rate all-reduce per step.
`--scaling weak` (default): every rank runs the workload's batch; `--scaling strong`: the workload's batch is the
GLOBAL batch, sharded with distributed.shard_range.
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step returned to its caller as DIR/<name>.npy
(see dump_outputs); inputs and weights are seeded, so two builds run with the same arguments can be compared array by array.
With --impl reference it writes the fp32 oracle's outputs, under the same names, for the inputs of the B200 path's last
timed step with the same arguments (the reference arm times a sample of other images), minus rate_sums and ids_shuffle.

--impl reference: the reference's CPU implementation of the same path (the in-repo fp32 oracle, bit-identical to the
reference's MCM.forward - tests/test_reference_exec.py) on all host cores, same images per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

VIT_L = dict(img_size=512, encoder_embed_dim=1024, encoder_depth=24, encoder_num_heads=16)
WORKLOADS = {
    # name: (model kwargs, batch, description, input kind)
    "B64": (dict(img_size=224, num_keep_patches=64), 64,
            "synthetic 224x224 batch 64/GPU, ViT-B/16, K=64 (67% masked; nearest valid to 0.75)", "uniform"),
    "B144": (dict(img_size=224, num_keep_patches=144), 64,
             "synthetic 224x224 batch 64/GPU, ViT-B/16, K=144 (shipped test.sh value)", "uniform"),
    "L256": (dict(num_keep_patches=256, **VIT_L), 32,
             "synthetic 512x512 batch 32/GPU, ViT-L/16, K=256 (75% masked)", "uniform"),
    "KODAK24": (dict(img_size=224, num_keep_patches=144), 24,
                "24 Kodak images, reference test transform (224x224) + reference-generated scores, ViT-B/16, K=144", "kodak"),
    "KODAK24_K64": (dict(img_size=224, num_keep_patches=64), 24,
                    "24 Kodak images, reference test transform (224x224) + reference-generated scores, ViT-B/16, K=64", "kodak"),
    "TILES288": (dict(img_size=224, num_keep_patches=144), 288,
                 "Kodak native-resolution tiling shape: 24 images x 12 tiles of 224x224 = 288 tiles (synthetic pixels, "
                 "heavy-tie scores), ViT-B/16, K=144", "ties"),
    "DIV2K_L400": (dict(num_keep_patches=400, **VIT_L), 12,
                   "DIV2K-shaped 2048x1080 -> 12 tiles of 512x512, ViT-L/16, K=400 (mask ratio 0.61)", "uniform"),
    "DIV2K_L256": (dict(num_keep_patches=256, **VIT_L), 12,
                   "DIV2K-shaped 2048x1080 -> 12 tiles of 512x512, ViT-L/16, K=256 (mask ratio 0.75)", "uniform"),
    "DIV2K_L144": (dict(num_keep_patches=144, **VIT_L), 12,
                   "DIV2K-shaped 2048x1080 -> 12 tiles of 512x512, ViT-L/16, K=144 (mask ratio 0.86)", "uniform"),
}
# reference-algorithmic GFLOP per image (SURVEY 6.2: embed all L patches, all 12 LRP nets); closed forms for the others
ALGO_GFLOP_PER_IMG = {"B64": 20.761, "B144": 46.636, "L256": 201.005, "KODAK24": 46.636, "KODAK24_K64": 20.761,
                      "TILES288": 46.636, "DIV2K_L256": 201.005}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm_sorted = sorted(sm)
        return {"sm_mhz": sm_sorted[len(sm_sorted) // 2], "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


def make_inputs(kwargs, batch, seed, n_rot, kind="uniform"):
    """n_rot batches of (imgs [batch,3,S,S], scores [batch,L]) on the host."""
    g = torch.Generator().manual_seed(seed)
    S = kwargs["img_size"]
    L = (S // 16) ** 2
    if kind == "kodak":
        import numpy as np
        z = np.load(ROOT / "tests" / "golden" / "kodak_224.npz")
        imgs = torch.from_numpy(z["imgs"]).permute(0, 3, 1, 2).float() / 255.0          # reference test transform, no normalise
        scores = torch.load(ROOT / "tests" / "golden" / "kodak_scores.pt")               # reference score generator
        reps = (batch + imgs.shape[0] - 1) // imgs.shape[0]
        imgs, scores = imgs.repeat(reps, 1, 1, 1)[:batch].contiguous(), scores.repeat(reps, 1)[:batch].contiguous()
        return [imgs.clone() for _ in range(n_rot)], [scores.clone() for _ in range(n_rot)]
    imgs = [torch.rand(batch, 3, S, S, generator=g) for _ in range(n_rot)]
    if kind == "ties":          # Kodak-like heavy-tie integer products, min-max normalised (SURVEY 8d config 2)
        scores = []
        for _ in range(n_rot):
            a = torch.randint(0, 40, (batch, L), generator=g).float() * torch.randint(0, 165, (batch, L), generator=g).float()
            lo, hi = a.min(1, keepdim=True)[0], a.max(1, keepdim=True)[0]
            scores.append((a - lo) / (hi - lo).clamp_min(1.0))
    else:
        scores = [torch.rand(batch, L, generator=g) for _ in range(n_rot)]
    return imgs, scores


DUMP_BUDGET_BYTES = 64 * 10**6


def dump_outputs(out, dirname):
    """Writes every tensor of a forward's result dict as <dirname>/<name>.npy, nested keys joined by "_"
    (likelihoods_y, latents_y_sym, bpp, ids_restore, ...): float32 outputs as float32, the rest (fp64 rate sums, integer
    symbols and indices) as float64, which holds them exactly.  When the files would exceed DUMP_BUDGET_BYTES in all,
    each array above 1 MiB is replaced by the same fraction of its elements, flattened, at indices drawn from a fixed
    seed: the same arguments give the same sample."""
    import numpy as np
    arrays = {}

    def collect(prefix, v):
        if isinstance(v, dict):
            for k, x in v.items():
                collect(f"{prefix}{k}_", x)
        elif torch.is_tensor(v):
            dt = torch.float32 if v.dtype == torch.float32 else torch.float64
            arrays[prefix[:-1]] = np.ascontiguousarray(v.detach().to("cpu", dt).numpy())

    collect("", out)
    room = DUMP_BUDGET_BYTES - 1024 * len(arrays)               # .npy headers
    if sum(a.nbytes for a in arrays.values()) > room:
        big = [n for n, a in arrays.items() if a.nbytes > 2**20]
        frac = (room - sum(a.nbytes for n, a in arrays.items() if n not in big)) / sum(arrays[n].nbytes for n in big)
        for name in big:
            a = arrays[name]
            idx = np.random.default_rng(0).choice(a.size, int(a.size * frac), replace=False)
            arrays[name] = a.reshape(-1)[np.sort(idx)]
    d = Path(dirname)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", a)


def algo_gflop_per_image(cfg, wl):
    """Reference-algorithmic GFLOP per image (2 x MAC; SURVEY 6.2 closed forms)."""
    if wl in ALGO_GFLOP_PER_IMG:
        return ALGO_GFLOP_PER_IMG[wl]
    K, T, C, D, L = cfg.num_keep_patches, cfg.tokens, cfg.encoder_embed_dim, cfg.encoder_depth, cfg.num_patches
    f = 2.0 * L * cfg.patch_dim * C + 24.0 * D * T * C * C + 4.0 * D * T * T * C
    ch = cfg.g_a_channels()
    f += 2.0 * K * sum(ch[i] * ch[i + 1] for i in range(4))
    side = cfg.side
    for cin, cout, st in cfg.h_a_layers():
        side = side // st
        f += 2.0 * side * side * 9 * cin * cout
    side = cfg.side // 4
    for cin, cout, r in cfg.h_s_layers():
        f += 2 * (2.0 * side * side * 9 * cin * cout * r * r)
        side *= r
    for i in range(cfg.num_slices):
        for chans, mult in ((cfg.cc_channels(i), 2), (cfg.lrp_channels(i), 1)):
            f += mult * sum(2.0 * K * 9 * chans[j] * chans[j + 1] for j in range(5))
    return f / 1e9


# ----------------------------------------------------------------------------------------------------------
def rotation_count(kwargs, batch):
    """Input batches the timed B200 loop rotates over: together > 126 MB L2 (with the weights)."""
    img_bytes = batch * 3 * kwargs["img_size"] ** 2 * 4
    return max(2, min(8, int(320e6 // max(img_bytes, 1)) + 1))


def run_reference(args, kwargs, batch, desc, kind):
    """The reference's CPU path (fp32 oracle == reference MCM.forward bit for bit) on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_model
    from textmae_image_compression_b200 import PathConfig, make_state_dict
    cfg = PathConfig(**kwargs)
    sd = make_state_dict(cfg, seed=0)
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    imgs, scores = make_inputs(kwargs, batch, 0, 1, kind)
    sample = batch if args.ref_sample <= 0 else min(batch, args.ref_sample)
    t0 = time.perf_counter()
    ref_model.forward_rate(sd, cfg, imgs[0][:sample], scores[0][:sample])                 # warm-up step (also sizes the run)
    t_step = time.perf_counter() - t0
    budget = 240.0                                                                         # the whole run ends within a few minutes
    planned = (args.steps + max(args.warmup - 1, 0)) * t_step
    if planned > budget:
        sample = max(1, int(sample * budget / planned))
    for _ in range(max(min(args.warmup, 2) - 1, 0)):
        ref_model.forward_rate(sd, cfg, imgs[0][:sample], scores[0][:sample])
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref_model.forward_rate(sd, cfg, imgs[0][:sample], scores[0][:sample])
    dt = time.perf_counter() - t0
    val = sample * args.steps / dt
    # the testing.py:29 configuration: one thread, batch 1
    torch.set_num_threads(1)
    ref_model.forward_rate(sd, cfg, imgs[0][:1], scores[0][:1])
    t1 = time.perf_counter()
    reps = 0
    while reps < 2 or (time.perf_counter() - t1 < 6.0 and reps < 10):
        ref_model.forward_rate(sd, cfg, imgs[0][:1], scores[0][:1])
        reps += 1
    one_thread = reps / (time.perf_counter() - t1)
    torch.set_num_threads(cores)
    line = {
        "impl": "reference", "metric": "images/s masked-ViT encode+rate", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic" if kind != "kodak" else "kodak",
        "config": {"workload": desc, "name": args.workload, "per_gpu_batch": batch, "sample": f"{sample} of {batch} images per step",
                   "same_config": sample == batch},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} images/step x {args.steps} steps, fp32 oracle (oracle/ref_model.py; bit-identical to the "
                                   f"reference MCM.forward executed in the build container), host python mask routine included",
                         "single_thread_batch1": {"value": one_thread, "unit": "images/s", "cores": 1,
                                                  "note": "testing.py:29 torch.set_num_threads(1), batch 1"}},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        n_rot = rotation_count(kwargs, batch)
        imgs_b, scores_b = make_inputs(kwargs, batch, 1000, n_rot, kind)
        r = ref_model.forward_rate(sd, cfg, imgs_b[(args.steps - 1) % n_rot], scores_b[(args.steps - 1) % n_rot])
        dump_outputs({"likelihoods": r["likelihoods"], "bpp": r["bpp"], "ids_restore": r["ids_restore"], "ids_keep": r["ids_keep"],
                      "latents": {k: r[k] for k in ("y_sym", "z_sym", "y_hat", "z_hat")}}, args.dump_outputs)


# ----------------------------------------------------------------------------------------------------------
class Runner:
    """S handles / streams of one model configuration on this rank's GPU and the timed loops over them."""

    def __init__(self, kwargs, batch, S, precise, dev, world):
        from textmae_image_compression_b200 import MCM, PathConfig, make_state_dict
        self.cfg = PathConfig(**kwargs)
        sd = make_state_dict(self.cfg, seed=0)                     # replicated weights
        self.models = []
        for _ in range(S):
            m_ = MCM(**kwargs, skip_dead_lrp=False, share_sm=S > 1, precise=precise)
            m_.load_state_dict(sd)
            m_.cuda().eval()
            m_.reserve(batch)
            self.models.append(m_)
        self.S, self.batch, self.dev, self.world = S, batch, dev, world
        self.stream = torch.cuda.current_stream()
        self.side = [torch.cuda.Stream(device=dev) for _ in range(S)]

    def fork(self, ev):
        ev.record(self.stream)
        for s_ in self.side:
            s_.wait_event(ev)

    def join(self, ev):
        for s_ in self.side:
            self.stream.wait_stream(s_)
        ev.record(self.stream)

    def barrier(self):
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, step_fn, steps):
        """EXACTLY `steps` steps between a barrier + synchronize on both sides; device time, max over ranks (ms)."""
        import torch.distributed as dist
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        self.fork(e0)
        out = None
        for i in range(steps):
            out = step_fn(i)
        self.join(e1)
        self.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item(), out


def run_b200(args, kwargs, batch_named, desc, wl, kind):
    import torch.distributed as dist
    from textmae_image_compression_b200 import distributed as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    strong = args.scaling == "strong"
    if strong:                                      # the named batch is the GLOBAL batch: this rank's shard of it
        lo, hi = D.shard_range(batch_named, rank, world)
        batch = hi - lo
        global_batch = batch_named
    else:
        batch, global_batch = batch_named, batch_named * world
    # `--streams S` pipelines S batches through S independent handles (own workspace, own CUDA stream): the serial
    # slice chain of one batch leaves most SMs idle, a second batch in flight fills them.  A step is still one batch.
    S = max(1, args.streams)
    R = Runner(kwargs, max(batch, 1), S, args.precise, dev, world)
    cfg, models, model = R.cfg, R.models, R.models[0]
    n_rot = rotation_count(kwargs, batch)
    imgs_h, scores_h = make_inputs(kwargs, batch, 1000 + rank, n_rot, kind)
    imgs_d = [t.cuda() for t in imgs_h]
    scores_d = [t.cuda() for t in scores_h]

    def step_dev(i):
        with torch.cuda.stream(R.side[i % S]):
            out = models[i % S](imgs_d[i % n_rot], scores_d[i % n_rot], need_recon=False)
            if world > 1:
                D.aggregate_rate(out["rate_sums"])            # the path's only collective (16 bytes)
        return out

    # ---- device-resident throughput -------------------------------------------------------------------
    # every handle needs 3 forwards before it is in steady state (plain launches, graph capture, first replay) and its
    # stream's allocator pool is populated: warm up max(W, 3 S) steps so none of that lands in the timed region
    warm_eff = max(args.warmup, 3 * S)
    # the clock sampler (nvidia-smi -lms 100) starts BEFORE the warm-up: its process start / NVML initialisation stalls
    # the GPU for tens of ms, which must not fall into a 40 ms timed region; it then samples through both timed regions
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for i in range(S):                                        # first call per handle: lazy initialisation (plans, NCCL)
        step_dev(i)
    torch.cuda.synchronize()
    t_warm = time.perf_counter()
    for i in range(S, warm_eff):
        step_dev(i)
    torch.cuda.synchronize()
    # at least ~1 s under load before timing (clocks / power state settle).  The number of extra steps is agreed across
    # ranks (every step carries the 16-byte rate all-reduce when world > 1, so all ranks must run the same count).
    el = time.perf_counter() - t_warm
    extra = 0 if el >= 1.0 else int((1.0 - el) / max(el / max(warm_eff - S, 1), 1e-5) / S + 1) * S
    if world > 1:
        t_extra = torch.tensor([extra], dtype=torch.int64, device=dev)
        dist.all_reduce(t_extra, op=dist.ReduceOp.MAX)
        extra = int(t_extra.item())
    for i in range(extra):
        step_dev(warm_eff + i)
    warm_eff += extra
    ms_max, out = R.timed(step_dev, args.steps)
    value = global_batch * args.steps / (ms_max / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)

    # ---- end to end through the host-buffer entry -------------------------------------------------------------------
    # pinned host images + scores -> H2D -> forward -> D2H of what the reference's forward returns to its caller
    # (likelihoods y / z, MCM.py:801) plus the int16 symbols, ids_restore and the per-image bpp, every step, all on the
    # step's stream.
    n_pin = min(3, n_rot)
    pin_i = [t.pin_memory() for t in imgs_h[:n_pin]]
    pin_s = [t.pin_memory() for t in scores_h[:n_pin]]
    res_pin = [[m_.host_result_buffers(batch) for _ in range(2)] for m_ in models]     # two result sets per handle

    def step_host(i):
        models[i % S].forward_host(pin_i[i % n_pin], pin_s[i % n_pin], res_pin[i % S][(i // S) % 2], stream=R.side[i % S])
        if world > 1:
            pass                                              # rate_sums travel to the host with the step; no device collective here
        return None

    for i in range(max(args.warmup, 2 * S)):
        step_host(i)
    ms_e2e, _ = R.timed(step_host, args.steps)
    e2e_value = global_batch * args.steps / (ms_e2e / 1e3)
    h2d = imgs_h[0].numel() * 4 + scores_h[0].numel() * 4
    d2h = sum(v.numel() * v.element_size() for v in res_pin[0][0].values())
    e2e_check = {"bpp_equal_device_path": bool(torch.allclose(res_pin[(args.steps - 1) % S][((args.steps - 1) // S) % 2]["bpp"],
                                                              models[(args.steps - 1) % S](imgs_d[(args.steps - 1) % n_pin],
                                                                                           scores_d[(args.steps - 1) % n_pin],
                                                                                           need_recon=False)["bpp"].cpu(), rtol=1e-5)),
                 "returns": sorted(res_pin[0][0].keys())}

    # ---- batch-1 latency (config 1: the testing.py call pattern) ------------------------------------------------------
    latency = None
    if rank == 0 and kind == "kodak":
        one_i, one_s = imgs_d[0][:1].contiguous(), scores_d[0][:1].contiguous()
        for _ in range(5):
            model(one_i, one_s, need_recon=False)
        torch.cuda.synchronize()
        ts = []
        for k in range(24):
            a = imgs_d[0][k % batch: k % batch + 1].contiguous(); b = scores_d[0][k % batch: k % batch + 1].contiguous()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o1 = model(a, b, need_recon=False)
            o1["bpp"].cpu()                                    # the caller reads the rate: host-visible latency
            ts.append((time.perf_counter() - t0) * 1e3)
        ts.sort()
        latency = {"batch1_ms_median": ts[len(ts) // 2], "batch1_ms_min": ts[0], "images_per_s": 1e3 / ts[len(ts) // 2],
                   "note": "wall clock, one image per call, device inputs -> bpp read on the host (testing.py call pattern)"}
    # ---- latency of one batch alone (one handle, nothing else in flight): wall clock around a forward whose bpp is read on the host
    batch_latency = None
    if rank == 0:
        ts = []
        for k in range(12):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ob = model(imgs_d[k % n_rot], scores_d[k % n_rot], need_recon=False)
            ob["bpp"].cpu()
            ts.append((time.perf_counter() - t0) * 1e3)
        ts = sorted(ts[2:])
        batch_latency = {"batch": batch, "ms_median": ts[len(ts) // 2], "ms_min": ts[0],
                         "note": "one batch, one handle, device inputs -> bpp on the host; the throughput figures keep S batches in flight"}
    clocks = sampler.stop() if rank == 0 else None

    # ---- roofline of the dominant kernel family: CUDA events inside the library --------------------------------
    peaks = load_peaks()
    peak = peaks["bf16_tflops_sustained"]
    # events bracket every RUN of consecutive launches of one kernel family (the launch-to-launch overlap (PDL) inside
    # a run is kept and the event gap between its members is not charged to the kernel).  `isolated`: one stream, nothing
    # else on the GPU.  `in_mode`: the same profiled forwards while the other S-1 handles keep running their forwards on
    # their own streams, i.e. under the contention of the benchmarked configuration.
    def profiled(by_run, loaded):
        model.profile(True, by_run=by_run)
        if loaded:
            for rep in range(3):
                for k in range(1, S):
                    with torch.cuda.stream(R.side[k]):
                        models[k](imgs_d[k % n_rot], scores_d[k % n_rot], need_recon=False)
        with torch.cuda.stream(R.side[0]):
            for i in range(2):
                model(imgs_d[i % n_rot], scores_d[i % n_rot], need_recon=False)
        torch.cuda.synchronize()
        f_ = model.profile_read()
        model.profile(False)
        return f_
    fams_launch = profiled(False, False)
    fams = profiled(True, False)
    fams_mode = profiled(True, True) if S > 1 else fams
    tot_ms = sum(f["ms"] for f in fams) or 1.0
    gemm = next((f for f in fams if f["name"] == "gemm_tc"), None)
    gemm_mode = next((f for f in fams_mode if f["name"] == "gemm_tc"), None)
    gemm_launch = next((f for f in fams_launch if f["name"] == "gemm_tc"), None)
    roofline = None
    traffic = None
    tr_path = ROOT / "profiles" / f"r02_launches_{wl}.json"      # ncu dram__bytes_read+write per launch (--cache-control none)
    if tr_path.exists():
        try:
            traffic = json.loads(tr_path.read_text())["families"]["gemm_tc_kernel"]["dram_MB_per_launch"] * 1e6
        except Exception:
            traffic = None
    exec_flops_step = 0.0
    if gemm and gemm["ms"] > 0:
        exec_flops_step = gemm["flops"]                        # the library keeps the events of the LAST forward it profiled
        mma_flops_step = gemm["mma_flops"]
        achieved = gemm["mma_flops"] / (gemm["ms"] * 1e-3) / 1e12
        roofline = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 GEMM / implicit-GEMM conv engine)",
                    "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": traffic, "traffic_note": "bytes per launch, ncu dram__bytes_read+write averaged over the gemm_tc launches of "
                    "one forward (profiles/r02_launches_*.json, --cache-control none); null until that capture exists",
                    "flops": "EXECUTED tensor-core flops (patch embed counts the K kept patches; precise layers count their 3 terms)",
                    "executed_flops_per_launch": mma_flops_step / gemm["launches"],
                    "useful_frac": gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12 / peak,
                    "peak_source": f"{peaks['source']} bf16_tflops_sustained (of measured)",
                    "launches_per_step": gemm["launches"], "avg_launch_us": gemm["ms"] * 1e3 / gemm["launches"],
                    "share_of_step": gemm["ms"] / tot_ms,
                    "timing": "CUDA events around each run of consecutive gemm_tc launches, inside the library, on the launching stream; "
                              "isolated = one stream, plain launches",
                    "per_launch_events": {"avg_launch_us": gemm_launch["ms"] * 1e3 / gemm_launch["launches"],
                                          "frac": gemm_launch["mma_flops"] / (gemm_launch["ms"] * 1e-3) / 1e12 / peak},
                    "in_mode": {"streams": S, "avg_launch_us": gemm_mode["ms"] * 1e3 / gemm_mode["launches"],
                                "frac": gemm_mode["mma_flops"] / (gemm_mode["ms"] * 1e-3) / 1e12 / peak,
                                "note": "same events while the other handles run their forwards concurrently (the benchmarked mode): "
                                        "a launch shares the SMs, so its own duration grows while the step's throughput rises"},
                    # the timed region itself: executed tensor-core flops of one step / measured ms_per_step (graph replay, S streams)
                    "step_aggregate": {"achieved": mma_flops_step * world / (ms_max / args.steps * 1e-3) / 1e12 / world,
                                       "frac": mma_flops_step / (ms_max / args.steps * 1e-3) / 1e12 / peak,
                                       "note": "executed flops of one step / ms_per_step of the timed region (CUDA graph + S streams)"},
                    "families": {f["name"]: {"ms": round(f["ms"], 4), "launches": f["launches"]} for f in fams}}

    # memory-bound kernel families against the measured HBM peak (algorithmic bytes / per-launch event time; these
    # launches move 0.1-19 MB each, i.e. they are launch-latency bound at batch 64 - SURVEY 8d)
    hbm_kernels = {f["name"]: {"GB/s": round(f["bytes"] / (f["ms"] * 1e-3) / 1e9, 1), "launches": f["launches"],
                               "MB_per_launch": round(f["bytes"] / f["launches"] / 1e6, 3),
                               "frac_of_hbm_peak": round(f["bytes"] / (f["ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)}
                   for f in fams_launch if f["bytes"] > 0 and f["ms"] > 0}
    launches = model.launch_count(max(batch, 1))

    # ---- score generation (SURVEY 8 f-3): what produces `total_scores` upstream of the path; Kodak-sized grey images ----
    score_gen = None
    if rank == 0 and world == 1:
        from textmae_image_compression_b200.scores import generate_scores
        gh, gw, gn = 512, 768, 64
        gg = torch.Generator(device="cpu").manual_seed(4)
        base = torch.nn.functional.interpolate(torch.rand(gn, 1, gh // 16, gw // 16, generator=gg), size=(gh, gw), mode="bilinear")
        gray = (base[:, 0] * 255 + torch.randn(gn, gh, gw, generator=gg) * 6).clamp(0, 255).to(torch.uint8).to(dev)
        for _ in range(3):
            generate_scores(gray)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(20):
            generate_scores(gray)
        ev1.record()
        torch.cuda.synchronize()
        g_ms = ev0.elapsed_time(ev1) / 20
        g_bytes = gn * (3 * gh * gw + 4 * 196)            # grey read by the split decisions and the segment pass, segmented image written
        score_gen = {"images_per_s": gn / (g_ms * 1e-3), "ms_per_batch": g_ms, "batch": gn, "image": [gh, gw], "kernels_per_batch": 4,
                     "algorithmic_MB_per_batch": g_bytes / 1e6, "GB/s": g_bytes / (g_ms * 1e-3) / 1e9,
                     "frac_of_hbm_peak": g_bytes / (g_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                     "note": "tmae_generate_scores (generate_scores_file.py:19-31 on the GPU): latency-bound byte work, 0.4 MB per image; "
                             "the reference's Python loops take 0.3-1.0 s per image"}

    # ---- CPU baseline beside it (rank 0, N=1 only): the oracle on a bounded sample ---------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import ref_model
        from textmae_image_compression_b200 import make_state_dict
        sdc = make_state_dict(cfg, seed=0)
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sample = min(batch, 16)
        ref_model.forward_rate(sdc, cfg, imgs_h[0][:sample], scores_h[0][:sample])          # warm-up
        reps, t0 = 0, time.perf_counter()
        while reps < 2 or (time.perf_counter() - t0 < 10.0 and reps < 50):
            ref_model.forward_rate(sdc, cfg, imgs_h[0][:sample], scores_h[0][:sample])
            reps += 1
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": sample * reps / dt, "unit": "images/s", "cores": torch.get_num_threads(),
                        "kind": "port", "sample": f"{sample} images x {reps} reps of the same workload, fp32 oracle "
                                                  f"(oracle/ref_model.py == reference MCM.forward bit for bit) incl. the host python mask routine"}
        torch.set_num_threads(1)
        ref_model.forward_rate(sdc, cfg, imgs_h[0][:1], scores_h[0][:1])
        reps, t0 = 0, time.perf_counter()
        while reps < 2 or (time.perf_counter() - t0 < 5.0 and reps < 10):
            ref_model.forward_rate(sdc, cfg, imgs_h[0][:1], scores_h[0][:1])
            reps += 1
        cpu_baseline["single_thread_batch1"] = {"value": reps / (time.perf_counter() - t0), "unit": "images/s", "cores": 1,
                                                "note": "testing.py:29 torch.set_num_threads(1), batch 1"}
        torch.set_num_threads(cores)

    if rank == 0:
        gfl = algo_gflop_per_image(cfg, wl)
        line = {
            "metric": "images/s masked-ViT encode+rate", "value": value, "unit": "images/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precise is None else ("bf16x6 (three bf16 planes per operand, fp32-exact products)" if args.precise.endswith("x6")
                                                           else "bf16x3 (two bf16 planes per operand, ~2^-17 products)"),
            "data": "kodak (tests/golden fixtures)" if kind == "kodak" else "synthetic",
            "config": {"workload": desc, "name": wl, "per_gpu_batch": batch, "global_batch": global_batch,
                       "parallelism": f"dp{world} (images sharded, weights replicated, 16-byte rate all-reduce)",
                       "precise": args.precise, "streams_per_gpu": S, "warmup_effective": warm_eff,
                       "l2_policy": f"inputs rotate over {n_rot} batches ({n_rot * imgs_h[0].numel() * 4 / 1e6:.0f} MB) "
                                    "+ >= 350 MB of weights per step > 126 MB L2",
                       "algorithmic_gflop_per_image": gfl, "executed_gflop_per_image": exec_flops_step / max(batch, 1) / 1e9},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "check": e2e_check},
            "gpu_launches": launches * args.steps,
            "roofline": roofline, "hbm_kernels": hbm_kernels, "cpu_baseline": cpu_baseline, "clocks": clocks,
            "latency": latency, "batch_latency": batch_latency, "score_generation": score_gen,
            "model_tflops": value * gfl / 1e3,
            "model_tflops_frac_of_peak": value / world * gfl / 1e3 / peak,
            "bpp_mean_last_step": out["bpp"].mean().item(),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree, which may be read-only
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="B64", choices=sorted(WORKLOADS))
    ap.add_argument("--precise", default=None, choices=["all", "rate", "all-x6", "rate-x6"],
                    help="accuracy mode: split-bf16 operands for the rate half / the whole path (symbols match the fp32 reference)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's batch per GPU; strong: the workload's batch is the global batch, sharded over the GPUs")
    ap.add_argument("--ref-sample", type=int, default=0, help="images per step for the CPU reference arm (0 = the full batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--streams", type=int, default=4, help="batches in flight per GPU (independent handles/streams)")
    ap.add_argument("--batch", type=int, default=0, help="experiment only: images per step instead of the workload's batch")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the last timed step returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    kwargs, batch, desc, kind = WORKLOADS[args.workload]
    if args.batch > 0:
        desc = desc.replace(f"batch {batch}", f"batch {args.batch} (EXPERIMENT, not the named workload)")
        batch = args.batch
    if args.impl == "reference":
        run_reference(args, kwargs, batch, desc, kind)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_b200(args, kwargs, batch, desc, args.workload, kind)


if __name__ == "__main__":
    main()
