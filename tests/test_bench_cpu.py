"""CPU: the reference arm of bench.py (the oracle port timed on the host cores) prints one JSON line that carries the
contract keys; the B200 arm refuses to run without a GPU (no CPU fallback); --dump-outputs writes what a forward
returns, within its size budget."""
import importlib.util
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent


def _run(*args, timeout=300):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_reference_arm_json_contract():
    p = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-sample", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["metric"] == "images/s masked-ViT encode+rate" and d["value"] > 0 and d["n_gpus"] == 1
    for key in ("steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly(monkeypatch):
    import os
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert p.returncode == 0 and not [ln for ln in p.stdout.splitlines() if ln.startswith("{")]


def test_b200_arm_needs_a_gpu():
    if torch.cuda.is_available():
        return
    p = _run("--steps", "1", "--no-cpu-baseline")
    assert p.returncode != 0 and "CUDA" in (p.stderr + p.stdout)


def test_reference_arm_dumps_the_b200_names(tmp_path):
    p = _run("--impl", "reference", "--steps", "3", "--warmup", "1", "--ref-sample", "1", "--dump-outputs", str(tmp_path / "d"))
    assert p.returncode == 0, p.stderr[-2000:]
    names = sorted(f.name for f in (tmp_path / "d").iterdir())
    assert names == ["bpp.npy", "ids_keep.npy", "ids_restore.npy", "latents_y_hat.npy", "latents_y_sym.npy", "latents_z_hat.npy",
                     "latents_z_sym.npy", "likelihoods_y.npy", "likelihoods_z.npy"]
    assert np.load(tmp_path / "d" / "likelihoods_y.npy").shape == (64, 384, 8, 8)      # the whole B64 batch of the last step


def test_steps_must_be_positive():
    p = _run("--steps", "0")
    assert p.returncode == 2 and "--steps" in p.stderr


def _bench_module():
    spec = importlib.util.spec_from_file_location("_bench", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _forward_like(n, side=8, cy=384):
    g = torch.Generator().manual_seed(2)
    return {"likelihoods": {"y": torch.rand(n, side, side, cy, generator=g).permute(0, 3, 1, 2), "z": torch.rand(n, 4, 1, 1, generator=g)},
            "latents": {"y_sym": torch.randint(-20, 20, (n, cy, side, side), generator=g, dtype=torch.int32)},
            "bpp": torch.rand(n, generator=g), "rate_sums": torch.tensor([-1234.5678901234, 4096.0], dtype=torch.float64),
            "ids_restore": torch.argsort(torch.rand(n, 196, generator=g), 1)}


def test_dump_outputs_names_dtypes_and_values(tmp_path):
    out = _forward_like(3)
    _bench_module().dump_outputs(out, tmp_path / "d")
    assert sorted(p.name for p in (tmp_path / "d").iterdir()) == [
        "bpp.npy", "ids_restore.npy", "latents_y_sym.npy", "likelihoods_y.npy", "likelihoods_z.npy", "rate_sums.npy"]
    y = np.load(tmp_path / "d" / "likelihoods_y.npy")
    assert y.dtype == np.float32 and np.array_equal(y, out["likelihoods"]["y"].numpy())           # NCHW, as returned
    sym = np.load(tmp_path / "d" / "latents_y_sym.npy")
    assert sym.dtype == np.float64 and np.array_equal(sym, out["latents"]["y_sym"].numpy())
    assert np.array_equal(np.load(tmp_path / "d" / "ids_restore.npy"), out["ids_restore"].numpy())
    assert np.load(tmp_path / "d" / "rate_sums.npy").tolist() == out["rate_sums"].tolist()


def test_dump_outputs_samples_within_budget(tmp_path):
    bench = _bench_module()
    bench.DUMP_BUDGET_BYTES = 8 * 10**6
    out = _forward_like(40)                                             # ~4 MB of likelihoods + ~8 MB of symbols (float64)
    for d in ("a", "b"):
        bench.dump_outputs(out, tmp_path / d)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= bench.DUMP_BUDGET_BYTES
    for f in files:                                                      # a fixed seed: the same sample every time
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    y = np.load(tmp_path / "a" / "likelihoods_y.npy")
    assert y.ndim == 1 and 0 < y.size < out["likelihoods"]["y"].numel() and np.isin(y, out["likelihoods"]["y"].numpy()).all()
    assert np.array_equal(np.load(tmp_path / "a" / "bpp.npy"), out["bpp"].numpy())                 # small outputs stay whole
