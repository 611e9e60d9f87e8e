"""ORACLE (test infrastructure only - never imported by the product path).

Score-guided patch ordering of the reference, `MCM.get_ids_shuffle`
(models/Compression/MCM.py:364-423) and the inverse
permutation / keep-set of `MCM.random_masking` (MCM.py:548-588).

Two implementations live here:

* `load_reference_get_ids_shuffle()` - pulls the *verbatim* reference function
  out of the reference checkout (oracle.REFERENCE_ROOT) with `ast` (the function
  only needs torch, F.softmax and collections.Counter, so it runs without
  timm/compressai).  Only usable where that checkout exists; it is what pins the
  restatement and what generates tests/golden/mask_*.pt.
* `ids_shuffle_spec()` - an index-level restatement in torch (same torch
  kernels, same fp32 arithmetic, so it equals the reference wherever torch's
  CPU kernels are the same build).

The bit-level, torch-free restatement (the one the CUDA kernel mirrors) is
oracle/mask_oracle.c; `mask_oracle_c()` binds it through ctypes.
"""
from __future__ import annotations

import ast
import collections
import ctypes
import os
import subprocess
import types
from pathlib import Path

import numpy as np
import torch
import torch.nn.functional as F

from . import REFERENCE_ROOT, reference_has

REFERENCE_MCM = REFERENCE_ROOT / "models/Compression/MCM.py"
_HERE = Path(__file__).resolve().parent


def reference_available() -> bool:
    return reference_has("models/Compression/MCM.py")


def load_reference_get_ids_shuffle():
    """Return the reference's own `get_ids_shuffle(self, total_scores)` function object,
    compiled from the reference source file where it lies (MCM.py:364-423)."""
    src = REFERENCE_MCM.read_text()
    tree = ast.parse(src)
    fn_node = None
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "get_ids_shuffle":
            fn_node = node
            break
    if fn_node is None:
        raise RuntimeError("get_ids_shuffle not found in reference MCM.py")
    mod = ast.Module(body=[fn_node], type_ignores=[])
    ns = {"torch": torch, "F": F, "Counter": collections.Counter}
    exec(compile(mod, str(REFERENCE_MCM), "exec"), ns)
    return ns["get_ids_shuffle"]


def reference_ids_shuffle(total_scores: torch.Tensor, num_keep_patches: int) -> torch.Tensor:
    """Run the verbatim reference routine.  Returns int64 CPU [N, L] (MCM.py:423)."""
    fn = load_reference_get_ids_shuffle()
    self_ns = types.SimpleNamespace(num_keep_patches=int(num_keep_patches))
    return fn(self_ns, total_scores.detach().cpu().float())


def ids_shuffle_spec(score: torch.Tensor, K: int) -> list:
    """Index-level restatement of MCM.py:379-421 for ONE sample (score: fp32 [L])."""
    score = score.detach().cpu().float()
    L = score.numel()
    q = torch.arange(0.1, 0.91, 0.1, dtype=torch.float32)                  # MCM.py:381
    thr = torch.quantile(score.unique(), q, dim=0)                          # :383-384
    cat = torch.bucketize(score, thr)                                       # :387
    means = torch.tensor([score[cat == g].mean() for g in range(10)],
                         dtype=torch.float32)                               # :390-393
    top = (cat == 9).nonzero().flatten().tolist()                           # :396
    cnt = torch.round(F.softmax(means[:-1], dim=0) * (K - len(top))).int().tolist()  # :399-402
    vals = [score[i].item() for i in top]
    for g in range(9):                                                      # :405-408
        gs, _ = torch.sort(score[cat == g])
        vals += gs[int(len(gs) - cnt[g]):].tolist()
    order = []
    for v, f in collections.Counter(vals).items():                          # :410-416
        order += (score == v).nonzero().flatten()[:f].tolist()
    chosen = set(order)
    order += [i for i in range(L) if i not in chosen]                       # :418-420
    return order


def ids_shuffle_spec_batch(total_scores: torch.Tensor, K: int) -> torch.Tensor:
    if K > total_scores.shape[1]:
        raise ValueError("Number of patches should not be greater than the length of scores")  # MCM.py:374-376
    return torch.tensor([ids_shuffle_spec(s, K) for s in total_scores])


def masking_from_shuffle(ids_shuffle: torch.Tensor, K: int):
    """MCM.py:579-583: ids_restore = argsort(ids_shuffle); ids_keep = ids_shuffle[:, :K]."""
    ids_restore = torch.argsort(ids_shuffle, dim=1)
    ids_keep = ids_shuffle[:, :K]
    return ids_keep, ids_restore


# ----------------------------------------------------------------------------------------------
# ctypes binding of the torch-free C restatement (oracle/mask_oracle.c)
# ----------------------------------------------------------------------------------------------
_C_LIB = None


def build_mask_oracle_c(force: bool = False) -> Path:
    out_dir = _HERE / "_build"
    out_dir.mkdir(exist_ok=True)
    so = out_dir / "libmask_oracle.so"
    src = _HERE / "mask_oracle.c"
    if force or not so.exists() or so.stat().st_mtime < src.stat().st_mtime:
        # -ffp-contract=off: every fused multiply-add in the routine is an explicit fmaf().
        subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fPIC",
                               "-shared", "-o", str(so), str(src), "-lm"])
    return so


def _c_lib():
    global _C_LIB
    if _C_LIB is None:
        lib = ctypes.CDLL(str(build_mask_oracle_c()))
        lib.tmae_oracle_ids_shuffle.restype = ctypes.c_int
        lib.tmae_oracle_ids_shuffle.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        _C_LIB = lib
    return _C_LIB


def torch_softmax_isa() -> int:
    """16 when this process' torch dispatches AVX512 CPU kernels, else 8."""
    return 16 if "AVX512" in torch.backends.cpu.get_cpu_capability().upper() else 8


def mask_oracle_c(total_scores: torch.Tensor, K: int, isa: int | None = None, return_debug: bool = False):
    """Bit-level C restatement.  isa = softmax lane-sum order of the torch CPU build being
    mirrored (16 = AVX512 kernels, 8 = AVX2); None = whatever this process' torch dispatches to.
    See mask_oracle.c header."""
    if isa is None:
        isa = torch_softmax_isa()
    sc = np.ascontiguousarray(total_scores.detach().cpu().float().numpy())
    N, L = sc.shape
    if K > L:
        raise ValueError("Number of patches should not be greater than the length of scores")
    out = np.empty((N, L), dtype=np.int64)
    dbg = np.zeros((N, 32), dtype=np.float32)
    rc = _c_lib().tmae_oracle_ids_shuffle(sc.ctypes.data, N, L, int(K), int(isa),
                                          out.ctypes.data, dbg.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"mask_oracle.c failed rc={rc}")
    if return_debug:
        return torch.from_numpy(out), torch.from_numpy(dbg)
    return torch.from_numpy(out)
