"""Generates tests/golden/kodak_gray6.npz and scores_refexec.npz.  Needs a checkout of the original project
(oracle.REFERENCE_ROOT) and cv2:

    python tests/golden/make_scores_golden.py

  * kodak_gray6.npz    - cv2.imread(path, IMREAD_GRAYSCALE) (generate_scores_file.py:19) of the first six bundled Kodak PNGs
                         (kodim04 is portrait): the INPUT of the score generator, for machines without the
                         reference checkout.  Their reference scores are rows 0..5 of kodak_scores.pt (make_golden.py).
  * scores_refexec.npz - outputs of the REFERENCE functions executed where they lie (utils/map.py Division_Merge_Segmented,
                         laplacian; utils/distribution.py cal_patch_score; the normalisation of generate_scores_file.py:24-31)
                         on seeded synthetic images (oracle.ref_scores.synthetic_gray) at several geometries: s_map, t_map,
                         scores per case.
"""
from __future__ import annotations

import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))

from oracle import REFERENCE_ROOT as REF, ref_scores  # noqa: E402

CASES = [(0, 256, 256, 1), (0, 300, 411, 2), (1, 225, 230, 3), (2, 256, 384, 4), (3, 256, 256, 77), (3, 301, 411, 9),
         (4, 512, 768, 5), (4, 333, 500, 6), (0, 768, 512, 7), (2, 230, 226, 8)]


def reference_functions():
    import cv2  # noqa: F401
    sys.path.insert(0, str(REF))
    stub = types.ModuleType("matplotlib")
    stub.pyplot = types.ModuleType("matplotlib.pyplot")
    sys.modules.setdefault("matplotlib", stub)
    sys.modules.setdefault("matplotlib.pyplot", stub.pyplot)
    from utils.distribution import cal_patch_score                # reference code
    from utils.map import Division_Merge_Segmented, laplacian      # reference code
    return Division_Merge_Segmented, laplacian, cal_patch_score


def reference_scores(img: np.ndarray, fns, side: int = 224):
    """generate_scores_file.py:19-31 on an already decoded grayscale image."""
    seg, lap, cps = fns
    img = img.copy()
    s_map = seg(img, (side, side))               # :21 (works in place on img)
    t_map = lap(img, (side, side))               # :22
    total = cps(t_map) * cps(s_map)              # :24-26
    with np.errstate(all="ignore"):
        total = (total - total.min()) / (total.max() - total.min())     # :28-29
    return torch.tensor(total, dtype=torch.float32).numpy(), s_map, t_map, img


def main():
    import cv2
    fns = reference_functions()
    paths = sorted((REF / "datasets" / "kodak").rglob("*.*"))[:6]
    np.savez_compressed(HERE / "kodak_gray6.npz", **{p.stem: cv2.imread(str(p), cv2.IMREAD_GRAYSCALE) for p in paths})
    blob = {}
    for k, (kind, h, w, seed) in enumerate(CASES):
        img = ref_scores.synthetic_gray(kind, h, w, seed)
        sc, s_map, t_map, seg = reference_scores(img, fns)
        blob[f"case{k}_scores"] = sc
        blob[f"case{k}_s_map"] = s_map
        blob[f"case{k}_t_map"] = t_map
    blob["cases"] = np.array(CASES)
    np.savez_compressed(HERE / "scores_refexec.npz", **blob)
    print("wrote", len(CASES), "cases")


if __name__ == "__main__":
    main()
