"""Generates the committed fixtures under tests/golden/.  Needs a checkout of the original project (oracle.REFERENCE_ROOT):

    python tests/golden/make_golden.py

What comes from REFERENCE CODE executed where it lies (the checkout, read-only):
  * kodak_scores.pt   - the reference's score generator (generate_scores_file.py:19-31 calling utils/map.py and
                        utils/distribution.py) on the 24 bundled Kodak PNGs (datasets/kodak).
  * kodak_224.npz     - the 24 Kodak images through the reference's test transform
                        (utils/dataloader.py:69-73: PIL RGB -> Resize((224,224), BICUBIC)), stored as uint8.
  * mask_golden.pt    - outputs of the verbatim `MCM.get_ids_shuffle` (MCM.py:364-423) on the Kodak scores and on
                        seeded fuzz vectors, for every valid K.
What comes from the in-repo oracle (oracle/ref_model.py; parity unpinned against reference outputs, see its header):
  * model_B64.pt / model_B144.pt - every intermediate of the rate path for two / one Kodak images with the
                        seeded synthetic checkpoint (seed 0).
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

from oracle import REFERENCE_ROOT as REF, SKIP_REASON, ref_mask, ref_model  # noqa: E402
from textmae_image_compression_b200.config import vit_base  # noqa: E402
from textmae_image_compression_b200.synthetic import make_state_dict  # noqa: E402


def kodak_scores_and_images():
    import cv2
    from PIL import Image
    sys.path.insert(0, str(REF))
    stub = types.ModuleType("matplotlib")
    stub.pyplot = types.ModuleType("matplotlib.pyplot")
    sys.modules.setdefault("matplotlib", stub)
    sys.modules.setdefault("matplotlib.pyplot", stub.pyplot)
    from utils.distribution import cal_patch_score           # reference code
    from utils.map import Division_Merge_Segmented, laplacian  # reference code

    paths = sorted((REF / "datasets" / "kodak").rglob("*.*"))
    assert len(paths) == 24, paths
    scores, imgs = [], []
    for p in paths:
        img = cv2.imread(str(p), cv2.IMREAD_GRAYSCALE)        # generate_scores_file.py:19
        s_map = Division_Merge_Segmented(img, (224, 224))     # :21
        t_map = laplacian(img, (224, 224))                    # :22
        total = cal_patch_score(t_map) * cal_patch_score(s_map)   # :24-26
        if total.size > 0:
            total = (total - total.min()) / (total.max() - total.min())   # :28-29
        scores.append(torch.tensor(total, dtype=torch.float32))           # :31
        pil = Image.open(p).convert("RGB").resize((224, 224), Image.BICUBIC)   # dataloader.py:38, 71
        imgs.append(np.asarray(pil, dtype=np.uint8))
    return torch.stack(scores), np.stack(imgs), [p.name for p in paths]


def fuzz_scores(kind: int, L: int, g: torch.Generator) -> torch.Tensor:
    if kind == 0:
        return torch.rand(L, generator=g)
    if kind == 1:      # Kodak-like heavy-tie integer products
        a = torch.randint(0, 40, (L,), generator=g).float() * torch.randint(0, 165, (L,), generator=g).float()
        return (a - a.min()) / (a.max() - a.min())
    if kind == 2:
        return torch.rand(L, generator=g) ** 4
    if kind == 3:      # 30 levels
        return torch.randint(0, 30, (L,), generator=g).float() / 29
    if kind == 4:      # 3 levels -> empty groups -> NaN means
        return torch.randint(0, 3, (L,), generator=g).float() / 2
    return torch.full((L,), 0.5)   # all equal


def main():
    assert ref_mask.reference_available(), SKIP_REASON
    scores, imgs_u8, names = kodak_scores_and_images()
    torch.save(scores, HERE / "kodak_scores.pt")
    np.savez_compressed(HERE / "kodak_224.npz", imgs=imgs_u8, names=np.array(names))
    print("kodak scores", tuple(scores.shape), "unique per image", [int(s.unique().numel()) for s in scores][:6], "...")

    # ---- mask goldens from the verbatim reference routine ----
    g = torch.Generator().manual_seed(1234)
    cases = []
    for K in (16, 64, 144):
        cases.append({"name": f"kodak_K{K}", "scores": scores, "K": K,
                      "ids_shuffle": ref_mask.reference_ids_shuffle(scores, K)})
    for L, Ks in ((196, (16, 64, 144)), (1024, (16, 64, 144, 256, 400, 576, 784, 1024))):
        for kind in range(6):
            sc = torch.stack([fuzz_scores(kind, L, g) for _ in range(6 if L == 196 else 2)])
            for K in Ks:
                cases.append({"name": f"fuzz_L{L}_kind{kind}_K{K}", "scores": sc, "K": K,
                              "ids_shuffle": ref_mask.reference_ids_shuffle(sc, K)})
    torch.save(cases, HERE / "mask_golden.pt")
    print("mask cases", len(cases))

    # ---- model goldens from the oracle ----
    imgs = torch.from_numpy(imgs_u8).permute(0, 3, 1, 2).float() / 255.0      # ToTensor()
    keep = ("ids_keep", "ids_restore", "x_remain", "y", "z", "z_sym", "z_lik", "mu", "sigma", "y_sym", "y_lik",
            "y_hat", "bpp")
    for K, n_img in ((64, 2), (144, 1)):
        cfg = vit_base(K)
        sd = make_state_dict(cfg, seed=0)
        out = ref_model.forward_rate(sd, cfg, imgs[:n_img], scores[:n_img])
        blob = {k: (out[k].half() if out[k].dtype == torch.float32 and k in ("x_remain",) else out[k]) for k in keep}
        blob["bpp_batch"] = out["bpp_batch"]
        blob["n_img"] = n_img
        torch.save(blob, HERE / f"model_B{K}.pt")
        print(f"B{K}: bpp", out["bpp"].tolist())


if __name__ == "__main__":
    main()
