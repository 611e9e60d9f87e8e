"""CPU: the score-generation oracle (oracle/ref_scores.py) against (1) OpenCV itself, (2) the reference's own functions
executed from the reference checkout when it is provided, (3) the committed reference-generated goldens."""
import sys
import types
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import REFERENCE_ROOT as REF, SKIP_REASON, ref_scores, reference_has

GOLDEN = Path(__file__).resolve().parent / "golden"
cv2 = pytest.importorskip("cv2")


@pytest.mark.parametrize("shape", [(512, 768), (510, 766), (224, 224), (100, 90), (64, 64), (200, 300), (223, 223), (30, 1000),
                                   (17, 19), (448, 448), (1078, 2046)])
@pytest.mark.parametrize("side", [224, 512, 64])
def test_resize_restatement_equals_cv2(shape, side):
    rng = np.random.default_rng(shape[0] * 7 + side)
    img = rng.integers(0, 256, shape, dtype=np.uint8)
    assert np.array_equal(cv2.resize(img, (side, side)), ref_scores.resize_linear_u8(img, side, side))
    view = img[1:-1, 1:-1]                                   # what Division_Merge_Segmented resizes (utils/map.py:51-53)
    assert np.array_equal(cv2.resize(view, (side, side)), ref_scores.resize_linear_u8(view, side, side))


@pytest.mark.parametrize("shape", [(512, 768), (37, 41), (3, 3), (2, 5), (64, 64)])
def test_laplacian_restatement_equals_cv2(shape):
    rng = np.random.default_rng(shape[0])
    for img in (rng.integers(0, 256, shape, dtype=np.uint8), (rng.integers(0, 2, shape) * 255).astype(np.uint8)):
        ref = cv2.convertScaleAbs(cv2.Laplacian(img, cv2.CV_16S, ksize=3))       # utils/map.py:58-59
        assert np.array_equal(ref, ref_scores.laplacian_abs_u8(img))


def test_oracle_equals_reference_generated_goldens():
    z = np.load(GOLDEN / "scores_refexec.npz")
    for k, (kind, h, w, seed) in enumerate(z["cases"]):
        sc, s_map, t_map, _ = ref_scores.generate_scores(ref_scores.synthetic_gray(int(kind), int(h), int(w), int(seed)), return_maps=True)
        assert np.array_equal(s_map, z[f"case{k}_s_map"]), k
        assert np.array_equal(t_map, z[f"case{k}_t_map"]), k
        assert np.array_equal(sc, z[f"case{k}_scores"], equal_nan=True), k
    assert np.isnan(z["case4_scores"]).all()                  # constant image: 0 / 0, like the reference
    gray = np.load(GOLDEN / "kodak_gray6.npz")
    gold = torch.load(GOLDEN / "kodak_scores.pt").numpy()     # reference generator on the Kodak PNGs (make_golden.py)
    for i, name in enumerate(sorted(gray.files)):
        assert np.array_equal(ref_scores.generate_scores(gray[name]), gold[i]), name


@pytest.mark.skipif(not reference_has("utils/map.py"), reason=SKIP_REASON)
def test_oracle_equals_reference_code_executed_in_place():
    sys.path.insert(0, str(GOLDEN))
    import make_scores_golden as mk
    fns = mk.reference_functions()
    paths = sorted((REF / "datasets" / "kodak").rglob("*.*"))
    gold = torch.load(GOLDEN / "kodak_scores.pt").numpy()
    for i in (6, 9, 13, 19, 23):                               # images outside the committed gray fixture
        img = cv2.imread(str(paths[i]), cv2.IMREAD_GRAYSCALE)
        assert np.array_equal(ref_scores.generate_scores(img), gold[i])
    for kind, h, w, seed in [(0, 231, 517, 11), (1, 260, 226, 12), (2, 400, 400, 13), (4, 226, 227, 14)]:
        img = ref_scores.synthetic_gray(kind, h, w, seed)
        sc, s_map, t_map, seg = mk.reference_scores(img, fns)
        o_sc, o_s, o_t, o_seg = ref_scores.generate_scores(img, return_maps=True)
        assert np.array_equal(seg, o_seg) and np.array_equal(s_map, o_s) and np.array_equal(t_map, o_t)
        assert np.array_equal(sc, o_sc, equal_nan=True)
