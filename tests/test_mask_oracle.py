"""CPU: the bit-level C restatement of MCM.get_ids_shuffle (oracle/mask_oracle.c) against
 (a) the committed outputs of the verbatim reference function (tests/golden/mask_golden.pt),
 (b) the verbatim function itself where the reference checkout is provided,
 (c) the ATen kernels it restates (cascade sum, softmax), bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import SKIP_REASON, ref_mask


@pytest.fixture(scope="module")
def cases(golden_dir):
    return torch.load(golden_dir / "mask_golden.pt")


def test_golden_cases_cover_edge_cases(cases):
    names = [c["name"] for c in cases]
    assert any("kodak" in n for n in names) and any("kind4" in n for n in names) and any("kind5" in n for n in names)
    assert any("L1024" in n and "K1024" in n for n in names)


def test_c_oracle_matches_reference_goldens(cases):
    bad = []
    for c in cases:
        got = ref_mask.mask_oracle_c(c["scores"], c["K"], isa=16)     # goldens were generated on an AVX512 torch
        if not torch.equal(got, c["ids_shuffle"]):
            bad.append(c["name"])
    assert not bad, bad


def test_torch_spec_matches_reference_goldens(cases):
    if ref_mask.torch_softmax_isa() != 16:
        pytest.skip("goldens were generated with AVX512 ATen kernels")
    for c in cases[:12]:
        got = ref_mask.ids_shuffle_spec_batch(c["scores"], c["K"])
        assert torch.equal(got, c["ids_shuffle"]), c["name"]


def test_every_output_is_a_permutation(cases):
    for c in cases:
        L = c["scores"].shape[1]
        srt = torch.sort(c["ids_shuffle"], dim=1)[0]
        assert torch.equal(srt, torch.arange(L).expand_as(srt))


@pytest.mark.skipif(not ref_mask.reference_available(), reason=SKIP_REASON)
def test_c_oracle_matches_live_reference_fuzz():
    g = torch.Generator().manual_seed(99)
    for L, K in ((196, 64), (196, 144), (1024, 256)):
        sc = torch.rand(8, L, generator=g)
        sc[4:] = torch.round(sc[4:] * 20) / 20          # ties
        ref = ref_mask.reference_ids_shuffle(sc, K)
        assert torch.equal(ref_mask.mask_oracle_c(sc, K), ref)


def test_k_greater_than_l_raises():
    with pytest.raises(ValueError):
        ref_mask.mask_oracle_c(torch.rand(1, 16), 17)
    with pytest.raises(ValueError):
        ref_mask.ids_shuffle_spec_batch(torch.rand(1, 16), 17)


def _lib():
    lib = ctypes.CDLL(str(ref_mask.build_mask_oracle_c()))
    lib.tmae_oracle_sum_f32.restype = ctypes.c_float
    lib.tmae_oracle_sum_f32.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    lib.tmae_oracle_softmax9.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    return lib


def test_cascade_sum_restatement_is_bit_exact():
    lib = _lib()
    g = torch.Generator().manual_seed(5)
    for n in list(range(1, 70)) + [127, 128, 129, 255, 511, 512, 513, 1000, 1024]:
        for _ in range(5):
            x = torch.rand(n, generator=g)
            mine = lib.tmae_oracle_sum_f32(x.numpy().ctypes.data, n, 8)
            assert np.float32(mine) == np.float32(x.sum().item()), n


def test_softmax9_restatement_is_bit_exact():
    lib = _lib()
    isa = ref_mask.torch_softmax_isa()
    g = torch.Generator().manual_seed(6)
    for t in range(500):
        x = torch.sort(torch.rand(9, generator=g))[0] if t % 2 else torch.randn(9, generator=g)
        out = np.empty(9, np.float32)
        lib.tmae_oracle_softmax9(x.numpy().ctypes.data, isa, out.ctypes.data)
        ref = torch.softmax(x, 0).numpy()
        assert np.array_equal(out.view(np.uint32), ref.view(np.uint32))
