"""CPU: the host-side side-information coder (csrc/huffman.cpp via textmae_image_compression_b200.huffman.HuffmanCoding)
against the reference's HuffmanCoding - executed from the reference checkout when provided, committed goldens otherwise - and the
oracle restatement.  Bit strings and code tables must be identical; decode must invert encode."""
from pathlib import Path

import pytest
import torch

from oracle import SKIP_REASON, ref_huffman
from textmae_image_compression_b200.huffman import HuffmanCoding, side_info_bits

GOLDEN = Path(__file__).resolve().parent / "golden"


def test_matches_reference_goldens():
    for case in torch.load(GOLDEN / "huffman_refexec.pt"):
        h = HuffmanCoding()
        text, shape, dev = h.compress(case["tensor"])
        assert text == case["text"], case["name"]
        assert h.codes == case["codes"], case["name"]
        assert list(h.codes) == list(case["codes"]), case["name"]          # key order of the reference's dict (pre-order walk)
        assert torch.equal(h.decompress(text, shape, dev), case["tensor"]), case["name"]
        packed, nbits, _, _ = h.compress_packed(case["tensor"])
        assert nbits == len(text) and len(packed) == (nbits + 7) // 8
        assert "".join(f"{b:08b}" for b in packed)[:nbits] == text
        assert torch.equal(h.decode((packed, nbits)), case["tensor"].reshape(-1))
        o = ref_huffman.HuffmanOracle()
        assert o.compress(case["tensor"].reshape(-1).tolist()) == text and o.codes == case["codes"]


def test_permutation_cost_is_closed_form():
    """ids_restore of one image is a permutation of L: every frequency is 1, so the cost the reference adds to the bpp
    (testing.py:89) is L floor(log2 L) + 2 (L - 2^floor(log2 L)) bits whatever the tie-breaking."""
    for L in (196, 1024, 50, 64):
        k = L.bit_length() - 1
        assert side_info_bits(torch.randperm(L)[None]) == L * k + 2 * (L - (1 << k))


def test_fuzz_against_oracle():
    g = torch.Generator().manual_seed(11)
    for trial in range(40):
        n = int(torch.randint(1, 600, (1,), generator=g))
        alphabet = int(torch.randint(2, 80, (1,), generator=g))
        t = (torch.rand(n, generator=g) ** (1 + trial % 4) * alphabet).long() - trial
        if t.unique().numel() < 2:
            continue
        h = HuffmanCoding()
        text, shape, dev = h.compress(t)
        o = ref_huffman.HuffmanOracle()
        assert o.compress(t.tolist()) == text, trial
        assert o.codes == h.codes
        assert torch.equal(h.decompress(text, shape, dev), t)
        assert h.encode(t) == text


def test_single_symbol_alphabet_behaves_like_the_reference():
    """One distinct value: the root is the leaf, its code is "" - zero bits, and decode returns nothing, so the reference's
    decompress fails in .view; same here."""
    h = HuffmanCoding()
    text, shape, dev = h.compress(torch.tensor([5, 5, 5]))
    assert text == "" and h.codes == {5: ""}
    with pytest.raises(RuntimeError):
        h.decompress(text, shape, dev)


@pytest.mark.skipif(not ref_huffman.reference_available(), reason=SKIP_REASON)
def test_matches_reference_class_executed_in_place():
    Ref = ref_huffman.load_reference_class()
    g = torch.Generator().manual_seed(3)
    for L in (196, 1024):
        for _ in range(4):
            t = torch.stack([torch.randperm(L, generator=g) for _ in range(2)])
            r = Ref()
            text, shape, _ = r.compress(t)
            h = HuffmanCoding()
            mine, _, _ = h.compress(t)
            assert mine == text and h.codes == r.codes and h.reverse_mapping == r.reverse_mapping
            assert torch.equal(h.decompress(mine, shape, "cpu"), r.decompress(text, shape, "cpu"))
