"""TEST INFRASTRUCTURE - the reference's HuffmanCoding (utils/huffman.py) for checking the host-side coder (SURVEY 8 f-4).

Only tests/ may import this.  `load_reference_class()` executes the reference file where it lies (it needs only torch and the
standard library); `HuffmanOracle` is a restatement for machines without the reference checkout: the same algorithm on
Python's own `heapq` (the library the reference calls, so the tie-breaking is the reference's by construction), nodes ordered by
frequency only (utils/huffman.py:28-38), values in first-appearance order (:55-62), pre-order walk left "0" / right "1"
(:76-93), decode by growing the current code (:120-139).  Pinned by tests/test_huffman.py against the executed reference
class and the committed goldens (tests/golden/huffman_refexec.pt).
"""
from __future__ import annotations

import heapq
import importlib.util

from . import REFERENCE_ROOT, reference_has

REF_FILE = REFERENCE_ROOT / "utils/huffman.py"


def reference_available() -> bool:
    return reference_has("utils/huffman.py")


def load_reference_class():
    spec = importlib.util.spec_from_file_location("_ref_huffman", REF_FILE)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.HuffmanCoding


class _Node:
    __slots__ = ("value", "freq", "left", "right")

    def __init__(self, value, freq):
        self.value, self.freq, self.left, self.right = value, freq, None, None

    def __lt__(self, other):
        return self.freq < other.freq


class HuffmanOracle:
    def __init__(self):
        self.codes, self.reverse_mapping = {}, {}

    def compress(self, values):
        freq = {}
        for v in values:
            freq[int(v)] = freq.get(int(v), 0) + 1
        heap = []
        for v, f in freq.items():
            heapq.heappush(heap, _Node(v, f))
        while len(heap) > 1:
            a, b = heapq.heappop(heap), heapq.heappop(heap)
            m = _Node(None, a.freq + b.freq)
            m.left, m.right = a, b
            heapq.heappush(heap, m)
        self.codes, self.reverse_mapping = {}, {}
        stack = [(heap[0], "")] if heap else []
        while stack:
            node, code = stack.pop()
            if node.value is not None:
                self.codes[node.value] = code
                self.reverse_mapping[code] = node.value
                continue
            stack.append((node.right, code + "1"))
            stack.append((node.left, code + "0"))
        return "".join(self.codes[int(v)] for v in values)

    def decode(self, text):
        out, cur = [], ""
        for bit in text:
            cur += bit
            if cur in self.reverse_mapping:
                out.append(self.reverse_mapping[cur])
                cur = ""
        return out
