"""GPU: one handle keeps the launch plans of every kind (forward, decode, decode from streams, synthesis) in one cache, and a
change drops exactly the plans that read what it changed.  One model runs a mixed sequence that grows each workspace and
installs a new scale table, new CDF tables and new weights.  Every call runs three times (plain launches, graph capture,
graph replay), and every result must equal that of a fresh model with the same weights and scale table running the call
alone."""
import ctypes as C

import pytest
import torch

from tests import gpu_util as G
from textmae_image_compression_b200 import MCM, PathConfig, _native, make_state_dict

pytestmark = pytest.mark.gpu

SMALL = dict(img_size=64, encoder_embed_dim=128, encoder_depth=2, encoder_num_heads=2, num_keep_patches=16,
             decoder_embed_dim=64, decoder_depth=2, decoder_num_heads=2)
CFG = PathConfig(**SMALL)
# reductions whose order is not fixed: bpp / rate_sums sum through fp64 atomics, and the loss is torch's on x_hat
_UNORDERED = ("bpp", "rate_sums", "loss")


@pytest.fixture(scope="module")
def weights():
    return [make_state_dict(CFG, seed=s, include_decoder=True) for s in (3, 4)]


@pytest.fixture(scope="module")
def inputs():
    g = torch.Generator().manual_seed(0)
    return {n: (torch.rand(n, 3, CFG.img_size, CFG.img_size, generator=g).cuda(),
                torch.rand(n, CFG.num_patches, generator=g).cuda()) for n in (2, 8, 16)}


def _model(sd, table=None):
    m = MCM(**SMALL, softmax_isa=16, native_synthesis=True)
    m.load_state_dict(sd)
    m.cuda().eval()
    if table is not None:
        m.update(scale_table=table)
    return m


def _assert_same(got, want, where, unordered=False):
    if isinstance(want, dict):
        assert got.keys() == want.keys(), where
        for k in want:
            _assert_same(got[k], want[k], f"{where}[{k!r}]", unordered or k in _UNORDERED)
    elif isinstance(want, (list, tuple)):
        assert len(got) == len(want), where
        for i, (a, b) in enumerate(zip(got, want)):
            _assert_same(a, b, f"{where}[{i}]", unordered)
    elif isinstance(want, torch.Tensor):
        assert got.dtype == want.dtype and got.shape == want.shape, where
        if unordered:
            assert torch.allclose(got, want, rtol=1e-6, atol=0), where
        else:
            assert torch.equal(got, want), where
    else:
        assert got == want, where


class _Run:
    """The model under test and what a fresh model returns: `call(name, fn)` runs fn(model) three times against one
    fn(fresh model), the fresh model built from the current weights and scale table."""

    def __init__(self, sd):
        self.sd, self.table = sd, None
        self.m = _model(sd)

    def call(self, name, fn):
        want = fn(_model(self.sd, self.table))
        for rep in range(3):
            got = fn(self.m)
            _assert_same(got, want, f"{name} call {rep}")
        return got


def _refinalize(m, sd):
    """New weights on the same handle, as a C caller re-loads them (tmae_set_weight, then tmae_finalize_weights);
    MCM.load_state_dict makes a new handle instead."""
    lib = _native.load()
    m._weights = {k: v.float().cuda() for k, v in sd.items()}
    m._entropy_tables = None                    # the bottleneck's CDF tables follow the weights
    ign = C.c_int(0)
    for name, t in m._weights.items():
        t = t.contiguous()
        shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
        _native.check(lib.tmae_set_weight(m._handle, name.encode(), G.ptr(t), 0, t.dim(), shape, C.byref(ign)), m._handle)
    _native.check(lib.tmae_finalize_weights(m._handle), m._handle, RuntimeError)


def test_invalidation_across_plan_kinds(cuda_dev, weights, inputs):
    sd_a, sd_b = weights
    run = _Run(sd_a)
    fwd = lambda n, recon=False: (lambda m: m(*inputs[n], need_recon=recon))

    def bitstream(n, lanes):
        bs = run.call(f"compress_bitstream N={n} lanes={lanes}", lambda m: m.compress_bitstream(*inputs[n], lanes=lanes))
        run.call(f"decompress_bitstream N={n} lanes={lanes}",
                 lambda m: m.decompress_bitstream(bs["strings"], bs["shape"], bs["ids_restore"], lanes=lanes))

    def symbols(n):
        sym = run.call(f"compress_symbols N={n}", lambda m: m.compress_symbols(*inputs[n]))
        run.call(f"decompress_symbols N={n}",
                 lambda m: m.decompress_symbols(sym["z_symbols"], sym["ids_restore"], y_symbols=sym["y_symbols"]))

    def every_call():
        run.call("forward N=2", fwd(2))
        symbols(2)
        for lanes in ((32, 4), None):
            bitstream(8, lanes)
        run.call("forward N=16 need_recon", fwd(16, True))

    run.call("forward N=2", fwd(2))
    bitstream(8, None)                          # grows the network and coder workspaces past N = 2
    run.call("forward N=2 after growth", fwd(2))
    # a shorter scale table with other values: the forward plans carry its length, the coder its CDF tables
    run.table = MCM.get_scale_table(0.2, 128.0, 48)
    run.m.update(scale_table=run.table)
    run.call("forward N=2 new table", fwd(2))
    symbols(2)
    for lanes in ((32, 4), None):
        bitstream(8, lanes)
    run.call("forward N=16 need_recon", fwd(16, True))        # grows the synthesis workspace
    bitstream(8, None)                          # synthesis at N = 8 again, on the regrown workspace
    # new weights through MCM (a new handle), then on the same handle (every plan dropped at finalize)
    run.sd = sd_b
    run.m.load_state_dict(sd_b)
    run.m.cuda()
    every_call()
    run.sd = sd_a
    _refinalize(run.m, sd_a)
    every_call()
