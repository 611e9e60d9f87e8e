"""`MCM` - host-side mirror of the reference module for the compression forward path.

Same constructor keywords, state-dict names and `forward(imgs, total_scores)` contract as
`models.Compression.MCM.MCM` (/root/reference/models/Compression/MCM.py:25-52, 445-452, 590-634, 714-803),
but everything up to the rate runs in libtmae_b200.so (hand-written sm_100a kernels) through the C ABI of
include/tmae.h.  PyTorch is used for device memory, streams and the module plumbing only.

`forward` returns a superset of the reference dict:
    "likelihoods": {"y": f32 [N,Cy,s,s], "z": f32 [N,Cz,s/4,s/4]}   (same keys / shapes as MCM.py:801,
                    channels-last strides); `RateDistortionLoss.forward` reads it at loss/rd_loss.py:19-20
    "latents":     {"y_sym": i32, "z_sym": i32, "y_hat": f32, "z_hat": f32}
    "bpp":         f32 [N]   per-image rate (rd_loss.py formula with N = 1)
    "rate_sums":   f64 [2]   {sum log2 likelihood, pixels} for the data-parallel aggregate
    "ids_restore": i64 [N,L], "ids_keep": i64 [N,K], "ids_shuffle": i64 [N,L]
    "loss": (ssim_loss, l1_loss, vgg_loss), "x_hat": f32 [N,3,S,S]   when the reconstruction half is requested
                    (`need_recon=True`, or by default when the loaded state dict carries the decoder-side tensors):
                    g_s + MAE decoder + unpatchify + distortion terms (MCM.py:789-797) in stock PyTorch on the
                    library's y_hat (recon.py) - with them `RateDistortionLoss` (rd_loss.py:21-23) and
                    `utils/engine.py:189-199 val_one_epoch` run against this module unchanged
                    (tests/test_recon_cpu.py drives both, executed from /root/reference).  The VGG term is a hook
                    (`feature_loss`), 0 when unset: the reference downloads pretrained weights for it.
`compress_symbols` is the front half of `MCM.compress` (MCM.py:805-873): symbols and scale-table indexes of y in the
order `encode_with_indexes` consumes, z symbols / channel indexes for `entropy_bottleneck.compress` (SURVEY 8f-1).
`compress_bitstream` / `decompress_bitstream` add the GPU rANS coder (entropy.py, csrc/rans.cu) on either side: images to
compressai-format byte strings and back.
`decompress_symbols` is the decoder side of `MCM.decompress` (MCM.py:896-968) around the range decoder: symbols in (all at
once, or group by group through a callback that receives the scale-table indexes), y_hat / z_hat / x_hat out, bit-exact
with the encoder of the same accuracy mode.

x_hat (g_s + MAE decoder + unpatchify) comes from one of two paths:
    native_synthesis=False (default): recon.synthesize, stock fp32 PyTorch - the reference arithmetic that the conformance
                    mode (`precise=`) and the parity tests rely on;
    native_synthesis=True: `tmae_synthesize` on the engine (bf16 operands, fp32 accumulation, residual stream, LayerNorm
                    statistics and softmax; one CUDA graph per batch size) on the call's stream, for forward(need_recon),
                    decompress_symbols and decompress_bitstream.  The same accuracy-for-throughput choice `precise` offers for
                    the rate path; it needs a decoder head dim of 32 (the reference's 512 / 16).
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, Iterator, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _native, entropy, recon
from .config import PathConfig


_NATIVE_PREFIXES = ("cls_token", "encoder_pos_embed", "encoder_embed.", "encoder_blocks.", "encoder_norm.", "g_a.", "h_a.",
                    "h_s_mean.", "h_s_scale.", "cc_transform_mean.", "cc_transform_scale.", "lrp_transform.",
                    "entropy_bottleneck.")


def _native_needs(name: str) -> bool:
    return name.startswith(_NATIVE_PREFIXES)


class MCM(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, encoder_embed_dim=768, encoder_depth=12,
                 encoder_num_heads=12, decoder_embed_dim=512, decoder_depth=8, decoder_num_heads=16, mlp_ratio=4.0,
                 norm_layer=None, norm_pix_loss=False, latent_depth=384, hyperprior_depth=192, num_slices=12,
                 num_keep_patches=144, *, skip_dead_lrp: bool = False, debug_simt: bool = False,
                 softmax_isa: Optional[int] = None, extra_outputs: bool = False, share_sm: bool = False,
                 precise: Optional[str] = None, native_synthesis: bool = False):
        super().__init__()
        self.cfg = PathConfig(img_size=img_size, patch_size=patch_size, in_chans=in_chans,
                              encoder_embed_dim=encoder_embed_dim, encoder_depth=encoder_depth,
                              encoder_num_heads=encoder_num_heads, decoder_embed_dim=decoder_embed_dim,
                              decoder_depth=decoder_depth, decoder_num_heads=decoder_num_heads, mlp_ratio=mlp_ratio,
                              latent_depth=latent_depth, hyperprior_depth=hyperprior_depth, num_slices=num_slices,
                              num_keep_patches=num_keep_patches)
        self.cfg.validate()                      # same failure classes as the reference (ValueError / RuntimeError)
        self.num_keep_patches = num_keep_patches
        self.norm_pix_loss = norm_pix_loss
        self.skip_dead_lrp = skip_dead_lrp
        self.debug_simt = debug_simt
        self.share_sm = share_sm                 # several handles/streams in flight on this GPU (see TMAE_FLAG_SHARE_SM)
        self.extra_outputs = extra_outputs       # also return y, z, mu, sigma, x_remain (parity tests)
        # accuracy mode: None = bf16 operands everywhere (throughput); "rate" = split-bf16 (fp32-equivalent products) for
        # g_a and every entropy-model conv; "all" = the encoder too -> symbols match the fp32 reference up to ties
        # "-x6" suffix: three bf16 planes / six terms per product = fp32-equivalent arithmetic (default: two planes / three terms)
        if precise not in (None, "rate", "all", "rate-x6", "all-x6"):
            raise ValueError("precise must be None, 'rate', 'all', 'rate-x6' or 'all-x6'")
        self.precise = precise
        self.native_synthesis = native_synthesis  # x_hat on the engine (tmae_synthesize) instead of recon.synthesize
        self._syn_on = False                     # the handle has synthesis enabled (native_synthesis and decoder weights)
        if softmax_isa is None:
            # lane order of the ATen CPU softmax the reference's host routine would have used on this machine
            softmax_isa = 16 if "AVX512" in torch.backends.cpu.get_cpu_capability().upper() else 8
        self.softmax_isa = softmax_isa
        self.feature_loss = None                 # optional callable(preds, imgs) -> scalar: the VGG term of forward_loss
        self._scale_table = None                 # GaussianConditional scale table for compress_symbols (update())
        self._entropy_tables = None              # quantised CDF tables (entropy_tables()), rebuilt after update() / new weights
        self._last_stream = None                 # stream of the previous call on this handle (one workspace per handle)
        self._last_event = None
        self._weights: Dict[str, torch.Tensor] = {}
        self._handle = None
        self._handle_device = None
        self._dirty = True

    # ------------------------------------------------------------------ module plumbing
    def parameters(self, recurse: bool = True) -> Iterator[torch.Tensor]:
        return iter(self._weights.values())

    def named_parameters(self, prefix: str = "", recurse: bool = True, remove_duplicate: bool = True):
        return iter(self._weights.items())

    def state_dict(self, *args, **kwargs):
        return dict(self._weights)

    def load_state_dict(self, state_dict, strict: bool = True):
        self._weights = {k: v.detach().clone().float() if v.is_floating_point() else v.detach().clone()
                         for k, v in state_dict.items()}
        self._dirty = True
        self._entropy_tables = None
        return self

    @classmethod
    def from_state_dict(cls, num_keep_patches, state_dict, **kwargs):     # MCM.py:448-452
        net = cls(num_keep_patches=num_keep_patches, **kwargs)
        net.load_state_dict(state_dict)
        return net

    def _apply(self, fn, recurse=True):
        self._weights = {k: fn(v) for k, v in self._weights.items()}
        self._dirty = True
        return self

    def train(self, mode: bool = True):
        if mode:
            raise NotImplementedError("MCM (B200 path) is inference-only: additive-noise quantisation and backward "
                                      "are outside the compression forward path (SURVEY H7)")
        return super().train(False)

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def _release(self):
        if self._handle is not None:
            _native.load().tmae_destroy(self._handle)
            self._handle = None

    # ------------------------------------------------------------------ native handle
    def _device(self) -> torch.device:
        for v in self._weights.values():
            return v.device
        raise RuntimeError("no weights loaded (call load_state_dict first)")

    def _ensure_handle(self):
        dev = self._device()
        if dev.type != "cuda":
            raise RuntimeError("MCM (B200 path) runs on CUDA only - move the module with .cuda(); there is no CPU path")
        if self._handle is not None and not self._dirty and self._handle_device == dev:
            return
        lib = _native.load()
        self._release()
        c = self.cfg
        flags = ((_native.FLAG_SKIP_DEAD_LRP if self.skip_dead_lrp else 0) | (_native.FLAG_DEBUG_SIMT if self.debug_simt else 0)
                 | (_native.FLAG_SHARE_SM if self.share_sm else 0)
                 | {None: 0, "rate": _native.FLAG_PRECISE_RATE, "all": _native.FLAG_PRECISE_ALL,
                    "rate-x6": _native.FLAG_PRECISE_RATE | _native.FLAG_PRECISE_X6,
                    "all-x6": _native.FLAG_PRECISE_ALL | _native.FLAG_PRECISE_X6}[self.precise])
        cfg = _native.TmaeConfig(c.img_size, c.patch_size, c.in_chans, c.encoder_embed_dim, c.encoder_depth,
                                 c.encoder_num_heads, c.decoder_embed_dim, c.mlp_ratio, c.latent_depth,
                                 c.hyperprior_depth, c.num_slices, c.num_keep_patches, c.ln_eps, self.softmax_isa, flags)
        with torch.cuda.device(dev):
            hp = C.c_void_p()
            _native.check(lib.tmae_create(C.byref(cfg), C.byref(hp)), None, RuntimeError)
            self._handle = hp
            self._handle_device = dev
            syn = self.native_synthesis and recon.has_decoder_weights(self._weights)
            if syn:
                _native.check(lib.tmae_enable_synthesis(hp, c.decoder_depth, c.decoder_num_heads), hp)
            ign = C.c_int(0)
            for name, t in self._weights.items():
                if not t.is_floating_point():
                    continue
                if not (_native_needs(name) or (syn and name.startswith(recon.DECODER_PREFIXES))):
                    continue                          # decoder-side tensors stay with recon.py unless synthesis is native
                t = t.float().contiguous()            # .half() / .bfloat16() modules: the ABI takes fp32 (dtype 0)
                shape = (C.c_int64 * max(t.dim(), 1))(*t.shape)
                _native.check(lib.tmae_set_weight(hp, name.encode(), C.c_void_p(t.data_ptr()), 0, t.dim(), shape,
                                                  C.byref(ign)), hp)
            _native.check(lib.tmae_finalize_weights(hp), hp, RuntimeError)
        self._dirty = False
        self._syn_on = syn
        self._scale_table_dirty = True           # a fresh handle has no scale table yet
        self._cdf_dirty = True                   # ... nor cdf tables
        self._last_stream = None

    # ------------------------------------------------------------------ helpers
    def _check_inputs(self, imgs, total_scores):
        c = self.cfg
        if imgs.dim() != 4 or imgs.shape[1] != c.in_chans:
            raise AssertionError(f"expected imgs [N,{c.in_chans},S,S], got {tuple(imgs.shape)}")
        if imgs.shape[2] != c.img_size or imgs.shape[3] != c.img_size:
            raise AssertionError(f"Input image size ({imgs.shape[2]}*{imgs.shape[3]}) doesn't match model "
                                 f"({c.img_size}*{c.img_size}).")                      # timm PatchEmbed assert
        if c.num_keep_patches > total_scores.shape[1]:
            raise ValueError("Number of patches should not be greater than the length of scores")   # MCM.py:374-376
        if total_scores.shape[1] != c.num_patches or total_scores.shape[0] != imgs.shape[0]:
            raise ValueError(f"total_scores must be [N,{c.num_patches}], got {tuple(total_scores.shape)}")

    def _alloc_outputs(self, N, dev, encoder=True, rate=True, extra=False, indexes=False):
        """Every output of one call is a view into ONE fresh allocation (a single caching-allocator request per forward
        instead of 11-15: it matters at the batch-1 `testing.py` configuration)."""
        c = self.cfg
        s, s4 = c.side, c.side // 4
        spec = []          # (name, shape, dtype)
        f32, i32, i64, f64 = torch.float32, torch.int32, torch.int64, torch.float64
        if rate:
            spec += [("y_likelihoods", (N, s, s, c.latent_depth), f32), ("z_likelihoods", (N, s4, s4, c.hyperprior_depth), f32),
                     ("y_symbols", (N, s, s, c.latent_depth), i32), ("z_symbols", (N, s4, s4, c.hyperprior_depth), i32),
                     ("y_hat", (N, s, s, c.latent_depth), f32), ("z_hat", (N, s4, s4, c.hyperprior_depth), f32),
                     ("bpp", (N,), f32), ("rate_sums", (2,), f64)]
            if indexes:
                spec += [("y_indexes", (N, s, s, c.latent_depth), i32)]
            if extra:
                spec += [("y", (N, s, s, c.latent_depth), f32), ("z", (N, s4, s4, c.hyperprior_depth), f32),
                         ("mu", (N, s, s, c.latent_depth), f32), ("sigma", (N, s, s, c.latent_depth), f32)]
        if encoder:
            spec += [("ids_shuffle", (N, c.num_patches), i64), ("ids_restore", (N, c.num_patches), i64),
                     ("ids_keep", (N, c.num_keep_patches), i64)]
            if extra or not rate:
                spec += [("x_remain", (N, c.num_keep_patches, c.encoder_embed_dim), f32)]
        sizes = []
        for _, shape, dt in spec:
            n = 1
            for d in shape:
                n *= d
            sizes.append((n * dt.itemsize + 255) // 256 * 256)
        arena = torch.empty((sum(sizes),), dtype=torch.uint8, device=dev)
        t: Dict[str, torch.Tensor] = {}
        off = 0
        for (name, shape, dt), sz in zip(spec, sizes):
            n = 1
            for d in shape:
                n *= d
            t[name] = arena[off: off + n * dt.itemsize].view(dt).view(shape)
            off += sz
        o = _native.TmaeOutputs()
        for k, v in t.items():
            setattr(o, k, v.data_ptr())
        return t, o

    def _enter_stream(self, dev, stream=None):
        """One handle owns one workspace, one device IoBlock and one captured graph, so its calls must be ordered: when
        a call arrives on a different stream than the previous one, the new stream first waits for that call's event."""
        cur = stream or torch.cuda.current_stream(dev)
        if self._last_stream is not None and self._last_stream != cur:
            cur.wait_event(self._last_event)
        return cur

    def _leave_stream(self, cur):
        if self._last_event is None:
            self._last_event = torch.cuda.Event()
        self._last_event.record(cur)
        self._last_stream = cur

    @staticmethod
    def _nchw(t):          # channels-last storage viewed with the reference's [N,C,h,w] shape
        return t.permute(0, 3, 1, 2)

    def _pack_result(self, t):
        out = {
            "likelihoods": {"y": self._nchw(t["y_likelihoods"]), "z": self._nchw(t["z_likelihoods"])},
            "latents": {"y_sym": self._nchw(t["y_symbols"]), "z_sym": self._nchw(t["z_symbols"]),
                        "y_hat": self._nchw(t["y_hat"]), "z_hat": self._nchw(t["z_hat"])},
            "bpp": t["bpp"], "rate_sums": t["rate_sums"],
        }
        for k in ("ids_restore", "ids_keep", "ids_shuffle", "x_remain"):
            if k in t:
                out[k] = t[k]
        for k in ("y", "z", "mu", "sigma", "y_indexes"):
            if k in t:
                out[k] = self._nchw(t[k])
        return out

    # ------------------------------------------------------------------ the path
    def _native_forward(self, imgs, total_scores, indexes=False):
        """imgs / scores on the handle's device -> dict of channels-last result tensors (one C-ABI call)."""
        dev = self._handle_device
        N = imgs.shape[0]
        lib = _native.load()
        with torch.cuda.device(dev):
            t, o = self._alloc_outputs(N, dev, extra=self.extra_outputs, indexes=indexes)
            cur = self._enter_stream(dev)
            _native.check(lib.tmae_forward(self._handle, C.c_void_p(imgs.data_ptr()), C.c_void_p(total_scores.data_ptr()),
                                           N, C.byref(o), C.c_void_p(cur.cuda_stream)), self._handle, RuntimeError)
            self._leave_stream(cur)
        return t

    @torch.no_grad()
    def forward(self, imgs: torch.Tensor, total_scores: torch.Tensor, need_recon: Optional[bool] = None):
        """MCM.forward (MCM.py:714-803).  The rate half runs in the library; with `need_recon` (default: whenever the
        decoder-side weights are loaded) the reconstruction half follows - x_hat in stock PyTorch, or on the engine with
        native_synthesis=True - and the dict also carries the reference's "loss" 3-tuple and "x_hat"."""
        if need_recon is None:
            need_recon = recon.has_decoder_weights(self._weights)
        if need_recon and not recon.has_decoder_weights(self._weights):
            raise RuntimeError("need_recon=True but the loaded state dict has no g_s / decoder tensors")
        self._ensure_handle()
        dev = self._handle_device
        self._check_inputs(imgs, total_scores)
        imgs = imgs.to(device=dev, dtype=torch.float32).contiguous()
        total_scores = total_scores.to(device=dev, dtype=torch.float32).contiguous()
        t = self._native_forward(imgs, total_scores)
        out = self._pack_result(t)
        if need_recon:
            self._add_recon(out, t, imgs)
        return out

    def _add_recon(self, out, t, imgs):
        c = self.cfg
        N = imgs.shape[0]
        if self._syn_on:
            with torch.cuda.device(self._handle_device):
                cur = self._enter_stream(self._handle_device)
                x_hat = self._synthesize(t["y_hat"], t["ids_restore"], cur)
                self._leave_stream(cur)
            out["loss"] = recon.forward_loss(imgs, x_hat, self.feature_loss)
            out["x_hat"] = x_hat
            return
        y_hat_tokens = t["y_hat"].reshape(N, c.num_keep_patches, c.latent_depth)      # NHWC == token matrix
        loss, x_hat = recon.reconstruct(self._weights, c, y_hat_tokens, t["ids_restore"], imgs, self.feature_loss)
        out["loss"] = loss
        out["x_hat"] = x_hat

    def _synthesize(self, y_hat, ids_restore, cur):
        """x_hat f32 [N,3,S,S] from channels-last y_hat [N,s,s,Cy] and ids_restore [N,L] on the engine (tmae_synthesize),
        enqueued on `cur` (inside the handle's device context)."""
        c = self.cfg
        N = y_hat.shape[0]
        ids = ids_restore.to(device=self._handle_device, dtype=torch.int64).contiguous()
        x_hat = torch.empty((N, c.in_chans, c.img_size, c.img_size), dtype=torch.float32, device=self._handle_device)
        _native.check(_native.load().tmae_synthesize(self._handle, C.c_void_p(y_hat.data_ptr()), C.c_void_p(ids.data_ptr()), N,
                                                     C.c_void_p(x_hat.data_ptr()), C.c_void_p(cur.cuda_stream)),
                      self._handle, RuntimeError)
        return x_hat

    def _ids_not_permutation(self, ids_restore):
        """Device bool [N]: rows of ids_restore that are not a permutation of 0..L-1 (no host synchronisation)."""
        L = self.cfg.num_patches
        ids = ids_restore.to(device=self._handle_device, dtype=torch.int64)
        return (ids.sort(dim=1).values != torch.arange(L, device=ids.device)).any(dim=1)

    @staticmethod
    def _raise_if_not_permutation(bad):
        rows = [i for i, b in enumerate(bad) if b]
        if rows:
            raise ValueError(f"ids_restore rows {rows} are not permutations of 0..L-1")

    @torch.no_grad()
    def forward_encoder(self, imgs, total_scores) -> Tuple[torch.Tensor, torch.Tensor]:
        """MCM.forward_encoder (MCM.py:590-634) -> (x_remain [N,K,C], ids_restore [N,L]).
        (The reference returns ids_restore on the CPU; here it stays on the device - no host sync.)"""
        self._ensure_handle()
        dev = self._handle_device
        self._check_inputs(imgs, total_scores)
        imgs = imgs.to(device=dev, dtype=torch.float32).contiguous()
        total_scores = total_scores.to(device=dev, dtype=torch.float32).contiguous()
        N = imgs.shape[0]
        lib = _native.load()
        with torch.cuda.device(dev):
            t, o = self._alloc_outputs(N, dev, encoder=True, rate=False)
            cur = self._enter_stream(dev)
            _native.check(lib.tmae_forward_encoder(self._handle, C.c_void_p(imgs.data_ptr()),
                                                   C.c_void_p(total_scores.data_ptr()), N, C.byref(o),
                                                   C.c_void_p(cur.cuda_stream)), self._handle, RuntimeError)
            self._leave_stream(cur)
        self._last_encoder = t
        return t["x_remain"], t["ids_restore"]

    @torch.no_grad()
    def forward_from_latent(self, y_nchw: torch.Tensor, y_hat_support: Optional[torch.Tensor] = None):
        """Teacher-forced rate half (MCM.py:739-787) from y = g_a(...) [N,Cy,s,s].  With `y_hat_support` (the reference's
        y_hat, [N,Cy,s,s]) the forcing is slice-wise: every slice takes the given y_hat of the slices before it as support,
        so a rounding-boundary flip in one slice cannot cascade into the later ones."""
        self._ensure_handle()
        dev = self._handle_device
        y = y_nchw.to(device=dev, dtype=torch.float32).permute(0, 2, 3, 1).contiguous()
        N = y.shape[0]
        lib = _native.load()
        with torch.cuda.device(dev):
            t, o = self._alloc_outputs(N, dev, encoder=False, rate=True, extra=True)
            cur = self._enter_stream(dev)
            if y_hat_support is None:
                rc = lib.tmae_forward_from_latent(self._handle, C.c_void_p(y.data_ptr()), N, C.byref(o), C.c_void_p(cur.cuda_stream))
            else:
                sup = y_hat_support.to(device=dev, dtype=torch.float32).permute(0, 2, 3, 1).contiguous()
                rc = lib.tmae_forward_from_latent_forced(self._handle, C.c_void_p(y.data_ptr()), C.c_void_p(sup.data_ptr()), N,
                                                         C.byref(o), C.c_void_p(cur.cuda_stream))
            _native.check(rc, self._handle, RuntimeError)
            self._leave_stream(cur)
        return self._pack_result(t)

    def host_result_buffers(self, N: int) -> Dict[str, torch.Tensor]:
        """Pinned host buffers for `forward_host`: what the reference's forward hands its caller (likelihoods,
        MCM.py:801) + int16 symbols + ids_restore + per-image bpp."""
        c = self.cfg
        s, s4 = c.side, c.side // 4
        mk = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory()
        return {"bpp": mk((N,), torch.float32), "rate_sums": mk((2,), torch.float64),
                "y_likelihoods": mk((N, s, s, c.latent_depth), torch.float32),
                "z_likelihoods": mk((N, s4, s4, c.hyperprior_depth), torch.float32),
                "y_symbols": mk((N, s, s, c.latent_depth), torch.int16),
                "z_symbols": mk((N, s4, s4, c.hyperprior_depth), torch.int16),
                "ids_restore": mk((N, c.num_patches), torch.int64)}

    @torch.no_grad()
    def forward_host(self, imgs_cpu: torch.Tensor, scores_cpu: torch.Tensor, result: Optional[Dict[str, torch.Tensor]] = None,
                     stream: Optional[torch.cuda.Stream] = None) -> Dict[str, torch.Tensor]:
        """End-to-end call with HOST buffers (pinned for full speed): H2D copies, the forward and the D2H read of the
        results - likelihoods, int16 symbols, ids_restore, per-image bpp - are all enqueued on `stream`.  `result` is a
        dict of host tensors (see `host_result_buffers`; a subset is fine, e.g. {"bpp": ...}); returned as is, valid
        after the stream is synchronised."""
        self._ensure_handle()
        dev = self._handle_device
        if imgs_cpu.device.type != "cpu" or scores_cpu.device.type != "cpu":
            raise ValueError("forward_host takes CPU tensors")
        self._check_inputs(imgs_cpu, scores_cpu)
        imgs_cpu = imgs_cpu.contiguous()
        scores_cpu = scores_cpu.contiguous()
        N = imgs_cpu.shape[0]
        if result is None:
            result = self.host_result_buffers(N)
        ho = _native.TmaeHostOutputs()
        for k, v in result.items():
            if k not in _native.HOST_OUTPUT_FIELDS:
                raise KeyError(f"unknown host result '{k}'")
            setattr(ho, k, v.data_ptr())
        lib = _native.load()
        with torch.cuda.device(dev):
            cur = self._enter_stream(dev, stream)
            _native.check(lib.tmae_forward_host(self._handle, C.c_void_p(imgs_cpu.data_ptr()),
                                                C.c_void_p(scores_cpu.data_ptr()), N, C.byref(ho), None,
                                                C.c_void_p(cur.cuda_stream)), self._handle, RuntimeError)
            self._leave_stream(cur)
        return result

    @torch.no_grad()
    def get_ids_shuffle(self, total_scores: torch.Tensor) -> torch.Tensor:
        """MCM.get_ids_shuffle (MCM.py:364-423) on the GPU: int64 [N, L] (device tensor)."""
        K = self.num_keep_patches
        if K > total_scores.shape[1]:
            raise ValueError("Number of patches should not be greater than the length of scores")
        dev = total_scores.device if total_scores.is_cuda else self._device()
        sc = total_scores.to(device=dev, dtype=torch.float32).contiguous()
        N, L = sc.shape
        out = torch.empty((N, L), dtype=torch.int64, device=dev)
        lib = _native.load()
        with torch.cuda.device(dev):
            st = torch.cuda.current_stream(dev).cuda_stream
            _native.check(lib.tmae_mask_select(C.c_void_p(sc.data_ptr()), N, L, K, self.softmax_isa,
                                               C.c_void_p(out.data_ptr()), None, None, C.c_void_p(st)))
        return out

    def random_masking(self, x, total_scores):
        """MCM.random_masking (MCM.py:548-588): gather of the kept tokens with GPU-computed ids."""
        ids_shuffle = self.get_ids_shuffle(total_scores)
        ids_restore = torch.argsort(ids_shuffle, dim=1)
        ids_keep = ids_shuffle[:, : self.num_keep_patches].to(x.device)
        x_remain = torch.gather(x, 1, ids_keep.unsqueeze(-1).repeat(1, 1, x.shape[-1]))
        return x_remain, ids_restore

    # ------------------------------------------------------------------ small host-side pieces of the interface
    def aux_loss(self) -> torch.Tensor:
        """compressai CompressionModel.aux_loss() == EntropyBottleneck.loss(): sum |logits(quantiles) - target|
        (called by utils/engine.py:194).  Pure function of 11.7 k parameters - evaluated with torch ops."""
        w = self._weights
        q = w["entropy_bottleneck.quantiles"]
        logits = q
        for i in range(5):
            logits = torch.matmul(F.softplus(w[f"entropy_bottleneck._matrix{i}"]), logits) + w[f"entropy_bottleneck._bias{i}"]
            if i < 4:
                logits = logits + torch.tanh(w[f"entropy_bottleneck._factor{i}"]) * torch.tanh(logits)
        import math
        t = math.log(2 / 1e-9 - 1)
        target = torch.tensor([-t, 0.0, t], device=q.device, dtype=q.dtype)
        return torch.abs(logits - target).sum()

    @staticmethod
    def get_scale_table(min_scale: float = 0.11, max_scale: float = 256.0, levels: int = 64) -> torch.Tensor:
        """compressai.models.utils / google.get_scale_table: the table `CompressionModel.update()` installs when
        called without one (testing.py:223 `model.update(force=True)`)."""
        import math
        return torch.exp(torch.linspace(math.log(min_scale), math.log(max_scale), levels))

    def update(self, scale_table=None, force: bool = False):
        """The part of `CompressionModel.update(scale_table, force)` that the symbol / index emission needs: install the
        GaussianConditional scale table (default `get_scale_table()`).  The quantised CDF tables of the range coder
        (`entropy_tables()`) are rebuilt from it and the weights on their next use."""
        self._scale_table = (self.get_scale_table() if scale_table is None else torch.as_tensor(scale_table)).float().contiguous()
        self._scale_table_dirty = True
        self._entropy_tables = None
        return True

    def _install_scale_table(self):
        """Hand the GaussianConditional scale table to the handle (the default table if `update()` was never called)."""
        if self._scale_table is None:
            self.update()
        self._ensure_handle()
        if getattr(self, "_scale_table_dirty", True):
            tab = self._scale_table
            with torch.cuda.device(self._handle_device):
                _native.check(_native.load().tmae_set_scale_table(self._handle, C.c_void_p(tab.data_ptr()), tab.numel()), self._handle)
            self._scale_table_dirty = False

    @torch.no_grad()
    def compress_symbols(self, imgs: torch.Tensor, total_scores: torch.Tensor):
        """Front half of `MCM.compress` (MCM.py:805-873), everything up to the `encode_with_indexes` call:
            "y_symbols", "y_indexes": i32 [N, Cy*s*s]  - per image, slice by slice in (c, y, x) order, exactly the lists the
                          reference extends per slice (MCM.py:872-873) and passes to the coder (:882-884);
                          indexes = GaussianConditional.build_indexes(sigma) (:867)
            "z_symbols": i32 [N, Cz, s/4, s/4], "z_indexes": i32 [same] - what `entropy_bottleneck.compress(z)` codes
                          (:827): quantize(z, "symbols", medians) and the channel index of every element
            "shape": z spatial size (:890), "ids_restore" (:891)
        `compress_bitstream` runs the range coder on these lists."""
        self._install_scale_table()
        dev = self._handle_device
        lib = _native.load()
        self._check_inputs(imgs, total_scores)
        imgs = imgs.to(device=dev, dtype=torch.float32).contiguous()
        total_scores = total_scores.to(device=dev, dtype=torch.float32).contiguous()
        t = self._native_forward(imgs, total_scores, indexes=True)
        c = self.cfg
        N, s, s4 = imgs.shape[0], c.side, c.side // 4
        packed = torch.empty((2, N, c.latent_depth * s * s), dtype=torch.int32, device=dev)
        zpacked = torch.empty((N, c.hyperprior_depth, s4, s4), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            for k, name in enumerate(("y_symbols", "y_indexes")):
                _native.check(lib.tmae_pack_nchw_i32(C.c_void_p(t[name].data_ptr()), C.c_void_p(packed[k].data_ptr()), N, s * s,
                                                     c.latent_depth, st))
            _native.check(lib.tmae_pack_nchw_i32(C.c_void_p(t["z_symbols"].data_ptr()), C.c_void_p(zpacked.data_ptr()), N, s4 * s4,
                                                 c.hyperprior_depth, st))
        z_idx = torch.arange(c.hyperprior_depth, dtype=torch.int32, device=dev).view(1, -1, 1, 1).expand(N, -1, s4, s4)
        return {"y_symbols": packed[0], "y_indexes": packed[1], "z_symbols": zpacked, "z_indexes": z_idx,
                "shape": (s4, s4), "ids_restore": t["ids_restore"], "bpp": t["bpp"]}

    @torch.no_grad()
    def decompress_symbols(self, z_symbols: torch.Tensor, ids_restore: torch.Tensor, y_symbols: Optional[torch.Tensor] = None,
                           decode_fn: Optional[Callable[[int, torch.Tensor], torch.Tensor]] = None,
                           need_recon: Optional[bool] = None) -> Dict[str, torch.Tensor]:
        """`MCM.decompress` (MCM.py:896-968) with the range decoder left to the caller: symbols -> y_hat, z_hat (-> x_hat).
            z_symbols  i32 [N, Cz, s/4, s/4]  (`compress_symbols()["z_symbols"]`)
            ids_restore  i64 [N, L]           (the side information; used for x_hat only)
        and exactly one of
            y_symbols  i32 [N, Cy*s*s]        every slice's symbols at once (`compress_symbols()["y_symbols"]`): the whole
                                              decode is enqueued on the current stream without a host synchronisation;
            decode_fn  callable(first_slice, indexes) -> symbols: called once per slice group (slices 0..5 one by one, then
                                              6..11 together) with the group's scale-table indexes, i32 [N, n_slices, Cs, s, s]
                                              on the device - the list the reference hands `decode_stream` for those slices -
                                              and returning the group's symbols of the same shape (any device).  This is
                                              where compressai's `RansDecoder.decode_stream` plugs in.
        The decode runs the encoder's own kernels and launch shapes, so it reproduces the y_hat / z_hat / indexes of a
        module of the same configuration (same `precise` mode) bit for bit.
        Returns {"y_hat": f32 [N,Cy,s,s], "z_hat": f32 [N,Cz,s/4,s/4], "y_indexes": i32 [N, Cy*s*s]} and, with `need_recon`
        (default: whenever the decoder-side weights are loaded), "x_hat": f32 [N,3,S,S] computed exactly as forward's
        x_hat (recon.synthesize, or tmae_synthesize with native_synthesis=True).  No post-processing (e.g. clamping) is
        applied to x_hat: it is forward's x_hat.  With native_synthesis=True the x_hat is enqueued on the same stream, and a
        row of ids_restore that is not a permutation of 0..L-1 raises ValueError (checked on the device, read once at the end)."""
        if (y_symbols is None) == (decode_fn is None):
            raise ValueError("give exactly one of y_symbols and decode_fn")
        if need_recon is None:
            need_recon = recon.has_decoder_weights(self._weights)
        if need_recon and not recon.has_decoder_weights(self._weights):
            raise RuntimeError("need_recon=True but the loaded state dict has no g_s / decoder tensors")
        self._install_scale_table()
        dev = self._handle_device
        c = self.cfg
        s, s4, sc, ns = c.side, c.side // 4, c.slice_ch, c.num_slices
        N = z_symbols.shape[0] if z_symbols.dim() == 4 else -1
        if z_symbols.dtype != torch.int32 or tuple(z_symbols.shape) != (N, c.hyperprior_depth, s4, s4) or N < 1:
            raise ValueError(f"z_symbols must be int32 [N, {c.hyperprior_depth}, {s4}, {s4}], got {z_symbols.dtype} {tuple(z_symbols.shape)}")
        if tuple(ids_restore.shape) != (N, c.num_patches):
            raise ValueError(f"ids_restore must be [{N}, {c.num_patches}], got {tuple(ids_restore.shape)}")
        if y_symbols is not None and (y_symbols.dtype != torch.int32 or tuple(y_symbols.shape) != (N, c.latent_depth * s * s)):
            raise ValueError(f"y_symbols must be int32 [{N}, {c.latent_depth * s * s}], got {y_symbols.dtype} {tuple(y_symbols.shape)}")
        lib = _native.load()
        firsts, counts = (C.c_int * ns)(), (C.c_int * ns)()
        n_groups = lib.tmae_decode_groups(ns, firsts, counts, ns)
        if n_groups < 1:
            raise RuntimeError(f"tmae_decode_groups({ns}) failed")
        groups = [(firsts[g], counts[g]) for g in range(n_groups)]
        zs = z_symbols.to(dev).contiguous()
        f32 = torch.float32
        y_hat = torch.empty((N, s, s, c.latent_depth), dtype=f32, device=dev)
        z_hat = torch.empty((N, s4, s4, c.hyperprior_depth), dtype=f32, device=dev)
        y_idx = torch.empty((N, c.latent_depth * s * s), dtype=torch.int32, device=dev)
        ys = y_symbols.to(dev).contiguous() if y_symbols is not None else torch.empty_like(y_idx)
        o = _native.TmaeOutputs()
        o.y_hat, o.z_hat, o.y_indexes = y_hat.data_ptr(), z_hat.data_ptr(), y_idx.data_ptr()
        by_slice = lambda t: t.view(N, ns, sc, s, s)
        with torch.cuda.device(dev):
            cur = self._enter_stream(dev)
            st = C.c_void_p(cur.cuda_stream)
            _native.check(lib.tmae_decode_begin(self._handle, C.c_void_p(zs.data_ptr()), N, C.byref(o), st), self._handle, RuntimeError)
            for g, (first, cnt) in enumerate(groups):
                if decode_fn is not None:
                    sym = decode_fn(first, by_slice(y_idx)[:, first:first + cnt])
                    sym = torch.as_tensor(sym)
                    if tuple(sym.shape) != (N, cnt, sc, s, s) or sym.is_floating_point() or sym.is_complex():
                        raise ValueError(f"decode_fn must return integer symbols [{N}, {cnt}, {sc}, {s}, {s}], got {sym.dtype} {tuple(sym.shape)}")
                    by_slice(ys)[:, first:first + cnt] = sym.to(device=dev, dtype=torch.int32)
                _native.check(lib.tmae_decode_step(self._handle, g, C.c_void_p(ys.data_ptr()), C.byref(o), st), self._handle, RuntimeError)
            x_hat = self._synthesize(y_hat, ids_restore, cur) if need_recon and self._syn_on else None
            self._leave_stream(cur)
        out = {"y_hat": self._nchw(y_hat), "z_hat": self._nchw(z_hat), "y_indexes": y_idx}
        if x_hat is not None:
            self._raise_if_not_permutation(self._ids_not_permutation(ids_restore).tolist())
            out["x_hat"] = x_hat
        elif need_recon:
            out["x_hat"] = recon.synthesize(self._weights, c, y_hat.reshape(N, c.num_keep_patches, c.latent_depth), ids_restore.to(dev))
        return out

    # ------------------------------------------------------------------ bitstreams (the GPU rANS coder)
    def entropy_tables(self) -> Dict[str, torch.Tensor]:
        """The quantised CDF tables compressai's `update(force=True)` would build for this module's weights and scale table,
        under compressai's buffer names (CPU int32): gaussian_conditional._quantized_cdf / _cdf_length / _offset (one table
        per scale-table entry) and entropy_bottleneck._quantized_cdf / _cdf_length / _offset (one per channel)."""
        if self._entropy_tables is None:
            if self._scale_table is None:
                self.update()
            t = {}
            for prefix, tabs in (("gaussian_conditional.", entropy.gaussian_tables(self._scale_table)),
                                 ("entropy_bottleneck.", entropy.bottleneck_tables(self._weights))):
                t.update({prefix + k: v for k, v in tabs.items()})
            self._entropy_tables = t
            self._cdf_dirty = True
        return self._entropy_tables

    def _install_coder_tables(self):
        self._install_scale_table()
        tabs = self.entropy_tables()
        if self._cdf_dirty:
            with torch.cuda.device(self._handle_device):
                for model, prefix in ((_native.MODEL_GAUSSIAN, "gaussian_conditional."), (_native.MODEL_BOTTLENECK, "entropy_bottleneck.")):
                    entropy.set_tables(self._handle, model, {k: tabs[prefix + k] for k in ("_quantized_cdf", "_cdf_length", "_offset")})
            self._cdf_dirty = False

    @staticmethod
    def _check_lanes(lanes):
        """None (compressai's format) or (W_y, W_z), each in 1..32 (the laned format, DESIGN.md section 7)."""
        if lanes is None:
            return None
        if (not isinstance(lanes, (tuple, list)) or len(lanes) != 2
                or not all(isinstance(w, int) and not isinstance(w, bool) and 1 <= w <= 32 for w in lanes)):
            raise ValueError(f"lanes must be None or (W_y, W_z) with integers in 1..32, got {lanes!r}")
        return int(lanes[0]), int(lanes[1])

    @torch.no_grad()
    def compress_bitstream(self, imgs: torch.Tensor, total_scores: torch.Tensor, lanes=None):
        """`MCM.compress` (MCM.py:805-893) on the GPU: {"strings": [y_strings, z_strings], "shape", "ids_restore"} with one
        `bytes` per image in each list (compressai's rANS format: the y stream codes every slice in order with the Gaussian
        tables, the z stream the z symbols with the bottleneck tables), plus "bpp" [N], the likelihood estimate of the rate.
        compress_symbols, one encode call per stream kind, then two reads to the host: the stream offsets and status (a few
        hundred bytes, which size the second read), then exactly the packed bytes.  Each encode call writes into an output of
        n_streams * tmae_rans_bound(n) bytes (the worst case, ~63 MB for the y streams at batch 64 and K=64), and the handle
        keeps an encode scratch of about the same size.
        lanes=(W_y, W_z) writes the laned format instead (every y stream in W_y lanes, every z stream in W_z, each lane a
        compressai stream; they decode in parallel) and adds "lanes": (W_y, W_z) to the dict."""
        lanes = self._check_lanes(lanes)
        self._ensure_handle()
        self._install_coder_tables()
        sym = self.compress_symbols(imgs, total_scores)
        N = sym["y_symbols"].shape[0]
        lib_h = self._handle
        with torch.cuda.device(self._handle_device):
            cur = self._enter_stream(self._handle_device)
            if lanes is None:
                y_out, y_off, y_st = entropy.encode(lib_h, _native.MODEL_GAUSSIAN, sym["y_symbols"], sym["y_indexes"])
                z_out, z_off, z_st = entropy.encode(lib_h, _native.MODEL_BOTTLENECK, sym["z_symbols"].reshape(N, -1),
                                                    sym["z_indexes"].reshape(N, -1))
            else:
                y_out, y_off, y_st = entropy.encode_lanes(lib_h, _native.MODEL_GAUSSIAN, sym["y_symbols"], sym["y_indexes"], lanes[0])
                z_out, z_off, z_st = entropy.encode_lanes(lib_h, _native.MODEL_BOTTLENECK, sym["z_symbols"].reshape(N, -1),
                                                          sym["z_indexes"].reshape(N, -1), lanes[1])
            self._leave_stream(cur)
            meta = torch.cat([y_off, z_off, y_st.long(), z_st.long()]).cpu()
            y_off, z_off = meta[: N + 1].tolist(), meta[N + 1: 2 * N + 2].tolist()
            bad = [i for i in range(N) if meta[2 * N + 2 + i] or meta[3 * N + 2 + i]]
            if bad:
                raise RuntimeError(f"rANS encode failed for images {bad} (status {meta[2 * N + 2:].tolist()})")
            host = torch.cat([y_out[: y_off[-1]], z_out[: z_off[-1]]]).cpu().numpy().tobytes()
        zb = y_off[-1]
        y_strings = [host[y_off[i]: y_off[i + 1]] for i in range(N)]
        z_strings = [host[zb + z_off[i]: zb + z_off[i + 1]] for i in range(N)]
        out = {"strings": [y_strings, z_strings], "shape": sym["shape"], "ids_restore": sym["ids_restore"], "bpp": sym["bpp"]}
        if lanes is not None:
            out["lanes"] = lanes
        return out

    @torch.no_grad()
    def decompress_bitstream(self, strings, shape, ids_restore: torch.Tensor, need_recon: Optional[bool] = None,
                             lanes=None) -> Dict[str, torch.Tensor]:
        """`MCM.decompress` (MCM.py:896-968) on the GPU from `compress_bitstream`'s strings: one copy of the concatenated bytes
        to the device, then the range decoder and the network in one enqueued decode (no host round trip in between).
        Returns {"y_hat": f32 [N,Cy,s,s], "z_hat": f32 [N,Cz,s/4,s/4]} and, with `need_recon` (default: whenever the
        decoder-side weights are loaded), "x_hat" exactly as forward computes it.  Raises ValueError for malformed arguments,
        and for images whose streams do not decode exactly to their end (naming them).  With native_synthesis=True the x_hat is
        enqueued before the status read, which also carries the check that every row of ids_restore is a permutation of 0..L-1
        (ValueError otherwise).  lanes=(W_y, W_z): the strings are in
        the laned format of `compress_bitstream(..., lanes=(W_y, W_z))`; a header with another lane count, or lane lengths
        that do not add up, is a stream that does not decode."""
        lanes = self._check_lanes(lanes)
        if need_recon is None:
            need_recon = recon.has_decoder_weights(self._weights)
        if need_recon and not recon.has_decoder_weights(self._weights):
            raise RuntimeError("need_recon=True but the loaded state dict has no g_s / decoder tensors")
        self._ensure_handle()
        c = self.cfg
        s, s4 = c.side, c.side // 4
        if not isinstance(strings, (list, tuple)) or len(strings) != 2:
            raise ValueError("strings must be [y_strings, z_strings]")
        y_strings, z_strings = list(strings[0]), list(strings[1])
        N = len(y_strings)
        if N < 1 or len(z_strings) != N:
            raise ValueError(f"need as many z strings as y strings (>= 1), got {N} and {len(z_strings)}")
        for k, (kind, lst) in enumerate((("y", y_strings), ("z", z_strings))):
            # shortest stream: 8 bytes, or with W lanes the header and W empty lanes, 4 (1 + W) + 8 W
            least = 8 if lanes is None else 4 * (1 + lanes[k]) + 8 * lanes[k]
            for i, b in enumerate(lst):
                if not isinstance(b, (bytes, bytearray, memoryview)) or len(b) % 4 or len(b) < least:
                    raise ValueError(f"{kind} string of image {i}: need bytes of a length that is a multiple of 4 and >= {least}")
        if tuple(shape) != (s4, s4):
            raise ValueError(f"shape must be ({s4}, {s4}) for this model, got {tuple(shape)}")
        if tuple(ids_restore.shape) != (N, c.num_patches):
            raise ValueError(f"ids_restore must be [{N}, {c.num_patches}], got {tuple(ids_restore.shape)}")
        self._install_coder_tables()
        dev = self._handle_device
        # one host buffer: y offsets | z offsets (int64 [N + 1] each) | y bytes | z bytes
        y_data, y_off = entropy.pack_strings([bytes(b) for b in y_strings])
        z_data, z_off = entropy.pack_strings([bytes(b) for b in z_strings])
        host = torch.cat([y_off.view(torch.uint8), z_off.view(torch.uint8), y_data, z_data])
        f32 = torch.float32
        y_hat = torch.empty((N, s, s, c.latent_depth), dtype=f32, device=dev)
        z_hat = torch.empty((N, s4, s4, c.hyperprior_depth), dtype=f32, device=dev)
        status = torch.empty(N, dtype=torch.int32, device=dev)
        o = _native.TmaeOutputs()
        o.y_hat, o.z_hat = y_hat.data_ptr(), z_hat.data_ptr()
        lib = _native.load()
        with torch.cuda.device(dev):
            cur = self._enter_stream(dev)
            buf = host.pin_memory().to(dev, non_blocking=True)
            b0 = buf.data_ptr()
            no = 8 * (N + 1)
            yp, yo, zp, zo = (C.c_void_p(b0 + 2 * no), C.c_void_p(b0), C.c_void_p(b0 + 2 * no + y_data.numel()), C.c_void_p(b0 + no))
            if lanes is None:
                rc = lib.tmae_decompress_streams(self._handle, yp, yo, zp, zo, N, C.byref(o), C.c_void_p(status.data_ptr()),
                                                 C.c_void_p(cur.cuda_stream))
            else:
                rc = lib.tmae_decompress_streams_lanes(self._handle, yp, yo, lanes[0], zp, zo, lanes[1], N, C.byref(o),
                                                       C.c_void_p(status.data_ptr()), C.c_void_p(cur.cuda_stream))
            _native.check(rc, self._handle, RuntimeError)
            x_hat = None
            if need_recon and self._syn_on:   # enqueued before the status read: the one host round trip covers both
                x_hat = self._synthesize(y_hat, ids_restore, cur)
                status = torch.cat([status, self._ids_not_permutation(ids_restore).int()])
            self._leave_stream(cur)
        st = status.cpu()
        bad = [i for i in range(N) if st[i]]
        if bad:
            raise ValueError(f"the streams of images {bad} do not decode (status {[int(st[i]) for i in bad]}: truncated or corrupt)")
        out = {"y_hat": self._nchw(y_hat), "z_hat": self._nchw(z_hat)}
        if x_hat is not None:
            self._raise_if_not_permutation(st[N:].tolist())
            out["x_hat"] = x_hat
        elif need_recon:
            out["x_hat"] = recon.synthesize(self._weights, c, y_hat.reshape(N, c.num_keep_patches, c.latent_depth), ids_restore.to(dev))
        return out

    def compress(self, *args, **kwargs):
        raise NotImplementedError("MCM.compress is not provided under the reference's name until the bitstream format has been "
                                  "checked against compressai itself; compress_bitstream() returns the reference's compress dict "
                                  "(rANS strings coded on the GPU), compress_symbols() the symbol / index lists")

    def decompress(self, *args, **kwargs):
        raise NotImplementedError("MCM.decompress is not provided under the reference's name until the bitstream format has been "
                                  "checked against compressai itself; decompress_bitstream() decodes compress_bitstream()'s "
                                  "strings on the GPU, decompress_symbols() rebuilds y_hat / x_hat from decoded symbols")

    # ------------------------------------------------------------------ profiling hooks (bench.py)
    def profile(self, enable: bool, by_run: bool = False):
        """Device timing of the next forwards: per launch, or per run of consecutive same-family launches (by_run)."""
        self._ensure_handle()
        _native.check(_native.load().tmae_profile_enable(self._handle, (2 if by_run else 1) if enable else 0), self._handle)

    def profile_read(self):
        arr = (_native.TmaeProfileEntry * 16)()
        n = C.c_int(0)
        _native.check(_native.load().tmae_profile_read(self._handle, arr, 16, C.byref(n)), self._handle, RuntimeError)
        return [{"name": arr[i].name.decode(), "launches": arr[i].launches, "ms": arr[i].ms, "flops": arr[i].flops,
                 "bytes": arr[i].bytes, "mma_flops": arr[i].mma_flops} for i in range(n.value)]

    def profile_read_steps(self):
        arr = (_native.TmaeProfileStep * 512)()
        n = C.c_int(0)
        _native.check(_native.load().tmae_profile_read_steps(self._handle, arr, 512, C.byref(n)), self._handle, RuntimeError)
        return [{"name": arr[i].name.decode(), "ms": arr[i].ms, "flops": arr[i].flops, "ctas": arr[i].ctas,
                 "block_n": arr[i].block_n} for i in range(n.value)]

    def launch_count(self, N: int) -> int:
        self._ensure_handle()
        return int(_native.load().tmae_launch_count(self._handle, N))

    def reserve(self, N: int):
        self._ensure_handle()
        with torch.cuda.device(self._handle_device):
            _native.check(_native.load().tmae_reserve(self._handle, N), self._handle, RuntimeError)
