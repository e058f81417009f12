"""The COTR network as an nn.Module shell around the native sm_100a implementation.

Reference contract (COTR/models/cotr_model.py:17-51):
  * `build(args)` -> module with attributes transformer (.d_model), corr_embed, query_proj, input_proj, backbone;
  * `state_dict()` has the reference's 381 keys / shapes (SURVEY.md appendix C) so `utils.safe_load_weights`
    (COTR/utils/utils.py:164-193) loads a reference checkpoint with strict=True; FrozenBN statistics are buffers
    (backbone.py:31-34) and `num_batches_tracked` is dropped on load (backbone.py:38-40);
  * `forward(samples, queries) -> {'pred_corrs': (B,Q,2)}` on the module's device; samples is a (B,3,256,512) tensor,
    a list of (3,256,512) tensors or a NestedTensor; the canvas size is asserted like backbone.py:80.

`batch_invariant` (off by default; `args.batch_invariant` or `set_batch_invariant`) makes every pair and query come out
bit-identical whatever else shares the call: batch size, query count, decode chunking, entry point, rank count
(cotr_set_batch_invariant in include/cotr_b200.h).  It is a property of the handle, not a parameter: the state_dict is
the same in both modes.

The arithmetic is NOT done by torch: forward hands device pointers to libcotr_b200.so (include/cotr_b200.h).
There is no CPU path; calling forward without a CUDA device or without the built library raises.
Unlike the reference constructor (backbone.py:106 `pretrained=True`) nothing is downloaded.
"""
import math

import torch
from torch import nn

from .. import capi
from .misc import NestedTensor, nested_tensor_from_tensor_list

MAX_SIZE = 256     # COTR/utils/constants.py:2
_BN_FIELDS = ("weight", "bias", "running_mean", "running_var")


class _Namespace(nn.Module):
    """A stateless container node of the module tree (children are added by name)."""

    def forward(self, *a, **k):   # pragma: no cover
        raise RuntimeError("this sub-module is a parameter container; call the COTR module itself")


class FrozenBatchNorm2d(_Namespace):
    """Parameter holder for backbone.py:21-56: statistics and affine terms are buffers, folded into the conv at pack time."""

    def __init__(self, n):
        super().__init__()
        self.register_buffer("weight", torch.ones(n))
        self.register_buffer("bias", torch.zeros(n))
        self.register_buffer("running_mean", torch.zeros(n))
        self.register_buffer("running_var", torch.ones(n))

    def _load_from_state_dict(self, state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs):
        state_dict.pop(prefix + 'num_batches_tracked', None)
        super()._load_from_state_dict(state_dict, prefix, local_metadata, strict, missing_keys, unexpected_keys, error_msgs)


class _Weight(_Namespace):
    def __init__(self, shape, bias=False, init="xavier"):
        super().__init__()
        w = torch.empty(*shape)
        if init == "kaiming":
            nn.init.kaiming_normal_(w, mode="fan_out", nonlinearity="relu")
        elif len(shape) >= 2:
            nn.init.xavier_uniform_(w.view(shape[0], -1))
        else:
            nn.init.ones_(w)
        self.weight = nn.Parameter(w, requires_grad=False)
        if bias:
            self.bias = nn.Parameter(torch.zeros(shape[0]), requires_grad=False)


class _MHA(_Namespace):
    def __init__(self, d):
        super().__init__()
        w = torch.empty(3 * d, d)
        nn.init.xavier_uniform_(w)
        self.in_proj_weight = nn.Parameter(w, requires_grad=False)
        self.in_proj_bias = nn.Parameter(torch.zeros(3 * d), requires_grad=False)
        self.out_proj = _Weight((d, d), bias=True)


def _norm(d):
    m = _Namespace()
    m.weight = nn.Parameter(torch.ones(d), requires_grad=False)
    m.bias = nn.Parameter(torch.zeros(d), requires_grad=False)
    return m


def _bottleneck(inplanes, planes, downsample):
    b = _Namespace()
    b.conv1 = _Weight((planes, inplanes, 1, 1), init="kaiming"); b.bn1 = FrozenBatchNorm2d(planes)
    b.conv2 = _Weight((planes, planes, 3, 3), init="kaiming"); b.bn2 = FrozenBatchNorm2d(planes)
    b.conv3 = _Weight((planes * 4, planes, 1, 1), init="kaiming"); b.bn3 = FrozenBatchNorm2d(planes * 4)
    if downsample:
        ds = _Namespace()
        ds.add_module("0", _Weight((planes * 4, inplanes, 1, 1), init="kaiming"))
        ds.add_module("1", FrozenBatchNorm2d(planes * 4))
        b.downsample = ds
    return b


def _resnet50_layer3_body():
    """torchvision resnet50 up to layer3 (what IntermediateLayerGetter keeps, backbone.py:70-71), as a parameter tree."""
    body = _Namespace()
    body.conv1 = _Weight((64, 3, 7, 7), init="kaiming")
    body.bn1 = FrozenBatchNorm2d(64)
    inplanes = 64
    for name, n_blocks, planes in (("layer1", 3, 64), ("layer2", 4, 128), ("layer3", 6, 256)):
        layer = _Namespace()
        for i in range(n_blocks):
            layer.add_module(str(i), _bottleneck(inplanes, planes, downsample=(i == 0)))
            inplanes = planes * 4
        body.add_module(name, layer)
    return body


def _transformer(d, ff, n_enc, n_dec):
    t = _Namespace()
    t.d_model = d
    t.nhead = 8
    enc = _Namespace(); enc_layers = _Namespace()
    for l in range(n_enc):
        e = _Namespace()
        e.self_attn = _MHA(d)
        e.linear1 = _Weight((ff, d), bias=True); e.linear2 = _Weight((d, ff), bias=True)
        e.norm1 = _norm(d); e.norm2 = _norm(d)
        enc_layers.add_module(str(l), e)
    enc.layers = enc_layers
    dec = _Namespace(); dec_layers = _Namespace()
    for l in range(n_dec):
        e = _Namespace()
        e.multihead_attn = _MHA(d)
        e.linear1 = _Weight((ff, d), bias=True); e.linear2 = _Weight((d, ff), bias=True)
        e.norm1 = _norm(d)      # present in the checkpoint, never used (transformer.py:173 vs :185-201)
        e.norm2 = _norm(d); e.norm3 = _norm(d)
        dec_layers.add_module(str(l), e)
    dec.layers = dec_layers
    dec.norm = _norm(d)
    t.encoder = enc
    t.decoder = dec
    return t


class Context:
    """Encoded image pairs: the 6-layer decoder K/V cache living on the device (see cotr_encode_context)."""

    def __init__(self, native_ctx, batch):
        self.native = native_ctx
        self.batch = batch


class COTR(nn.Module):
    def __init__(self, args=None):
        super().__init__()
        cfg = dict(backbone="resnet50", hidden_dim=256, dilation=False, nheads=8, layer="layer3", enc_layers=6,
                   dec_layers=6, position_embedding="lin_sine", dim_feedforward=1024)
        if args is not None:
            for k, v in cfg.items():
                got = getattr(args, k, v)
                if got != v:
                    raise NotImplementedError(
                        f"cotr_b200 implements the configuration every reference demo uses ({k}={v!r}); got {k}={got!r}")
        d = cfg["hidden_dim"]
        self.transformer = _transformer(d, cfg["dim_feedforward"], 6, 6)
        head = _Namespace(); head.num_layers = 3
        layers = _Namespace()
        for i, shp in enumerate(((d, d), (d, d), (2, d))):
            layers.add_module(str(i), _Weight(shp, bias=True))
        head.layers = layers
        self.corr_embed = head
        self.query_proj = _Namespace()            # NerfPositionalEncoding(64): stateless
        self.input_proj = _Weight((d, 1024, 1, 1), bias=True)
        backbone = _Namespace()
        b0 = _Namespace(); b0.body = _resnet50_layer3_body(); b0.num_channels = 1024
        backbone.add_module("0", b0)
        backbone.add_module("1", _Namespace())    # PositionEmbeddingSine: stateless
        backbone.num_channels = 1024
        self.backbone = backbone
        self._native = None
        self._ctx_cache = {}
        self._batch_invariant = bool(getattr(args, "batch_invariant", False)) if args is not None else False

    # ---- native handle management ---------------------------------------------------------------------
    def _invalidate(self):
        for ctx in self._ctx_cache.values():
            ctx.close()
        self._ctx_cache = {}
        if self._native is not None:
            self._native.close()
        self._native = None

    def _apply(self, fn, *a, **k):                # .cuda() / .to() / .float(): weights move -> repack lazily
        self._invalidate()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, state_dict, *a, **k):
        self._invalidate()
        return super().load_state_dict(state_dict, *a, **k)

    def refresh_native(self):
        """Call after editing parameters in place: the packed device copy is rebuilt on the next forward."""
        self._invalidate()

    def native(self):
        if self._native is None:
            dev = next(self.parameters()).device
            if dev.type != "cuda":
                raise RuntimeError("cotr_b200.COTR runs only on a CUDA device (sm_100a): call model.cuda() first; "
                                   "there is no CPU fallback")
            idx = dev.index if dev.index is not None else torch.cuda.current_device()
            nat = capi.NativeModel(self.state_dict(), idx)
            if self._batch_invariant:
                nat.set_batch_invariant(True)
            self._native = nat
        return self._native

    @property
    def batch_invariant(self):
        """True: predictions are bit-identical for any batch size, query count, chunking, entry point or rank count."""
        return self._batch_invariant

    def set_batch_invariant(self, enabled):
        """Switch the batch-invariant mode.  Cached encode_context(reuse=True) contexts are closed (a context is only
        valid under the mode it was encoded in); the packed weights are kept."""
        enabled = bool(enabled)
        if enabled == self._batch_invariant:
            return
        self._batch_invariant = enabled
        for ctx in self._ctx_cache.values():
            ctx.close()
        self._ctx_cache = {}
        if self._native is not None:
            self._native.set_batch_invariant(enabled)

    # ---- reference API --------------------------------------------------------------------------------
    def _canvas(self, samples):
        if isinstance(samples, NestedTensor):
            x = samples.tensors
        elif isinstance(samples, (list, tuple, torch.Tensor)):
            x = nested_tensor_from_tensor_list(samples).tensors
        elif hasattr(samples, "tensors"):
            x = samples.tensors
        else:
            raise TypeError(f"unsupported samples type {type(samples)}")
        assert tuple(x.shape[-2:]) == (MAX_SIZE, MAX_SIZE * 2), f"canvas must be 256x512, got {tuple(x.shape[-2:])}"  # backbone.py:80
        assert x.ndim == 4 and x.shape[1] == 3
        dev = next(self.parameters()).device
        return x.to(device=dev, dtype=torch.float32).contiguous()

    def _queries(self, queries, batch):
        dev = next(self.parameters()).device
        q = queries.to(device=dev, dtype=torch.float32).contiguous()
        assert q.ndim == 3 and q.shape[-1] == 2 and q.shape[0] == batch, f"queries must be (B,Q,2), got {tuple(q.shape)}"
        return q

    @torch.no_grad()
    def forward(self, samples, queries):
        x = self._canvas(samples)
        q = self._queries(queries, x.shape[0])
        return {'pred_corrs': self.native().forward(x, q)}

    # ---- extensions used by cotr_b200.inference ---------------------------------------------------------
    supports_device_preprocess = True

    @torch.no_grad()
    def preprocess_canvases(self, img_from_u8, img_to_u8, rects):
        """Device-side `RefinementTask.get_task` pixels: uint8 HWC CUDA images + (n,6) int32 rectangles
        [x_from, y_from, size_from, x_to, y_to, size_to] -> (n,3,256,512) normalised fp32 canvases, bit-identical to
        the PIL resize + to_tensor + normalize of the reference (cotr_preprocess in include/cotr_b200.h)."""
        assert img_from_u8.dtype == torch.uint8 and img_to_u8.dtype == torch.uint8
        assert img_from_u8.ndim == 3 and img_from_u8.shape[2] == 3 and img_to_u8.ndim == 3 and img_to_u8.shape[2] == 3
        return self.native().preprocess(img_from_u8.contiguous(), img_to_u8.contiguous(), rects)

    @torch.no_grad()
    def dense_postprocess(self, pred):
        """Device-side tail of the dense pass (inference_helper.py:131-145): (n,131072,2) predictions of the canvas grid
        queries -> (n,256,512,3) [x in the other image, y, cycle confidence] (cotr_dense_postprocess)."""
        assert pred.dtype == torch.float32 and pred.ndim == 3 and pred.shape[1] == 256 * 512 and pred.shape[2] == 2
        return self.native().dense_postprocess(pred)

    @torch.no_grad()
    def flow_tile_merge(self, tile, affine, patch, flow, conf, first):
        """Device-side `c @ A + t` -> `float_image_resize` -> `merge_flow_patches` step for one 256x256x3 tile answer
        (inference_helper.py:155-160, :61-75): see cotr_flow_tile_merge in include/cotr_b200.h."""
        self.native().flow_tile_merge(tile, affine, patch, flow, conf, first)

    @torch.no_grad()
    def encode_context(self, samples, reuse=False):
        x = self._canvas(samples)
        nat = self.native()
        if reuse:
            # one cached device K/V buffer per batch size: no cudaMalloc / device-synchronising cudaFree per call.
            # The returned Context is only valid until the next encode_context(reuse=True) of the same batch size.
            native_ctx = self._ctx_cache.get(x.shape[0])
            if native_ctx is None:
                if len(self._ctx_cache) >= 4:
                    for old in self._ctx_cache.values():
                        old.close()
                    self._ctx_cache = {}
                native_ctx = self._ctx_cache[x.shape[0]] = capi.NativeContext(nat, x.shape[0])
        else:
            native_ctx = capi.NativeContext(nat, x.shape[0])
        ctx = Context(native_ctx, x.shape[0])
        nat.encode_context(x, ctx.native)
        return ctx

    @torch.no_grad()
    def decode(self, ctx, queries):
        q = self._queries(queries, ctx.batch)
        return {'pred_corrs': self.native().decode(ctx.native, q)}


def build(args):
    return COTR(args)
