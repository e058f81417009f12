"""ctypes binding of the C ABI declared in include/cotr_b200.h.

There is deliberately no CPU fallback: if the shared library is missing or no sm_100 GPU is visible the calls raise.
"""
import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcotr_b200.so")

_lib = None


class CotrTensor(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char_p), ("data", ctypes.POINTER(ctypes.c_float)),
                ("ndim", ctypes.c_int32), ("shape", ctypes.c_int64 * 4)]


class TestGemmDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "path", "M", "N", "K", "a_mode", "lda", "H", "W", "C", "OH", "OW", "KH", "KW", "stride", "pad",
        "relu", "add_period", "ld_add", "ldr", "ldc", "a_ln", "res_ln", "emit_part", "reserved")] + [("a_elems", ctypes.c_int64)]


class LaunchRecord(ctypes.Structure):
    _fields_ = [("kernel", ctypes.c_int32), ("M", ctypes.c_int32), ("N", ctypes.c_int32), ("K", ctypes.c_int32),
                ("ms", ctypes.c_float)]


KERNEL_NAMES = ("gemm_tc", "gemm_simt", "attention_tc", "attention_simt", "layernorm", "maxpool", "query_encode", "stem_canvas")

# name -> (restype, argtypes); every symbol include/cotr_b200.h declares
_PROTOTYPES = {
    "cotr_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(CotrTensor), ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "cotr_destroy": (None, [ctypes.c_void_p]),
    "cotr_context_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "cotr_context_destroy": (None, [ctypes.c_void_p]),
    "cotr_encode_context": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_decode": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_forward_host": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "cotr_preprocess": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_dense_postprocess": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_flow_tile_merge": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 6 +
                             [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]),
    "cotr_group_tasks": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_rasterize_triangles": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_exchange_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_size_t, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "cotr_exchange_handle": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_exchange_connect": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "cotr_exchange_connect_local": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]),
    "cotr_exchange_push": (ctypes.c_longlong, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "cotr_exchange_wait": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p, ctypes.POINTER(ctypes.c_size_t), ctypes.c_void_p]),
    "cotr_exchange_status": (ctypes.c_int, [ctypes.c_void_p]),
    "cotr_exchange_destroy": (None, [ctypes.c_void_p]),
    "cotr_set_graph_mode": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "cotr_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "cotr_last_launch_count": (ctypes.c_int, [ctypes.c_void_p]),
    "cotr_profile_begin": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "cotr_profile_end": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(LaunchRecord), ctypes.c_int]),
    "cotr_debug_read": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64]),
    "cotr_set_gemm_path": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "cotr_set_batch_invariant": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "cotr_test_gemm": (ctypes.c_int, [ctypes.POINTER(TestGemmDesc)] + [ctypes.c_void_p] * 9),
    "cotr_test_attention": (ctypes.c_int, [ctypes.c_int] + [ctypes.c_void_p] * 4 + [ctypes.c_int, ctypes.c_int]),
    "cotr_debug_set_variant": (None, [ctypes.c_int]),
    "cotr_debug_set_timestamps": (None, [ctypes.c_void_p]),
    "cotr_last_error": (ctypes.c_char_p, []),
    "cotr_version": (ctypes.c_char_p, []),
}


def lib():
    """The loaded shared library (loads on first use; raises if it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m cotr_b200.build` "
                               "(cotr_b200 has no CPU / PyTorch fallback by design)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (restype, argtypes) in _PROTOTYPES.items():
            try:
                fn = getattr(handle, name)
            except AttributeError:
                if os.environ.get("COTR_B200_ALLOW_OLD_LIB"):       # tools/ab_libs.py: A/B against a build of an older revision
                    continue
                raise
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def last_error():
    return lib().cotr_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed: {last_error()}")


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


class NativeContext:
    """Decoder K/V cache of up to `max_pairs` encoded image pairs (cotr_context)."""

    def __init__(self, model, max_pairs):
        self.model = model
        self.max_pairs = max_pairs
        self.pairs = 0
        h = ctypes.c_void_p()
        check(lib().cotr_context_create(model.handle, int(max_pairs), ctypes.byref(h)), "cotr_context_create")
        self.handle = h

    def close(self):
        # cotr_context_destroy only frees the context's own K/V buffers; it never touches the (possibly already
        # destroyed) model, so it is called unconditionally - skipping it leaked 12.6 MB per pair.
        if self.handle is not None:
            lib().cotr_context_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class NativeModel:
    """Owner of a `cotr_model` handle built from a reference-schema state dict (CPU fp32 tensors / arrays)."""

    def __init__(self, state_dict, device_index):
        if not torch.cuda.is_available():
            raise RuntimeError("cotr_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        names, arrays = [], []
        for k, v in state_dict.items():
            a = v.detach().to("cpu", torch.float32).contiguous().numpy() if isinstance(v, torch.Tensor) else np.ascontiguousarray(v, np.float32)
            if a.ndim > 4:
                continue
            names.append(k.encode())
            arrays.append(a)
        arr = (CotrTensor * len(arrays))()
        for i, (n, a) in enumerate(zip(names, arrays)):
            arr[i].name = n
            arr[i].data = a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
            arr[i].ndim = a.ndim
            for d in range(a.ndim):
                arr[i].shape[d] = a.shape[d]
        h = ctypes.c_void_p()
        self.handle = None
        self.device_index = int(device_index)
        check(lib().cotr_create(self.device_index, arr, len(arrays), ctypes.byref(h)), "cotr_create")
        self.handle = h

    # ---- calls ------------------------------------------------------------------------------------
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device_index).cuda_stream)

    def forward(self, img, queries):
        B, Q = queries.shape[0], queries.shape[1]
        pred = torch.empty((B, Q, 2), dtype=torch.float32, device=img.device)
        check(lib().cotr_forward(self.handle, _ptr(img), _ptr(queries), B, Q, _ptr(pred), self._stream()), "cotr_forward")
        return pred

    def encode_context(self, img, ctx):
        check(lib().cotr_encode_context(self.handle, _ptr(img), img.shape[0], ctx.handle, self._stream()), "cotr_encode_context")
        ctx.pairs = img.shape[0]

    def decode(self, ctx, queries):
        B, Q = queries.shape[0], queries.shape[1]
        pred = torch.empty((B, Q, 2), dtype=torch.float32, device=queries.device)
        check(lib().cotr_decode(self.handle, ctx.handle, _ptr(queries), B, Q, _ptr(pred), self._stream()), "cotr_decode")
        return pred

    def forward_host(self, img_np, queries_np, out_np=None):
        """Host buffers in, host buffer out (H2D + forward + D2H inside the C call)."""
        B, Q = queries_np.shape[0], queries_np.shape[1]
        if out_np is None:
            out_np = np.empty((B, Q, 2), dtype=np.float32)
        check(lib().cotr_forward_host(self.handle, ctypes.c_void_p(img_np.ctypes.data), ctypes.c_void_p(queries_np.ctypes.data),
                                      B, Q, ctypes.c_void_p(out_np.ctypes.data)), "cotr_forward_host")
        return out_np

    def preprocess(self, img_from_dev, img_to_dev, rects):
        """uint8 HWC device images + (n,6) int32 crop rectangles -> (n,3,256,512) fp32 normalised canvases (device)."""
        rects = np.ascontiguousarray(rects, dtype=np.int32)
        n = rects.shape[0]
        canvas = torch.empty((n, 3, 256, 512), dtype=torch.float32, device=img_from_dev.device)
        check(lib().cotr_preprocess(self.handle, _ptr(img_from_dev), img_from_dev.shape[0], img_from_dev.shape[1],
                                    _ptr(img_to_dev), img_to_dev.shape[0], img_to_dev.shape[1],
                                    ctypes.c_void_p(rects.ctypes.data), n, _ptr(canvas), self._stream()), "cotr_preprocess")
        return canvas

    def dense_postprocess(self, pred_dev):
        """(n, 131072, 2) fp32 predictions of the dense grid queries -> (n, 256, 512, 3) [x, y, confidence] (device)."""
        pred_dev = pred_dev.contiguous()
        n = pred_dev.shape[0]
        out = torch.empty((n, 256, 512, 3), dtype=torch.float32, device=pred_dev.device)
        check(lib().cotr_dense_postprocess(self.handle, _ptr(pred_dev), n, _ptr(out), self._stream()), "cotr_dense_postprocess")
        return out

    def flow_tile_merge(self, tile, affine, patch, flow, conf, first):
        """One 256 x 256 x 3 tile answer (a view into dense_postprocess' output) -> affine, Pillow-exact float resize to
        the patch size, confidence merge into the (oh,ow,2) / (oh,ow) device canvases (cotr_flow_tile_merge)."""
        assert tile.is_cuda and tile.dtype == torch.float32 and tile.shape == (256, 256, 3) and tile.stride(2) == 1 and tile.stride(1) == 3
        aff = np.ascontiguousarray(affine, dtype=np.float64).reshape(6)
        check(lib().cotr_flow_tile_merge(self.handle, _ptr(tile), int(tile.stride(0)), ctypes.c_void_p(aff.ctypes.data),
                                         int(patch.x), int(patch.y), int(patch.w), int(patch.h), int(patch.ow), int(patch.oh),
                                         _ptr(flow), _ptr(conf), int(bool(first)), self._stream()), "cotr_flow_tile_merge")

    def set_graph_mode(self, enabled):
        check(lib().cotr_set_graph_mode(self.handle, int(bool(enabled))), "cotr_set_graph_mode")

    def set_gemm_path(self, path):
        check(lib().cotr_set_gemm_path(self.handle, int(path)), "cotr_set_gemm_path")

    def set_batch_invariant(self, enabled):
        """Batch-invariant mode (cotr_set_batch_invariant): the headline schedule for every pair and query."""
        check(lib().cotr_set_batch_invariant(self.handle, int(bool(enabled))), "cotr_set_batch_invariant")

    def last_launch_count(self):
        return lib().cotr_last_launch_count(self.handle)

    def profile_begin(self, max_records=4096):
        check(lib().cotr_profile_begin(self.handle, int(max_records)), "cotr_profile_begin")
        self._prof_max = int(max_records)

    def profile_end(self):
        """-> list of (kernel name, M, N, K, ms) for every launch since profile_begin, in launch order."""
        buf = (LaunchRecord * self._prof_max)()
        rc = lib().cotr_profile_end(self.handle, buf, self._prof_max)
        if rc > 0:
            raise RuntimeError(f"cotr_profile_end failed: {last_error()}")
        n = -rc - 1
        return [(KERNEL_NAMES[buf[i].kernel], buf[i].M, buf[i].N, buf[i].K, buf[i].ms) for i in range(n)]

    def debug_read(self, name, n_elems):
        out = np.empty(int(n_elems), dtype=np.float32)
        n = lib().cotr_debug_read(self.handle, name.encode(), ctypes.c_void_p(out.ctypes.data), int(n_elems))
        if n < 0:
            raise RuntimeError(f"cotr_debug_read({name}) failed")
        return out[:n]

    def close(self):
        if self.handle is not None:
            lib().cotr_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


EXCHANGE_HANDLE_BYTES = 64


class NativeExchange:
    """One rank's end of the peer-memory result exchange (cotr_exchange, include/cotr_b200.h): `push` writes this rank's
    block into every peer's buffer over NVLink, `wait` gathers one step's blocks in rank order.  Connecting is the
    caller's job: `handle()` -> all-gather the 64-byte handles between the processes -> `connect(handles)`; exchanges
    living in one process use `connect_local(all_exchanges)`."""

    def __init__(self, device_index, rank, world, block_bytes, slots=4):
        self.device_index, self.rank, self.world, self.block_bytes, self.slots = int(device_index), int(rank), int(world), int(block_bytes), int(slots)
        h = ctypes.c_void_p()
        check(lib().cotr_exchange_create(self.device_index, self.rank, self.world, self.block_bytes, self.slots, ctypes.byref(h)), "cotr_exchange_create")
        self.handle_ = h

    def handle(self):
        buf = ctypes.create_string_buffer(EXCHANGE_HANDLE_BYTES)
        check(lib().cotr_exchange_handle(self.handle_, buf), "cotr_exchange_handle")
        return buf.raw

    def connect(self, handles):
        """handles: the `handle()` of every rank, in rank order."""
        blob = b"".join(handles)
        assert len(blob) == self.world * EXCHANGE_HANDLE_BYTES
        check(lib().cotr_exchange_connect(self.handle_, ctypes.create_string_buffer(blob, len(blob))), "cotr_exchange_connect")

    def connect_local(self, exchanges):
        arr = (ctypes.c_void_p * self.world)(*[e.handle_ for e in exchanges])
        check(lib().cotr_exchange_connect_local(self.handle_, arr), "cotr_exchange_connect_local")

    def _stream(self, stream):
        s = stream if stream is not None else torch.cuda.current_stream(self.device_index)
        return ctypes.c_void_p(s.cuda_stream)

    def push(self, block, stream=None):
        """block: contiguous CUDA tensor of this rank (at most block_bytes, a multiple of 16 bytes).  Returns the step number."""
        assert block.is_cuda and block.is_contiguous() and block.device.index == self.device_index
        seq = lib().cotr_exchange_push(self.handle_, _ptr(block), block.numel() * block.element_size(), self._stream(stream))
        if seq < 0:
            raise RuntimeError(f"cotr_exchange_push failed: {last_error()}")
        return int(seq)

    def wait(self, seq, out=None, bytes_per_rank=None, stream=None):
        """Enqueue the wait for step `seq`; `out` (contiguous CUDA tensor, or None) receives the blocks in rank order."""
        sizes = None
        if bytes_per_rank is not None:
            sizes = (ctypes.c_size_t * self.world)(*[int(b) for b in bytes_per_rank])
        need = sum(int(b) for b in bytes_per_rank) if bytes_per_rank is not None else self.world * self.block_bytes
        if out is not None:
            assert out.is_cuda and out.is_contiguous() and out.numel() * out.element_size() >= need
        check(lib().cotr_exchange_wait(self.handle_, int(seq), _ptr(out) if out is not None else None, sizes, self._stream(stream)), "cotr_exchange_wait")

    def status(self):
        return int(lib().cotr_exchange_status(self.handle_))

    def close(self):
        if self.handle_:
            lib().cotr_exchange_destroy(self.handle_)
            self.handle_ = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def group_tasks(pts, boxes, batch_size, max_load, device):
    """(n,4) end points + (n,8) pilot boxes (float64 numpy, list order) -> (squad (n,), rank (n,), n_squads): the device
    version of FasterSparseEngine's squad formation (cotr_group_tasks)."""
    n = int(pts.shape[0])
    dev = torch.device(device)
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    p = torch.from_numpy(np.ascontiguousarray(pts, dtype=np.float64)).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(boxes, dtype=np.float64)).to(dev)
    out = torch.empty(2 * n + 1, dtype=torch.int32, device=dev)
    stream = ctypes.c_void_p(torch.cuda.current_stream(idx).cuda_stream)
    check(lib().cotr_group_tasks(idx, _ptr(p), _ptr(b), n, int(batch_size), int(max_load), _ptr(out), ctypes.c_void_p(out.data_ptr() + 4 * n),
                                 ctypes.c_void_p(out.data_ptr() + 8 * n), stream), "cotr_group_tasks")
    host = out.cpu().numpy()
    return host[:n], host[n:2 * n], int(host[2 * n])


def rasterize_triangles(tris, H, W):
    """(n_tri,3,4) fp32 CUDA tensor [x, y, u, v] per vertex -> (H,W,2) fp32 CUDA tensor (cotr_rasterize_triangles)."""
    tris = tris.contiguous()
    assert tris.is_cuda and tris.dtype == torch.float32 and tris.ndim == 3 and tris.shape[1:] == (3, 4)
    out = torch.empty((H, W, 2), dtype=torch.float32, device=tris.device)
    dev = tris.device.index if tris.device.index is not None else torch.cuda.current_device()
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib().cotr_rasterize_triangles(dev, _ptr(tris), tris.shape[0], int(H), int(W), _ptr(out), stream), "cotr_rasterize_triangles")
    return out


def test_gemm(path, A, w_host, *, bias=None, addmat=None, add_period=1, residual=None, relu=False, ln=None,
              a_mode=0, conv=None, M=None, ldc=None, a_ln=False, res_ln=False, part_out=None):
    """Kernel-level hook: out = epilogue(A W^T).  A and optional epilogue operands are CUDA fp32 tensors.
    a_ln / res_ln: `ln` = (gamma, beta) is a DEFERRED LayerNorm of the A rows / of the residual rows (tcgen05 path)."""
    N, K = w_host.shape
    d = TestGemmDesc()
    d.path = path
    d.N, d.K = N, K
    d.a_mode = a_mode
    if a_mode == 0:
        d.M = A.shape[0] if M is None else M
        d.lda = A.stride(0)
    else:
        d.M = M
        for k_, v_ in conv.items():
            setattr(d, k_, v_)
        d.lda = conv.get("C", 0) if a_mode != 3 else A.shape[-1]
    d.a_elems = A.numel()
    d.relu = int(relu)
    d.a_ln = int(a_ln)
    d.res_ln = int(res_ln)
    d.emit_part = int(part_out is not None)
    d.add_period = add_period
    d.ld_add = addmat.stride(0) if addmat is not None else 0
    d.ldr = residual.stride(0) if residual is not None else 0
    d.ldc = N if ldc is None else ldc
    out = torch.zeros((d.M, d.ldc), dtype=torch.float32, device=A.device)
    w_np = np.ascontiguousarray(w_host, np.float32)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None
    check(lib().cotr_test_gemm(ctypes.byref(d), p(A), ctypes.c_void_p(w_np.ctypes.data), p(bias), p(addmat), p(residual),
                               p(ln[0]) if ln else None, p(ln[1]) if ln else None, p(out), p(part_out)), "cotr_test_gemm")
    return out


def test_attention(path, q, k, v, nq, npairs):
    out = torch.zeros_like(q)
    check(lib().cotr_test_attention(path, _ptr(q), _ptr(k), _ptr(v), _ptr(out), nq, npairs), "cotr_test_attention")
    return out
