"""Multi-GPU data parallelism over independent image pairs / contexts (SURVEY.md section 8e).

One process per GPU (torchrun).  Pairs (and the zoom-in engines' contexts) are independent, so the only exchange is
the gather of the (B,Q,2) fp32 predictions - 8 KB per 1024 queries.  Works with the `nccl` backend on CUDA tensors and
with `gloo` on CPU tensors (used by the CPU tests); the pipelined gather of `AsyncGather` uses this library's own
peer-memory exchange over NVLink when the ranks share a node.

Two entry points:
  * `forward_sharded(model, img, queries)`: BASELINE.json configs[3] - one batch of independent pairs, each rank runs
    its contiguous block, everybody receives all predictions;
  * `ShardedCOTR(model)`: a drop-in for the model object the engines drive (`SparseEngine(ShardedCOTR(model), ...)`,
    BASELINE.json configs[4], reference call site demo_reconstruction.py:44-49).  The host scheduler runs replicated
    (SPMD): every rank executes the same engine code with the same seeds, every model call is split over the ranks
    (contexts contiguously; the single-context dense pass of cotr_flow over its 131 072 queries) and all-gathered, so
    every rank sees identical predictions and takes identical decisions.  Task state therefore needs no broadcast,
    and rank 0's return value is the job's result.  That holds bit for bit only if a rank's predictions for a pair or a
    query do not depend on which other pairs / queries share its call: with the wrapped model in batch-invariant mode
    (`COTR.batch_invariant`) the job's result is the same on any number of ranks.  The ranks must agree on the mode,
    which `ShardedCOTR` checks when it is constructed.
"""
import numpy as np
import torch
import torch.distributed as dist
from torch import nn

MIN_QUERIES_TO_SPLIT = 4096      # below this a single context is not worth splitting over its queries


def pair_range(n_pairs, rank, world):
    """Contiguous block of pairs owned by `rank` (sizes differ by at most one)."""
    base, extra = divmod(n_pairs, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def _active(group=None):
    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


def _gather_blocks(local, total, dim, group=None):
    """All-gather per-rank blocks of `total` items split contiguously (pair_range) along `dim`, in order."""
    if not _active(group):
        return local
    world = dist.get_world_size(group)
    counts = [pair_range(total, r, world) for r in range(world)]
    widest = max(e - s for s, e in counts)
    local = local.movedim(dim, 0).contiguous()
    padded = local.new_zeros((widest,) + tuple(local.shape[1:]))
    padded[: local.shape[0]] = local
    out = local.new_empty((world * widest,) + tuple(local.shape[1:]))
    dist.all_gather_into_tensor(out, padded, group=group)
    parts = [out[r * widest: r * widest + (e - s)] for r, (s, e) in enumerate(counts)]
    return torch.cat(parts, dim=0).movedim(0, dim).contiguous()


def gather_predictions(local_pred, n_pairs, group=None):
    """All-gather per-rank (b_r,Q,2) predictions into the full (n_pairs,Q,2) tensor on every rank, in pair order."""
    return _gather_blocks(local_pred, n_pairs, 0, group)


def forward_sharded(model, img, queries, group=None):
    """BASELINE.json configs[3]: every rank holds the full (B,3,256,512) / (B,Q,2) batch description, runs its own
    block of pairs through `model` and receives everybody's predictions."""
    if not _active(group):
        return model(img, queries)['pred_corrs']
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    s, e = pair_range(img.shape[0], rank, world)
    if e > s:
        local = model(img[s:e], queries[s:e])['pred_corrs']
    else:
        local = queries.new_zeros((0, queries.shape[1], 2))
    return gather_predictions(local, img.shape[0], group)


def open_exchange(block_bytes, device, group=None, slots=4):
    """This rank's end of a peer-memory result exchange (`cotr_exchange`, csrc/peer_exchange.cu) connected to all ranks
    of `group`, or None when the ranks cannot map each other's device memory (different nodes, no peer access, block size
    not a multiple of 16 bytes).  Collective: every rank calls it, and all ranks get the same kind of answer."""
    import socket
    from cotr_b200 import capi
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    ex, handle, ok = None, b"\0" * capi.EXCHANGE_HANDLE_BYTES, int(block_bytes % 16 == 0 and device.type == "cuda")
    if ok:
        try:
            ex = capi.NativeExchange(device.index if device.index is not None else torch.cuda.current_device(), rank, world, block_bytes, slots)
            handle = ex.handle()
        except (RuntimeError, OSError, AttributeError):
            ok = 0
    infos = [None] * world
    dist.all_gather_object(infos, (socket.gethostname(), handle, ok), group=group)
    if ok and len({host for host, _, _ in infos}) == 1 and all(o for _, _, o in infos):
        try:
            ex.connect([h for _, h, _ in infos])
        except RuntimeError:
            ok = 0
    else:
        ok = 0
    agreed = torch.tensor([ok], dtype=torch.int32, device=device)
    dist.all_reduce(agreed, op=dist.ReduceOp.MIN, group=group)        # also: nobody pushes before everybody has mapped
    if int(agreed.item()) == 0:
        if ex is not None:
            ex.close()
        return None
    return ex


class AsyncGather:
    """The result gather of a stream of independent steps, kept off the compute stream's critical path.

    `submit(pred)` hands this rank's (b,Q,2) block to a side stream that waits (CUDA event) for the kernels that produce
    `pred`; the compute stream continues with the next step at once.  `wait()` joins the side stream into the current
    stream and returns the most recent gathered tensor.  Two transports:
      * "peer" (default on one node): `cotr_exchange` - the side stream runs this library's push kernel, which stores the
        block into every peer's symmetric buffer over NVLink and never waits for anybody; only `wait()` polls for the
        other ranks' blocks of that step.  Steps that are never waited for are simply overwritten `slots` steps later;
      * "nccl": `all_gather_into_tensor` on the side stream into alternating buffers (every rank's collective kernel
        waits for every other rank, step by step) - the fallback across nodes.
    Calls are issued in the same order on every rank."""

    def __init__(self, block_shape, device, group=None, backend="auto", slots=4):
        assert backend in ("auto", "peer", "nccl")
        self.group = group
        self.world = dist.get_world_size(group) if _active(group) else 1
        self.side = torch.cuda.Stream(device=device) if self.world > 1 else None
        self.block_shape = tuple(block_shape)
        self.bufs = [torch.empty((self.world * block_shape[0],) + tuple(block_shape[1:]), dtype=torch.float32, device=device) for _ in range(2)]
        self.turn = 0
        self.last = None
        self.seq = 0
        self.exchange = None
        if self.world > 1 and backend != "nccl":
            block_bytes = 4 * int(np.prod(block_shape))
            self.exchange = open_exchange(block_bytes, torch.device(device), group, slots)
            if self.exchange is None and backend == "peer":
                raise RuntimeError("AsyncGather(backend='peer'): the ranks cannot map each other's device memory")
        self.backend = "local" if self.world == 1 else ("peer" if self.exchange is not None else "nccl")

    def submit(self, pred):
        if self.world == 1:
            self.last = pred
            return
        pred = pred.contiguous()
        ready = torch.cuda.Event()
        ready.record()                                   # after the kernels of this step on the compute stream
        pred.record_stream(self.side)
        if self.exchange is not None:
            assert tuple(pred.shape) == self.block_shape and pred.dtype == torch.float32
            self.side.wait_event(ready)
            self.seq = self.exchange.push(pred, stream=self.side)
            self.last = None
            return
        out = self.bufs[self.turn]
        self.turn ^= 1
        with torch.cuda.stream(self.side):
            self.side.wait_event(ready)
            dist.all_gather_into_tensor(out, pred, group=self.group)
        self.last = out

    def wait(self):
        if self.exchange is not None and self.last is None and self.seq > 0:
            out = self.bufs[self.turn]
            self.turn ^= 1
            self.exchange.wait(self.seq, out=out, stream=self.side)
            self.last = out
        if self.side is not None:
            torch.cuda.current_stream().wait_stream(self.side)
        return self.last

    def check(self):
        """Host-synchronising health check of the peer transport (0 = fine); raises on a missed or overwritten step."""
        if self.exchange is None:
            return 0
        self.side.synchronize()
        status = self.exchange.status()
        if status != 0:
            raise RuntimeError("peer result exchange: " + ("a rank never published the step" if status == 1 else "a waited step was overwritten"))
        return 0

    def close(self):
        """Collective: no rank may free its buffer while another one can still push into it."""
        if self.exchange is not None:
            torch.cuda.synchronize()
            dist.barrier(group=self.group)
            self.exchange.close()
            self.exchange = None


class LazyCanvases:
    """What `ShardedCOTR.preprocess_canvases` returns: the recipe of n network canvases (two uint8 device images and
    n crop rectangles), materialised per rank for its own block only when the forward is issued."""

    def __init__(self, img_from, img_to, rects):
        self.img_from, self.img_to = img_from, img_to
        self.rects = np.ascontiguousarray(rects, dtype=np.int32)
        self.shape = (self.rects.shape[0], 3, 256, 512)

    def to(self, *a, **k):
        return self

    def __len__(self):
        return self.shape[0]


class ShardedCOTR(nn.Module):
    """The model object of the engines, with every call split over the ranks of `group` (see the module docstring)."""

    def __init__(self, model, group=None):
        super().__init__()
        self.model = model
        self.group = group
        if _active(group):
            # collective: a rank whose model runs another schedule would make other decisions and silently diverge
            mine = bool(getattr(model, 'batch_invariant', False))
            modes = [None] * dist.get_world_size(group)
            dist.all_gather_object(modes, mine, group=group)
            if len(set(modes)) != 1:
                raise RuntimeError(f"ShardedCOTR: the ranks' models disagree on batch_invariant (by rank: {modes}); "
                                   "set the same mode on every rank")

    @property
    def supports_device_preprocess(self):
        return getattr(self.model, 'supports_device_preprocess', False)

    def preprocess_canvases(self, img_from_u8, img_to_u8, rects):
        if not _active(self.group):
            return self.model.preprocess_canvases(img_from_u8, img_to_u8, rects)
        return LazyCanvases(img_from_u8, img_to_u8, rects)

    def _local_canvases(self, samples, s, e):
        if isinstance(samples, LazyCanvases):
            return self.model.preprocess_canvases(samples.img_from, samples.img_to, samples.rects[s:e])
        return samples[s:e]

    @torch.no_grad()
    def forward(self, samples, queries):
        if not _active(self.group):
            if isinstance(samples, LazyCanvases):
                samples = self._local_canvases(samples, 0, samples.shape[0])
            return self.model(samples, queries)
        rank, world = dist.get_rank(self.group), dist.get_world_size(self.group)
        B, Q = int(queries.shape[0]), int(queries.shape[1])
        if B == 1 and Q >= MIN_QUERIES_TO_SPLIT and not isinstance(samples, LazyCanvases):
            # one context, many queries (cotr_flow's dense pass): every rank encodes the (cheap) context itself and
            # decodes its slice of the queries - no broadcast of the 6 MB K/V cache
            s, e = pair_range(Q, rank, world)
            local = self.model(samples, queries[:, s:e].contiguous())['pred_corrs']
            return {'pred_corrs': _gather_blocks(local, Q, 1, self.group)}
        s, e = pair_range(B, rank, world)
        if e > s:
            local = self.model(self._local_canvases(samples, s, e), queries[s:e])['pred_corrs']
        else:
            dev = next(self.model.parameters()).device
            local = torch.zeros((0, Q, 2), dtype=torch.float32, device=dev)
        return {'pred_corrs': gather_predictions(local, B, self.group)}

    # The remaining extensions of cotr_b200.models.COTR (dense_postprocess, encode_context, decode) run replicated:
    # identical on every rank, no exchange.  They exist on the wrapper exactly when the wrapped model has them.
    def __getattr__(self, name):
        try:
            return super().__getattr__(name)
        except AttributeError:
            return getattr(super().__getattr__('model'), name)
