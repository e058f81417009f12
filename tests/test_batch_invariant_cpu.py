"""CPU: the batch-invariant mode's Python surface - the flag on COTR, the unchanged parameter schema, and the agreement
check of ShardedCOTR across ranks (world size 2 over gloo)."""
import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from torch import nn


def _args(**kw):
    return SimpleNamespace(**kw)


def test_build_model_reads_the_flag():
    from cotr_b200.models import build_model
    assert build_model(None).batch_invariant is False
    assert build_model(_args()).batch_invariant is False
    assert build_model(_args(batch_invariant=False)).batch_invariant is False
    assert build_model(_args(batch_invariant=True)).batch_invariant is True


def test_state_dict_is_unchanged_by_the_flag():
    from cotr_b200.models import build_model
    plain, inv = build_model(None), build_model(_args(batch_invariant=True))
    a, b = plain.state_dict(), inv.state_dict()
    assert len(a) == 381 and list(a) == list(b)
    assert all(a[k].shape == b[k].shape for k in a)
    assert sum(p.numel() for p in plain.parameters()) == sum(p.numel() for p in inv.parameters())
    assert [n for n, _ in plain.named_buffers()] == [n for n, _ in inv.named_buffers()]
    inv.load_state_dict(a, strict=True)            # strict loading across modes
    plain.load_state_dict(b, strict=True)


def test_toggle_on_cpu_module_raises_only_at_forward():
    from cotr_b200.models import build_model
    m = build_model(None)
    m.set_batch_invariant(True)
    assert m.batch_invariant is True
    m.set_batch_invariant(True)                    # no change: nothing to do
    m.set_batch_invariant(False)
    assert m.batch_invariant is False
    m.set_batch_invariant(1)
    assert m.batch_invariant is True
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 256, 512), torch.zeros(1, 4, 2))


class _Flagged(nn.Module):
    def __init__(self, flag):
        super().__init__()
        self.anchor = nn.Parameter(torch.zeros(1), requires_grad=False)
        if flag is not None:
            self.batch_invariant = flag


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, flags, results):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from cotr_b200.inference.sharding import ShardedCOTR
    try:
        ShardedCOTR(_Flagged(flags[rank]))
        results[rank] = "ok"
    except RuntimeError as e:
        results[rank] = "raised: " + str(e)
    dist.destroy_process_group()


@pytest.mark.parametrize("flags,agree", [((True, True), True), ((False, None), True), ((None, None), True),
                                         ((True, False), False), ((None, True), False)],
                         ids=["both-on", "off-and-absent", "absent", "on-off", "absent-on"])
def test_sharded_cotr_requires_the_ranks_to_agree(flags, agree):
    """A model without the attribute counts as "off"; disagreeing ranks raise on every rank instead of diverging."""
    world = 2
    port = _free_port()
    with mp.Manager() as mgr:
        results = mgr.dict()
        mp.spawn(_worker, args=(world, port, flags, results), nprocs=world, join=True)
        results = dict(results)
    if agree:
        assert results == {0: "ok", 1: "ok"}, results
    else:
        assert all(results[r].startswith("raised") and "batch_invariant" in results[r] for r in range(world)), results
