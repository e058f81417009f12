"""Worker of tests/test_batch_invariant_gpu.py::test_config5_job_identical_on_two_gpus (one process per GPU under
torchrun): a small config-5 job (forced queries, FasterSparseEngine with rescue_stranded, cycle-consistency filter) in
batch-invariant mode, once through ShardedCOTR over all ranks and once on rank 0's GPU alone."""
import contextlib
import io
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def job(model):
    from cotr_b200.inference.sparse_engine import FasterSparseEngine
    from cotr_b200.utils.utils import fix_randomness
    from tools.engine_bench import _pair, _queries, forced_cycle_consistency
    img_a, img_b = _pair(512)
    fix_randomness(0)
    eng = FasterSparseEngine(model, 32, mode='tile', rescue_stranded=True)
    with contextlib.redirect_stdout(io.StringIO()):
        return forced_cycle_consistency(eng, img_a, img_b, _queries(300, 512), 100)


def main(out_dir):
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend="nccl", device_id=dev)
    from cotr_b200.inference.sharding import ShardedCOTR
    from tools.engine_bench import _model
    native = _model(dev)
    native.set_batch_invariant(True)
    sharded = job(ShardedCOTR(native))
    dist.barrier()
    if rank == 0:
        single = job(native)
        same = all(np.array_equal(a, b) for a, b in zip(sharded, single)) and sharded[0].shape[0] > 0
        with open(os.path.join(out_dir, "rank0.txt"), "w") as f:
            f.write("identical\n" if same else f"differ: {sharded[0].shape} vs {single[0].shape}\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1])
