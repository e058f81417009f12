"""What the batch-invariant mode costs (COTR.set_batch_invariant, include/cotr_b200.h cotr_set_batch_invariant).

    python tools/invariance_cost.py [--out DIR] [--steps N] [--skip-engine]

Prints JSON lines (and writes them to DIR/invariance_cost.jsonl when --out is given):
  * "forward": default vs invariant forward time for (B, Q) in (1, 1024), (8, 1024), (32, 1), (1, 131 072) - bench.py's
    conventions: CUDA events around each call, graph replay (warmed up), L2 overwritten between steps, median;
  * "decoder_attention": per-launch CUDA-event times of the 6 decoder attention launches at B = 32, Q = 1 (eager, the
    library's per-launch profiler): the default schedule's SIMT kernel vs the tcgen05 kernel with idle lane quarters
    skipped;
  * "engine_config5": engine config 5 (tools/engine_bench.py: FasterSparseEngine with rescue_stranded, forced queries,
    cycle-consistency filter, 1024 x 1024 synthetic pair) in both modes on one GPU, plus the invariant job with every
    model call divided as ShardedCOTR divides it over 2 and 8 ranks, compared with compare_runs.  With several GPUs
    visible the 2-GPU job also runs for real (torchrun, ShardedCOTR, nccl).
The GPU name and power limit are recorded in every line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch
from torch import nn

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

SHAPES = ((1, 1024), (8, 1024), (32, 1), (1, 131072))


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        return "unknown"


class SplitCalls(nn.Module):
    """One-process stand-in for ShardedCOTR over `world` ranks: every model call is split exactly as ShardedCOTR splits
    it (pairs contiguously, or the queries of one large single-context call) and run as `world` separate calls."""

    def __init__(self, model, world):
        super().__init__()
        self.model, self.world = model, world

    @property
    def supports_device_preprocess(self):
        return True

    def preprocess_canvases(self, *a):
        return self.model.preprocess_canvases(*a)

    @torch.no_grad()
    def forward(self, samples, queries):
        from cotr_b200.inference.sharding import MIN_QUERIES_TO_SPLIT, pair_range
        B, Q = int(queries.shape[0]), int(queries.shape[1])
        if B == 1 and Q >= MIN_QUERIES_TO_SPLIT:
            parts = [self.model(samples, queries[:, s:e].contiguous())['pred_corrs']
                     for s, e in (pair_range(Q, r, self.world) for r in range(self.world))]
            return {'pred_corrs': torch.cat(parts, dim=1)}
        parts = [self.model(samples[s:e], queries[s:e])['pred_corrs']
                 for s, e in (pair_range(B, r, self.world) for r in range(self.world)) if e > s]
        return {'pred_corrs': torch.cat(parts, dim=0)}

    def __getattr__(self, name):
        try:
            return super().__getattr__(name)
        except AttributeError:
            return getattr(super().__getattr__('model'), name)


def _models(device):
    from tools.engine_bench import _model
    default, inv = _model(device), _model(device)
    inv.set_batch_invariant(True)
    return default, inv


def time_forward(models, steps):
    from cotr_b200.utils import synthetic as fixtures
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")      # > the 126 MB L2
    out = []
    for B, Q in SHAPES:
        img, q = fixtures.make_inputs(1, B, Q)
        img, q = torch.from_numpy(img).cuda(), torch.from_numpy(q).cuda()
        n = max(4, steps // 4) if Q > 32768 else steps
        res, preds = {}, {}
        for name, m in models.items():
            for _ in range(4):                                # eager, capture, replays
                m(img, q)
            torch.cuda.synchronize()
        times = {name: [] for name in models}
        for _ in range(n):                                    # alternate the modes step by step
            for name, m in models.items():
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                preds[name] = m(img, q)["pred_corrs"]
                b.record()
                torch.cuda.synchronize()
                times[name].append(a.elapsed_time(b))
        for name in models:
            res[name] = {"median_ms": statistics.median(times[name]), "min_ms": min(times[name]),
                         "launches": models[name].native().last_launch_count()}
        res["invariant_over_default"] = res["invariant"]["median_ms"] / res["default"]["median_ms"]
        res["max_abs_diff_between_modes"] = float((preds["default"] - preds["invariant"]).abs().max().item())
        out.append({"B": B, "Q": Q, "steps": n, **res})
    return out


def decoder_attention(models, reps=20):
    from cotr_b200.utils import synthetic as fixtures
    img, q = fixtures.make_inputs(2, 32, 1)
    img, q = torch.from_numpy(img).cuda(), torch.from_numpy(q).cuda()
    res = {}
    for name, m in models.items():
        nat = m.native()
        m(img, q)
        per, kernels = [], set()
        for _ in range(reps):
            nat.profile_begin(512)
            m(img, q)
            recs = nat.profile_end()
            dec = [r for r in recs if r[0].startswith("attention") and r[1] == 32]
            kernels.update(r[0] for r in dec)
            per.extend(r[4] * 1e3 for r in dec)
        res[name] = {"kernel": sorted(kernels), "launches_per_forward": len(per) // reps,
                     "median_us_per_launch": statistics.median(per), "min_us_per_launch": min(per)}
    return res


def engine_config5(models):
    from cotr_b200.inference.sparse_engine import FasterSparseEngine
    from cotr_b200.utils.utils import fix_randomness
    from tools.engine_bench import _pair, _queries, _quiet, compare_runs, forced_cycle_consistency
    img_a, img_b = _pair()
    n_corr = 2048
    queries = _queries(int(n_corr / 0.3))

    def job(model):
        fix_randomness(0)
        eng = FasterSparseEngine(model, 32, mode='tile', rescue_stranded=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        corrs, _ = _quiet(lambda: forced_cycle_consistency(eng, img_a, img_b, queries, n_corr))
        torch.cuda.synchronize()
        return corrs, time.perf_counter() - t0

    fix_randomness(0)                                         # warm-up: graphs, workspace, tables
    for m in models.values():
        _quiet(lambda: FasterSparseEngine(m, 32, mode='tile').cotr_corr_multiscale(img_a, img_b, np.linspace(0.5, 0.0625, 4), 1,
                                                                                    max_corrs=64, queries_a=queries[:64].copy(), force=True))
    res = {}
    base = {}
    for name, m in models.items():
        corrs, dt = job(m)
        base[name] = corrs
        res[name] = {"n_ranks": 1, "seconds": dt, "correspondences": int(corrs.shape[0])}
    res["invariant_over_default"] = res["invariant"]["seconds"] / res["default"]["seconds"]
    for world in (2, 8):
        corrs, dt = job(SplitCalls(models["invariant"], world))
        res[f"invariant_calls_split_{world}_ways_one_gpu"] = {"seconds": dt, "vs_unsplit": compare_runs(base["invariant"], corrs)}
        corrs, dt = job(SplitCalls(models["default"], world))
        res[f"default_calls_split_{world}_ways_one_gpu"] = {"seconds": dt, "vs_unsplit": compare_runs(base["default"], corrs)}
    return res, base["invariant"]


def engine_multi_gpu(out_dir, single):
    """The invariant config-5 job on 2 GPUs for real: torchrun, ShardedCOTR, nccl."""
    if torch.cuda.device_count() < 2:
        return {"skipped": f"{torch.cuda.device_count()} GPU visible"}
    np.save(os.path.join(out_dir, "single.npy"), single)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29545", os.path.abspath(__file__), "--rank-job", out_dir]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, cwd=REPO)
    if r.returncode != 0:
        return {"failed": r.stderr[-2000:]}
    return json.load(open(os.path.join(out_dir, "ranks2.json")))


def rank_job(out_dir):
    import torch.distributed as dist
    from cotr_b200.inference.sharding import ShardedCOTR
    from cotr_b200.inference.sparse_engine import FasterSparseEngine
    from cotr_b200.utils.utils import fix_randomness
    from tools.engine_bench import _model, _pair, _queries, _quiet, compare_runs, forced_cycle_consistency
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group(backend="nccl", device_id=dev)
    native = _model(dev)
    native.set_batch_invariant(True)
    model = ShardedCOTR(native)
    img_a, img_b = _pair()
    queries = _queries(int(2048 / 0.3))
    times = []
    for _ in range(2):                                        # the first run warms up
        fix_randomness(0)
        eng = FasterSparseEngine(model, 32, mode='tile', rescue_stranded=True)
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        corrs, _ = _quiet(lambda: forced_cycle_consistency(eng, img_a, img_b, queries, 2048))
        torch.cuda.synchronize()
        dist.barrier()
        times.append(time.perf_counter() - t0)
    if rank == 0:
        single = np.load(os.path.join(out_dir, "single.npy"))
        json.dump({"n_ranks": 2, "seconds": times[-1], "vs_single_gpu": compare_runs(single, corrs)},
                  open(os.path.join(out_dir, "ranks2.json"), "w"))
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--skip-engine", action="store_true")
    ap.add_argument("--rank-job", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.rank_job:
        return rank_job(a.rank_job)
    assert torch.cuda.is_available(), "tools/invariance_cost.py measures on the GPU"
    gpu = gpu_info()
    out_dir = a.out or os.path.join(os.environ.get("TMPDIR", "/tmp"), "invariance_cost")
    os.makedirs(out_dir, exist_ok=True)
    default, inv = _models(torch.device("cuda", 0))
    models = {"default": default, "invariant": inv}
    lines = [{"what": "forward", "gpu": gpu, "shapes": time_forward(models, a.steps)},
             {"what": "decoder_attention", "gpu": gpu, "B": 32, "Q": 1, **decoder_attention(models)}]
    for line in lines:
        print(json.dumps(line), flush=True)
    if not a.skip_engine:
        eng, single = engine_config5(models)
        line = {"what": "engine_config5", "gpu": gpu, **eng, "invariant_2_gpus": engine_multi_gpu(out_dir, single)}
        lines.append(line)
        print(json.dumps(line), flush=True)
    if a.out:
        with open(os.path.join(a.out, "invariance_cost.jsonl"), "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
