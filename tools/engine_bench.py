"""Engine-level benchmarks on the GPU: BASELINE.json configs[2] and configs[4].

    python bench.py --config 3 [--gpus N]     # 10 000 forced queries x 4 zoom levels (SparseEngine + FasterSparseEngine)
    python bench.py --config 5 [--gpus N]     # FasterSparseEngine, 2048 correspondences, cycle-consistency filter
    python tools/engine_bench.py [n_queries]  # quick single-GPU comparison of device-side vs host-side crop pixels

`run_config` is what bench.py calls; one "step" is one complete engine run (dense first guess + all zoom levels) on a
synthetic 1024x1024 pair with seeded synthetic weights.  With N > 1 ranks (torchrun) the engines drive
`cotr_b200.inference.sharding.ShardedCOTR`: the scheduler runs replicated, every model call is split over the ranks.
Random weights reject every task in the reference's acceptance tests (SURVEY.md section 8c), so - like the survey's
config-1 probe - the queries are FORCED (`force=True`): every query is followed through all zoom levels.
"""
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

ZOOMS = np.linspace(0.5, 0.0625, 4)        # demo_single_pair.py:37


def _model(device):
    import torch
    from cotr_b200.models import build_model
    from cotr_b200.utils import synthetic as fixtures
    sd = fixtures.make_state_dict(0)
    model = build_model(None)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return model.to(device).eval()


def _pair(size=1024):
    from cotr_b200.utils.synthetic import synthetic_image
    return synthetic_image(51, size, size), synthetic_image(52, size, size)


def _queries(n, size=1024, seed=1):
    rs = np.random.RandomState(seed)
    return np.stack([rs.uniform(10, size - 10, n), rs.uniform(10, size - 10, n)], axis=1)


def _quiet(fn):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn()


def forced_cycle_consistency(engine, img_a, img_b, queries_a, max_corrs):
    """`cotr_corr_multiscale_with_cycle_consistency` (sparse_engine.py:235-264) with forced queries: a -> b for every
    query, b -> a from the answers, keep the max_corrs smallest cycle errors."""
    corr_f, idx_f = engine.cotr_corr_multiscale(img_a, img_b, ZOOMS, 1, max_corrs=queries_a.shape[0], queries_a=queries_a.copy(),
                                                return_idx=True, force=True)
    corr_b, idx_b = engine.cotr_corr_multiscale(img_b, img_a, ZOOMS, 1, max_corrs=corr_f.shape[0], queries_a=corr_f[:, 2:].copy(),
                                                return_idx=True, force=True)
    err = np.linalg.norm(corr_f[idx_b][:, :2] - corr_b[:, 2:], axis=1)
    order = np.argsort(err)
    return corr_f[idx_b][order][:max_corrs], err[order][:max_corrs]


def compare_runs(single, sharded):
    """Two runs of the same job whose model calls were batched differently (1 rank vs N ranks).  In the default mode the
    network's answers agree to ~1e-6 of the image, not bit for bit (the GEMM tile shapes follow the rows per launch), so
    the 2048 survivors of the cycle-error ranking may differ near the cut: report the overlap and the differences on the
    common points.  In batch-invariant mode (COTR.set_batch_invariant) the two runs must be identical."""
    same_order = single.shape == sharded.shape and bool(np.array_equal(single[:, :2], sharded[:, :2]))
    a = {tuple(r[:2]): r[2:] for r in single}
    common = [(a[tuple(r[:2])], r[2:]) for r in sharded if tuple(r[:2]) in a]
    diff = np.array([np.abs(x - y).max() for x, y in common]) if common else np.zeros(0)
    return {"same_source_points": same_order, "common_source_points": len(common), "of": int(sharded.shape[0]),
            "max_abs_diff_px": float(diff.max()) if diff.size else None,
            "median_abs_diff_px": float(np.median(diff)) if diff.size else None}


def run_config(config, rank, local_rank, world, steps=2, cpu_rate=None):
    """One JSON line on rank 0 (same keys as bench.py's headline line where they apply)."""
    import torch
    import torch.distributed as dist
    from cotr_b200.inference.sharding import ShardedCOTR
    from cotr_b200.inference.sparse_engine import FasterSparseEngine, SparseEngine
    from cotr_b200.utils.utils import fix_randomness
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    native = _model(dev)
    model = ShardedCOTR(native) if world > 1 else native
    img_a, img_b = _pair()
    runs = {}

    def timed(fn):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = _quiet(fn)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return out, float(dt.item())

    if config == 3:
        n_q = 10000
        queries = _queries(n_q)
        workload = "configs[2]: dense cotr_flow first guess + 10 000 forced queries through 4 zoom levels, 1024x1024 synthetic pair"
        cases = (("SparseEngine", lambda: SparseEngine(model, 32, mode='tile')),
                 ("FasterSparseEngine", lambda: FasterSparseEngine(model, 32, mode='tile')),
                 ("FasterSparseEngine+rescue_stranded", lambda: FasterSparseEngine(model, 32, mode='tile', rescue_stranded=True)))
        fix_randomness(0)                       # warm-up: graphs, workspace, resampling tables
        _quiet(lambda: SparseEngine(model, 32, mode='tile').cotr_corr_multiscale(img_a, img_b, ZOOMS, 1, max_corrs=64, queries_a=queries[:64].copy(), force=True))
        for name, make in cases:
            times, n_out, contexts = [], 0, 0
            for _ in range(steps if name == "SparseEngine" else max(steps, 2)):
                fix_randomness(0)
                eng = make()
                corrs, dt = timed(lambda: eng.cotr_corr_multiscale(img_a, img_b, ZOOMS, 1, max_corrs=n_q, queries_a=queries.copy(), force=True))
                times.append(dt); n_out = int(corrs.shape[0]); contexts = int(eng.total_tasks)
            runs[name] = {"seconds": float(np.median(times)), "correspondences": n_out, "contexts_encoded": contexts,
                          "query_points_per_s": n_out / float(np.median(times)), "query_steps_per_s": n_q * 4 / float(np.median(times))}
        head = runs["SparseEngine"]
        value, n_points = head["query_points_per_s"], head["correspondences"]
        metric = "query-points/sec (10 000 queries x 4 zoom levels + dense first guess, 1024x1024 pair)"
    else:
        n_corr = 2048
        n_q = int(n_corr / 0.3)                 # EXTRACTION_RATE of sparse_engine.py:237
        queries = _queries(n_q)
        workload = ("configs[4]: FasterSparseEngine, 2048 correspondences after the cycle-consistency filter "
                    f"({n_q} forced queries a->b, back b->a, 4 zoom levels each), contexts sharded over the ranks")
        fix_randomness(0)
        _quiet(lambda: FasterSparseEngine(model, 32, mode='tile').cotr_corr_multiscale(img_a, img_b, ZOOMS, 1, max_corrs=64, queries_a=queries[:64].copy(), force=True))
        times, result = [], None
        for _ in range(max(steps, 2)):
            fix_randomness(0)
            eng = FasterSparseEngine(model, 32, mode='tile', rescue_stranded=True)
            (corrs, err), dt = timed(lambda: forced_cycle_consistency(eng, img_a, img_b, queries, n_corr))
            times.append(dt); result = (corrs, err, int(eng.total_tasks))
        corrs, err, contexts = result
        runs["FasterSparseEngine+cycle"] = {"seconds": float(np.median(times)), "correspondences": int(corrs.shape[0]),
                                            "contexts_encoded_single_query_phase": contexts, "median_cycle_error_px": float(np.median(err)),
                                            "query_points_per_s": corrs.shape[0] / float(np.median(times))}
        if world > 1:
            # the same job on rank 0's GPU alone: identical scheduler, so the correspondences should agree to a pixel fraction
            fix_randomness(0)
            eng1 = FasterSparseEngine(native, 32, mode='tile', rescue_stranded=True)
            single = _quiet(lambda: forced_cycle_consistency(eng1, img_a, img_b, queries, n_corr))[0] if rank == 0 else None
            if rank == 0:
                runs["vs_single_gpu"] = compare_runs(single, corrs)
            dist.barrier()
        value, n_points = runs["FasterSparseEngine+cycle"]["query_points_per_s"], int(corrs.shape[0])
        metric = "query-points/sec (FasterSparseEngine, 2048 cycle-consistent correspondences, 1024x1024 pair)"
    if rank != 0:
        return
    line = {"metric": metric, "value": value, "unit": "query-points/s", "n_gpus": world, "steps": steps,
            "ms_per_step": 1e3 * n_points / value, "higher_is_better": True, "scaling": "strong",
            "dtype": "f32 (fp16 hi/lo split operands, fp32 accumulate on tcgen05)", "data": "synthetic",
            "config": {"workload": workload, "zoom_ins": [float(z) for z in ZOOMS], "batch_size": 32,
                       "parallelism": f"{world} rank(s), SPMD scheduler, contexts split contiguously per model call"},
            "engines": runs, "timing": "wall clock around the whole engine run (host scheduler included), max over ranks, median of the runs"}
    if cpu_rate is not None:
        line["cpu_baseline"] = cpu_rate
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    import torch
    from cotr_b200.inference.sparse_engine import FasterSparseEngine, SparseEngine
    from cotr_b200.utils.utils import fix_randomness
    n_queries = int(sys.argv[1]) if len(sys.argv) > 1 else 512
    model = _model(torch.device("cuda", 0))
    img_a, img_b = _pair()
    queries = _queries(n_queries)

    def run(engine_cls, on_device, **kw):
        fix_randomness(0)
        eng = engine_cls(model, 32, mode='tile', device_preprocess=on_device, **kw)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        corrs = _quiet(lambda: eng.cotr_corr_multiscale(img_a, img_b, ZOOMS, 1, max_corrs=n_queries, queries_a=queries.copy(), force=True))
        torch.cuda.synchronize()
        return corrs, time.perf_counter() - t0

    run(SparseEngine, True)       # warm-up: graphs, workspace, coefficient tables
    for cls, kw in ((SparseEngine, {}), (FasterSparseEngine, {})):
        base = None
        for on_device in (True, False):
            corrs, dt = run(cls, on_device, **kw)
            tag = "device pixels" if on_device else "host PIL pixels"
            same = "" if base is None else f"  identical to device path: {np.array_equal(base, corrs)}"
            base = corrs if base is None else base
            print(f"{cls.__name__:18s} {tag:16s}: {len(corrs)} correspondences from {n_queries} queries x 4 zoom levels in {dt:.2f} s "
                  f"({n_queries * 4 / dt:.0f} query-steps/s){same}", flush=True)
