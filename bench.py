"""Benchmark of the COTR correspondence hot path on B200 (contract: see the task statement / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1], the one `metric` is quoted on): per GPU one synthetic 256x256 image pair laid side
by side (1,3,256,512) and 1024 random queries, no zoom; a "step" is one pass of the hot path over that batch
(COTR.forward: backbone -> input_proj -> encoder -> decoder -> head).  Weak scaling: every rank processes its own pair
(independent pairs shard with no data-path collective); for N > 1 every step hands its (1,1024,2) result to the result
exchange on a side stream (the path's only exchange: this library's peer-memory push over NVLink, cotr_exchange; NCCL
all-gather when the ranks cannot map each other's memory).

One JSON line on rank 0:
  value      query-points/s, whole job, inputs resident in HBM, CUDA-event timed per step, L2 flushed between steps
  e2e        same metric end to end from pinned HOST buffers: N = 1 through the C-ABI host-buffer call
             (cotr_forward_host: H2D + forward + D2H inside); N > 1 through the Python API with the result exchange
             (push, wait for all ranks) and the D2H read of the gathered (N,1024,2) block inside the timed region
  result_exchange  (N > 1) transport used, the last step's gathered block checked against a plain NCCL all-gather, and
             the per-rank step times with and without the exchange (what, if anything, the exchange costs the step)
  roofline   dominant kernel family of the step: its share of the kernel time comes from a per-launch CUDA-event pass
             (library profiler, eager), its time from share x the TIMED graph-replayed step - so kernel_ms_per_step
             can never exceed ms_per_step; `whole_step` = algorithmic FLOP / timed step
  config4    BASELINE.json configs[3] per GPU (8 pairs x 1024 queries in one forward), device-timed, whole-step roofline
  cpu_baseline  the oracle port (CPU restatement of the reference, oracle/cotr_oracle.py) on the host cores, rank 0, N=1
`--impl reference` times that CPU path alone (all host threads) and prints the same line shape with "impl": "reference".
`--config 3` / `--config 5` time the zoom-in engines instead (see DESIGN.md section 6).
`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (float32): `pred_corrs`
(1,1024,2) of rank 0, and for N > 1 `pred_corrs_gathered` (N,1024,2), the block the result exchange delivered.  Weights
and inputs are seeded, so runs with the same arguments see the same inputs and two builds can be compared output for
output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

N_QUERIES = 1024
METRIC = "query-points/sec (256x256 pair, 1024 queries)"
UNIT = "query-points/s"
WORKLOAD = "configs[1]: single 256x256 synthetic pair, 1024 random queries, no zoom (per GPU)"
CTX_FLOP = 24.641536e9          # per pair (BASELINE.md section 3)
QUERY_FLOP = 11273216.0         # per query


def algorithmic_flop(pairs, queries):
    return pairs * (CTX_FLOP + queries * QUERY_FLOP)


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_tflops": float(p["bf16_tflops"]), "hbm_gbs": float(p["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json, burst)"}
    return {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def samples(self):
        return len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
    """CPU threads this process may really use: min(os.cpu_count, sched affinity, cgroup cpu quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, quota // period))
            break
        except Exception:
            continue
    return max(1, n)


def config_dict(world):
    """The `config` object of the JSON line - the SAME object in the native and in the reference arm."""
    return {"workload": WORKLOAD, "pairs_per_gpu": 1, "queries_per_pair": N_QUERIES,
            "parallelism": f"dp{world} (independent pairs)",
            "l2": "GPU arm: flushed between timed steps by writing a 256 MiB buffer; CPU arm: not applicable",
            "weights": "seeded synthetic (cotr_b200/utils/synthetic.py seed 0)",
            "result_gather": "GPU arm, N > 1: every step hands its (1,1024,2) block to the result exchange on a side stream "
                             "(cotr_b200.inference.sharding.AsyncGather: peer-memory push over NVLink on one node, NCCL all_gather "
                             "otherwise; overlaps the next step, joined before the closing barrier; the synchronous push + wait is "
                             "inside `e2e`; the transport used is reported in `result_exchange`); CPU arm (rank 0 runs one pair per "
                             "step on the host cores): none"}


def committed_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture of this round (profiles/r02_traffic.json, written by tools/ncu_summary.py)."""
    path = os.path.join(REPO, "profiles", "r02_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        return float(t["gemm_tc"]["dram_bytes_per_launch"]), t.get("source", path)
    except Exception:
        return None, "no committed ncu --set full capture for this build"


def cpu_reference_rate(budget_s, warmup=1, max_iters=30):
    """The oracle port (validated bit-exact against the reference on CPU) on all host threads, same workload."""
    import torch
    from oracle import cotr_oracle, fixtures
    torch.set_num_threads(host_threads())
    sd = cotr_oracle.cast_state_dict(fixtures.make_state_dict(0), torch.float32)
    img, queries = fixtures.make_inputs(1, 1, N_QUERIES)
    for _ in range(warmup):
        cotr_oracle.forward(sd, img, queries, torch.float32)
    times = []
    t_start = time.perf_counter()
    while len(times) < max_iters and (time.perf_counter() - t_start < budget_s or len(times) < 3):
        t0 = time.perf_counter()
        cotr_oracle.forward(sd, img, queries, torch.float32)
        times.append(time.perf_counter() - t0)
    med = float(np.median(times))
    return {"value": N_QUERIES / med, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{len(times)} forwards of the same workload (1 pair, 1024 queries), median {med * 1e3:.1f} ms, "
                      f"fp32 eager torch {torch.__version__} on {torch.get_num_threads()} threads (os.cpu_count {os.cpu_count()})"}


def cpu_engine_rate(n_queries_full, n_sample=16):
    """CPU baseline of the engine configs: the oracle port driving the same SparseEngine on a BOUNDED sample (one dense
    first-guess pass + n_sample forced queries x 4 zoom levels), extrapolated to the full query count."""
    import contextlib
    import io
    import torch
    from torch import nn
    from oracle import cotr_oracle, fixtures
    from cotr_b200.inference.sparse_engine import SparseEngine
    from cotr_b200.utils.utils import fix_randomness
    from tools import engine_bench
    torch.set_num_threads(host_threads())

    class OracleCOTR(nn.Module):
        def __init__(self):
            super().__init__()
            self.anchor = nn.Parameter(torch.zeros(1), requires_grad=False)
            self.sd = cotr_oracle.cast_state_dict(fixtures.make_state_dict(0), torch.float32)
            self.seconds = []

        @torch.no_grad()
        def forward(self, img, queries):
            t0 = time.perf_counter()
            out = cotr_oracle.forward(self.sd, img, queries, torch.float32)
            self.seconds.append((int(queries.shape[0]) * int(queries.shape[1]), time.perf_counter() - t0))
            return {'pred_corrs': out}

    model = OracleCOTR()
    img_a, img_b = engine_bench._pair()
    q = engine_bench._queries(n_sample)
    fix_randomness(0)
    t0 = time.perf_counter()
    with contextlib.redirect_stdout(io.StringIO()):
        SparseEngine(model, n_sample, mode='tile').cotr_corr_multiscale(img_a, img_b, engine_bench.ZOOMS, 1, max_corrs=n_sample,
                                                                         queries_a=q.copy(), force=True)
    total = time.perf_counter() - t0
    dense = sum(t for n, t in model.seconds if n > 100000)
    per_step = (total - dense) / (n_sample * 4)
    full = dense + per_step * n_queries_full * 4
    return {"value": n_queries_full / full, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"oracle port under the same SparseEngine: 1 dense pass ({dense:.1f} s) + {n_sample} forced queries x 4 zoom levels "
                      f"({per_step * 1e3:.0f} ms per query-step incl. host PIL work), extrapolated to {n_queries_full} queries "
                      f"({full:.0f} s); {total:.1f} s of CPU work measured"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port), rank 0 only."""
    if rank != 0:
        return
    steps = []
    base = None
    import torch
    from oracle import cotr_oracle, fixtures
    torch.set_num_threads(host_threads())
    sd = cotr_oracle.cast_state_dict(fixtures.make_state_dict(0), torch.float32)
    img, queries = fixtures.make_inputs(1, 1, N_QUERIES)
    for _ in range(max(args.warmup, 1)):
        cotr_oracle.forward(sd, img, queries, torch.float32)
    for _ in range(args.steps):
        t0 = time.perf_counter()
        pred = cotr_oracle.forward(sd, img, queries, torch.float32)
        steps.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pred_corrs": pred})
    # the host is shared and noisy (round 1: 8.3-9.9 k q/s across records): the median step is the robust figure
    ms = float(np.median(steps)) * 1e3
    value = N_QUERIES / (ms * 1e-3)
    base = {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{args.steps} forwards of 1 pair x 1024 queries per step (the whole workload of one GPU), median step "
                      f"(mean {float(np.mean(steps)) * 1e3:.1f} ms, min {float(np.min(steps)) * 1e3:.1f} ms), fp32 eager torch on "
                      f"{torch.get_num_threads()} threads (os.cpu_count {os.cpu_count()})"}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": base, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array (torch tensor or numpy) as out_dir/<name>.npy in float32."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if not isinstance(a, np.ndarray):
            a = a.detach().cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def _timed_steps(step, flush, n, barrier):
    """n steps, each bracketed by CUDA events on the launching stream, L2 flushed before each; mean ms per step."""
    import torch
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(n)]
    barrier()
    for i in range(n):
        flush.zero_()
        starts[i].record()
        step()
        stops[i].record()
    barrier()
    return sum(s.elapsed_time(e) for s, e in zip(starts, stops)) / n


def run_native(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from cotr_b200.models import build_model
    from cotr_b200.utils import synthetic as fixtures   # seeded synthetic weights / inputs (nothing under oracle/ on this path)

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    sd = fixtures.make_state_dict(0)
    model = build_model(None)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    model = model.to(dev).eval()
    img_np, q_np = fixtures.make_inputs(100 + rank, 1, N_QUERIES)
    img = torch.from_numpy(img_np).to(dev)
    queries = torch.from_numpy(q_np).to(dev)
    img_pin = torch.from_numpy(img_np).pin_memory()
    q_pin = torch.from_numpy(q_np).pin_memory()
    out_pin = torch.empty((1, N_QUERIES, 2), dtype=torch.float32).pin_memory()
    gathered_pin = torch.empty((world, N_QUERIES, 2), dtype=torch.float32).pin_memory() if world > 1 else None
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2

    from cotr_b200.inference.sharding import AsyncGather
    # N > 1: the 8 KB blocks are exchanged on a side stream - this library's peer-memory push over NVLink on one node, NCCL otherwise
    gather = AsyncGather((1, N_QUERIES, 2), dev)
    last = {}

    def step():
        pred = model(img, queries)["pred_corrs"]
        gather.submit(pred)
        last["pred"] = pred
        return pred

    def step_solo():                          # control: the same step without handing the result to the exchange
        return model(img, queries)["pred_corrs"]

    def barrier():
        gather.wait()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    nat = model.native()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                      # nvidia-smi needs ~1 s to deliver its first sample: start it before the warm-up
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    # ---- value: K steps, each bracketed by CUDA events on the launching stream, L2 flushed between steps ----------
    dev_ms = _timed_steps(step, flush, args.steps, barrier)
    launches_per_step = nat.last_launch_count()
    gather_ok, solo_ms, rank_ms = None, dev_ms, [dev_ms]
    if world > 1:
        got = gather.wait()                    # the last step's blocks of all ranks, checked against a plain collective
        gather.check()
        want = torch.empty_like(got)
        dist.all_gather_into_tensor(want, last["pred"])
        gather_ok = bool(torch.equal(got, want))
        if not args.quick:
            solo_ms = _timed_steps(step_solo, flush, args.steps, barrier)
        per_rank = torch.zeros((world, 2), dtype=torch.float64, device=dev)
        per_rank[rank, 0], per_rank[rank, 1] = dev_ms, solo_ms
        dist.all_reduce(per_rank)
        rank_ms = per_rank.tolist()
    if args.dump_outputs and rank == 0:
        outputs = {"pred_corrs": last["pred"]}
        if world > 1:
            outputs["pred_corrs_gathered"] = got
        dump_outputs(args.dump_outputs, outputs)

    # ---- e2e: host buffers in, host result out, every copy inside the timed region ----------------------------------
    img_h, q_h, out_h = img_pin.numpy(), q_pin.numpy(), out_pin.numpy()
    if world == 1:
        def e2e_step():                      # the C-ABI host-buffer call: H2D + forward + D2H + sync inside
            nat.forward_host(img_h, q_h, out_h)
        e2e_api = "cotr_forward_host (C ABI, pinned host buffers)"
        d2h = int(out_pin.numel() * 4)
    else:
        def e2e_step():                      # the multi-GPU job as a user runs it: H2D, forward, result exchange, D2H of the gathered block
            pred = model(img_pin.to(dev, non_blocking=True), q_pin.to(dev, non_blocking=True))["pred_corrs"]
            gather.submit(pred)
            gathered_pin.copy_(gather.wait(), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e2e_api = f"COTR.forward on pinned host tensors + result exchange ({gather.backend}) + D2H of the gathered (N,1024,2) block"
        d2h = int(gathered_pin.numel() * 4)
    for _ in range(3):
        e2e_step()
    barrier()
    e2e_times = []
    for i in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e2e_step()
        e2e_times.append(time.perf_counter() - t0)
    barrier()
    e2e_ms = float(np.mean(e2e_times)) * 1e3

    # ---- BASELINE.json configs[3] per GPU: 8 pairs x 1024 queries in one forward (64 pairs over 8 GPUs) --------------
    B4 = 8
    img4_np, q4_np = fixtures.make_inputs(200 + rank, B4, N_QUERIES)
    img4 = torch.from_numpy(img4_np).to(dev)
    q4 = torch.from_numpy(q4_np).to(dev)

    gather4 = AsyncGather((B4, N_QUERIES, 2), dev)

    def step4():
        gather4.submit(model(img4, q4)["pred_corrs"])

    c4_steps = max(5, min(args.steps, 20))
    c4_ms, c4_launches = float("nan"), 0
    if not args.quick:
        for _ in range(3):
            step4()
        c4_ms = _timed_steps(step4, flush, c4_steps, barrier)
        c4_launches = nat.last_launch_count()
    # The timed regions above last ~0.1 s in total - shorter than nvidia-smi's 200 ms sampling period.  Keep the same step
    # loop running (untimed) until at least 5 samples under load exist, so the clock record describes this workload.
    clocks = None
    if rank == 0:
        t_end = time.perf_counter() + 6.0
        while not args.quick and sampler.proc is not None and sampler.samples() < 5 and time.perf_counter() < t_end:
            for _ in range(50):
                model(img, queries)
            torch.cuda.synchronize()
        clocks = sampler.stop()
        clocks["note"] = "sampled every 200 ms from before the warm-up to after the timed regions; the step loop is continued untimed until >= 5 samples exist"

    # ---- kernel shares: per-launch events (library profiler, eager launches), rank 0 ---------------------------------
    per_kernel = {}
    prof_steps = min(args.steps, 10)
    if rank == 0 and args.quick:
        per_kernel["gemm_tc"] = {"ms": 1.0, "launches": 0, "flop": 0.0}      # (no profiling pass under ncu)
    if rank == 0 and not args.quick:
        for _ in range(prof_steps):
            flush.zero_()
            nat.profile_begin(1024)
            model(img, queries)
            for name, M, N, K, ms in nat.profile_end():
                d = per_kernel.setdefault(name, {"ms": 0.0, "launches": 0, "flop": 0.0})
                d["ms"] += ms; d["launches"] += 1
                if name.startswith("gemm"):
                    d["flop"] += 2.0 * M * N * K
                elif name.startswith("attention"):
                    d["flop"] += 2.0 * 2.0 * M * N * K        # QK^T + PV over 8 heads x 32 dims
    # max over ranks
    t = torch.tensor([dev_ms, e2e_ms, c4_ms], dtype=torch.float64, device=dev)
    if world > 1:
        gather.check(); gather4.check()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, c4_ms = t.tolist()
    backends = (gather.backend, gather4.backend)
    gather.close(); gather4.close()          # collective: buffers are unmapped only after every rank has stopped pushing
    if rank != 0:
        return

    peaks = measured_peaks()
    total_q = world * N_QUERIES
    value = total_q / (dev_ms * 1e-3)
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms"])
    d = per_kernel[dom]
    share = d["ms"] / sum(v["ms"] for v in per_kernel.values())
    kernel_ms = dev_ms * share                      # the family's time inside the TIMED (graph-replayed) step
    achieved_tf = (d["flop"] / prof_steps) / (kernel_ms * 1e-3) / 1e12
    step_tf = algorithmic_flop(1, N_QUERIES) / (dev_ms * 1e-3) / 1e12
    whole_step = {"algorithmic_gflop": algorithmic_flop(1, N_QUERIES) / 1e9, "achieved": step_tf, "unit": "TFLOP/s",
                  "frac": step_tf / peaks["bf16_tflops"]}
    traffic, traffic_src = committed_traffic()
    roofline = {
        "bound": "tensor", "kernel": dom, "achieved": achieved_tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": achieved_tf / peaks["bf16_tflops"],
        "traffic": traffic, "traffic_source": traffic_src,
        "peak_source": peaks["source"],
        "launches_per_step": d["launches"] // prof_steps, "kernel_ms_per_step": kernel_ms,
        "kernel_share_of_step": share,
        "whole_step": whole_step,
        "eager_pass_ms_per_step": {k: v["ms"] / prof_steps for k, v in sorted(per_kernel.items())},
        "note": "achieved = algorithmic FLOPs of the family's launches (2*M*N*K per GEMM; the 3 split-precision MMAs per product are NOT "
                "counted) / (timed step x the family's share of the summed per-launch CUDA-event times of an eager profiling pass); "
                "eager_pass_ms_per_step are those un-overlapped eager launch times (context only: they exceed the graph-replayed step)",
    }
    c4_flop = algorithmic_flop(B4, N_QUERIES)
    c4_tf = c4_flop / (c4_ms * 1e-3) / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (fp16 hi/lo split operands, fp32 accumulate on tcgen05)", "data": "synthetic",
        "config": config_dict(world),
        "e2e": {"value": total_q / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
                "h2d_bytes_per_step": int(img_np.nbytes + q_np.nbytes), "d2h_bytes_per_step": d2h, "api": e2e_api},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": roofline,
        "whole_step": whole_step,
        "config4": {"workload": "configs[3]: 64 independent pairs x 1024 queries over 8 GPUs = 8 pairs per GPU in one forward",
                    "pairs_per_gpu": B4, "queries_per_pair": N_QUERIES, "value": world * B4 * N_QUERIES / (c4_ms * 1e-3), "unit": UNIT,
                    "ms_per_step": c4_ms, "steps": c4_steps, "launches_per_step": c4_launches,
                    "roofline": {"bound": "tensor", "algorithmic_gflop": c4_flop / 1e9, "achieved": c4_tf, "peak": peaks["bf16_tflops"],
                                 "unit": "TFLOP/s", "frac": c4_tf / peaks["bf16_tflops"]},
                    "result_gather": f"AsyncGather on a side stream, transport: {backends[1]}" if world > 1 else "none (single GPU)"},
        "clocks": clocks,
    }
    if world > 1:
        line["result_exchange"] = {
            "transport": backends[0], "last_step_equals_nccl_all_gather": gather_ok,
            "ms_per_step_by_rank": [r[0] for r in rank_ms], "ms_per_step_by_rank_without_exchange": [r[1] for r in rank_ms],
            "note": "peer = cotr_exchange: this library's push kernel stores each rank's block into every peer's buffer over NVLink on a side "
                    "stream; the second list is a control run of the same steps that never hands its result over"}
    if args.quick:
        line.pop("config4")
        line["roofline"] = None
    if world == 1 and not args.quick:
        line["cpu_baseline"] = cpu_reference_rate(budget_s=10.0)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps (at least 1)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["native", "reference"], default="native")
    ap.add_argument("--quick", action="store_true",
                    help="headline steps only (no configs[3] block, no CPU baseline, no clock continuation): the form to run under ncu")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 5],
                    help="2 = the headline (default); 3 / 5 = the zoom-in engines of BASELINE.json configs[2] / configs[4]")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (float32); headline config only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.config != 2:
        ap.error("--dump-outputs is available for the headline config (--config 2) only")
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # `python bench.py --gpus N` without a launcher: become `torch.distributed.run` with N ranks on this node
        os.execvp(sys.executable, [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
                                   "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
                                   os.path.abspath(__file__)] + sys.argv[1:])
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device; there is no CPU fallback")
    if args.gpus != world:
        raise SystemExit(f"bench.py: --gpus {args.gpus} but the launcher started {world} rank(s)")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.config != 2:
            from tools import engine_bench
            cpu = cpu_engine_rate(10000 if args.config == 3 else int(2048 / 0.3) * 2) if (rank == 0 and world == 1) else None
            engine_bench.run_config(args.config, rank, local_rank, world, steps=max(1, min(args.steps, 3)), cpu_rate=cpu)
        else:
            run_native(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
