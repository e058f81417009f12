"""GPU: batch-invariant mode (cotr_set_batch_invariant, COTR.set_batch_invariant).  Every pair and every query is
computed by the kernel sequence of the headline forward (B = 1, Q = 1024), so every comparison here is bitwise:
torch.equal / np.array_equal, never a tolerance."""
import glob
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import fixtures

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = 1e-3              # the bounds test_model_gpu.py applies to the goldens
TOL_INTERNAL = 3e-4
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(REPO, "tests", "golden", "model_*.npz")))


def _build(sd, invariant):
    from cotr_b200.models import build_model
    model = build_model(None)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    model.set_batch_invariant(invariant)
    return model.cuda().eval()


def _inputs(seed, B, Q):
    img, q = fixtures.make_inputs(seed, B, Q)
    return torch.from_numpy(img).cuda(), torch.from_numpy(q).cuda()


@pytest.fixture(scope="module")
def inv_model(built_lib):
    return _build(fixtures.make_state_dict(0), True)


def _fwd(model, img, q):
    return model(img, q)["pred_corrs"].clone()


def test_pair_alone_equals_pair_in_any_batch(inv_model):
    img, q = _inputs(41, 8, 64)
    alone = [_fwd(inv_model, img[p:p + 1], q[p:p + 1]) for p in range(8)]
    for B in (2, 3, 4, 8):
        out = _fwd(inv_model, img[:B], q[:B])
        for p in range(B):
            assert torch.equal(out[p:p + 1], alone[p]), (B, p)
    for B in (32, 64):
        idx = [(5 * i + 3 + i // 8) % 8 for i in range(B)]       # every pair, repeated, in mixed order
        out = _fwd(inv_model, img[idx].contiguous(), q[idx].contiguous())
        for j, p in enumerate(idx):
            assert torch.equal(out[j:j + 1], alone[p]), (B, j, p)


def test_query_alone_equals_query_among_any_others(inv_model):
    img, q = _inputs(42, 1, 1024)
    ref = _fwd(inv_model, img, q)
    rs = np.random.RandomState(0)
    for Q in (1, 7, 31, 32, 33, 100, 1024):
        for _ in range(2):
            idx = rs.choice(1024, Q, replace=False)            # other queries, other row positions
            out = _fwd(inv_model, img, q[:, idx].contiguous())
            assert torch.equal(out, ref[:, idx]), Q
    # 40 000 queries: two decode chunks of one pair
    idx = (np.arange(40000) * 7 + 11) % 1024
    out = _fwd(inv_model, img, q[:, idx].contiguous())
    assert torch.equal(out, ref[:, idx])
    # next to zero-padded queries (FasterSparseEngine pads its squads)
    padded = torch.cat([q[:, 200:250], torch.zeros(1, 207, 2, device="cuda")], dim=1)
    out = _fwd(inv_model, img, padded)
    assert torch.equal(out[:, :50], ref[:, 200:250])
    zero = _fwd(inv_model, img, torch.zeros(1, 1, 2, device="cuda"))
    assert torch.equal(out[:, 50:], zero.expand(1, 207, 2))


def test_queries_of_a_batch_equal_single_queries(inv_model):
    """B = 32, Q = 1 (the engines' single-query phase) == each pair alone with its query inside a 1024-query set."""
    img8, q8 = _inputs(43, 8, 1024)
    idx = [i % 8 for i in range(32)]
    rows = [(7 * i) % 1024 for i in range(32)]
    qs = torch.stack([q8[p, r] for p, r in zip(idx, rows)])[:, None, :].contiguous()
    out = _fwd(inv_model, img8[idx].contiguous(), qs)
    full = [_fwd(inv_model, img8[p:p + 1], q8[p:p + 1]) for p in range(8)]
    for j, (p, r) in enumerate(zip(idx, rows)):
        assert torch.equal(out[j, 0], full[p][0, r]), j


def test_entry_points_agree(inv_model):
    img, q = _inputs(44, 2, 333)
    runs = [_fwd(inv_model, img, q) for _ in range(3)]          # eager, capture, replay
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])
    ctx = inv_model.encode_context(img)
    parts = [inv_model.decode(ctx, q[:, s:e].contiguous())["pred_corrs"] for s, e in ((0, 100), (100, 101), (101, 333))]
    assert torch.equal(torch.cat(parts, dim=1), runs[0])
    ctx.native.close()
    host = inv_model.native().forward_host(img.cpu().numpy(), q.cpu().numpy())
    assert np.array_equal(host, runs[0].cpu().numpy())
    inv_model.native().set_graph_mode(False)
    try:
        assert torch.equal(_fwd(inv_model, img, q), runs[0])
    finally:
        inv_model.native().set_graph_mode(True)
    # the same pair through the cached context of another batch size
    ctx1 = inv_model.encode_context(img[1:2], reuse=True)
    assert torch.equal(inv_model.decode(ctx1, q[1:2, 5:9].contiguous())["pred_corrs"], runs[0][1:2, 5:9])


def test_headline_shape_is_the_default_schedule(built_lib):
    sd = fixtures.make_state_dict(0)
    default, inv = _build(sd, False), _build(sd, True)
    img, q = _inputs(1, 1, 1024)
    a, b = _fwd(default, img, q), _fwd(inv, img, q)
    assert torch.equal(a, b)
    assert default.native().last_launch_count() == 136
    for B, Q in ((1, 1024), (8, 1024), (32, 1)):
        img, q = _inputs(2, B, Q)
        _fwd(inv, img, q)
        assert inv.native().last_launch_count() == 136, (B, Q)


def test_attention_never_falls_back_to_simt(built_lib):
    """The per-launch profiler names the kernel that really ran: the default decoder of a 1-query launch is SIMT,
    the invariant one tcgen05."""
    sd = fixtures.make_state_dict(0)
    img, q = _inputs(3, 4, 1)
    for invariant, want in ((False, "attention_simt"), (True, "attention_tc")):
        m = _build(sd, invariant)
        nat = m.native()
        nat.profile_begin(512)
        m(img, q)
        recs = nat.profile_end()
        dec_attn = [r[0] for r in recs if r[0].startswith("attention") and r[1] == 4]
        assert dec_attn == [want] * 6, (invariant, dec_attn)


@pytest.mark.parametrize("name", CASES)
def test_goldens_in_invariant_mode(golden_dir, built_lib, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    params = g["params"]
    wseed, qk, hg, iseed, b, nq = params[:6]
    stem_gain, q_stride = (float(params[6]), int(params[7])) if len(params) > 6 else (1.0, 1)
    sd = fixtures.make_state_dict(int(wseed), float(qk), float(hg), stem_gain)
    img, queries = fixtures.make_inputs(int(iseed), int(b), int(nq))
    model = _build(sd, True)
    pred = model(torch.from_numpy(img).cuda(), torch.from_numpy(queries).cuda())["pred_corrs"].cpu().numpy()
    assert np.isfinite(pred).all()
    pred = pred[:, ::q_stride]
    err32 = np.abs(pred - g["ref_pred_fp32"]).max()
    err64 = np.abs(pred - g["ref_pred_fp64"]).max()
    assert err32 < TOL and err64 < TOL, (err32, err64)
    assert err64 < TOL_INTERNAL, err64


def test_toggle_drops_graphs_and_restores_the_default(built_lib):
    sd = fixtures.make_state_dict(0)
    m = _build(sd, False)
    img, q = _inputs(45, 8, 300)
    for _ in range(3):                                          # the shape's graph is captured and replayed
        _fwd(m, img, q)
    m.set_batch_invariant(True)
    after = _fwd(m, img, q)
    m.native().set_graph_mode(False)
    eager = _fwd(m, img, q)
    m.native().set_graph_mode(True)
    assert torch.equal(after, eager)
    assert torch.equal(after[3:4], _fwd(m, img[3:4], q[3:4]))
    m.set_batch_invariant(False)
    back = [_fwd(m, img, q) for _ in range(3)]
    fresh = _fwd(_build(sd, False), img, q)
    assert all(torch.equal(x, fresh) for x in back)


def test_context_of_the_other_mode_is_refused(built_lib):
    m = _build(fixtures.make_state_dict(0), True)
    img, q = _inputs(46, 2, 16)
    for mode in (True, False):
        m.set_batch_invariant(mode)
        ctx = m.encode_context(img)
        m.set_batch_invariant(not mode)
        with pytest.raises(RuntimeError, match="batch-invariant"):
            m.decode(ctx, q)
        m.set_batch_invariant(mode)
        dec = m.decode(ctx, q)["pred_corrs"]
        if mode:
            assert torch.equal(dec, _fwd(m, img, q))
        ctx.native.close()


@pytest.mark.parametrize("npairs", [1, 3])
def test_tcgen05_attention_any_query_count(built_lib, npairs):
    """cotr_test_attention path 2: tcgen05 for every nq (idle lane quarters skipped below 32 rows) - within the
    attention bound of test_kernels_gpu.py, and row r of a pair bit-identical whatever nq is."""
    from cotr_b200 import capi
    g = torch.Generator(device="cpu").manual_seed(50 + npairs)
    nmax = 100
    q_all = torch.randn(npairs, nmax, 256, generator=g) * 2.0
    k = torch.randn(npairs * 512, 256, generator=g).cuda()
    v = torch.randn(npairs * 512, 256, generator=g).cuda()
    kh = k.double().view(npairs, 512, 8, 32).transpose(1, 2)
    vh = v.double().view(npairs, 512, 8, 32).transpose(1, 2)
    outs = {}
    for nq in (1, 5, 31, 32, 100):
        q = q_all[:, :nq].reshape(npairs * nq, 256).contiguous().cuda()
        qh = q.double().view(npairs, nq, 8, 32).transpose(1, 2)
        ref = (torch.softmax(qh @ kh.transpose(-1, -2), -1) @ vh).transpose(1, 2).reshape(npairs * nq, 256)
        out = capi.test_attention(2, q, k, v, nq, npairs)
        rel = ((out.double() - ref).norm() / ref.norm()).item()
        assert rel < 5e-6, (nq, rel)
        outs[nq] = out.view(npairs, nq, 256)
    for nq, out in outs.items():
        assert torch.equal(out, outs[nmax][:, :nq]), nq


def test_sparse_engine_batch_size_does_not_matter(inv_model):
    from cotr_b200.inference.sparse_engine import SparseEngine
    from cotr_b200.utils.synthetic import synthetic_image
    from cotr_b200.utils.utils import fix_randomness
    img_a, img_b = synthetic_image(61, 512, 512), synthetic_image(62, 512, 512)
    rs = np.random.RandomState(7)
    queries = np.stack([rs.uniform(10, 502, 48), rs.uniform(10, 502, 48)], axis=1)
    zooms = np.linspace(0.5, 0.0625, 4)
    out = []
    for bs in (32, 5):
        fix_randomness(0)
        out.append(SparseEngine(inv_model, bs, mode='tile').cotr_corr_multiscale(
            img_a, img_b, zooms, 1, max_corrs=48, queries_a=queries.copy(), force=True))
    assert out[0].shape[0] > 0 and np.array_equal(out[0], out[1])


def _config5_job(model, n_queries=300):
    from cotr_b200.inference.sparse_engine import FasterSparseEngine
    from cotr_b200.utils.utils import fix_randomness
    from tools.engine_bench import _pair, _queries, forced_cycle_consistency
    img_a, img_b = _pair(512)
    fix_randomness(0)
    eng = FasterSparseEngine(model, 32, mode='tile', rescue_stranded=True)
    corrs, err = forced_cycle_consistency(eng, img_a, img_b, _queries(n_queries, 512), n_queries // 3)
    return corrs, err


def test_config5_job_is_identical_for_any_split_of_the_calls(inv_model):
    """What 2 and 8 ranks compute (each model call divided as ShardedCOTR divides it), here on one GPU."""
    from tools.invariance_cost import SplitCalls
    base = _config5_job(inv_model)
    assert base[0].shape[0] > 0
    for world in (2, 8):
        got = _config5_job(SplitCalls(inv_model, world))
        assert np.array_equal(got[0], base[0]) and np.array_equal(got[1], base[1]), world


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_config5_job_identical_on_two_gpus(built_lib, tmp_path):
    """torchrun / nccl: the config-5 job through ShardedCOTR on 2 ranks == rank 0 alone, bit for bit."""
    worker = os.path.join(REPO, "tests", "batch_invariant_worker.py")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29543", worker, str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=REPO)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert open(tmp_path / "rank0.txt").read().strip() == "identical"


@pytest.mark.parametrize("invariant", [False, True], ids=["default", "invariant"])
def test_repeatable(built_lib, invariant):
    m = _build(fixtures.make_state_dict(0), invariant)
    m.native().set_graph_mode(False)
    img, q = _inputs(47, 3, 77)
    assert torch.equal(_fwd(m, img, q), _fwd(m, img, q))
