"""CPU: the oracle restatement against the golden vectors produced by the REAL reference (oracle/make_golden.py)."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import cotr_oracle, fixtures
from oracle.make_golden import GOLDEN_THREADS

CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "model_*.npz")))


def _load(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    params = g["params"]
    wseed, qk, hg, iseed, b, q = params[:6]
    stem_gain, q_stride = (float(params[6]), int(params[7])) if len(params) > 6 else (1.0, 1)   # round-2 cases
    sd = fixtures.make_state_dict(int(wseed), float(qk), float(hg), stem_gain)
    img, queries = fixtures.make_inputs(int(iseed), int(b), int(q))
    return g, sd, img, queries, q_stride


def test_golden_files_exist():
    assert len(CASES) >= 4


@pytest.fixture
def golden_threads():
    """The intra-op thread count the fp32 goldens were recorded with (their round-off depends on it)."""
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", CASES)
def test_oracle_fp32_matches_reference_fp32(golden_dir, golden_threads, name):
    g, sd, img, queries, q_stride = _load(golden_dir, name)
    pred = cotr_oracle.forward(sd, img, queries, torch.float32).numpy()[:, ::q_stride]
    # same arithmetic, same library kernels: the restatement reproduces the reference to fp32 round-off
    assert np.abs(pred - g["ref_pred_fp32"]).max() < 5e-6


@pytest.mark.parametrize("name", [c for c in CASES if "q1024" not in c])
def test_oracle_fp64_matches_reference_fp64(golden_dir, name):
    g, sd, img, queries, q_stride = _load(golden_dir, name)
    pred = cotr_oracle.forward(sd, img, queries, torch.float64).numpy()[:, ::q_stride]
    assert np.abs(pred - g["ref_pred_fp64"]).max() < 1e-10
    assert float(g["oracle_vs_ref_fp64"]) < 1e-10          # recorded when the goldens were generated


def test_fixture_is_well_conditioned(golden_dir):
    """SURVEY.md appendix E.3: a parity fixture must be query-sensitive AND numerically benign."""
    g = np.load(os.path.join(golden_dir, "model_b1_q1024.npz"))
    assert g["ref_pred_fp64"].std(axis=1).min() > 0.05                       # >> the 1e-3 parity bar
    assert np.abs(g["ref_pred_fp32"] - g["ref_pred_fp64"]).max() < 2e-4      # << the 1e-3 parity bar


def test_queries_are_independent():
    """No decoder self-attention (transformer.py:185-201): a query alone == the same query inside a batch."""
    sd = fixtures.make_state_dict(0)
    img, queries = fixtures.make_inputs(5, 1, 64)
    full = cotr_oracle.forward(sd, img, queries, torch.float64)
    one = cotr_oracle.forward(sd, img, queries[:, 17:18], torch.float64)
    assert (full[:, 17:18] - one).abs().max() < 1e-10


def test_schema_has_381_entries():
    sch = fixtures.schema()
    assert len(sch) == 381
    n_params = sum(int(np.prod(s)) for k, s in sch if "running" not in k and ".bn" not in k and "downsample.1" not in k)
    assert n_params == 18387906
