"""BASELINE.json configs[0]: the reference's `demo_single_pair.py` against this repository, held to what the reference
itself did with the same inputs.

tests/golden/demo_single_pair.npz was made by running that script, unmodified, against the reference's own package
(oracle/make_demo_golden.py) on seeded synthetic stand-ins for the sample pair and a seeded synthetic checkpoint.
`_demo_main` below makes the script's calls in the script's order, but through the alias package `COTR/` -> `cotr_b200`
(`from COTR.models import build_model`, `from COTR.inference.sparse_engine import SparseEngine`, `from
COTR.options.options import *` ...), with the same inputs:

  * the CPU test puts the deterministic stand-in network of `oracle/fake_model.py` behind `build_model` - same
    parameter schema (so the strict checkpoint load is the real one), same `model(img, queries)['pred_corrs']`
    contract - and demands the reference's network calls, correspondences and final blended image;
  * the GPU test runs the real native model; seeded random weights accept no task, and the reference ends in
    `assert corr_f.shape[0] > 0` (sparse_engine.py:247, SURVEY.md section 8c).  The native run must end there too,
    after the dense passes and the zoom-in batches have run on the device.
"""
import argparse
import os
import sys
import traceback

import numpy as np
import pytest
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _golden(golden_dir):
    return np.load(os.path.join(golden_dir, "demo_single_pair.npz"))


def _demo_main(tmp_path, max_corrs, prepare_model=None, triangulate=None):
    """What demo_single_pair.py does between its imports and plt.show(), through the `COTR` alias package.
    Returns (model, corrs, blended image)."""
    import cv2
    sys.path.insert(0, REPO)
    from COTR.inference import inference_helper
    from COTR.inference.sparse_engine import SparseEngine
    from COTR.models import build_model
    from COTR.options.options import set_COTR_arguments
    from COTR.utils import utils
    from cotr_b200.utils import synthetic
    from oracle.make_demo_golden import demo_image

    ckpt = tmp_path / "out" / "default" / "checkpoint.pth.tar"
    ckpt.parent.mkdir(parents=True)
    sd = {k: torch.from_numpy(v) for k, v in synthetic.make_state_dict(0).items()}
    torch.save({"epoch": 0, "iteration": 0, "optim_state_dict": {}, "model_state_dict": sd}, ckpt)
    parser = argparse.ArgumentParser()
    set_COTR_arguments(parser)
    opt = parser.parse_args([])
    opt.dim_feedforward = 1024                         # layer3
    utils.fix_randomness(0)
    with torch.set_grad_enabled(False):
        model = build_model(opt)
        if prepare_model is not None:
            prepare_model(model)
        model = model.cuda()
        utils.safe_load_weights(model, torch.load(ckpt, map_location='cpu')['model_state_dict'])
        model = model.eval()
        img_a, img_b = demo_image("cathedral_1.jpg"), demo_image("cathedral_2.jpg")
        engine = SparseEngine(model, 32, mode='tile')
        corrs = engine.cotr_corr_multiscale_with_cycle_consistency(img_a, img_b, np.linspace(0.5, 0.0625, 4), 1,
                                                                   max_corrs=max_corrs, queries_a=None)
        utils.visualize_corrs(img_a, img_b, corrs)
        dense = (triangulate or inference_helper.triangulate_corr)(corrs, img_a.shape, img_b.shape)
        warped = cv2.remap(img_b, dense[..., 0].astype(np.float32), dense[..., 1].astype(np.float32),
                           interpolation=cv2.INTER_LINEAR, borderMode=cv2.BORDER_CONSTANT)
        return model, corrs, warped / 255 * 0.5 + img_a / 255 * 0.5


def test_demo_single_pair_matches_reference_cpu(golden_dir, tmp_path, capsys):
    from oracle import triangulate_oracle
    from oracle.fake_model import FakeCOTR
    from oracle.make_demo_golden import FAKE_MAX_CORRS, blend_summary
    from oracle.make_engine_golden import call_log_array
    gold = _golden(golden_dir)

    def fake_network(model):
        object.__setattr__(model, "fake", FakeCOTR())      # not a registered sub-module: the schema stays the reference's
        model.forward = model.fake.forward
        model.supports_device_preprocess = False
        model.cuda = lambda *a, **k: model                 # no GPU needed: the stand-in runs on the host

    # the product triangulate_corr renders with CUDA; on the host the script gets the CPU restatement, as the reference did
    model, corrs, shown = _demo_main(tmp_path, FAKE_MAX_CORRS, fake_network,
                                     lambda corr, a, b: triangulate_oracle.triangulate_corr(corr, a, b)[0])
    assert "weights safely loaded" in capsys.readouterr().out      # utils.safe_load_weights, strict path
    calls = call_log_array(model.fake)
    assert calls.shape == gold["fake_calls"].shape                 # 4 dense passes + the zoom-in batches
    assert np.array_equal(calls[:, :2], gold["fake_calls"][:, :2])
    np.testing.assert_allclose(calls[:, 2:], gold["fake_calls"][:, 2:], rtol=1e-12, atol=1e-9)
    assert corrs.shape == (FAKE_MAX_CORRS, 4)
    np.testing.assert_array_equal(corrs, gold["fake_corrs"])
    got = blend_summary(shown)
    np.testing.assert_array_equal(got["shown_shape"], gold["shown_shape"])        # warped image blended over image a
    np.testing.assert_allclose(got["shown_sum"], gold["shown_sum"], rtol=1e-12)
    np.testing.assert_allclose(got["shown_abs"], gold["shown_abs"], rtol=1e-12)
    np.testing.assert_allclose(got["shown_sample"], gold["shown_sample"], rtol=1e-12, atol=1e-12)


@pytest.mark.gpu
def test_demo_single_pair_native_ends_like_reference_gpu(golden_dir, tmp_path, capsys, built_lib):
    """The same calls, native model on the GPU, 100 correspondences requested (the demo's default).  Seeded random
    weights are rejected by the engine's own acceptance tests: the run must end where the reference's ended."""
    from oracle.make_demo_golden import NETWORK_MAX_CORRS, failure_site
    gold = _golden(golden_dir)
    built = []
    with pytest.raises(AssertionError) as info:
        _demo_main(tmp_path, NETWORK_MAX_CORRS, built.append)
    assert failure_site(info.value) == (str(gold["network_failure_function"]), str(gold["network_failure_line"])), \
        traceback.format_exception(info.value)
    assert "weights safely loaded" in capsys.readouterr().out
    assert built and next(built[0].parameters()).is_cuda
    assert built[0].native().last_launch_count() > 50            # the device really ran the network


@pytest.mark.gpu
def test_demo_call_sequence_native_gpu(tmp_path, capsys, built_lib):
    """What `demo_single_pair.py:25-45` does, with the changes SURVEY.md section 8(d) prescribes for random weights:
    synthetic images instead of the sample pair and 100 FORCED queries (`cotr_corr_multiscale(..., queries_a=q,
    force=True)`), so every query comes back.  Everything goes through the alias package `COTR`, as in the script:
    build_model -> cuda -> checkpoint file -> safe_load_weights -> SparseEngine(model, 32, mode='tile') ->
    visualize_corrs -> triangulate_corr (CUDA rasteriser) -> cv2.remap."""
    import cv2
    sys.path.insert(0, REPO)
    from COTR.utils import utils
    from COTR.models import build_model
    from COTR.inference.inference_helper import triangulate_corr
    from COTR.inference.sparse_engine import SparseEngine
    from cotr_b200.utils import synthetic

    utils.fix_randomness(0)
    torch.set_grad_enabled(False)
    ckpt = tmp_path / "checkpoint.pth.tar"
    torch.save({"model_state_dict": {k: torch.from_numpy(v) for k, v in synthetic.make_state_dict(0).items()}}, ckpt)
    model = build_model(None).cuda()
    utils.safe_load_weights(model, torch.load(ckpt, map_location='cpu')['model_state_dict'])
    model = model.eval()
    img_a = synthetic.synthetic_image(61, 783, 1064)          # the shapes of cathedral_1.jpg / cathedral_2.jpg
    img_b = synthetic.synthetic_image(62, 1053, 689)
    rs = np.random.RandomState(0)
    queries = np.stack([rs.uniform(0, img_a.shape[1], 100), rs.uniform(0, img_a.shape[0], 100)], axis=1)
    engine = SparseEngine(model, 32, mode='tile')
    corrs = engine.cotr_corr_multiscale(img_a, img_b, np.linspace(0.5, 0.0625, 4), 1, max_corrs=100, queries_a=queries, force=True)
    assert corrs.shape == (100, 4) and np.isfinite(corrs).all()
    assert np.allclose(np.sort(corrs[:, 0]), np.sort(queries[:, 0]))            # every forced query came back
    canvas = utils.visualize_corrs(img_a, img_b, corrs)
    assert canvas.shape == (1053, 1064 + 689, 3)
    dense = triangulate_corr(corrs, img_a.shape, img_b.shape)
    assert dense.shape == (783, 1064, 2) and dense.dtype == np.float32 and (dense != 0).any()
    warped = cv2.remap(img_b, dense[..., 0].astype(np.float32), dense[..., 1].astype(np.float32), interpolation=cv2.INTER_LINEAR,
                       borderMode=cv2.BORDER_CONSTANT)
    assert warped.shape == img_a.shape
    assert "weights safely loaded" in capsys.readouterr().out
