"""Generate tests/golden/demo_single_pair.npz by running the reference's `demo_single_pair.py`, unmodified, against the
reference's own package (needs a checkout of the reference, located by oracle/ref_shim.py).

    python -m oracle.make_demo_golden

Both runs read seeded synthetic stand-ins for the sample pair (`DEMO_IMAGES`: the shapes of cathedral_1.jpg /
cathedral_2.jpg) and load the seeded synthetic checkpoint (cotr_b200/utils/synthetic.py seed 0) from
`out/default/checkpoint.pth.tar`, as the script expects:

  * fake: the deterministic stand-in network of oracle/fake_model.py answers in place of the reference network (the
    parameter tree, and so the strict checkpoint load, stays the reference's), `--max_corrs 40`.  Stored: the
    correspondences the script hands to `triangulate_corr`, the network call log and the blended image it shows.
  * network: the reference network itself on CPU, `--max_corrs 100` (the script's default).  Random weights yield no
    accepted correspondence and the run ends in the engine's `assert corr_f.shape[0] > 0`; stored: where it ended.

The reference renders `triangulate_corr` with OpenGL, which cannot run offline; both runs use the CPU restatement
of oracle/triangulate_oracle.py.  `imageio` and `matplotlib` are not installed offline and get stand-ins.
tests/test_demo_dropin.py drives the script's call sequence through the `COTR` alias package and compares.
"""
import os
import runpy
import sys
import tempfile
import traceback

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)

from cotr_b200.utils.synthetic import make_state_dict, synthetic_image  # noqa: E402
from oracle.make_engine_golden import call_log_array  # noqa: E402

DEMO_IMAGES = {"cathedral_1.jpg": (61, 783, 1064), "cathedral_2.jpg": (62, 1053, 689)}   # name -> (seed, h, w)
FAKE_MAX_CORRS = 40
NETWORK_MAX_CORRS = 100


def demo_image(name):
    seed, h, w = DEMO_IMAGES[name]
    return synthetic_image(seed, h, w)


def blend_summary(shown):
    """Checksums and a strided sample of the (h, w, 3) float image the script passes to plt.imshow."""
    shown = np.asarray(shown, dtype=np.float64)
    return {"shown_shape": np.array(shown.shape), "shown_sum": np.array(shown.sum()),
            "shown_abs": np.array(np.abs(shown).sum()), "shown_sample": shown[::17, ::13].copy()}


def failure_site(exc):
    """(function, source line) of the frame that raised `exc`."""
    frame = traceback.extract_tb(exc.__traceback__)[-1]
    return frame.name, frame.line.strip()


class _Inert:
    """Answers every attribute access and call with itself: the figure / axes calls of the reference's plotting."""

    def __getattr__(self, name):
        return self

    def __call__(self, *a, **k):
        return self


def _run_reference_demo(workdir, max_corrs, fake):
    import torch
    import COTR.models as ref_models
    from COTR.inference import inference_helper
    from oracle import ref_shim, triangulate_oracle
    from oracle.fake_model import FakeCOTR

    ref_build = ref_models.build_model
    built, shown, handed = [], [], []

    def build_model(opt):
        model = ref_build(opt)
        model.cuda = lambda *a, **k: model             # no GPU here: the reference network (or the stand-in) runs on CPU
        if fake:
            object.__setattr__(model, "fake", FakeCOTR())   # not a registered sub-module: the schema stays the reference's
            model.forward = model.fake.forward
        built.append(model)
        return model

    def triangulate_corr(corr, from_shape, to_shape):
        handed.append(np.array(corr, copy=True))
        return triangulate_oracle.triangulate_corr(corr, from_shape, to_shape)[0]

    sys.modules["imageio"].imread = lambda path, pilmode="RGB": demo_image(os.path.basename(path))
    plt = sys.modules["matplotlib.pyplot"]                 # the module the reference bound at import: patched in place
    plt.imshow = lambda img, *a, **k: shown.append(np.asarray(img)) or _Inert()
    plt.__getattr__ = lambda name: _Inert()
    ref_models.build_model = build_model
    inference_helper.triangulate_corr = triangulate_corr
    cwd, argv = os.getcwd(), sys.argv
    os.chdir(workdir)
    sys.argv = ["demo_single_pair.py", "--load_weights", "default", "--max_corrs", str(max_corrs), "--out_dir", os.path.join(workdir, "out")]
    try:
        runpy.run_path(os.path.join(ref_shim.REF_ROOT, "demo_single_pair.py"), run_name="__main__")
        return built[0], shown, handed, None
    except AssertionError as e:
        return built[0], shown, handed, e
    finally:
        os.chdir(cwd)
        sys.argv = argv
        ref_models.build_model = ref_build
        torch.set_grad_enabled(True)


def main():
    import torch
    from oracle import ref_shim
    ref_shim.import_reference()
    import COTR.inference.inference_helper  # noqa: F401  (imported from the reference tree while CWD is its root)
    import COTR.inference.sparse_engine  # noqa: F401
    import COTR.options.options  # noqa: F401
    import COTR.utils.utils  # noqa: F401
    payload = {}
    with tempfile.TemporaryDirectory() as workdir:
        os.makedirs(os.path.join(workdir, "out", "default"))
        sd = {k: torch.from_numpy(v) for k, v in make_state_dict(0).items()}
        torch.save({"epoch": 0, "iteration": 0, "optim_state_dict": {}, "model_state_dict": sd},
                   os.path.join(workdir, "out", "default", "checkpoint.pth.tar"))

        model, shown, handed, err = _run_reference_demo(workdir, FAKE_MAX_CORRS, fake=True)
        assert err is None and len(handed) == 1 and len(shown) == 2, err      # visualize_corrs' canvas, then the blend
        payload["fake_corrs"] = handed[0]
        payload["fake_calls"] = call_log_array(model.fake)
        payload.update(blend_summary(shown[1]))
        print("fake:", handed[0].shape, "network calls:", len(model.fake.calls))

        model, shown, handed, err = _run_reference_demo(workdir, NETWORK_MAX_CORRS, fake=False)
        assert err is not None and not handed and not shown
        name, line = failure_site(err)
        payload["network_failure_function"] = np.array(name)
        payload["network_failure_line"] = np.array(line)
        print("network:", name, "|", line)
    np.savez_compressed(os.path.join(REPO, "tests", "golden", "demo_single_pair.npz"), **payload)


if __name__ == "__main__":
    main()
