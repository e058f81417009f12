"""Generate tests/golden/model_*.npz from the REAL reference (run in the authoring container only).

    python -m oracle.make_golden            # needs /root/reference

For each case the unmodified reference model (imported through oracle/ref_shim.py) is run on CPU in
fp32 and in fp64 on the seeded fixture of oracle/fixtures.py; the predictions are stored together with
the fixture parameters so tests can rebuild the exact inputs anywhere (TEST INFRASTRUCTURE).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)
sys.path.insert(0, REPO)

from oracle import cotr_oracle, fixtures, ref_shim  # noqa: E402

# name: (weight_seed, qk_gain, head_gain, input_seed, batch, n_queries)
CASES = {
    "model_b1_q1024": (0, 3.0, 1.35, 1, 1, 1024),      # BASELINE.json configs[1] shape
    "model_b2_q100": (0, 3.0, 1.35, 2, 2, 100),        # ragged Q (not a multiple of any tile)
    "model_b3_q1": (0, 3.0, 1.35, 3, 3, 1),            # default engine step shape (one query per context)
    "model_peaked_b1_q257": (7, 4.0, 1.0, 4, 1, 257),  # sharper attention, FasterSparseEngine max load + pilot
    # round 2 (params grow two fields: stem_gain, q_stride = only every q_stride-th query is stored)
    "model_b32_q1": (0, 3.0, 1.35, 5, 32, 1, 1.0, 1),            # a full engine batch: 32 contexts x 1 query
    "model_b16_q1024": (0, 3.0, 1.35, 6, 16, 1024, 1.0, 8),      # >= 64 row tiles in the encoder GEMMs
    "model_b64_q1024": (0, 3.0, 1.35, 7, 64, 1024, 1.0, 16),     # BASELINE.json configs[3] (64 pairs x 1024 queries)
    "model_bigact_b1_q256": (0, 3.0, 1.35, 8, 1, 256, 160.0, 1),  # backbone activations up to ~4e4 (fp16 hi/lo range)
}
# The fp32 round-off of a CPU forward depends on torch's intra-op thread count (model_b1_q1024 moves by 9e-5 at 1
# thread and by 5e-5 at 16 or more against 4 or 8), so the fp32 vectors are recorded, and checked, with this many.
GOLDEN_THREADS = 8


def main():
    torch.set_grad_enabled(False)
    torch.set_num_threads(GOLDEN_THREADS)
    out_dir = os.path.join(REPO, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    only = sys.argv[1:]
    for name, case in CASES.items():
        if only and name not in only:
            continue
        wseed, qk, hg, iseed, b, q = case[:6]
        stem_gain, q_stride = (case[6], case[7]) if len(case) > 6 else (1.0, 1)
        sd = fixtures.make_state_dict(wseed, qk, hg, stem_gain)
        img, queries = fixtures.make_inputs(iseed, b, q)
        model = ref_shim.build_reference_model(sd)
        ref32 = model(torch.from_numpy(img), torch.from_numpy(queries))["pred_corrs"].numpy()
        model = model.double()
        ref64 = model(torch.from_numpy(img).double(), torch.from_numpy(queries).double())["pred_corrs"].numpy()
        o64, inter = cotr_oracle.forward(sd, img, queries, torch.float64, return_intermediates=True)
        o32 = cotr_oracle.forward(sd, img, queries, torch.float32)
        d_oracle = float(np.abs(o64.numpy() - ref64).max())
        print(f"{name}: std over queries {ref64.std(axis=1).max():.4f}  |ref32-ref64| {np.abs(ref32 - ref64).max():.2e}  "
              f"|oracle64-ref64| {d_oracle:.2e}  |oracle32-ref32| {np.abs(o32.numpy() - ref32).max():.2e}")
        np.savez_compressed(
            os.path.join(out_dir, name + ".npz"),
            params=np.array(case, dtype=np.float64),
            ref_pred_fp32=ref32.astype(np.float32)[:, ::q_stride], ref_pred_fp64=ref64.astype(np.float64)[:, ::q_stride],
            feat_absmax=np.array(float(inter["feat"].abs().max())),
            oracle_vs_ref_fp64=np.array(d_oracle),
            feat_rms=np.array(float(inter["feat"].pow(2).mean().sqrt())),
            mem_head=inter["mem"][0, :4, :16].numpy(), hs_head=inter["hs"][0, :4, :16].numpy(),
        )


if __name__ == "__main__":
    main()
