"""Per-GEMM-group precision switches, measured on the B200 against the REFERENCE's golden tracks (VERDICT r1 item 6).

For every (prec.corr, prec.fc1) setting: max |d pred_tracks| (pixels) and visibility mismatches on the committed
reference-generated fixtures at BASELINE scale -- unit-gain and amplified-head ("stress", ~20 px of motion) -- plus
the headline step time.  The table goes to profiles/ and picks the library default (csrc/api.cu kDefPrec*).

    python tests/tools/precision_sweep.py > profiles/r2_precision_sweep.txt
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cases import golden_view, load_golden, run_cuda  # noqa: E402
from cotracker_b200 import engine  # noqa: E402

CASES = ["c2_grid30", "c2_grid30_stress", "headline_grid80", "headline_grid80_stress", "c1_apple_grid10_stress",
         "c4_online_grid50", "offline_stress", "predictor_grid"]
SETTINGS = [(3, 3), (2, 3), (1, 3), (3, 2), (2, 2), (1, 2), (2, 1), (1, 1)]


def step_ms():
    from cotracker_b200.predictor import CoTrackerPredictor
    from cotracker_b200.synthetic import seeded_state_dict, texture_video
    p = CoTrackerPredictor(checkpoint=None, window_len=60)
    p.model.load_state_dict(seeded_state_dict(1234))
    p = p.to("cuda:0")
    v = texture_video(16, 512, 512, seed=0).to("cuda:0")
    for _ in range(3):
        p(v, grid_size=80)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(5):
        p(v, grid_size=80)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / 5 * 1e3


def main():
    cases = [c for c in CASES if os.path.exists(os.path.join(ROOT, "tests", "golden", c + ".npz"))]
    print("prec.corr prec.fc1 | headline ms/step | " + " | ".join(cases))
    for corr, fc1 in SETTINGS:
        engine.set_option("prec.corr", corr)
        engine.set_option("prec.fc1", fc1)
        cells = []
        for name in cases:
            got, want = golden_view(run_cuda(name), load_golden(name))
            err, flips = 0.0, 0
            for k, w in want.items():
                if k.startswith("prob_"):
                    continue
                if w.dtype == torch.bool:
                    flips += int((got[k] != w).sum())
                elif "tracks" in k or "coords" in k:
                    err = max(err, float((got[k].float() - w.float()).abs().max()))
            cells.append(f"{err:.2e}/{flips}")
        print(f"{corr:9d} {fc1:8d} | {step_ms():16.2f} | " + " | ".join(cells), flush=True)


if __name__ == "__main__":
    main()
