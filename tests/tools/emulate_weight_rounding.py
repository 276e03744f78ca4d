"""CPU emulation (reference model, $COTRACKER_REFERENCE): what would a 2-product transformer GEMM cost in track error?

A 2-product GEMM on fp16 planes keeps the activation exact to ~2^-22 (hi + lo) and rounds the WEIGHT to one fp16 plane
(2^-12).  That is exactly the unmodified reference run with its transformer weights rounded to fp16, so the error of
the scheme can be measured without writing the kernel.  Prints max |d tracks| against the committed golden of the case.

    python tests/tools/emulate_weight_rounding.py c2_grid30 c2_grid30_stress c4_online_grid50
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import make_golden as mg  # noqa: E402


def rounded(sd, mode, groups):
    out = {}
    for k, v in sd.items():
        hit = v.ndim == 2 and any(g in k for g in groups)
        if not hit:
            out[k] = v
        elif mode == "fp16":
            out[k] = v.half().float()
        elif mode == "bf16":
            out[k] = v.bfloat16().float()
        elif mode == "fp16x2":
            hi = v.half().float()
            out[k] = hi + (v - hi).half().float()
        else:
            raise ValueError(mode)
    return out


def main():
    mode = os.environ.get("ROUND", "fp16")
    groups = os.environ.get("WGROUPS", "updateformer.").split(",")
    for name in sys.argv[1:]:
        cfg = dict(mg.DEFAULTS, **mg.CASES[name]) if hasattr(mg, "DEFAULTS") else mg.CASES[name]
        orig = mg.seeded_state_dict

        def patched(*a, **k):
            return rounded(orig(*a, **k), mode, groups)
        mg.seeded_state_dict = patched
        try:
            got = mg.run_reference(cfg)
        finally:
            mg.seeded_state_dict = orig
        with np.load(os.path.join(ROOT, "tests", "golden", name + ".npz")) as z:
            if "track_sample" in z.files:
                got = mg.take_tracks(got, z["track_sample"])
            worst, flips = 0.0, 0
            for k in got:
                if k.startswith("tracks") or k.startswith("coords"):
                    worst = max(worst, float(np.abs(got[k] - z[k]).max()))
                if k.startswith("visibility"):
                    flips += int((got[k] != z[k]).sum())
        print(f"{name}: weights of {groups} -> {mode}: max |d tracks| = {worst:.2e} px, visibility flips = {flips}", flush=True)


if __name__ == "__main__":
    main()
