"""Shared case runners: the same seeded case through (a) the CPU oracle, (b) the CUDA product path."""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ct3_oracle as O  # noqa: E402  (tests may use the oracle; product code may not)
from oracle.make_golden import CASES, case_inputs, predictor_kwargs, take_tracks  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def load_golden(name):
    with np.load(os.path.join(GOLDEN_DIR, name + ".npz")) as z:
        return {k: torch.from_numpy(z[k]) for k in z.files}


def golden_view(got, want):
    """(got, want) on the tracks the golden keeps: all of them, or the fixed sample stored as `track_sample`."""
    if "track_sample" not in want:
        return got, want
    want = dict(want)
    return take_tracks(got, want.pop("track_sample")), want


def run_oracle(name):
    cfg = CASES[name]
    sd, video, queries = case_inputs(cfg)
    kind = cfg["kind"]
    with torch.no_grad():
        if kind == "model_offline":
            c, v, q = O.offline_forward(sd, video, queries, iters=cfg["iters"])
            return dict(coords=c, vis=v, conf=q)
        if kind == "model_online_slide":
            c, v, q = O.online_forward(sd, None, video, queries, iters=cfg["iters"], window_len=cfg["window_len"])
            return dict(coords=c, vis=v, conf=q)
        if kind == "model_online_stream":
            st, out, S = O.OnlineState(), {}, cfg["window_len"]
            for k, ind in enumerate(range(0, cfg["T"] - S // 2, S // 2)):
                c, v, q = O.online_forward(sd, st, video[:, ind:ind + S], queries, iters=cfg["iters"], window_len=S,
                                           is_online=True)
                out[f"coords{k}"], out[f"vis{k}"], out[f"conf{k}"] = c.clone(), v.clone(), q.clone()
            return out
        if kind in ("predictor_offline", "predictor_dense"):
            tr, vi = O.predict_offline(sd, video, **predictor_kwargs(cfg, video, queries))
            return dict(tracks=tr, visibility=vi)
        if kind == "predictor_online":
            st, out, step = O.OnlinePredictorState(), {}, cfg["window_len"] // 2
            O.predict_online(sd, st, video, is_first_step=True, window_len=cfg["window_len"],
                             **predictor_kwargs(cfg, video, queries))
            for k, ind in enumerate(range(0, video.shape[1] - step, step)):
                tr, vi = O.predict_online(sd, st, video[:, ind:ind + 2 * step], window_len=cfg["window_len"],
                                          add_support_grid=cfg.get("add_support_grid", False))
                out[f"tracks{k}"], out[f"visibility{k}"] = tr.clone(), vi.clone()
            return out
    raise ValueError(kind)


def run_cuda(name, device="cuda:0"):
    """The product path: cotracker_b200 models / predictors on the GPU (libct3_b200.so)."""
    from cotracker_b200.build import build_cotracker
    from cotracker_b200.predictor import CoTrackerOnlinePredictor, CoTrackerPredictor

    cfg = CASES[name]
    sd, video, queries = case_inputs(cfg)
    kind = cfg["kind"]
    video = video.to(device)
    if queries is not None:
        queries = queries.to(device)
    out = {}
    with torch.no_grad():
        if kind in ("model_offline", "model_online_slide", "model_online_stream"):
            m = build_cotracker(None, offline=(kind == "model_offline"), window_len=cfg["window_len"]).eval()
            m.load_state_dict(sd)
            m = m.to(device)
            if kind == "model_offline":
                c, v, q, _ = m(video, queries, iters=cfg["iters"])
                out = dict(coords=c, vis=v, conf=q)
            elif kind == "model_online_slide":
                c, v, q, _ = m(video, queries, iters=cfg["iters"], is_online=False)
                out = dict(coords=c, vis=v, conf=q)
            else:
                m.init_video_online_processing()
                S = cfg["window_len"]
                for k, ind in enumerate(range(0, cfg["T"] - S // 2, S // 2)):
                    c, v, q, _ = m(video[:, ind:ind + S], queries, iters=cfg["iters"], is_online=True)
                    out[f"coords{k}"], out[f"vis{k}"], out[f"conf{k}"] = c.clone(), v.clone(), q.clone()
        elif kind in ("predictor_offline", "predictor_dense"):
            p = CoTrackerPredictor(checkpoint=None, window_len=cfg["window_len"])
            p.model.load_state_dict(sd)
            p = p.to(device)
            tr, vi = p(video, **predictor_kwargs(cfg, video, queries))
            out = dict(tracks=tr, visibility=vi)
        elif kind == "predictor_online":
            p = CoTrackerOnlinePredictor(checkpoint=None, window_len=cfg["window_len"])
            p.model.load_state_dict(sd)
            p = p.to(device)
            p(video_chunk=video, is_first_step=True, **predictor_kwargs(cfg, video, queries))
            k = 0
            for ind in range(0, video.shape[1] - p.step, p.step):
                tr, vi = p(video_chunk=video[:, ind:ind + p.step * 2],
                           add_support_grid=cfg.get("add_support_grid", False))
                out[f"tracks{k}"], out[f"visibility{k}"] = tr.clone(), vi.clone()
                k += 1
        else:
            raise ValueError(kind)
    return {k: v.cpu() for k, v in out.items()}


THRESHOLD_BAND = 2e-4   # |probability - threshold| below which a boolean flip is rounding, not a defect


def _threshold_margin(want, k):
    """Distance of the REFERENCE's own probabilities from the decision threshold for the boolean output `k`
    (stored next to the booleans by oracle/make_golden.py); None when the fixture carries no probabilities."""
    n = want[k].shape[-1]
    if k == "visibility" and "prob_vis" in want:
        m = (want["prob_vis"][..., :n] - 0.9).abs()
        if "prob_vis_inv" in want:   # backward tracking: either pass may have produced the value
            m = torch.minimum(m, (want["prob_vis_inv"][..., :n] - 0.9).abs())
        return m
    if k.startswith("visibility") and ("prob_visconf" + k[len("visibility"):]) in want:
        return (want["prob_visconf" + k[len("visibility"):]][..., :n] - 0.6).abs()
    return None


def compare(got, want, tol_px=1e-3, tol_logit=1e-3):
    """pred_tracks within tol_px (north-star: 1e-3 abs), vis/conf within tol_logit, bool visibility exact: every
    mismatch must sit where the reference's own probability is within THRESHOLD_BAND of the threshold (reported
    as `<key>_on_threshold`; 0 in every committed fixture run so far), anything else fails."""
    report = {}
    got, want = golden_view(got, want)
    for k, w in want.items():
        if k.startswith("prob_"):
            continue
        g = got[k]
        assert g.shape == w.shape, (k, g.shape, w.shape)
        if w.dtype == torch.bool:
            bad = g != w
            margin = _threshold_margin(want, k)
            if margin is not None and bool(bad.any()):
                report[k + "_on_threshold"] = int((bad & (margin < THRESHOLD_BAND)).sum())
                bad = bad & ~(margin < THRESHOLD_BAND)
            report[k] = int(bad.sum())
            assert report[k] == 0, f"{k}: {report[k]} visibility mismatches"
        else:
            err = float((g.float() - w.float()).abs().max())
            report[k] = err
            tol = tol_px if ("coords" in k or "tracks" in k) else tol_logit
            assert err <= tol, f"{k}: max abs err {err:.3e} > {tol:.1e}"
    return report
