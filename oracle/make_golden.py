"""Generate tests/golden/*.npz by running the UNMODIFIED reference (a facebookresearch/co-tracker checkout, given as
$COTRACKER_REFERENCE) on seeded weights and seeded synthetic inputs.  The tests only read the stored files:

    COTRACKER_REFERENCE=<checkout> python oracle/make_golden.py                 # every golden (minutes each for
                                                                                # the BASELINE-scale cases)
    COTRACKER_REFERENCE=<checkout> python oracle/make_golden.py c2_grid30 ...   # selected ones

Only the *outputs* are stored (tiny); weights and inputs are re-created from their seeds by
cotracker_b200.synthetic on whichever machine runs the tests (the one real clip, BASELINE.json config 1's
assets/apple.mp4, travels as a 60x108 area-downsampled uint8 copy of its 50 decoded frames:
tests/golden/apple_frames_60x108.npz, made by `make_apple_fixture()` below).  Cases are listed in CASES below
and are the single source of truth for tests/test_golden*.py.  Predictor cases also store the model's visibility
(and confidence) probabilities -- captured with a forward hook on the unmodified reference model -- so a test
can tell a genuine visibility mismatch from a value sitting on the threshold.  Every golden file stays below 1 MB:
a case whose full output would not keeps a fixed, seeded sample of its tracks (TRACK_SAMPLE), and the stage-level
golden (`reference_units`, make_unit_golden) keeps every k-th element of its larger arrays (`thin`).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cotracker_b200.synthetic import random_queries, seeded_state_dict, texture_video  # noqa: E402


def reference_dir():
    """The reference checkout named by $COTRACKER_REFERENCE, put first on sys.path (generation only)."""
    ref = os.environ.get("COTRACKER_REFERENCE", "")
    if not os.path.isfile(os.path.join(ref, "cotracker", "predictor.py")):
        raise SystemExit("set COTRACKER_REFERENCE to a facebookresearch/co-tracker checkout")
    if ref not in sys.path:
        sys.path.insert(0, ref)
    return ref


# name -> config.  kind: model_offline | model_online_stream | model_online_slide | predictor_offline | predictor_online
CASES = {
    # small feature maps (24x32 ... 3x4): every pyramid level hits the border-clamp path
    "offline_small": dict(kind="model_offline", T=6, H=96, W=128, N=20, iters=3, wseed=1234, vseed=1, qseed=2,
                          head_gain=1.0, vis_gain=1.0, window_len=60),
    # amplified heads: ~10-20 px of motion, vis/conf logits swing (stress regime of SURVEY.md 8c)
    "offline_stress": dict(kind="model_offline", T=8, H=128, W=160, N=24, iters=4, wseed=4321, vseed=3, qseed=4,
                           head_gain=10.0, vis_gain=100.0, window_len=60),
    # T == window_len: no time-embedding interpolation
    "offline_T_eq_window": dict(kind="model_offline", T=8, H=96, W=128, N=12, iters=2, wseed=99, vseed=5, qseed=6,
                                head_gain=3.0, vis_gain=10.0, window_len=8),
    # streaming online model: 3 chunks of a 32-frame video, queries entering in later windows
    "online_stream": dict(kind="model_online_stream", T=32, H=96, W=128, N=18, iters=3, wseed=77, vseed=7, qseed=8,
                          head_gain=5.0, vis_gain=30.0, window_len=16),
    # the online model sliding over a whole video in one call (is_online=False)
    "online_slide": dict(kind="model_online_slide", T=27, H=96, W=128, N=10, iters=2, wseed=78, vseed=9, qseed=10,
                         head_gain=5.0, vis_gain=30.0, window_len=16),
    # public predictor API at the model resolution (384x512 internally), regular grid
    "predictor_grid": dict(kind="predictor_offline", T=4, H=240, W=320, grid=5, iters=6, wseed=5, vseed=11,
                           head_gain=10.0, vis_gain=100.0, window_len=60),
    # public predictor API with explicit queries (adds the 6x6 support grid)
    "predictor_queries": dict(kind="predictor_offline", T=3, H=200, W=256, N=7, iters=6, wseed=6, vseed=12, qseed=13,
                              head_gain=10.0, vis_gain=100.0, window_len=60),
    # online predictor: first step + 2 steps of 16-frame chunks with stride 8
    "predictor_online": dict(kind="predictor_online", T=24, H=192, W=256, grid=4, iters=6, wseed=8, vseed=14,
                             head_gain=5.0, vis_gain=30.0, window_len=16),
    # T > 64: the multi-chunk time-attention path (ADVICE r1), odd T, time-embedding interpolation 60 -> 70
    "offline_long_T": dict(kind="model_offline", T=70, H=64, W=96, N=14, iters=2, wseed=21, vseed=22, qseed=23,
                           head_gain=5.0, vis_gain=30.0, window_len=60),
    # ---- predictor paths (reference predictor.py:70-98, :132-140, :161-164, :192-209, :255-264) --------------
    "pred_segm_mask": dict(kind="predictor_offline", T=4, H=160, W=224, grid=9, mask="box", iters=6, wseed=31,
                           vseed=32, head_gain=10.0, vis_gain=100.0, window_len=60),
    "pred_backward": dict(kind="predictor_offline", T=7, H=144, W=192, N=9, backward=True, iters=6, wseed=33,
                          vseed=34, qseed=35, head_gain=10.0, vis_gain=100.0, window_len=60),
    "pred_grid_query_frame": dict(kind="predictor_offline", T=8, H=144, W=192, grid=6, grid_query_frame=3,
                                  backward=True, iters=6, wseed=36, vseed=37, head_gain=10.0, vis_gain=100.0,
                                  window_len=60),
    "pred_dense": dict(kind="predictor_dense", T=3, H=48, W=160, iters=6, wseed=38, vseed=39, head_gain=10.0,
                       vis_gain=100.0, window_len=60),
    "pred_online_support_grid": dict(kind="predictor_online", T=24, H=160, W=224, N=6, add_support_grid=True,
                                     iters=6, wseed=40, vseed=41, qseed=42, head_gain=5.0, vis_gain=30.0,
                                     window_len=16),
    # ---- BASELINE.json configs at full size (reference CPU run: 16 s ... 2 min each) -------------------------
    # C1: assets/apple.mp4 (50 frames), grid_size=10, the demo.py:92-98 call pattern
    "c1_apple_grid10": dict(kind="predictor_offline", video="apple", grid=10, iters=6, wseed=1234, head_gain=1.0,
                            vis_gain=1.0, window_len=60),
    "c1_apple_grid10_stress": dict(kind="predictor_offline", video="apple", grid=10, iters=6, wseed=1234,
                                   head_gain=10.0, vis_gain=100.0, window_len=60),
    # C2: synthetic 512x512x16, grid_size=30
    "c2_grid30": dict(kind="predictor_offline", T=16, H=512, W=512, grid=30, iters=6, wseed=1234, vseed=0,
                      head_gain=1.0, vis_gain=1.0, window_len=60),
    "c2_grid30_stress": dict(kind="predictor_offline", T=16, H=512, W=512, grid=30, iters=6, wseed=1234, vseed=0,
                             head_gain=10.0, vis_gain=100.0, window_len=60),
    # headline: synthetic 512x512x16, grid_size=80 (N=6400) -- exactly bench.py's workload (same seeds)
    "headline_grid80": dict(kind="predictor_offline", T=16, H=512, W=512, grid=80, iters=6, wseed=1234, vseed=0,
                            head_gain=1.0, vis_gain=1.0, window_len=60),
    "headline_grid80_stress": dict(kind="predictor_offline", T=16, H=512, W=512, grid=80, iters=6, wseed=1234,
                                   vseed=0, head_gain=10.0, vis_gain=100.0, window_len=60),
    # C4: online predictor, 512x512 stream, window 16 / step 8, grid_size=50 (N=2500), 4 steps
    "c4_online_grid50": dict(kind="predictor_online", T=40, H=512, W=512, grid=50, iters=6, wseed=1234, vseed=0,
                             head_gain=5.0, vis_gain=30.0, window_len=16),
}
APPLE_FIXTURE = os.path.join(ROOT, "tests", "golden", "apple_frames_60x108.npz")

# tracks kept in the golden of a case whose full output would exceed 1 MB (C4: 4 steps x up to 40 frames x 2500 tracks)
TRACK_SAMPLE = {"c4_online_grid50": 640}


def track_sample(name, n):
    """The fixed, seeded, sorted subset of the n tracks that the golden of `name` keeps."""
    g = torch.Generator().manual_seed(0)
    return torch.randperm(n, generator=g)[:TRACK_SAMPLE[name]].sort().values


def take_tracks(out, idx):
    """Every output of a predictor case restricted to the tracks `idx` (axis 2 of tracks, visibility, probabilities)."""
    return {k: v[:, :, idx] for k, v in out.items()}


def make_apple_fixture():
    """Decode assets/apple.mp4 (BASELINE.json config 1) and store an area-downsampled uint8 copy."""
    import cv2
    cap, frames = cv2.VideoCapture(os.path.join(reference_dir(), "assets", "apple.mp4")), []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        frames.append(cv2.resize(cv2.cvtColor(f, cv2.COLOR_BGR2RGB), (108, 60), interpolation=cv2.INTER_AREA))
    np.savez_compressed(APPLE_FIXTURE, frames=np.stack(frames))


def box_mask(H, W):
    """[1,1,H,W] segmentation mask: an off-centre rectangle (keeps ~1/3 of a regular grid)."""
    m = torch.zeros(1, 1, H, W)
    m[:, :, H // 5: H // 5 * 4, W // 3: W // 8 * 7] = 1.0
    return m


def case_inputs(cfg):
    offline = cfg["kind"] in ("model_offline", "predictor_offline", "predictor_dense")
    sd = seeded_state_dict(cfg["wseed"], offline=offline, window_len=cfg["window_len"],
                           head_gain=cfg["head_gain"], vis_gain=cfg["vis_gain"])
    if cfg.get("video") == "apple":
        with np.load(APPLE_FIXTURE) as z:
            video = torch.from_numpy(z["frames"]).permute(0, 3, 1, 2)[None].float().contiguous()
        cfg = dict(cfg, T=video.shape[1], H=video.shape[3], W=video.shape[4])
    else:
        video = texture_video(cfg["T"], cfg["H"], cfg["W"], seed=cfg["vseed"])
    queries = None
    if "N" in cfg:
        queries = random_queries(cfg["N"], cfg["T"], cfg["H"], cfg["W"], seed=cfg["qseed"])
    return sd, video, queries


def predictor_kwargs(cfg, video, queries):
    """Keyword arguments of the public predictor call of a case (shared with tests/cases.py)."""
    kw = {}
    if cfg["kind"] == "predictor_dense":
        return kw
    if queries is not None:
        kw["queries"] = queries
    else:
        kw["grid_size"] = cfg["grid"]
    if cfg.get("grid_query_frame"):
        kw["grid_query_frame"] = cfg["grid_query_frame"]
    if cfg["kind"] == "predictor_online":
        if cfg.get("add_support_grid"):
            kw["add_support_grid"] = True
        return kw
    if cfg.get("mask") == "box":
        kw["segm_mask"] = box_mask(video.shape[3], video.shape[4]).to(video.device)
    if cfg.get("backward"):
        kw["backward_tracking"] = True
    return kw


def record_model_outputs(model):
    """Record (vis, conf) of every call of the unmodified reference model (the predictors call model.forward
    directly, so an instance-level wrapper rather than a forward hook)."""
    rec, fwd = [], model.forward

    def wrapped(*a, **k):
        o = fwd(*a, **k)
        rec.append((o[1].clone(), o[2].clone()))
        return o
    model.forward = wrapped
    return rec


def run_reference(cfg):
    reference_dir()
    from cotracker.models.build_cotracker import build_cotracker
    from cotracker.predictor import CoTrackerOnlinePredictor, CoTrackerPredictor

    sd, video, queries = case_inputs(cfg)
    kind = cfg["kind"]
    out = {}
    with torch.no_grad():
        if kind == "model_offline":
            m = build_cotracker(None, offline=True, window_len=cfg["window_len"]).eval()
            m.load_state_dict(sd)
            c, v, q, _ = m(video, queries, iters=cfg["iters"])
            out = dict(coords=c, vis=v, conf=q)
        elif kind == "model_online_slide":
            m = build_cotracker(None, offline=False, window_len=cfg["window_len"]).eval()
            m.load_state_dict(sd)
            c, v, q, _ = m(video, queries, iters=cfg["iters"], is_online=False)
            out = dict(coords=c, vis=v, conf=q)
        elif kind == "model_online_stream":
            m = build_cotracker(None, offline=False, window_len=cfg["window_len"]).eval()
            m.load_state_dict(sd)
            m.init_video_online_processing()
            S = cfg["window_len"]
            for k, ind in enumerate(range(0, cfg["T"] - S // 2, S // 2)):
                c, v, q, _ = m(video[:, ind:ind + S], queries, iters=cfg["iters"], is_online=True)
                out[f"coords{k}"], out[f"vis{k}"], out[f"conf{k}"] = c.clone(), v.clone(), q.clone()
        elif kind in ("predictor_offline", "predictor_dense"):
            p = CoTrackerPredictor(checkpoint=None, window_len=cfg["window_len"])
            p.model.load_state_dict(sd)
            probs = record_model_outputs(p.model)   # (vis, conf) probabilities of every model call, in call order
            tr, vi = p(video, **predictor_kwargs(cfg, video, queries))
            out = dict(tracks=tr, visibility=vi)
            if kind == "predictor_offline":
                out["prob_vis"] = probs[0][0]          # forward pass; support-grid columns still attached
                if cfg.get("backward"):
                    out["prob_vis_inv"] = probs[1][0].flip(1)
        elif kind == "predictor_online":
            p = CoTrackerOnlinePredictor(checkpoint=None, window_len=cfg["window_len"])
            p.model.load_state_dict(sd)
            probs = record_model_outputs(p.model)
            p(video_chunk=video, is_first_step=True, **predictor_kwargs(cfg, video, queries))
            k = 0
            for ind in range(0, video.shape[1] - p.step, p.step):
                tr, vi = p(video_chunk=video[:, ind:ind + p.step * 2],
                           add_support_grid=cfg.get("add_support_grid", False))
                out[f"tracks{k}"], out[f"visibility{k}"] = tr.clone(), vi.clone()
                out[f"prob_visconf{k}"] = probs[k][0] * probs[k][1]
                k += 1
        else:
            raise ValueError(kind)
    return {k: v.numpy() for k, v in out.items()}


def eval_case_inputs():
    """Seeded inputs of the EvaluationPredictor golden (tests/test_evaluation.py)."""
    sd = seeded_state_dict(51, offline=True, window_len=60, head_gain=10.0, vis_gain=100.0)
    video = texture_video(6, 160, 224, seed=52)
    queries = random_queries(5, 6, 160, 224, seed=53)
    return sd, video, queries


def make_eval_golden():
    """reference cotracker/models/evaluation_predictor.py:25-199, single-point (TAP-Vid protocol) and joint mode."""
    reference_dir()
    from cotracker.models.build_cotracker import build_cotracker
    from cotracker.models.evaluation_predictor import EvaluationPredictor
    sd, video, queries = eval_case_inputs()
    m = build_cotracker(None, offline=True, window_len=60).eval()
    m.load_state_dict(sd)
    out = {}
    with torch.no_grad():
        for key, single in (("single", True), ("joint", False)):
            ev = EvaluationPredictor(m, single_point=single, grid_size=5, local_grid_size=8)
            tr, vi = ev(video, queries)
            out[f"tracks_{key}"], out[f"vis_{key}"] = tr.numpy(), vi.numpy()
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "eval_predictor.npz"), **out)
    print("eval_predictor", {k: v.shape for k, v in out.items()})


THIN = 13   # odd and prime to every axis length below: the kept elements cover every row and every channel


def thin(t):
    """Every THIN-th element of `t`, flattened: what reference_units.npz keeps of an array larger than a few KB."""
    return t.reshape(-1)[::THIN]


UNIT_TIME_LENGTHS = (60, 16, 7)     # time-embedding lengths: the stored 60, and two interpolations of it
UNIT_GRID_SIZES = (1, 5, 30)
UNIT_SINCOS_LENGTHS = (16, 60)
CENTRED_GRIDS = ((8, (50, 50), (120.5, 77.25)), (5, (384, 512), None), (1, (384, 512), None))


def unit_inputs():
    """Seeded weights and inputs of the stage-level golden (reference_units.npz; tests/test_oracle_vs_reference.py).
    Amplified heads and correlation volumes x10 reach the regimes where end-to-end parity is blind (e.g. erf vs tanh
    GELU in corr_mlp, SURVEY Appendix A)."""
    sd = seeded_state_dict(2024, offline=True, window_len=60, head_gain=10.0, vis_gain=100.0)
    x = {"updateformer": torch.randn(1, 33, 7, 1110, generator=torch.Generator().manual_seed(1)) * 2}
    g = torch.Generator().manual_seed(2)
    T, N, H, W = 3, 11, 12, 16
    x["corr_fmap"] = torch.randn(1, T, 128, H, W, generator=g)
    x["corr_coords"] = torch.rand(T, N, 2, generator=g) * torch.tensor([W + 4.0, H + 4.0]) - 2.0   # some outside
    x["corr_support"] = torch.randn(1, 49, N, 128, generator=g)
    x["corr_mlp_in"] = torch.randn(T, N, 2401, generator=g) * 10.0     # x10: where erf and tanh GELU differ
    g = torch.Generator().manual_seed(3)
    T, N, H, W = 4, 9, 12, 16
    x["sup_fmap"] = torch.randn(1, T, 128, H, W, generator=g)
    x["sup_qf"] = torch.randint(0, T, (1, N), generator=g)
    x["sup_qc"] = torch.rand(1, N, 2, generator=g) * torch.tensor([W - 1.0, H - 1.0])
    x["posenc"] = torch.randn(5, 3, 4, generator=torch.Generator().manual_seed(4)) * 0.1
    x["encoder"] = texture_video(2, 64, 96, seed=5)[0] / 255 * 2 - 1
    x["video"] = texture_video(5, 64, 96, seed=6)
    x["queries"] = random_queries(9, 5, 64, 96, seed=7)
    return sd, x


def tapvid_problem(seed, b=2, n=17, t=11):
    """Seeded TAP-Vid metric inputs (query_points, gt_occluded, gt_tracks, pred_occluded, pred_tracks)."""
    r = np.random.default_rng(seed)
    q = np.concatenate([r.integers(0, t, (b, n, 1)).astype(np.float64), r.uniform(0, 256, (b, n, 2))], axis=-1)
    gt = r.uniform(0, 256, (b, n, t, 2))
    pred = gt + r.normal(0, 3.0, gt.shape) * (r.uniform(size=(b, n, t, 1)) < 0.7)
    occ = r.uniform(size=(b, n, t)) < 0.3
    pocc = occ ^ (r.uniform(size=(b, n, t)) < 0.2)
    return q, occ, gt, pocc, pred


def make_unit_golden():
    """Stage by stage, the reference on unit_inputs(), plus its query grids, sin-cos embeddings and TAP-Vid metrics."""
    reference_dir()
    from cotracker.evaluation.core.eval_utils import compute_tapvid_metrics
    from cotracker.models.build_cotracker import build_cotracker
    from cotracker.models.core.cotracker.cotracker3_online import posenc
    from cotracker.models.core.embeddings import get_1d_sincos_pos_embed_from_grid
    from cotracker.models.core.model_utils import get_points_on_a_grid
    sd, x = unit_inputs()
    m = build_cotracker(None, offline=True, window_len=60).eval()
    m.load_state_dict(sd)
    out = {}
    with torch.no_grad():
        out["updateformer"] = thin(m.updateformer(x["updateformer"]))
        N = x["corr_coords"].shape[1]
        feat = m.get_correlation_feat(x["corr_fmap"], x["corr_coords"])
        s = x["corr_support"].view(1, 1, 7, 7, N, 128).squeeze(1).permute(0, 3, 1, 2, 4)
        out["corr_volume"] = thin(torch.einsum("btnhwc,bnijc->btnhwij", feat, s))
        out["corr_mlp"] = thin(m.corr_mlp(x["corr_mlp_in"]))
        out["support"] = thin(m.get_track_feat(x["sup_fmap"], x["sup_qf"], x["sup_qc"], support_radius=3)[1][0])
        out["posenc"] = posenc(x["posenc"], 0, 10)
        for t in UNIT_TIME_LENGTHS:
            out[f"time_embed{t}"] = thin(m.interpolate_time_embed(torch.zeros(1, t, 1110), t))
        out["encoder"] = thin(m.fnet(x["encoder"]))
        out["coords"], out["vis"], _, _ = m(x["video"], x["queries"], iters=3)
    for size in UNIT_GRID_SIZES:
        out[f"grid{size}"] = get_points_on_a_grid(size, (384, 512))
    for L in UNIT_SINCOS_LENGTHS:
        pos = torch.linspace(0, L - 1, L).reshape(1, L, 1)[0]
        out[f"sincos{L}"] = thin(get_1d_sincos_pos_embed_from_grid(1110, pos))
    for i, (size, extent, centre) in enumerate(CENTRED_GRIDS):
        out[f"centred_grid{i}"] = get_points_on_a_grid(size, extent, centre)
    for mode in ("first", "strided"):
        for seed in range(4):
            for k, v in compute_tapvid_metrics(*tapvid_problem(seed), mode).items():
                out[f"tapvid_{mode}{seed}_{k}"] = v
    path = os.path.join(ROOT, "tests", "golden", "reference_units.npz")
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in out.items()})
    print("reference_units", len(out), "arrays", os.path.getsize(path), "bytes")


def main():
    import time
    os.makedirs(os.path.join(ROOT, "tests", "golden"), exist_ok=True)
    if not os.path.exists(APPLE_FIXTURE):
        make_apple_fixture()
    names = sys.argv[1:] or (list(CASES) + ["eval_predictor", "reference_units"])
    if "eval_predictor" in names:
        names.remove("eval_predictor")
        make_eval_golden()
    if "reference_units" in names:
        names.remove("reference_units")
        make_unit_golden()
    for name in names:
        cfg = CASES[name]
        t0 = time.perf_counter()
        out = run_reference(cfg)
        print(f"{name}: reference ran {time.perf_counter() - t0:.1f} s")
        if name in TRACK_SAMPLE:
            idx = track_sample(name, out[next(iter(out))].shape[2]).numpy()
            out = dict(take_tracks(out, idx), track_sample=idx)
        path = os.path.join(ROOT, "tests", "golden", name + ".npz")
        np.savez_compressed(path, **out)
        print(name, {k: v.shape for k, v in out.items()}, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
