"""Evaluation harness (SURVEY 8(f4)): the numpy TAP-Vid metrics against the reference implementation's results
(pinned in tests/golden/reference_units.npz) and, on the GPU, EvaluationPredictor against the reference's
EvaluationPredictor output pinned in a golden."""
import numpy as np
import pytest
import torch

from cases import load_golden
from cotracker_b200.evaluation import EvaluationPredictor, points_on_a_grid, tapvid_metrics
from oracle.make_golden import CENTRED_GRIDS, tapvid_problem


def test_perfect_prediction_scores_one():
    q, occ, gt, _, _ = tapvid_problem(0)
    m = tapvid_metrics(q, occ, gt, occ, gt, "strided")
    assert np.allclose(m["average_jaccard"], 1.0) and np.allclose(m["average_pts_within_thresh"], 1.0)
    assert np.isclose(m["occlusion_accuracy"].sum(), 1.0)      # the reference normalises by the batch total


def test_hand_computed_case():
    # one video, one track, 4 frames, query at frame 0 ("first": frames 1..3 scored)
    q = np.array([[[0.0, 5.0, 5.0]]])
    gt = np.array([[[[5, 5], [6, 5], [7, 5], [8, 5]]]], dtype=np.float64)
    pred = gt + np.array([0, 0.5, 3.0, 20.0])[None, None, :, None] * np.array([1.0, 0.0])
    occ = np.array([[[False, False, False, True]]])
    pocc = np.array([[[False, False, True, False]]])
    m = tapvid_metrics(q, occ, gt, pocc, pred, "first")
    assert np.isclose(m["occlusion_accuracy"][0], 1 / 3)
    assert np.isclose(m["pts_within_1"][0], 0.5) and np.isclose(m["pts_within_4"][0], 1.0)
    # thr 1: TP = frame 1; FP = frame 3 (pred visible, gt occluded) -> 1 / (2 + 1)
    assert np.isclose(m["jaccard_1"][0], 1 / 3)


@pytest.mark.parametrize("mode", ["first", "strided"])
def test_metrics_match_live_reference(mode):
    ref = load_golden("reference_units")
    for seed in range(4):
        prefix = f"tapvid_{mode}{seed}_"
        want = {k[len(prefix):]: v.numpy() for k, v in ref.items() if k.startswith(prefix)}
        got = tapvid_metrics(*tapvid_problem(seed), mode)
        assert set(want) == set(got)
        for k in want:
            assert np.allclose(got[k], want[k], rtol=0, atol=1e-12), k


def test_grid_with_centre_matches_live_reference():
    ref = load_golden("reference_units")
    for i, (size, extent, centre) in enumerate(CENTRED_GRIDS):
        assert torch.equal(points_on_a_grid(size, extent, centre), ref[f"centred_grid{i}"])


@pytest.mark.gpu
@pytest.mark.parametrize("single_point", [True, False])
def test_evaluation_predictor_matches_reference_golden(single_point):
    """tests/golden/eval_predictor.npz: the reference's EvaluationPredictor on a seeded clip (oracle/make_golden.py);
    tracks within 1e-3 px, and the TAP-Vid metrics of B200-vs-reference tracks are exactly 1."""
    from cases import load_golden
    from cotracker_b200.build import build_cotracker
    from oracle.make_golden import eval_case_inputs
    sd, video, queries = eval_case_inputs()
    want = load_golden("eval_predictor")
    model = build_cotracker(None, offline=True, window_len=60).eval()
    model.load_state_dict(sd)
    ev = EvaluationPredictor(model.to("cuda:0"), single_point=single_point, grid_size=5, local_grid_size=8)
    tracks, vis = ev(video.to("cuda:0"), queries.to("cuda:0"))
    key = "single" if single_point else "joint"
    wt, wv = want[f"tracks_{key}"], want[f"vis_{key}"]
    assert float((tracks.cpu() - wt).abs().max()) < 1e-3
    assert float((vis.cpu() - wv).abs().max()) < 1e-3
    q = queries[0].numpy()[None][..., [0, 2, 1]]                                     # (t, y, x)
    # random-init weights give visibility*confidence far below the usual 0.6 cut: threshold in the widest gap around
    # the median of the reference's values, so both classes are populated and no value sits on the threshold
    vals = np.sort(wv.numpy().ravel())
    mid = vals[len(vals) // 4: 3 * len(vals) // 4 + 1]
    i = int(np.argmax(np.diff(mid)))
    thr = 0.5 * (mid[i] + mid[i + 1])
    occ_w = (wv[0].numpy().T < thr)[None]
    occ_g = (vis[0].cpu().numpy().T < thr)[None]
    assert occ_w.any() and not occ_w.all()
    tw = wt[0].permute(1, 0, 2).numpy()[None].astype(np.float64)
    tg = tracks[0].cpu().permute(1, 0, 2).numpy()[None].astype(np.float64)
    m = tapvid_metrics(q, occ_w, tw, occ_g, tg, "first")
    assert m["average_pts_within_thresh"][0] == 1.0 and m["average_jaccard"][0] == 1.0
