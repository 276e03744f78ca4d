"""Two devices driven from ONE process (SURVEY 8(b) threading contract, ADVICE r1): function attributes and the SM
count are per device inside libct3_b200.so, so the same predictor code must work on cuda:1 after cuda:0 has run,
and from two host threads at once.  Needs >= 2 GPUs in one process; skipped on a single-GPU machine."""
import threading

import pytest
import torch

from cases import CASES, compare, load_golden, run_cuda

pytestmark = pytest.mark.gpu

needs2 = pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs in one process")


@needs2
def test_second_device_after_first():
    for dev in ("cuda:0", "cuda:1", "cuda:0"):
        for name in ("predictor_grid", "c2_grid30"):
            compare(run_cuda(name, device=dev), load_golden(name))


@needs2
def test_two_host_threads_two_devices():
    """Two host threads, each driving its own GPU through the same library at the same time.  Weights and inputs are
    built in the main thread (seeded_state_dict seeds torch's GLOBAL generator, which two threads would race on);
    the threads only run the predictor -- concurrently, several times -- and every result must match the golden."""
    from cotracker_b200.predictor import CoTrackerPredictor
    from oracle.make_golden import case_inputs, predictor_kwargs
    name = "c2_grid30_stress"
    cfg = CASES[name]
    sd, video, queries = case_inputs(cfg)
    want = load_golden(name)
    jobs = []
    for i in range(2):
        p = CoTrackerPredictor(checkpoint=None, window_len=cfg["window_len"])
        p.model.load_state_dict(sd)
        jobs.append((p.to(f"cuda:{i}"), video.to(f"cuda:{i}")))
    errs = []

    def work(p, v):
        try:
            for _ in range(3):
                with torch.no_grad():
                    tr, vi = p(v, **predictor_kwargs(cfg, v, queries))
                compare(dict(tracks=tr.cpu(), visibility=vi.cpu()), want)
        except Exception as e:  # noqa: BLE001
            errs.append((str(v.device), repr(e)))

    ts = [threading.Thread(target=work, args=j) for j in jobs]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errs, errs
