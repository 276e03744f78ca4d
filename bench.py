#!/usr/bin/env python
"""bench.py -- headline benchmark: tracked points*frames / second, CoTracker3 offline predictor,
synthetic 512x512x16 video, grid_size=80 (N=6400 tracks), 6 refinement iterations (BASELINE.json `metric`).

    python bench.py --gpus 1 --steps 5 --warmup 3                 # this repo (libct3_b200.so on the B200)
    python bench.py --impl reference --gpus 1 --steps 2 --warmup 1  # CPU arm: the UNMODIFIED reference on the host cores
    python bench.py --grid 30 | --frames 48 | --online --grid 50    # BASELINE.json configs C2 / C3 / C4
    python bench.py --dump-outputs DIR                              # + the last timed step's outputs as DIR/*.npy
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                    # N replicas, one clip per GPU (weak scaling)

One JSON line on stdout (rank 0).  A "step" = one CoTrackerPredictor.forward over one clip; --steps K times exactly K.
  value : whole-job points*frames/s with the clip resident in HBM when the timed region starts
  e2e   : same call with the clip in pinned HOST memory (H2D copy + D2H of tracks/visibility inside the region)
  roofline     : dominant kernel (the tcgen05 split-bf16x3 GEMM) -- algorithmic FLOPs / live CUDA-event time
  roofline_corr: the fused sampling+correlation kernel against the HBM roofline (4.71 GB/iteration, SURVEY 8d)
  cpu_baseline : the reference's own PyTorch-CPU path on a bounded sample of the same workload (rank 0, N=1 only)

--dump-outputs DIR writes what the last timed step (the `value` path) returned on rank 0, tracks.npy and
visibility.npy (float32, visibility as 0/1), so that two builds can be compared output for output: inputs and weights
are seeded, so the same arguments give the same inputs.  Above 64 MB in all, a fixed seeded sample of the tracks is
written instead, with their indices as track_sample.npy.

CPU arm: the unmodified reference package is looked up in $COTRACKER_REFERENCE and baseline/_ref (pip --target
install of the reference; DESIGN.md section 5) and driven through its own CoTrackerPredictor with the shared seeded
state dict ("kind": "reference").  Only when neither exists does the arm fall back to the oracle port ("kind": "port").
Synthetic clip: cotracker_b200.synthetic.texture_video (integer-valued random texture, nearest-upsampled x8,
translated per frame) -- NOT BASELINE.md section 3's bicubic recipe: integer-only construction is bit-identical
on every machine, which the committed full-size goldens (tests/golden/headline_grid80*.npz) rely on.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_FRAMES, SIZE, GRID, ITERS = 16, 512, 80, 6
METRIC = "tracked points*frames/sec at N=6400, T=16, 512^2"
UNIT = "points*frames/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops_sustained"], bf16_burst=d["bf16_tflops"], source="measured")
    return dict(hbm=6650.0, bf16=1400.0, bf16_burst=1590.0, source="fallback")



def usable_cores() -> int:
    """CPU threads this process may actually use: affinity mask and cgroup quota, not the host's core count
    (oversubscribing OpenMP threads in a CPU-limited container is catastrophically slow)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 64))

def find_reference():
    """Directory holding the unmodified reference package (`cotracker/predictor.py`), or None."""
    for p in (os.environ.get("COTRACKER_REFERENCE"), os.path.join(ROOT, "baseline", "_ref")):
        if p and os.path.isfile(os.path.join(p, "cotracker", "predictor.py")):
            return p
    return None


def reference_predictor(ref_dir, sd, online=False):
    """The reference's own predictor (CPU, fp32) with the shared seeded state dict loaded."""
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    import cotracker.predictor as RP
    assert os.path.abspath(RP.__file__).startswith(os.path.abspath(ref_dir)), RP.__file__
    p = (RP.CoTrackerOnlinePredictor(checkpoint=None, window_len=16) if online
         else RP.CoTrackerPredictor(checkpoint=None, window_len=60))
    p.model.load_state_dict(sd)
    return p.eval()


def workload_config(T, G, world, online=False):
    """`config` of the JSON line -- identical for the B200 arm and the CPU reference arm."""
    N = G * G
    if online:
        w = (f"cotracker3_online predictor, synthetic {SIZE}x{SIZE} texture stream, window 16 / step 8, "
             f"grid_size={G} ({N} tracks), 6 iters, one step = one 16-frame chunk (8 new frames), one stream per GPU")
    else:
        w = (f"cotracker3_offline predictor, synthetic {SIZE}x{SIZE}x{T} texture video, grid_size={G} "
             f"({N} tracks), 6 iters, one clip per GPU")
    return {"workload": w, "global_batch": world, "parallelism": f"replicas x{world} (no hot-loop collective)",
            "l2": "no explicit flush: per-step working set of several GB >> 126 MB L2"}


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        if sm:
            # "under load": the upper half of the samples (idle samples sit at the low clock)
            sm_sorted = sorted(sm)
            out["sm_mhz"] = statistics.median(sm_sorted[len(sm_sorted) // 2:])
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        return out


# ---------------------------------------------------------------------------------------------------
def cpu_run(sd, video, G, online, ref_dir):
    """One timed CPU pass of the workload: the unmodified reference if present, else the oracle port.
    Offline: one predictor call.  Online: is_first_step + one 16-frame chunk (the unit bench.py's B200 arm times)."""
    with torch.no_grad():
        if ref_dir:
            p = reference_predictor(ref_dir, sd, online)
            t0 = time.perf_counter()
            if online:
                p(video_chunk=video, is_first_step=True, grid_size=G)
                p(video_chunk=video[:, :16])
            else:
                p(video, grid_size=G)
            return time.perf_counter() - t0
        from oracle import ct3_oracle as O
        t0 = time.perf_counter()
        if online:
            st = O.OnlinePredictorState()
            O.predict_online(sd, st, video, is_first_step=True, grid_size=G)
            O.predict_online(sd, st, video[:, :16])
        else:
            O.predict_offline(sd, video, grid_size=G, iters=ITERS)
        return time.perf_counter() - t0


def bench_reference(args, rank):
    """CPU arm: the reference's own PyTorch-CPU implementation on all usable host cores, on the SAME config as the
    B200 arm (grid/frames as given; default = the headline shape).  One repetition takes 1-2 minutes there, so the
    warm-up runs at grid_size=10; the timed repetitions are exactly `steps`."""
    if rank != 0:
        return
    from cotracker_b200.synthetic import seeded_state_dict, texture_video

    cores = usable_cores()
    torch.set_num_threads(cores)
    ref_dir = find_reference()
    T, G, online = args.frames, args.grid, args.online
    sd = seeded_state_dict(1234, offline=not online, window_len=16 if online else 60)
    video = texture_video(T, SIZE, SIZE, seed=0)
    for _ in range(min(args.warmup, 1)):
        cpu_run(sd, video, 10, online, ref_dir)            # thread pool, allocator, oneDNN primitive caches
    times = [cpu_run(sd, video, G, online, ref_dir) for _ in range(args.steps)]
    ms = 1e3 * sum(times) / len(times)
    units = G * G * (8 if online else T)
    value = units / (ms / 1e3)
    kind = "reference" if ref_dir else "port"
    sample = (f"{'unmodified reference (' + ref_dir + ')' if ref_dir else 'oracle port'}, full workload "
              f"(grid_size={G}, {G * G} tracks, T={T}), {len(times)} timed repetition(s) of {ms / 1e3:.1f} s, "
              f"warm-up at grid_size=10")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": len(times),
        "steps_requested": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(T, G, 1, online),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT = 64 * 10**6 - 4096     # bytes of array data: 64 MB in all with the .npy headers


def dump_outputs(out_dir, outputs):
    """outputs: name -> [B, T, N, ...] tensor of one predictor call; written as out_dir/<name>.npy in float32.  Above
    DUMP_LIMIT bytes in all, only a fixed seeded sample of the N tracks is written, its indices as track_sample.npy."""
    outputs = {k: v.float().cpu() for k, v in outputs.items()}
    n = outputs["tracks"].shape[2]
    per_track = sum(v.numel() * 4 for v in outputs.values()) // n + 8
    if per_track * n > DUMP_LIMIT:
        keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_LIMIT // per_track].sort().values
        outputs = {k: v[:, :, keep] for k, v in outputs.items()}
        outputs["track_sample"] = keep.double()
    os.makedirs(out_dir, exist_ok=True)
    for k, v in outputs.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.numpy())


# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--grid", type=int, default=GRID)
    ap.add_argument("--frames", type=int, default=T_FRAMES)
    ap.add_argument("--online", action="store_true", help="BASELINE config C4: cotracker3_online, window 16 / step 8")
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="library option for A/B runs, e.g. --opt fuse=1 --opt prec.fc1=2 (ct3_set_option)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's tracks and visibility to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        bench_reference(args, rank)
        return

    import torch.distributed as dist

    from cotracker_b200 import engine
    from cotracker_b200.predictor import CoTrackerOnlinePredictor, CoTrackerPredictor
    from cotracker_b200.sharding import broadcast_state_dict
    from cotracker_b200.synthetic import seeded_state_dict, texture_video

    assert torch.cuda.is_available(), "bench.py (impl b200) needs a GPU; there is no CPU fallback"
    for kv in args.opt:
        name, value = kv.split("=")
        engine.set_option(name, int(value))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    T, G, online = args.frames, args.grid, args.online
    N = G * G
    predictor = (CoTrackerOnlinePredictor(checkpoint=None, window_len=16) if online
                 else CoTrackerPredictor(checkpoint=None, window_len=60))
    sd = seeded_state_dict(1234, offline=not online, window_len=16 if online else 60) if rank == 0 else None
    if world > 1:
        # weights travel once, rank 0 -> all, over NCCL/NVLink; no collective in the hot loop (replicas only)
        predictor = predictor.to(dev)
        if rank == 0:
            predictor.model.load_state_dict(sd)
        broadcast_state_dict(predictor.model, src=0)
    else:
        predictor.model.load_state_dict(sd)
        predictor = predictor.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if online:
        # a stream long enough for every call of the run; chunk k = frames [8k, 8k+16): consecutive chunks overlap by 8
        n_calls = 2 * (args.warmup + args.steps) + 4
        stream_host = texture_video(8 * n_calls + 8, SIZE, SIZE, seed=rank).pin_memory()
        stream_dev = stream_host.to(dev)
        pos = [0]

        def restart():
            predictor(video_chunk=stream_dev[:, :16], is_first_step=True, grid_size=G)
            pos[0] = 0

        def run_resident():
            k = pos[0]; pos[0] += 1
            return predictor(video_chunk=stream_dev[:, 8 * k:8 * k + 16])

        def run_e2e():
            k = pos[0]; pos[0] += 1
            tr, vis = predictor(video_chunk=stream_host[:, 8 * k:8 * k + 16].to(dev, non_blocking=True))
            return tr[:, -16:].cpu(), vis[:, -16:].cpu()     # the window this call refined

        restart()
        h2d_bytes = 16 * 3 * SIZE * SIZE * 4
        units_per_step = N * 8                                 # new frames x tracks per call
    else:
        video_host = texture_video(T, SIZE, SIZE, seed=rank).pin_memory()   # one clip per GPU
        video_dev = video_host.to(dev)

        def run_resident():
            return predictor(video_dev, grid_size=G)

        def run_e2e():
            v = video_host.to(dev, non_blocking=True)
            tr, vis = predictor(v, grid_size=G)
            return tr.cpu(), vis.cpu()

        h2d_bytes = video_host.numel() * 4
        units_per_step = N * T

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, out

    for _ in range(args.warmup):
        run_resident()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_step, last = timed(run_resident, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tracks": last[0], "visibility": last[1]})
    for _ in range(1):
        run_e2e()
    ms_e2e, (tr, vis) = timed(run_e2e, args.steps)

    units = units_per_step * world
    value = units / (ms_step / 1e3)
    e2e_value = units / (ms_e2e / 1e3)

    # ---- instrumented step (live CUDA events per kernel category inside the library) -----------------
    engine.profile_enable(True)
    run_resident()
    torch.cuda.synchronize()
    cat_ms, cat_n, gemm_flops = engine.profile_read()
    engine.profile_enable(False)
    pk = peaks()
    prec = engine.precision_summary()
    traffic, traffic_src = {}, None
    for name in ("r2_dram_traffic.json", "r1_dram_traffic.json"):   # ncu-measured DRAM bytes of one headline step
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp) and T == T_FRAMES and G == GRID and not online:
            with open(tp) as f:
                traffic = json.load(f)
            traffic_src = "profiles/" + name + " (ncu --set full capture of this command; NOT measured in this run)"
            break
    gemm_tflops = gemm_flops / (cat_ms["gemm"] / 1e3) / 1e12 if cat_ms["gemm"] > 0 else 0.0
    # SURVEY 8d: pyramid read once (16320 texels/frame at the 384x512 model resolution) + support + coords + volume
    # write; the volume is written with `vol_bytes` bytes per element (4 = split bf16 hi|lo, 2 = single fp16 plane)
    Tw = 16 if online else T
    vol_bytes = prec["volume_bytes_per_element"]
    corr_bytes = ITERS * (Tw * 16320 * 128 * 4 + N * 4 * 49 * 128 * 4 + Tw * N * 8 + Tw * N * 4 * 2401 * vol_bytes)
    corr_gbs = corr_bytes / (cat_ms["corr_sample"] / 1e3) / 1e9 if cat_ms["corr_sample"] > 0 else 0.0
    lib_ms = sum(cat_ms.values())
    # the fused q|k|v projection + time attention kernel: its projection FLOPs over its own time (3 blocks x ITERS calls)
    Tw_rows = (N + 64) * Tw
    qkva_tflops = (ITERS * 3 * 2.0 * Tw_rows * 1152 * 384) / (cat_ms["qkv_time_attention"] / 1e3) / 1e12 \
        if cat_ms.get("qkv_time_attention", 0) > 0 else 0.0

    line = {
        "metric": METRIC if not online else "tracked points*new frames/sec, cotracker3_online, 512^2 stream, step 8",
        "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": prec["dtype"], "data": "synthetic",
        "config": dict(workload_config(T, G, world, online), **({"options": args.opt} if args.opt else {})),
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": tr.numel() * 4 + vis.numel()},
        "gpu_launches": int(sum(cat_n.values())),
        "clocks": clocks,
        "roofline": {"kernel": "gemm_split3_pair_kernel / gemm_split3_tc_kernel (tcgen05, all linear layers)",
                     "bound": "tensor", "achieved": gemm_tflops, "peak": pk["bf16"], "unit": "TFLOP/s",
                     "frac": gemm_tflops / pk["bf16"],
                     "traffic": traffic.get("gemm", {}).get("dram_bytes_per_step"),
                     "traffic_source": traffic_src,
                     "note": "algorithmic fp32-equivalent FLOPs (2*M*N*K per linear layer) / live CUDA-event time of "
                             "the GEMM launches; products per FLOP: " + prec["products"] + "; peak = sustained cuBLAS "
                             "bf16 (" + pk["source"] + ")",
                     "ms_per_step": cat_ms["gemm"], "launches_per_step": cat_n["gemm"]},
        "roofline_corr": {"kernel": "corr_patch_t_kernel (corr_tc3.cu; fused bilinear sampling + 4-D correlation)",
                          "bound": "hbm", "achieved": corr_gbs, "peak": pk["hbm"],
                          "unit": "GB/s", "frac": corr_gbs / pk["hbm"],
                          "traffic": traffic.get("corr_sample", {}).get("dram_bytes_per_step"),
                          "traffic_source": traffic_src,
                          "algorithmic_bytes_per_step": corr_bytes, "volume_bytes_per_element": vol_bytes,
                          "ms_per_step": cat_ms["corr_sample"], "launches_per_step": cat_n["corr_sample"]},
        "roofline_qkv_attention": {"kernel": "gemm_qkv_time_attn_kernel (q|k|v projection + per-track time attention, one "
                                             "kernel)", "bound": "tensor", "achieved": qkva_tflops, "peak": pk["bf16"],
                                   "unit": "TFLOP/s", "frac": qkva_tflops / pk["bf16"],
                                   "note": "projection FLOPs only (the T x T attention runs as fp32 FMA in the epilogue); "
                                           "ncu tensor-pipe active 52 % (profiles/r2_ncu_qkv_time_attn.txt)",
                                   "ms_per_step": cat_ms.get("qkv_time_attention", 0.0)},
        "kernel_ms_per_step": cat_ms, "library_ms_per_step": lib_ms,
    }

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded CPU sample of the same workload through the reference's own PyTorch-CPU path (reported baseline)
        cores = usable_cores()
        torch.set_num_threads(cores)
        ref_dir = find_reference()
        g = min(G, 30 if ref_dir else 20)
        sd_cpu = seeded_state_dict(1234, offline=not online, window_len=16 if online else 60)
        vh = texture_video(24 if online else T, SIZE, SIZE, seed=0)
        cpu_run(sd_cpu, vh[:, :2] if not online else vh, 4, online, ref_dir)   # warm the thread pool
        dt = cpu_run(sd_cpu, vh, g, online, ref_dir)
        line["cpu_baseline"] = {"value": g * g * (8 if online else T) / dt, "unit": UNIT, "cores": cores,
                                "kind": "reference" if ref_dir else "port",
                                "sample": f"{'unmodified reference (' + ref_dir + ')' if ref_dir else 'oracle port'}, "
                                          f"same clip, grid_size={g} ({g * g} of {N} tracks), 6 iters, one full "
                                          f"predictor call, {dt:.1f} s; the full-size CPU run is `--impl reference`"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
