"""CPU tests of the host side: ABI surface, state-dict contract, query construction, replica sharding (gloo)."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from cotracker_b200 import engine
    lib = engine.lib()  # raises if the .so is missing: build it first (__graft_entry__.build)
    header = open(os.path.join(ROOT, "include", "ct3_b200.h")).read()
    declared = set(re.findall(r"\b(ct3_[a-z0-9_]+)\s*\(", header))
    declared -= {"ct3_update_iter"}  # mentioned in a comment only
    assert declared == set(engine.EXPORTED_SYMBOLS), declared ^ set(engine.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.ct3_version() >= 100


def test_abi_argument_validation_without_gpu():
    from cotracker_b200 import engine
    lib = engine.lib()
    n = ctypes.c_size_t(0)
    assert lib.ct3_workspace_bytes(16, 6400, 96, 128, ctypes.byref(n)) == 0 and n.value > 6e9
    assert lib.ct3_workspace_bytes(0, 10, 0, 0, ctypes.byref(n)) == -1          # CT3_EINVAL
    assert b"T and N" in lib.ct3_last_error()
    assert lib.ct3_workspace_bytes(4, 4, 0, 0, None) == -1
    off, h, w, total = engine.pyramid_layout(16, 96, 128)
    assert h == [96, 48, 24, 12] and w == [128, 64, 32, 16] and total == 16 * 16320 * 128
    with pytest.raises(engine.EngineError):
        engine.pyramid_layout(2, 4, 4)                                      # level 3 would be 0x0
    assert lib.ct3_set_option(b"nope", 1) == -1
    assert engine.get_option("gemm") == 0
    assert lib.ct3_update_loop(None, None, 1, 1, None, None, None, None, None, None, 1, 1, 1, None, 0, None) == -1
    # the split-bf16 pyramid copy of the correlation kernel is part of the workspace iff every level is >= 8x8 texels
    *_, total = engine.pyramid_layout(16, 96, 128)
    assert engine.workspace_bytes(16, 6400, 96, 128) - engine.workspace_bytes(16, 6400) == total * 4
    assert engine.workspace_bytes(4, 10, 24, 32) == engine.workspace_bytes(4, 10)       # level 3 is 3x4
    assert lib.ct3_workspace_bytes(4, 10, 4, 4, ctypes.byref(n)) == -1                    # level 3 would be 0x0
    # stage entry: argument checks come before any launch
    one = ctypes.c_void_p(256)
    assert lib.ct3_corr_sample(None, 96, 128, one, None, one, 2, 5, one, None, 0, None) == -1
    assert lib.ct3_corr_sample(one, 96, 128, one, None, one, 2, 5, one, ctypes.c_void_p(264), 1 << 30, None) == -1
    assert b"256-byte aligned" in lib.ct3_last_error()
    assert lib.ct3_corr_sample(one, 96, 128, one, None, one, 2, 5, one, ctypes.c_void_p(512), 1024, None) == -3   # CT3_ENOSPC


def test_weight_names_match_state_dict():
    from cotracker_b200 import engine
    from cotracker_b200.build import build_cotracker
    names = engine.weight_names()
    sd = build_cotracker(None, offline=True, window_len=60).state_dict()
    hot = [k for k in sd if k.startswith(("updateformer.", "corr_mlp."))]
    assert sorted(names) == sorted(hot)
    assert len(names) == 143
    assert sum(sd[k].numel() for k in sd if k != "time_emb") == 25385700      # SURVEY Appendix B
    assert sd["time_emb"].shape == (1, 60, 1110)
    assert "updateformer.virual_tracks" in sd                                   # (sic)


def test_v2_and_training_are_rejected():
    from cotracker_b200.build import build_cotracker
    with pytest.raises(NotImplementedError):
        build_cotracker(None, v2=True)


def test_grid_queries_match_reference_contract():
    from cotracker_b200.predictor import get_points_on_a_grid
    g = get_points_on_a_grid(80, (384, 512))
    assert g.shape == (1, 6400, 2)
    assert float(g[0, :, 0].min()) == 8.0 and float(g[0, :, 0].max()) == 504.0   # margin W/64
    assert float(g[0, :, 1].min()) == 8.0 and float(g[0, :, 1].max()) == 376.0
    assert torch.equal(g[0, 1] - g[0, 0], torch.tensor([g[0, 1, 0] - 8.0, 0.0]))     # row-major, x fastest
    assert get_points_on_a_grid(1, (384, 512)).tolist() == [[[256.0, 192.0]]]


def test_grid_and_time_embedding_match_live_reference():
    """Query grids and sin-cos time embeddings against the reference's (pinned in tests/golden/reference_units.npz)."""
    from cases import load_golden
    from cotracker_b200.model import sincos_time_embedding
    from cotracker_b200.predictor import get_points_on_a_grid
    from oracle.make_golden import UNIT_GRID_SIZES, UNIT_SINCOS_LENGTHS, thin
    ref = load_golden("reference_units")
    for size in UNIT_GRID_SIZES:
        assert torch.equal(get_points_on_a_grid(size, (384, 512)), ref[f"grid{size}"])
    for L in UNIT_SINCOS_LENGTHS:
        assert torch.equal(thin(sincos_time_embedding(1110, L)), ref[f"sincos{L}"])


def test_shard_clips():
    from cotracker_b200.sharding import shard_clips
    assert [shard_clips(8, 8, r) for r in range(8)] == [[r] for r in range(8)]
    assert shard_clips(10, 4, 1) == [1, 5, 9]
    assert sorted(sum((shard_clips(13, 4, r) for r in range(4)), [])) == list(range(13))


_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from cotracker_b200.build import build_cotracker
from cotracker_b200.sharding import broadcast_state_dict, shard_clips, gather_results
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
torch.manual_seed(100 + rank)                      # different random weights per rank before the broadcast
m = build_cotracker(None, offline=False, window_len=16)
sent = broadcast_state_dict(m, src=0)
ref = torch.cat([v.reshape(-1).float() for _, v in sorted(m.state_dict().items())])
chk = ref.clone(); dist.broadcast(chk, src=0)
assert torch.equal(ref, chk), "weights differ after broadcast"
assert sent >= 25385700 * 4
mine = shard_clips(5, world, rank)
tr = torch.full((1, 2, 3, 2), float(rank)); vi = torch.ones(1, 2, 3, dtype=torch.bool)
tl, vl = gather_results(tr, vi, dst=0)
if rank == 0:
    assert [float(t.mean()) for t in tl] == [0.0, 1.0] and all(v.all() for v in vl)
print("OK", rank, mine)
"""


def test_replica_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29613", str(script), ROOT],
                       capture_output=True, text=True, timeout=240, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "OK 0 [0, 2, 4]" in r.stdout and "OK 1 [1, 3]" in r.stdout


def test_corr_patch_taps_stay_in_box():
    """fp32 restatement of box_origin8 / tap_pair (csrc/corr_tc2.cu): for every map size >= 8 and every coordinate --
    far outside, on texel centres, one ulp either side of them -- both bilinear taps of all 7 border-clamped samples
    lie inside the 8-texel box the TMA load fetches, once a zero-weight second tap is folded onto the first (the case
    `c + offset` rounding up to an integer in fp32).  The kernel relies on this to index the box without a fallback."""
    import numpy as np
    f32 = np.float32
    rng = np.random.default_rng(0)
    for size in (8, 9, 12, 16, 24, 48, 96, 128, 1000):
        ints = np.arange(-6, size + 7).astype(f32)
        near = [ints]
        lo, hi = ints.copy(), ints.copy()
        for _ in range(6):
            lo, hi = np.nextafter(lo, f32(-1e9)), np.nextafter(hi, f32(1e9))
            near += [lo.copy(), hi.copy()]
        c = np.concatenate([rng.uniform(-40, size + 40, 100000).astype(f32), np.array([-1e9, 1e9], dtype=f32)] + near)
        cc = np.minimum(np.maximum(c, f32(-16)), f32(size + 16)).astype(f32)
        origin = np.clip(np.floor(cc).astype(np.int64) - 3, 0, size - 8)
        for a in range(7):
            x = np.minimum(np.maximum((c + f32(a - 3)).astype(f32), f32(0)), f32(size - 1)).astype(f32)
            xf = np.floor(x)
            x0 = xf.astype(np.int64)
            w = (x - xf).astype(f32)
            x1 = np.minimum(x0 + 1, size - 1)
            s0 = x0 - origin
            s1 = np.where(w > 0, x1 - origin, s0)
            assert s0.min() >= 0 and s0.max() <= 7 and s1.min() >= 0 and s1.max() <= 7, (size, a)


def test_dropin_package_and_hub_entry_points():
    """The import-path shim (dropin/cotracker/...) and hubconf.py expose the reference's names (INTEGRATION.md 1):
    `from cotracker.predictor import CoTrackerPredictor`, `build_cotracker`, `torch.hub.load(..., source="local")`."""
    code = (
        "import torch, cotracker\n"
        "from cotracker.predictor import CoTrackerPredictor, CoTrackerOnlinePredictor\n"
        "from cotracker.models.build_cotracker import build_cotracker\n"
        "from cotracker.models.core.cotracker.cotracker3_offline import CoTrackerThreeOffline\n"
        "from cotracker.models.core.cotracker.cotracker3_online import CoTrackerThreeOnline\n"
        "import cotracker_b200.predictor as P\n"
        "assert CoTrackerPredictor is P.CoTrackerPredictor and CoTrackerOnlinePredictor is P.CoTrackerOnlinePredictor\n"
        "m = build_cotracker(None, offline=False, window_len=16)\n"
        "assert isinstance(m, CoTrackerThreeOnline) and m.window_len == 16 and m.model_resolution == (384, 512)\n"
        "on = torch.hub.load(%r, 'cotracker3_online', source='local', pretrained=False)\n"
        "off = torch.hub.load(%r, 'cotracker3_offline', source='local', pretrained=False)\n"
        "assert type(on).__name__ == 'CoTrackerOnlinePredictor' and on.step == 8 and on.model.window_len == 16\n"
        "assert type(off).__name__ == 'CoTrackerPredictor' and off.model.window_len == 60 and off.interp_shape == (384, 512)\n"
        "print('HUB_OK')\n" % (ROOT, ROOT))
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "dropin") + os.pathsep + ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=240, env=env, cwd="/tmp")
    assert r.returncode == 0 and "HUB_OK" in r.stdout, r.stdout + r.stderr


def test_non_default_model_resolution_is_rejected():
    """tokens.cu normalises the relative-motion posenc by (128, 96) = (512, 384)/4 (ADVICE r1)."""
    from cotracker_b200.model import CoTrackerThreeOffline
    with pytest.raises(NotImplementedError):
        CoTrackerThreeOffline(window_len=60, model_resolution=(256, 320))


def test_options_are_validated_and_thread_local():
    import threading
    from cotracker_b200 import engine
    lib = engine.lib()
    assert lib.ct3_set_option(b"corr", 7) == -1 and b"out of range" in lib.ct3_last_error()
    assert lib.ct3_set_option(b"attn", -1) == -1
    assert lib.ct3_set_option(b"gemm", 1) == 0 and engine.get_option("gemm") == 1
    seen = []
    t = threading.Thread(target=lambda: seen.append(engine.get_option("gemm")))   # another host thread: defaults
    t.start(); t.join()
    assert seen == [0]
    assert lib.ct3_set_option(b"gemm", 0) == 0


def test_corr_shift_pattern_covers_every_sample():
    """fp32 restatement of box_origin8 / tap_weights (csrc/corr_tc3.cu).  The transposed correlation kernel blends the
    8x8 raw correlations with STATIC register indices: per frame and axis the two taps of sample a are box entries
    clamp07(a + d) and clamp07(a + d + 1) for one shift d = clamp(floor(clamp(c)) - 3 - origin, -7, 7).  This test
    brute-forces, for every map size >= 8 and every coordinate class (far outside, on texel centres, a few ulps either
    side), that the border-clamped bilinear taps of all 7 samples -- computed exactly as grid_sample does -- ARE that
    pattern with weights (1 - w, w), or (0, 1) when c + offset rounded up to an integer; and that the blend value equals
    the straightforward two-tap evaluation.  The kernel traps otherwise; this is the proof that it never does."""
    import numpy as np
    f32 = np.float32
    rng = np.random.default_rng(1)
    for size in (8, 9, 12, 16, 24, 48, 96, 128, 1000):
        ints = np.arange(-20, size + 21).astype(f32)
        near = [ints]
        lo, hi = ints.copy(), ints.copy()
        for _ in range(6):
            lo, hi = np.nextafter(lo, f32(-1e9)), np.nextafter(hi, f32(1e9))
            near += [lo.copy(), hi.copy()]
        c = np.concatenate([rng.uniform(-40, size + 40, 200000).astype(f32), np.array([-1e9, 1e9, 0.5, size - 0.5], dtype=f32)] + near)
        cc = np.minimum(np.maximum(c, f32(-16)), f32(size + 16)).astype(f32)
        base = np.floor(cc).astype(np.int64) - 3
        origin = np.clip(base, 0, size - 8)
        d = np.clip(base - origin, -7, 7)
        box = rng.standard_normal((len(c), 8)).astype(f32)            # the 8 box entries along this axis
        rows = np.arange(len(c))
        for a in range(7):
            x = np.minimum(np.maximum((c + f32(a - 3)).astype(f32), f32(0)), f32(size - 1)).astype(f32)
            xf = np.floor(x)
            x0 = xf.astype(np.int64)
            fr = (x - xf).astype(f32)
            s0 = np.clip(x0 - origin, 0, 7)
            s1 = np.where(fr > 0, np.clip(np.minimum(x0 + 1, size - 1) - origin, 0, 7), s0)
            i0, i1 = np.clip(a + d, 0, 7), np.clip(a + d + 1, 0, 7)
            direct = (s0 == i0) & ((fr == 0) | (s1 == i1))
            rounded = (~direct) & (fr == 0) & (s0 == i1)
            assert bool((direct | rounded).all()), (size, a, c[~(direct | rounded)][:5])
            u = np.where(direct, f32(1) - fr, f32(0)).astype(f32)
            w = np.where(direct, fr, f32(1)).astype(f32)
            want = (f32(1) - fr) * box[rows, s0] + fr * box[rows, s1]
            got = u * box[rows, i0] + w * box[rows, i1]
            assert np.array_equal(want.astype(f32), got.astype(f32)), (size, a)
