"""Host-side logic: problem containers, synthetic scenes, pair sharding, the pybundle-style
API's bookkeeping, and the N>1 plumbing on gloo (world_size 2, CPU)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from opensfm_b200 import ba_problem as bp
from opensfm_b200 import bundle, matching, synthetic as syn
from opensfm_b200 import types as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_cube_scene_is_deterministic_and_shaped():
    a = syn.cube_scene(5, 300, 1.0)
    b = syn.cube_scene(5, 300, 1.0)
    assert np.array_equal(a.obs_xy, b.obs_xy) and np.array_equal(a.track_descriptors, b.track_descriptors)
    assert a.track_descriptors.dtype == np.float32 and a.track_descriptors.shape == (300, 128)
    assert ((a.track_descriptors == np.round(a.track_descriptors)).all() and a.track_descriptors.max() <= 255)
    assert (np.count_nonzero(a.track_descriptors, axis=1) <= 5).all()
    # every camera sits on the r=2 sphere and looks at the origin
    assert np.allclose(np.linalg.norm(a.origins, axis=1), 2.0)
    for s in range(5):
        assert np.allclose(a.R_wc[s] @ (-a.origins[s]) / 2.0, [0, 0, 1], atol=1e-12)
    assert np.abs(a.obs_xy[:, 0]).max() < 0.5 + 0.01 and np.abs(a.obs_xy[:, 1]).max() < 0.375 + 0.01


def test_thinned_visibility_is_exact():
    sc = syn.cube_scene(30, 500, 1.0, with_descriptors=False, max_obs_per_point=10)
    counts = np.bincount(sc.obs_point, minlength=500)
    assert counts.max() == 10


def test_problem_validation_and_offsets():
    sc = syn.cube_scene(4, 100, 1.0, with_descriptors=False)
    pb = syn.scene_to_problem(sc)
    assert list(pb.cam_off) == [0, 3, 6, 9, 12]
    assert pb.loss_name == "SoftLOneLoss" and pb.max_iterations == 100
    assert np.allclose(pb.cam_prior_sigma, 0.01) and list(pb.cam_prior_log[:3]) == [0, 0, 1]
    pb.obs_point[0] = 10 ** 6
    with pytest.raises(AssertionError):
        pb.validate()


def test_default_sigma_follows_reference_map():
    # k4..k6, s0..s3 read a default-inserted 0 (bundle_adjuster.cc:46-67)
    s = bp.default_prior_sigma(bp.FISHEYE624)
    names = bp.CAMERA_PARAM_NAMES[bp.FISHEYE624]
    assert [s[names.index(n)] for n in ("k1", "k2", "k3", "p1", "focal", "cx")] == [1.0] * 6
    assert [s[names.index(n)] for n in ("k4", "k5", "k6", "s0", "s3")] == [0.0] * 5


def test_pose_conversion_roundtrip():
    rng = np.random.RandomState(0)
    p = T.Pose(rng.normal(0, 1, 3), rng.normal(0, 1, 3))
    q = T.Pose.from_ba_params(p.to_ba_params())
    assert np.allclose(p.rotation, q.rotation) and np.allclose(p.translation, q.translation)
    assert np.allclose(p.to_ba_params()[3:], p.get_origin())


def test_camera_factories_follow_camera_cc_order():
    c = T.Camera.create_brown(0.4, 1.0, [0.1, -0.05], [-0.1, 0.03, 0.001, 0.001, 0.002])
    assert c.get_parameters_types() == ["k1", "k2", "k3", "p1", "p2", "focal", "aspect_ratio", "cx", "cy"]
    assert c.focal == 0.4 and c.cy == -0.05 and c.k3 == 0.001
    assert T.Camera.create_spherical().get_parameters_values().tolist() == [0.0]
    assert T.Camera.create_dual(0.5, 0.4, 0.1, 0.2).get_parameters_values().tolist() == [0.5, 0.1, 0.2, 0.4]


def test_bundle_adjuster_bookkeeping_without_gpu():
    ba = bundle.BundleAdjuster()
    cam = T.Camera.create_perspective(0.4, 0.1, -0.01)
    ba.add_camera("A\xb2", cam, cam, True)      # unicode id (test_bundle.py:20-34)
    ba.add_camera(b"A_2", cam, cam, True)       # bytes id
    ba.add_camera("cam1", cam, cam, False)
    ba.add_rig_camera("rc", T.Pose(), T.Pose(), True)
    ba.add_rig_instance("1", T.Pose([0.5, 0, 0], [0, 0, 0]), {"s1": "cam1"}, {"s1": "rc"}, False)
    ba.add_point("p", [0, 0, 5.0], False)
    ba.add_point_projection_observation("s1", "p", [0.01, 0.02], 0.004)
    with pytest.raises(RuntimeError, match="doesn't exist"):
        ba.add_rig_instance("2", T.Pose(), {"s2": "missing"}, {"s2": "rc"}, False)
    with pytest.raises(IndexError):
        ba.add_point_projection_observation("s1", "missing", [0, 0], 1.0)
    pb = ba.to_problem()
    assert pb.num_observations == 1 and pb.shot_use_rc.tolist() == [0]  # identity fixed rig camera is not useful
    assert pb.loss_name == "CauchyLoss" and pb.max_iterations == 500      # bundle_adjuster.cc:24-44
    assert pb.cam_const.tolist() == [1, 1, 0]
    assert ba.has_point("p") and not ba.has_point("q")
    assert np.allclose(ba.get_rig_instance_pose("1").rotation, [0.5, 0, 0])
    # secondary residuals become side terms of the problem (bundle_adjuster.cc:956-971); std <= 0 adds nothing
    ba.add_absolute_up_vector("s1", [0, 0, -2.0], 1e-3)
    ba.add_absolute_pan("s1", 0.3, 0.0)
    pb = ba.to_problem()
    assert [t.type for t in pb.side_terms] == [bp.SIDE_UP_VECTOR]
    assert np.allclose(pb.side_terms[0].consts, [0, 0, -1, 1e3]) and pb.side_terms[0].loss == bp.LOSS_CAUCHY
    with pytest.raises(RuntimeError, match="already exist"):
        ba.add_rig_camera("rc", T.Pose(), T.Pose(), True)   # bundle_adjuster.cc:155-158
    with pytest.raises(NotImplementedError):
        ba.add_heatmap("h", [0.0] * 16, 4, 1.0)


def test_shard_pairs_balances_work():
    sizes = {i: 1000 + 100 * i for i in range(12)}
    pairs = [(i, j) for i in range(12) for j in range(i + 1, 12)]
    shards = matching.shard_pairs(pairs, sizes, 4)
    assert sorted(p for s in shards for p in s) == sorted(pairs)
    loads = [sum(sizes[a] * sizes[b] for a, b in s) for s in shards]
    assert max(loads) / min(loads) < 1.1


GLOO_WORKER = r"""
import os, sys, ctypes
import numpy as np
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
from opensfm_b200 import dist as odist, matching
rank, world, _ = odist.init_from_env("gloo")
assert world == 2
# all-reduce on a raw host pointer, as the BA library calls it
buf = np.arange(6, dtype=np.float64) * (rank + 1)
ar = odist.make_allreduce()
ar(buf.ctypes.data, 6, 0)
assert np.allclose(buf, np.arange(6) * 3.0), buf
# pair sharding + host gather
pairs = [(i, j) for i in range(5) for j in range(i + 1, 5)]
sizes = {i: 100 + i for i in range(5)}
mine = matching.shard_pairs(pairs, sizes, world)[rank]
local = {p: np.array([[p[0], p[1]]]) for p in mine}
allr = odist.gather_pair_results(local, world)
assert sorted(allr) == sorted(pairs)
dist.barrier()
if rank == 0:
    print("GLOO_OK")
"""


def test_world_size_2_gloo_plumbing(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER % {"root": ROOT})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29617", str(script)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "GLOO_OK" in out.stdout


def test_split_match_lists_matches_the_per_pair_loop():
    from opensfm_b200.matching import split_match_lists

    rng = np.random.default_rng(3)
    assert split_match_lists(np.zeros(0, np.int32), np.zeros(0, np.int64)) == []
    for _ in range(200):
        npairs = int(rng.integers(1, 7))
        counts = rng.integers(0, 9, size=npairs).astype(np.int64)
        raw = rng.integers(-1, 6, size=int(counts.sum())).astype(np.int32)
        parts = split_match_lists(raw, counts)
        assert len(parts) == npairs
        off = 0
        for n, got in zip(counts, parts):
            idx = raw[off:off + n]
            off += n
            q = np.nonzero(idx >= 0)[0]
            want = np.stack([q, idx[q]], axis=1).astype(np.int64) if len(q) else np.zeros((0, 2), dtype=np.int64)
            assert got.dtype == np.int64 and got.shape == want.shape and np.array_equal(got, want)


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm: oracle port for BA, cv2 for MATCH) needs no GPU."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--workload", "tiny",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["higher_is_better"] is True
    for key in ("metric", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config", "e2e",
                "cpu_baseline"):
        assert key in line, key
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["kind"] in ("port", "reference")
    assert line["match"]["value"] > 0


def test_unfilter_matches_follows_the_reference():
    m1 = np.array([1, 0, 1, 1, 0, 1], dtype=bool)
    m2 = np.array([0, 1, 1, 0, 1], dtype=bool)
    matches = np.array([[0, 2], [3, 0], [1, 1]])
    # reference: [(flatnonzero(m1)[a], flatnonzero(m2)[b])] (matching.py:932-936)
    i1, i2 = np.flatnonzero(m1), np.flatnonzero(m2)
    want = np.array([(i1[a], i2[b]) for a, b in matches])
    assert np.array_equal(matching.unfilter_matches(matches, m1, m2), want)
    assert matching.unfilter_matches(np.zeros((0, 2)), m1, m2).shape == (0, 2)


def test_bench_submodel_workload_host_logic(monkeypatch):
    """bench.py run_c5 (BASELINE configs[4] stand-in) with the GPU calls stubbed out: the four sub-problems and the
    alignment problem it builds are valid, every shot is added once and constrained once per submodel it belongs to."""
    import importlib
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    bench = importlib.import_module("bench")
    from opensfm_b200 import alignment, bundle

    seen = {"solve": 0, "problems": []}

    def fake_solve(pb, **kw):
        pb.validate()
        seen["solve"] += 1
        return {"inst": pb.inst.copy(), "summary": {"iterations": 5, "time_device_ms": 1.0}}

    def fake_run(self):
        pb = self.to_problem()
        pb.validate()
        seen["problems"].append((len(pb.inst), len(pb.ext_size), len(pb.side_terms)))

    monkeypatch.setattr(bundle, "solve", fake_solve)
    monkeypatch.setattr(alignment.ReconstructionAlignment, "run", fake_run)
    monkeypatch.setattr(alignment.ReconstructionAlignment, "brief_report", lambda self: "stub")
    out = bench.run_c5("c2")
    cams = [m["cameras"] for m in out["submodels"]]
    assert cams == [14, 14, 15, 13] and seen["solve"] == 8            # warm-up + timed solve per submodel
    assert seen["problems"] == [(50, 4, 50 + sum(cams))] * 2          # 50 GPS terms + one relative motion per (submodel, shot)
    assert out["alignment_terms"] == 50 + sum(cams)


def _bench():
    import importlib

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    return importlib.import_module("bench")


def test_bench_dump_outputs_layout_and_sample(tmp_path):
    """bench.dump_outputs: float64 .npy files, matches tagged with their pair in pair-list order, and a sample of the
    outgrown outputs that depends on the row count only."""
    bench = _bench()
    rng = np.random.default_rng(1)
    pairs = [(0, 1), (0, 2), (1, 2)]
    lists = {(0, 1): np.array([[0, 3], [2, 1]], np.int32), (0, 2): np.zeros((0, 2), np.int32),
             (1, 2): np.array([[5, 4]], np.int32)}
    ba = {"summary": {"initial_cost": 2.0, "final_cost": 1.0, "iterations": 7}, "points": rng.normal(size=(4, 3)),
          "inst": rng.normal(size=(3, 6)), "rigcam": np.zeros((1, 6)), "cam_params": rng.normal(size=9),
          "reprojection_errors": rng.normal(size=(10, 3))}
    names = bench.dump_outputs(str(tmp_path / "out"), ba, lists, pairs)
    got = {n: np.load(str(tmp_path / "out" / (n + ".npy"))) for n in names}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["ba_summary"].tolist() == [2.0, 1.0, 7.0]
    assert np.array_equal(got["ba_points"], ba["points"]) and np.array_equal(got["ba_cam_params"], ba["cam_params"])
    assert np.array_equal(got["ba_reprojection_errors"], ba["reprojection_errors"])
    assert got["match_counts"].tolist() == [2, 0, 1]
    assert got["matches"].tolist() == [[0, 1, 0, 3], [0, 1, 2, 1], [1, 2, 5, 4]]

    keep = bench.sample_rows(1000, 100)
    assert len(keep) == 100 and np.all(np.diff(keep) > 0) and keep[-1] < 1000
    assert np.array_equal(keep, bench.sample_rows(1000, 100))
    assert np.array_equal(bench.sample_rows(50, 100), np.arange(50))


def test_bench_rejects_zero_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                         text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_timed_results(tmp_path):
    """`bench.py --dump-outputs` writes what the timed steps computed: the BA solution and the match lists the public
    API returns for the same workload."""
    import json

    from opensfm_b200 import matching

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "2",
                          "--warmup", "1", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == 2
    bench = _bench()
    pb, feats, pairs, _ = bench.build_workload("tiny")
    got = {f[:-4]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    ref = bundle.solve(pb)
    assert got["ba_summary"][2] == ref["summary"]["iterations"]
    assert abs(got["ba_summary"][1] - ref["summary"]["final_cost"]) <= 1e-12 * ref["summary"]["final_cost"]
    assert np.abs(got["ba_points"] - ref["points"]).max() < 1e-9
    assert np.abs(got["ba_reprojection_errors"] - ref["reprojection_errors"]).max() < 1e-9
    pm = matching.PairMatcher()
    pm.add_many([(i, f.astype(np.uint8)) for i, f in enumerate(feats)], uint8_is_l2=True)
    lists = pm.match_pairs(pairs, {"lowes_ratio": 0.8})
    assert got["match_counts"].tolist() == [len(lists[p]) for p in pairs]
    want = np.concatenate([np.column_stack([np.tile(p, (len(lists[p]), 1)), lists[p]]) for p in pairs])
    assert np.array_equal(got["matches"], want)
