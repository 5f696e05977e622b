"""GPU parity of the bundle-adjustment engine against the oracle (restated Ceres path)."""
import numpy as np
import pytest

from oracle import ba_lm as oracle
from opensfm_b200 import ba_problem as bp
from opensfm_b200 import bundle, synthetic as syn
from opensfm_b200 import types as T

pytestmark = pytest.mark.gpu

POINT = [1.0, 2.0, 3.0]
RT = [0.1, 0.2, 0.3, 0.4, 0.5, 0.6]
OBS = [0.5, 0.5]
SIGMA = 10.0  # scale 0.1 in the reference test
# opensfm/src/bundle/test/reprojection_errors_test.cc:114-174
CAMS = {
    bp.BROWN: [0.3, 1.0, 0.001, -0.02, 0.1, -0.03, 0.001, -0.005, 0.001],
    bp.PERSPECTIVE: [0.3, 0.1, -0.03],
    bp.FISHEYE: [0.3, 0.1, -0.03],
    bp.FISHEYE_OPENCV: [0.3, 1.0, 0.001, -0.02, 0.1, -0.03, 0.001, -0.005],
    bp.FISHEYE62: [0.3, 1.0, 0.001, -0.02, 0.1, -0.03, 0.001, -0.005, 0.01, 0.006, 0.02, 0.003],
    bp.FISHEYE624: [0.3, 1.0, 0.001, -0.02, 0.1, -0.03, 0.001, -0.005, 0.01, 0.006, 0.02, 0.003, 0.001, -0.009,
                    -0.01, 0.03],
    bp.DUAL: [0.5, 0.3, 0.1, -0.03],
    bp.RADIAL: [0.1, -0.03, 0.3, 1.0, 0.001, -0.02],
    bp.SIMPLE_RADIAL: [0.1, 0.3, 1.0, 0.001, -0.02],
    bp.SPHERICAL: [0.0],
}


@pytest.mark.parametrize("ptype", sorted(CAMS))
@pytest.mark.parametrize("use_rc", [True, False])
def test_device_jacobian_matches_autodiff_on_reference_vectors(ptype, use_rc):
    """Same inputs and tolerance (1e-14) as the reference's analytic-vs-autodiff tests."""
    got = bundle.eval_observation(ptype, CAMS[ptype], RT, RT, use_rc, POINT, OBS, SIGMA)
    ref = oracle.reprojection(ptype, CAMS[ptype], RT, RT, use_rc, POINT, OBS, SIGMA, autodiff=True)
    for g, r in zip(got, ref):
        if not use_rc and g.shape == (r.shape[0], 6) and np.all(r == 0):
            continue
        assert np.abs(g - r).max() < 1e-14


def _compare(pb, tol_cost=1e-6, tol_param=2e-5, compare_params=True, tol_rmse=1e-6):
    ref = oracle.solve(pb)
    got = bundle.solve(pb)
    s = got["summary"]
    assert s["termination"] == "CONVERGENCE", s
    assert abs(s["initial_cost"] - ref["initial_cost"]) <= 1e-9 * ref["initial_cost"]
    assert abs(s["final_cost"] - ref["final_cost"]) <= tol_cost * ref["final_cost"], (s, ref["final_cost"])
    rm_ref = np.sqrt((ref["reprojection_errors"] ** 2).sum(1).mean())
    rm_got = np.sqrt((got["reprojection_errors"] ** 2).sum(1).mean())
    assert abs(rm_ref - rm_got) <= tol_rmse * rm_ref
    if not compare_params:
        return ref, got
    assert np.abs(got["points"] - ref["points"]).max() < tol_param
    assert np.abs(got["inst"] - ref["inst"]).max() < tol_param
    assert np.abs(got["cam_params"] - ref["cam_params"]).max() < tol_param
    return ref, got


def test_cube_scene_small_matches_oracle():
    sc = syn.cube_scene(10, 1000, 1.0, with_descriptors=False)
    _compare(syn.scene_to_problem(sc))


def test_cube_scene_shared_intrinsics_and_fixed_cameras():
    sc = syn.cube_scene(8, 600, 1.0, with_descriptors=False)
    _compare(syn.scene_to_problem(sc, shared_intrinsics=True))
    _compare(syn.scene_to_problem(sc, optimize_cameras=False))


@pytest.mark.parametrize("loss", ["TrivialLoss", "HuberLoss", "CauchyLoss", "ArctanLoss"])
def test_losses(loss):
    sc = syn.cube_scene(6, 300, 2.0, with_descriptors=False)
    # ArctanLoss saturates: the cost is flat along the (free) similarity gauge, so two solvers agree on
    # cost / reprojection RMSE but may stop at different gauge representatives.
    # (6 cameras without GPS: the similarity gauge is free, so the two solvers' iterates drift along it by a few
    # 1e-5 when they stop on the function tolerance; 5e-5 like the other gauge-free scenes)
    # ArctanLoss (non-convex, 48 iterations until the 1e-6 function tolerance stops both solvers): the two final
    # costs agree to a few times that tolerance, not better -- a different summation order in the Schur kernel
    # moves the last digits of every iterate.
    _compare(syn.scene_to_problem(sc, loss_name=loss, loss_threshold=1.0), compare_params=loss != "ArctanLoss",
             tol_rmse=1e-5 if loss == "ArctanLoss" else 1e-6, tol_param=5e-5,
             tol_cost=5e-6 if loss == "ArctanLoss" else 1e-6)


def test_async_observation_upload_gives_the_same_solve():
    """pinned_inputs=True: image coordinates / standard deviations travel on a copy stream while run() sorts the indices
    (osfm_ba_set_observations_async); with page-locked and with pageable arrays the solve is the one of the default path."""
    import torch

    sc = syn.cube_scene(10, 1000, 1.0, with_descriptors=False)
    pb = syn.scene_to_problem(sc)
    ref = bundle.solve(pb)
    got = bundle.solve(pb, pinned_inputs=True)   # pageable: the driver stages the copies
    # (not bit-equal: the fp64 atomics of the Schur flush land in a different order from run to run)
    assert abs(got["summary"]["final_cost"] - ref["summary"]["final_cost"]) <= 1e-12 * ref["summary"]["final_cost"]
    for name in ("obs_shot", "obs_point", "obs_xy", "obs_sigma"):
        setattr(pb, name, torch.from_numpy(np.ascontiguousarray(getattr(pb, name))).pin_memory().numpy())
    for _ in range(3):
        got = bundle.solve(pb, pinned_inputs=True)
        assert abs(got["summary"]["final_cost"] - ref["summary"]["final_cost"]) <= 1e-12 * ref["summary"]["final_cost"]
        assert np.abs(got["points"] - ref["points"]).max() < 1e-9


def test_pose_only_and_point_only():
    sc = syn.cube_scene(6, 400, 1.0, with_descriptors=False)
    pb = syn.scene_to_problem(sc, optimize_cameras=False)
    pb.point_const[:] = 1  # bundle_shot_poses: only poses free (ba_helpers.cc:408-579)
    _compare(pb)
    pb2 = syn.scene_to_problem(sc, optimize_cameras=False)
    pb2.inst_const[:] = 1
    _compare(pb2)


def test_position_prior_and_thinned_visibility():
    sc = syn.cube_scene(12, 800, 1.0, with_descriptors=False, max_obs_per_point=5)
    pb = syn.scene_to_problem(sc)
    pb.inst_has_prior[:] = 1
    pb.inst_prior_pos = sc.origins + np.random.RandomState(1).normal(0, 0.01, sc.origins.shape)
    pb.inst_prior_std = np.full((12, 3), 0.05)
    _compare(pb)


def test_bundle_adjuster_api_roundtrip():
    sc = syn.cube_scene(5, 200, 1.0, with_descriptors=False)
    pb = syn.scene_to_problem(sc)
    ba = bundle.BundleAdjuster()
    for i in range(5):
        cam = T.Camera.create_perspective(0.9, -0.1, 0.01)
        ba.add_camera("cam%d" % i, cam, cam, False)
    ba.add_rig_camera("rc", T.Pose(), T.Pose(), True)
    for i in range(5):
        ba.add_rig_instance("inst%d" % i, T.Pose.from_ba_params(pb.inst[i]), {"shot%d" % i: "cam%d" % i},
                            {"shot%d" % i: "rc"}, False)
    for p in range(len(pb.points)):
        ba.add_point("p%d" % p, pb.points[p], False)
    for k in range(pb.num_observations):
        ba.add_point_projection_observation("shot%d" % pb.obs_shot[k], "p%d" % pb.obs_point[k], pb.obs_xy[k], 0.004)
    ba.set_point_projection_loss_function("SoftLOneLoss", 1.0)
    ba.set_internal_parameters_prior_sd(0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01, 0.01)
    ba.set_max_num_iterations(100)
    ba.run()
    ref = oracle.solve(pb)
    pts = np.array([ba.get_point("p%d" % p).p for p in range(len(pb.points))])
    assert np.abs(pts - ref["points"]).max() < 2e-5
    errs = ba.get_point("p0").reprojection_errors
    assert set(errs) <= {"shot%d" % i for i in range(5)} and all(len(v) == 2 for v in errs.values())
    assert "Termination" in ba.brief_report()
    with pytest.raises(RuntimeError):
        ba.get_camera("nope")
    with pytest.raises(IndexError):
        ba.add_point_projection_observation("nope", "p0", [0, 0], 1.0)
    with pytest.raises(RuntimeError):
        ba.set_point_projection_loss_function("NopeLoss", 1.0)
        ba.run()


def _mixed_problem(seed=0, rig=False, free_rig=False, only=None):
    """6 instances looking at a point cloud through different camera models (and, optionally, a
    two-camera rig so that the two-pose path of projection_errors.h:95-149 runs)."""
    from scipy.spatial.transform import Rotation

    rng = np.random.RandomState(seed)
    types = [bp.PERSPECTIVE, bp.BROWN, bp.FISHEYE, bp.FISHEYE_OPENCV, bp.RADIAL, bp.SPHERICAL, bp.DUAL,
             bp.SIMPLE_RADIAL, bp.FISHEYE62, bp.FISHEYE624]
    if only is not None:
        types = [only] * 6
    params = {
        bp.PERSPECTIVE: [-0.05, 0.01, 0.8], bp.BROWN: [-0.05, 0.01, 0.001, 0.001, -0.001, 0.8, 1.0, 0.01, -0.01],
        bp.FISHEYE: [-0.02, 0.005, 0.7], bp.FISHEYE_OPENCV: [-0.02, 0.005, 0.001, 0.0, 0.7, 1.0, 0.0, 0.01],
        bp.RADIAL: [-0.05, 0.01, 0.8, 1.0, 0.0, 0.0], bp.SPHERICAL: [0.0], bp.DUAL: [0.4, -0.03, 0.005, 0.75],
        bp.SIMPLE_RADIAL: [-0.04, 0.8, 1.0, 0.0, 0.0],
        bp.FISHEYE62: [-0.02, 0.005, 0.0, 0.0, 0.0, 0.0, 0.001, -0.001, 0.7, 1.0, 0.0, 0.0],
        bp.FISHEYE624: [-0.02, 0.005, 0.0, 0.0, 0.0, 0.0, 0.001, -0.001, 0.001, 0.0, -0.001, 0.0, 0.7, 1.0, 0.0, 0.0],
    }
    K = len(types)
    NI = K
    pts = rng.uniform(-0.5, 0.5, (300, 3))
    inst = np.zeros((NI, 6))
    for i in range(NI):
        ang = 2 * np.pi * i / NI
        origin = 2.5 * np.array([np.cos(ang), np.sin(ang), 0.2 * np.sin(3 * ang)])
        ez = -origin / np.linalg.norm(origin)
        ex = np.cross(ez, [0, 0, 1.0]); ex /= np.linalg.norm(ex)
        ey = np.cross(ez, ex)
        R_wc = np.array([ex, ey, ez])
        inst[i] = np.concatenate([Rotation.from_matrix(R_wc.T).as_rotvec(), origin])
    if rig:
        rigcam = np.array([[0.0, 0.0, 0.0, 0.0, 0.0, 0.0], [0.02, -0.03, 0.01, 0.1, 0.0, 0.02]])
        shot_inst = np.repeat(np.arange(NI), 2)
        shot_cam = np.repeat(np.arange(K), 2)
        shot_rc = np.tile([0, 1], NI)
        shot_use = np.tile([0, 1], NI)  # rig camera 0 is the identity: not "useful" (bundle_adjuster.cc:17-20)
    else:
        rigcam = np.zeros((1, 6))
        shot_inst = np.arange(NI); shot_cam = np.arange(K); shot_rc = np.zeros(NI, int); shot_use = np.zeros(NI, int)
    S = len(shot_inst)
    obs_shot, obs_point, obs_xy = [], [], []
    for s in range(S):
        i, k = shot_inst[s], shot_cam[s]
        for p in range(len(pts)):
            xc = Rotation.from_rotvec(-inst[i, :3]).apply(pts[p] - inst[i, 3:])
            if shot_use[s]:
                rc = rigcam[shot_rc[s]]
                xc = Rotation.from_rotvec(-rc[:3]).apply(xc - rc[3:])
            if types[k] != bp.SPHERICAL and xc[2] < 0.5:
                continue
            if types[k] == bp.SPHERICAL:
                lon, lat = np.arctan2(xc[0], xc[2]), np.arctan2(-xc[1], np.hypot(xc[0], xc[2]))
                px = np.array([lon / (2 * np.pi), -lat / (2 * np.pi)])
            else:
                px = oracle.project(types[k], params[types[k]], xc)
            obs_shot.append(s); obs_point.append(p); obs_xy.append(px + rng.normal(0, 5e-4, 2))
    pb = bp.make_problem(types, [params[t] for t in types], inst, pts + rng.normal(0, 0.01, pts.shape), obs_shot,
                         obs_point, np.array(obs_xy), np.full(len(obs_shot), 0.004), shot_inst=shot_inst,
                         shot_cam=shot_cam, rigcam=rigcam, shot_rc=shot_rc, shot_use_rc=shot_use,
                         rigcam_const=[1, 0 if free_rig else 1],
                         prior_sd=dict(focal_sd=0.01, aspect_ratio_sd=0.01, c_sd=0.01, k1_sd=0.01, k2_sd=0.01,
                                       p1_sd=0.01, p2_sd=0.01, k3_sd=0.01, k4_sd=0.01),
                         loss_name="SoftLOneLoss", loss_threshold=1.0, max_iterations=50)
    pb.inst[:, 3:] += rng.normal(0, 0.01, (NI, 3))
    return pb


def test_all_camera_models_in_one_problem():
    _compare(_mixed_problem(0), tol_param=5e-5)


@pytest.mark.parametrize("ptype", ["PERSPECTIVE", "BROWN", "FISHEYE"])
def test_uniform_camera_type_uses_the_specialised_linearisation(ptype):
    """One projection type for every camera and no rig cameras: ba_linearize<.., TYPE> (compile-time model) runs;
    it must agree with the oracle like the generic kernel does."""
    _compare(_mixed_problem(3, only=getattr(bp, ptype)), tol_param=5e-5)


def test_rig_cameras_two_pose_path():
    _compare(_mixed_problem(1, rig=True), tol_param=5e-5)
    _compare(_mixed_problem(2, rig=True, free_rig=True), tol_param=5e-5)


def test_degenerate_inputs():
    sc = syn.cube_scene(4, 60, 1.0, with_descriptors=False)
    pb = syn.scene_to_problem(sc)
    # everything constant: nothing to optimise, reprojection errors still produced
    pb.cam_const[:] = 1; pb.inst_const[:] = 1; pb.point_const[:] = 1
    got = bundle.solve(pb)
    assert got["summary"]["termination"] == "CONVERGENCE" and got["summary"]["iterations"] == 0
    assert np.allclose(got["points"], pb.points)
    ref_cost, ref_rep = oracle.OracleBA(pb).cost(want_reproj=True)
    assert abs(got["summary"]["final_cost"] - ref_cost) <= 1e-9 * ref_cost
    assert np.abs(got["reprojection_errors"] - ref_rep).max() < 1e-12
    # no observations at all
    pb2 = syn.scene_to_problem(sc)
    pb2.obs_shot = pb2.obs_shot[:0]; pb2.obs_point = pb2.obs_point[:0]
    pb2.obs_xy = pb2.obs_xy[:0]; pb2.obs_sigma = pb2.obs_sigma[:0]
    got2 = bundle.solve(pb2)
    assert got2["reprojection_errors"].shape == (0, 3)
    assert np.allclose(got2["points"], pb2.points)
    # dangling index -> error, like std::map::at / "doesn't exist" in the reference
    pb3 = syn.scene_to_problem(sc)
    pb3.obs_point = pb3.obs_point.copy(); pb3.obs_point[0] = 10 ** 6
    with pytest.raises((AssertionError, ValueError, RuntimeError)):
        bundle.solve(pb3)


def test_kernel_variants_agree(tmp_path):
    """The default path (persistent fp64 tensor-core segment Schur, pipelined PCG with S resident in shared memory) and the
    kernels it replaces (per-point ba_schur, SIMT segment kernel, classic / streamed PCG) must give the same solve."""
    import os
    import subprocess
    import sys

    code = (
        "import sys; sys.path.insert(0, %r)\n"
        "import numpy as np\n"
        "from opensfm_b200 import bundle, synthetic as syn\n"
        "sc = syn.cube_scene(30, 4000, 1.0, with_descriptors=False, max_obs_per_point=8)\n"
        "r = bundle.solve(syn.scene_to_problem(sc))\n"
        "np.save(sys.argv[1], np.concatenate([[r['summary']['final_cost'], r['summary']['iterations']], r['points'].ravel()]))\n"
    ) % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {}
    variants = {"default": {}, "generic_schur": {"OSFM_BA_SEGMENT_SCHUR": "0"}, "simt_seg_schur": {"OSFM_BA_SCHUR_MMA": "0"}, "cta_per_segment_schur": {"OSFM_BA_SCHUR_PIPE": "0"}, "generic_linearize": {"OSFM_BA_LIN_SPECIAL": "0"}, "undeflated_pcg": {"OSFM_BA_PCG_DEFLATE": "0"}, "explicit_model_change": {"OSFM_BA_MODEL_CHANGE_EXPLICIT": "1"}, "classic_pcg": {"OSFM_BA_PCG_PIPELINED": "0"}, "b128_barrier": {"OSFM_BA_PCG_B128": "1"},
                "streamed_pcg": {"OSFM_BA_PCG_PIPELINED": "0", "OSFM_BA_PCG_RESIDENT": "0"}}
    for name, extra in variants.items():
        path = str(tmp_path / ("%s.npy" % name))
        env = dict(os.environ, **extra)
        subprocess.run([sys.executable, "-c", code, path], check=True, env=env, timeout=600)
        out[name] = np.load(path)
    for name in ("generic_schur", "simt_seg_schur", "cta_per_segment_schur", "generic_linearize", "undeflated_pcg", "explicit_model_change", "classic_pcg", "b128_barrier", "streamed_pcg"):
        assert out["default"][1] == out[name][1]
        assert abs(out["default"][0] - out[name][0]) <= 1e-9 * out["default"][0]
        # the solvers that do not deflate the gauge directions stop with a different (larger) error along those
        # weakly determined directions: same cost to 1e-9, points to 2e-6; everything else is the same solve
        plain = name in ("undeflated_pcg", "classic_pcg", "b128_barrier", "streamed_pcg")
        assert np.abs(out["default"][2:] - out[name][2:]).max() < (2e-6 if plain else 1e-8)   # measured 3e-7 / 1e-9
