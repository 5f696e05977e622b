#!/usr/bin/env python
"""Headline benchmark: BA observations/sec + descriptor-pairs/sec (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this engine (one rank per GPU)
    python bench.py --impl reference --gpus N ...            # the reference's CPU path, host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's results (dump_outputs)

Workload (config.workload): the synthetic cube scene of BASELINE.json configs[3],
500 cameras / 200k points / 2M observations (exactly 10 observations per point), which fits
one B200 and is the configuration the north-star target is quoted on.  One *step* is

  BA     one full `bundle()` of that scene: Levenberg-Marquardt to convergence (SoftLOneLoss,
         cameras optimised, <= 100 iterations) from the seed-43 perturbed start;
  MATCH  symmetric brute-force matching of every image with its 8 nearest cameras
         (unique unordered pairs), 128-D integer-valued descriptors (HAHOG / SIFT as OpenSfM
         stores them: uint8 on disk, float32 in memory), ratio 0.8.

`value` = BA observations/sec = N_obs x LM iterations / CUDA-event time of the LM loop with the
problem resident in HBM; `value_run` = the same over the wall time of run() (the reference's
`wall_times["run"]`, SURVEY 8d); `match.value` = descriptor pairs (2 directions) / device time of the
batch with descriptors resident.  `e2e` is the same metric through the public Python API with
page-locked host buffers (H2D of the problem / descriptors and D2H of the results inside the timed
region; descriptors travel as the uint8 they are stored as).
Multi-GPU: BA shards observations by point (all-reduce of the reduced camera system per LM
iteration), MATCH shards the pair list (pairs sharing images on the same GPU); total work is fixed
=> "scaling": "strong".

Sub-records measured once per run at N = 1 (`extras`, outside the K timed steps): guided matching on the
BASELINE configs[2] stand-in (29 images x 8000 HAHOG-like descriptors, epipolar mask built on the device),
AKAZE- / ORB-size Hamming (fp8 tensor-core kernel), general float32 (cv2-order exact kernel), the configs[1] scene
(50 cameras / 5k points) and a configs[4] stand-in (`c5`: four overlapping submodels of the scene, a bundle adjustment
each, then the ReconstructionAlignment problem of opensfm/large/tools.py).  The e2e BA leg uploads its page-locked
observation arrays with osfm_ba_set_observations_async (`pinned_inputs=True`).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The CPU arms use every host thread: torchrun exports OMP_NUM_THREADS=1, and libgomp reads the variable when the
# oracle library is loaded, so it is forced here, before anything is imported (VERDICT r1 #9).
_CORES = os.cpu_count() or 1
if "--impl" in sys.argv and "reference" in sys.argv or int(os.environ.get("WORLD_SIZE", "1")) == 1:
    os.environ["OMP_NUM_THREADS"] = str(_CORES)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: cameras, points, obs/point, neighbours per image for matching
    "c4": dict(cameras=500, points=200000, obs_per_point=10, neighbours=8,
               label="synthetic cube 500 cameras / 200k points / 2M observations (BASELINE configs[3])"),
    "c2": dict(cameras=50, points=5000, obs_per_point=None, neighbours=49,
               label="synthetic cube 50 cameras / 5k points, all pairs (BASELINE configs[1])"),
    "tiny": dict(cameras=12, points=1500, obs_per_point=6, neighbours=4, label="tiny smoke workload"),
}
CPU_BA_ITERATIONS = {"c4": 2}   # bounded CPU sample: LM iterations per step (5 for the small scenes)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


FP64_TENSOR_PEAK_TFLOPS = 37.2   # scripts/bench_dmma.cu on this pool's B200 (DMMA = DFMA = 64 FMA/clk/SM); not in MEASURED_PEAKS
POPC_PER_CLK_PER_SM = 16.0       # CUDA programming guide, arithmetic-instruction throughput table (population count)


def build_workload(name):
    from opensfm_b200 import synthetic as syn

    w = WORKLOADS[name]
    sc = syn.cube_scene(w["cameras"], w["points"], 1.0, seed=42, with_descriptors=True,
                        max_obs_per_point=w["obs_per_point"])
    pb = syn.scene_to_problem(sc)
    # per-image descriptor matrices (rows of the visible points); observations are shot-major
    starts = np.searchsorted(sc.obs_shot, np.arange(sc.num_shots + 1))
    feats = [np.ascontiguousarray(sc.track_descriptors[sc.obs_point[starts[s]:starts[s + 1]]]) for s in range(sc.num_shots)]
    # pair list: each image with its k nearest cameras, unique unordered pairs (pairs_selection-style)
    k = min(w["neighbours"], sc.num_shots - 1)
    d = np.linalg.norm(sc.origins[:, None, :] - sc.origins[None, :, :], axis=2)
    np.fill_diagonal(d, np.inf)
    nn = np.argsort(d, axis=1, kind="stable")[:, :k]
    pairs = sorted({(min(i, int(j)), max(i, int(j))) for i in range(sc.num_shots) for j in nn[i]})
    pairs = [p for p in pairs if len(feats[p[0]]) and len(feats[p[1]])]
    return pb, feats, pairs, w


def config_of(w, pb, pairs, feats, world):
    """The `config` object of the JSON line -- identical keys and values in both arms."""
    return {"workload": w["label"], "observations": int(pb.num_observations), "cameras": int(len(pb.cam_type)),
            "points": int(len(pb.points)), "loss": pb.loss_name, "max_lm_iterations": int(pb.max_iterations),
            "image_pairs": len(pairs), "descriptors": int(sum(len(f) for f in feats)), "descriptor_dim": 128,
            "lowes_ratio": 0.8, "symmetric_matching": True,
            "parallelism": "points sharded over %d GPU(s); pair list sharded" % world}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------
# reference arm: the reference's CPU implementation of the path on the host cores
# --------------------------------------------------------------------------------------
def cpu_ba_sample(pb, iterations):
    """CPU restatement of the Ceres path (oracle, OpenMP over all host threads): LM iterations on the
    same problem, stopped after `iterations` (bounded sample)."""
    from oracle import ba_lm

    res = ba_lm.solve(pb, stop_after_iterations=iterations)
    its = max(res["iterations"], 1)
    return pb.num_observations * its / res["time_run"], its, res["time_run"]


def cpu_match_sample(feats, pairs, npairs, threads, masks=None):
    """The reference matcher itself (cv2 BFMatcher through opensfm/matching.py:723-777 semantics) on a
    bounded sample of the pair list, in a joblib *threading* pool like opensfm/context.py:47-67."""
    import cv2
    from joblib import Parallel, delayed

    from oracle import match_oracle as mo

    sample = pairs[:npairs]
    cfg = {"lowes_ratio": 0.8}
    cv2.setNumThreads(0)  # context.py:52-53

    def one(k, p):
        return len(mo.match_brute_force_symmetric(feats[p[0]], feats[p[1]], cfg, None if masks is None else masks(k, p)))

    t0 = time.perf_counter()
    Parallel(n_jobs=threads, backend="threading")(delayed(one)(k, p) for k, p in enumerate(sample))
    dt = time.perf_counter() - t0
    work = sum(2 * len(feats[a]) * len(feats[b]) for a, b in sample)
    return work / dt, len(sample), dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    pb, feats, pairs, w = build_workload(args.workload)
    cores = _CORES
    ba_vals, mt_vals = [], []
    ba_its = CPU_BA_ITERATIONS.get(args.workload, 5)
    npairs = min(len(pairs), max(cores // 2, 16))
    for _ in range(args.warmup):
        cpu_match_sample(feats, pairs, min(npairs, 8), cores)
    t_all = time.perf_counter()
    for _ in range(args.steps):
        v, its, dt = cpu_ba_sample(pb, ba_its)
        ba_vals.append((v, dt))
        m, n, dtm = cpu_match_sample(feats, pairs, npairs, cores)
        mt_vals.append((m, dtm))
    total = time.perf_counter() - t_all
    ba_v = float(np.mean([v for v, _ in ba_vals]))
    mt_v = float(np.mean([v for v, _ in mt_vals]))
    line = {
        "impl": "reference", "metric": "BA observations/sec", "value": ba_v, "unit": "observations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_of(w, pb, pairs, feats, args.gpus),
        "cpu_baseline": {"value": ba_v, "unit": "observations/s", "cores": cores,
                         "omp_threads": int(os.environ.get("OMP_NUM_THREADS", "0")), "kind": "port",
                         "sample": "%d LM iterations of the same problem per step (restated Ceres path, OpenMP; "
                                   "Ceres itself cannot be built in this image)" % ba_its},
        "e2e": {"value": ba_v, "unit": "observations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "match": {"metric": "descriptor-pairs/sec", "value": mt_v, "unit": "descriptor-pairs/s",
                  "cpu_baseline": {"value": mt_v, "unit": "descriptor-pairs/s", "cores": cores, "kind": "reference",
                                   "sample": "%d symmetric pairs per step through cv2 BFMatcher in a joblib threading pool"
                                             % npairs},
                  "e2e": {"value": mt_v, "unit": "descriptor-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------
# extras (N = 1): the other BASELINE configs and the non-tensor-core matcher paths
# --------------------------------------------------------------------------------------
def run_c5(workload="c4"):
    """BASELINE configs[4] stand-in ("opensfm/large" submodel split): the C4 scene's 500 cameras in 4 overlapping
    submodels, one bundle adjustment per submodel, each result moved into a gauge of its own (what independent
    reconstructions come back in), then opensfm.large.tools.align_reconstructions' problem (soft camera constraints:
    one relative-motion term per (submodel, shot) + one absolute GPS position per shot, opensfm/large/tools.py:120-159)
    through opensfm_b200.alignment.ReconstructionAlignment.  Pair-list matching of the submodels is the sharded matching
    of the headline line.  Reports times; the alignment is checked against the similarities that were applied."""
    from scipy.spatial.transform import Rotation

    from opensfm_b200 import alignment, ba_problem as bp, bundle

    pb, _, _, _ = build_workload(workload)
    S = len(pb.inst)
    # four overlapping index ranges: (0, 140), (120, 265), (245, 390), (370, 500) for the 500 cameras of C4
    ranges = [(0, int(0.28 * S)), (int(0.24 * S), int(0.53 * S)), (int(0.49 * S), int(0.78 * S)), (int(0.74 * S), S)]
    off = np.asarray(pb.cam_off)
    out = {"workload": "BASELINE configs[4] stand-in: the C4 scene in 4 overlapping submodels (%s cameras), BA per submodel, "
                       "then ReconstructionAlignment with soft camera constraints + GPS" % "/".join(str(b - a) for a, b in ranges),
           "submodels": []}
    rng = np.random.RandomState(5)
    results = []
    t_ba = 0.0
    for m, (a, b) in enumerate(ranges):
        sel = (pb.obs_shot >= a) & (pb.obs_shot < b)
        o_shot, o_pt = pb.obs_shot[sel] - a, pb.obs_point[sel]
        cnt = np.bincount(o_pt, minlength=len(pb.points))
        keep_pt = cnt >= 2
        ok = keep_pt[o_pt]
        remap = np.cumsum(keep_pt) - 1
        sub = bp.make_problem(
            [bp.PERSPECTIVE] * (b - a), [pb.cam_params[off[k]:off[k + 1]] for k in range(a, b)], pb.inst[a:b], pb.points[keep_pt],
            o_shot[ok].astype(np.int32), remap[o_pt[ok]].astype(np.int32), pb.obs_xy[sel][ok], pb.obs_sigma[sel][ok],
            prior_sd=dict(focal_sd=0.01, aspect_ratio_sd=0.01, c_sd=0.01, k1_sd=0.01, k2_sd=0.01, p1_sd=0.01, p2_sd=0.01,
                          k3_sd=0.01, k4_sd=0.01),
            loss_name=pb.loss_name, loss_threshold=pb.loss_threshold, max_iterations=pb.max_iterations)
        bundle.solve(sub)   # warm-up (allocations)
        t0 = time.perf_counter()
        r = bundle.solve(sub)
        dt = time.perf_counter() - t0
        t_ba += dt
        s = r["summary"]
        out["submodels"].append({"cameras": b - a, "points": int(keep_pt.sum()), "observations": int(ok.sum()),
                                 "lm_iterations": s["iterations"], "device_ms": s["time_device_ms"], "wall_ms": 1e3 * dt,
                                 "obs_per_s": ok.sum() * s["iterations"] / (s["time_device_ms"] * 1e-3)})
        results.append((a, b, r["inst"]))
    # every submodel comes back in its own gauge: X' = s Q X + T
    gauges = [(float(rng.uniform(0.8, 1.25)), Rotation.from_rotvec(rng.normal(0, 0.2, 3)).as_matrix(), rng.normal(0, 2.0, 3))
              for _ in results]
    gps_noise = rng.normal(0, 0.05, (S, 3))
    cov = np.diag([1e-5, 1e-5, 1e-5, 1e-2, 1e-2, 1e-2])
    sm = np.linalg.inv(np.linalg.cholesky(cov)).T   # scale_matrix of opensfm/large/tools.py

    def make_alignment():
        ra = alignment.ReconstructionAlignment()
        added = set()
        for m, (a, b, inst) in enumerate(results):
            sc, Q, T = gauges[m]
            ra.add_reconstruction("rec%d" % m, 0, 0, 0, 0, 0, 0, 1, False)
            for k in range(a, b):
                R_cw = Rotation.from_rotvec(inst[k - a, :3]).as_matrix()
                origin = inst[k - a, 3:]
                R_cw2, origin2 = Q @ R_cw, sc * Q @ origin + T          # pose of the shot in the submodel's own gauge
                R_wc2 = R_cw2.T
                rv, tv = Rotation.from_matrix(R_wc2).as_rotvec(), -R_wc2 @ origin2   # OpenSfM pose: x_cam = R x_world + t
                name = "shot%d" % k
                if name not in added:
                    ra.add_shot(name, rv[0], rv[1], rv[2], tv[0], tv[1], tv[2], False)
                    gps = origin + gps_noise[k]   # positions in the common (GPS) frame
                    ra.add_absolute_position_constraint(name, gps[0], gps[1], gps[2], 1.0)
                    added.add(name)
                rmc = alignment.RARelativeMotionConstraint("rec%d" % m, name, rv[0], rv[1], rv[2], tv[0], tv[1], tv[2])
                for i in range(6):
                    for j in range(6):
                        rmc.set_scale_matrix(i, j, sm[i, j])
                ra.add_relative_motion_constraint(rmc)
        return ra, len(added)

    make_alignment()[0].run()   # warm-up
    ra, n_shots = make_alignment()
    t0 = time.perf_counter()
    ra.run()
    t_ra = time.perf_counter() - t0
    # the reconstruction similarity must undo the gauge: compare the recovered scale with 1 / s
    err = 0.0
    for m, (sc, Q, T) in enumerate(gauges):
        rec = ra.get_reconstruction("rec%d" % m)
        err = max(err, min(abs(rec.scale * sc - 1.0), abs(rec.scale / sc - 1.0)))   # either direction convention
    out.update({"ba_wall_ms": 1e3 * t_ba, "alignment_wall_ms": 1e3 * t_ra, "alignment_terms": n_shots + sum(b - a for a, b in ranges),
                "alignment_report": ra.brief_report().strip().splitlines()[-1] if ra.brief_report() else "",
                "alignment_scale_error": float(err), "total_wall_ms": 1e3 * (t_ba + t_ra)})
    return out


def run_extras(pk, clocks_mhz, with_cpu):
    import torch

    from opensfm_b200 import bundle, matching, synthetic as syn

    cfg = {"lowes_ratio": 0.8}
    out = {}
    reps = 3

    def timed(pm, fn):
        fn()
        tot = ker = 0.0
        for _ in range(reps):
            fn()
            a, b = pm.device_ms()
            tot += a
            ker += b
        return tot / reps, ker / reps

    # ---- configs[2] stand-in: guided matching, 29 images x 8000 HAHOG-like descriptors ----
    n_img, n_desc = 29, 8000
    descs, bears, Rs, Os = syn.guided_scene(n_img, n_desc, seed=11)
    pairs = [(i, j) for i in range(n_img) for j in range(i + 1, min(i + 6, n_img))]
    poses = [syn.relative_pose(Rs[a], Os[a], Rs[b], Os[b]) for a, b in pairs]
    pm = matching.PairMatcher()
    pm.add_many([(i, descs[i].astype(np.uint8)) for i in range(n_img)], uint8_is_l2=True)
    for i in range(n_img):
        pm.set_bearings(i, bears[i])
    res = {}

    def guided():
        res["m"] = pm.match_pairs_guided(pairs, poses, 0.006, cfg, mask_budget_bytes=1 << 31)

    tot, ker = timed(pm, guided)
    work = sum(2 * n_desc * n_desc for _ in pairs)
    d8 = [d.astype(np.uint8) for d in descs]
    e2e_s = 1e30
    for _ in range(2):   # long-lived matcher like the headline e2e leg: descriptors, bearings re-uploaded every time
        t0 = time.perf_counter()
        pm.clear()
        pm.add_many([(i, d8[i]) for i in range(n_img)], uint8_is_l2=True)
        for i in range(n_img):
            pm.set_bearings(i, bears[i])
        pm.match_pairs_guided(pairs, poses, 0.006, cfg, mask_budget_bytes=1 << 31)
        e2e_s = min(e2e_s, time.perf_counter() - t0)
    g = {"workload": "BASELINE configs[2] stand-in: %d images x %d HAHOG-like descriptors, %d sequence pairs, guided "
                     "(epipolar threshold 0.006), symmetric" % (n_img, n_desc, len(pairs)),
         "value": work / (tot * 1e-3), "unit": "descriptor-pairs/s", "device_ms": tot, "distance_kernel_ms": ker,
         "mask_and_finalize_ms": tot - ker, "matches": int(sum(len(v) for v in res["m"].values())),
         "kernel": "bf_top2_tc<masked> + epi_mask_bits" if pm.last_kernel() == 2 else "bf_top2_f32_cv",
         "e2e": {"value": work / e2e_s, "unit": "descriptor-pairs/s",
                 "h2d_bytes_per_step": int(n_img * n_desc * (128 + 12)), "d2h_bytes_per_step": int(4 * n_desc * len(pairs))},
         "roofline": {"bound": "tensor", "achieved": 2.0 * 128 * work / (ker * 1e-3) / 1e12, "peak": pk["bf16_sustained"],
                      "unit": "TFLOP/s", "frac": 2.0 * 128 * work / (ker * 1e-3) / 1e12 / pk["bf16_sustained"]}}
    if with_cpu:
        from oracle import match_oracle as mo

        def masks(k, p):
            return mo.epipolar_mask(bears[p[0]], bears[p[1]], poses[k][0], poses[k][1], 0.006)

        v, n, dt = cpu_match_sample(descs, pairs, min(len(pairs), max(_CORES // 8, 8)), _CORES, masks)
        g["cpu_baseline"] = {"value": v, "unit": "descriptor-pairs/s", "cores": _CORES, "kind": "reference",
                             "sample": "%d guided pairs via cv2 BFMatcher + numpy epipolar mask (%.1f s)" % (n, dt)}
    out["match_guided"] = g
    del pm

    # ---- Hamming (AKAZE 61-byte MLDB, ORB 32 bytes) and general float32 ----
    n_img, n_desc = 8, 8000
    pairs8 = [(i, j) for i in range(n_img) for j in range(i + 1, n_img)][:16]
    work8 = 2 * len(pairs8) * n_desc * n_desc
    sm_clock = (clocks_mhz or 1965.0) * 1e6

    def simt(name, make, extra):
        pm = matching.PairMatcher()
        for i in range(n_img):
            pm.add(i, make(i))

        def go():
            pm.submit(pairs8, 0.8, True)
            pm.sync()

        tot, ker = timed(pm, go)
        rec = {"workload": "%d images x %d descriptors, %d symmetric pairs" % (n_img, n_desc, len(pairs8)),
               "value": work8 / (tot * 1e-3), "unit": "descriptor-pairs/s", "distance_kernel_ms": ker,
               "kernel": {1: "bf_top2_simt<u8>" if name != "float" else "bf_top2_f32_cv", 2: "bf_top2_tc",
                          3: "bf_top2_tc_h8"}[pm.last_kernel()]}
        rec.update(extra(ker, pm.last_kernel()))
        if with_cpu:
            f = [make(i) for i in range(n_img)]
            v, n, dt = cpu_match_sample(f, pairs8, len(pairs8), _CORES)
            rec["cpu_baseline"] = {"value": v, "unit": "descriptor-pairs/s", "cores": _CORES, "kind": "reference",
                                   "sample": "%d pairs via cv2 BFMatcher (%.1f s)" % (n, dt)}
        out["match_" + name] = rec

    def popc_roof(words):
        def f(ker, kid):
            if kid == 3:
                # +-1 fp8 contraction, K padded to 512 per descriptor pair; no measured fp8 figure in
                # MEASURED_PEAKS.json -> the nominal dense fp8 peak (4.5 PFLOP/s), said so in the note
                ach = 2.0 * 512 * work8 / (ker * 1e-3) / 1e12
                return {"roofline": {"bound": "tensor", "achieved": ach, "peak": 4500.0, "unit": "TFLOP/s", "frac": ach / 4500.0,
                                     "note": "fp8 (E4M3 +-1) tcgen05 kind::f8f6f4, K = 512 per pair (%d useful bits); peak = "
                                             "nominal dense fp8; the epilogue (top-2 over 128x128 accumulators), not "
                                             "the tensor pipe, bounds this kernel" % (words * 32)}}
            ach = work8 * words / (ker * 1e-3)
            peak = 148 * POPC_PER_CLK_PER_SM * sm_clock
            return {"roofline": {"bound": "alu-popc", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "Tpopc/s",
                                 "frac": ach / peak,
                                 "note": "%d 32-bit XOR+POPC per descriptor pair; peak = 148 SMs x 16 POPC/clk x SM clock "
                                         "(CUDA programming guide throughput table)" % words}}
        return f

    def fp32_roof(ker, kid):
        ach = work8 * 128 * 3 / (ker * 1e-3)   # sub, mul, add per element: cv2's order forbids FMA
        peak = 148 * 128 * sm_clock
        return {"roofline": {"bound": "alu-fp32", "achieved": ach / 1e12, "peak": peak / 1e12, "unit": "Tinst/s",
                             "frac": ach / peak, "note": "3 fp32 instructions per element (no FMA: bit-exact cv2 order)"}}

    simt("hamming_akaze61", lambda i: syn.binary_descriptors(n_desc, 50 + i, 61), popc_roof(16))
    simt("hamming_orb32", lambda i: syn.binary_descriptors(n_desc, 70 + i, 32), popc_roof(8))
    simt("float", lambda i: np.random.RandomState(i).rand(n_desc, 128).astype(np.float32), fp32_roof)

    # ---- configs[1]: cube 50 cameras / 5k points, one full BA + all-pairs matching ----
    pb, feats, pairs2, w2 = build_workload("c2")
    bundle.solve(pb)
    t0 = time.perf_counter()
    r = bundle.solve(pb)
    wall = time.perf_counter() - t0
    s = r["summary"]
    pmc = matching.PairMatcher()
    pmc.add_many([(i, f.astype(np.uint8)) for i, f in enumerate(feats)], uint8_is_l2=True)

    def allpairs():
        pmc.submit(pairs2, 0.8, True)
        pmc.sync()

    tot, ker = timed(pmc, allpairs)
    work2 = sum(2 * len(feats[a]) * len(feats[b]) for a, b in pairs2)
    out["c2"] = {"workload": w2["label"], "observations": int(pb.num_observations), "lm_iterations": s["iterations"],
                 "ba_value": pb.num_observations * s["iterations"] / (s["time_device_ms"] * 1e-3),
                 "ba_e2e": pb.num_observations * s["iterations"] / wall, "ba_unit": "observations/s",
                 "image_pairs": len(pairs2), "match_value": work2 / (tot * 1e-3), "match_unit": "descriptor-pairs/s"}
    torch.cuda.synchronize()
    return out


# --------------------------------------------------------------------------------------
# --dump-outputs: what the timed path returned, for comparing two builds output for output
# --------------------------------------------------------------------------------------
DUMP_BUDGET_BYTES = 64 << 20
# row caps of the two outputs that outgrow the budget at C4 (2M reprojection errors, ~4M matches); the rest is whole
DUMP_MAX_ROWS = {"ba_reprojection_errors": 1 << 20, "matches": 1 << 19}


def sample_rows(n, max_rows, seed=0):
    """Sorted indices of a fixed sample of `max_rows` out of `n` rows (all of them when n <= max_rows): the same
    indices for the same n, whatever the values, so two builds that agree on the shapes are compared row for row."""
    if n <= max_rows:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, max_rows, replace=False))


def dump_outputs(dirname, ba, match_lists, pairs):
    """Write one step's results as DIR/<name>.npy, float64:

    ba_summary              [initial cost, final cost, LM iterations]
    ba_points, ba_rig_instances, ba_rig_cameras, ba_cam_params   the solved parameters, whole
    ba_reprojection_errors  rows sample_rows(N_obs, ...) of the (N_obs, 3) reprojection errors
    match_counts            matches of every pair, in the order of the pair list
    matches                 rows sample_rows(total, ...) of (image 1, image 2, feature 1, feature 2), the match lists of
                            the pair list concatenated in its order
    """
    s = ba["summary"]
    rep = ba["reprojection_errors"]
    counts = np.array([len(match_lists[p]) for p in pairs], dtype=np.int64)
    rows = np.concatenate([match_lists[p] for p in pairs]) if pairs else np.zeros((0, 2), dtype=np.int64)
    keep = sample_rows(len(rows), DUMP_MAX_ROWS["matches"])
    pair_of = np.searchsorted(np.cumsum(counts), keep, side="right")
    arrays = {
        "ba_summary": [s["initial_cost"], s["final_cost"], s["iterations"]],
        "ba_points": ba["points"], "ba_rig_instances": ba["inst"], "ba_rig_cameras": ba["rigcam"],
        "ba_cam_params": ba["cam_params"],
        "ba_reprojection_errors": rep[sample_rows(len(rep), DUMP_MAX_ROWS["ba_reprojection_errors"])],
        "match_counts": counts,
        "matches": np.column_stack([np.asarray(pairs, dtype=np.int64).reshape(-1, 2)[pair_of], rows[keep]]),
    }
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BUDGET_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte budget" % (total, DUMP_BUDGET_BYTES))
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)
    return sorted(arrays)


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the BA solution and match lists of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the CUDA arm (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch

    from opensfm_b200 import _lib, bundle, dist as odist, matching

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    allreduce = None
    if world > 1:
        odist.init_from_env("nccl")
        import torch.distributed as tdist

        allreduce = "nccl"  # the library's own NCCL communicator (opensfm_b200.dist.make_allreduce is the callback form)
    L = _lib.load()
    pk = peaks()

    pb, feats, pairs, w = build_workload(args.workload)
    nobs = pb.num_observations
    sizes = {i: len(f) for i, f in enumerate(feats)}
    my_pairs = matching.shard_pairs(pairs, sizes, world)[rank] if world > 1 else pairs
    pair_work_total = sum(2 * sizes[a] * sizes[b] for a, b in pairs)
    my_pair_work = sum(2 * sizes[a] * sizes[b] for a, b in my_pairs)
    cfg = {"lowes_ratio": 0.8, "symmetric_matching": True}

    # the descriptors are integers 0..255 (HAHOG-like): they travel as the uint8 OpenSfM stores them as
    feats8 = [f.astype(np.uint8) for f in feats]
    assert all(np.array_equal(f8.astype(np.float32), f) for f8, f in zip(feats8[:4], feats[:4]))

    # resident descriptors for the device-timed leg
    pm = matching.PairMatcher(device=local)
    needed = sorted({i for p in my_pairs for i in p})
    pm.add_many([(i, feats8[i]) for i in needed], uint8_is_l2=True)

    # e2e legs: host buffers are page-locked (the contract's "pinned host memory"); every step copies
    # them to the device and reads the results back into page-locked arrays
    def pinned(a):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()

    for name in ("obs_shot", "obs_point", "obs_xy", "obs_sigma", "points"):
        setattr(pb, name, pinned(getattr(pb, name)))
    feats8 = [pinned(f) for f in feats8]
    ba_out = {"points": pinned(np.zeros((len(pb.points), 3))), "reprojection_errors": pinned(np.zeros((nobs, 3)))}

    def ba_step():
        t0 = time.perf_counter()
        res = bundle.solve(pb, device=local, rank=rank, world=world, allreduce=allreduce, out=ba_out, pinned_inputs=True)
        return res, time.perf_counter() - t0

    def match_resident():
        pm.submit(my_pairs, cfg["lowes_ratio"], True)
        pm.sync()
        return pm.device_ms()

    pm2 = matching.PairMatcher(device=local)  # long-lived matcher; every step re-uploads all descriptors

    def match_e2e():
        t0 = time.perf_counter()
        pm2.clear()
        pm2.add_many([(i, feats8[i]) for i in needed], uint8_is_l2=True)  # H2D of every descriptor matrix
        out = pm2.match_pairs(my_pairs, cfg)  # kernels + D2H of the match lists
        return time.perf_counter() - t0, out

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        ba_step()
        match_resident()
    if args.warmup:
        match_e2e()

    launches0 = L.osfm_kernel_launch_count()
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    t_begin = time.perf_counter()
    ba_dev_ms, ba_wall, ba_run_s, ba_iters, ba_sum = 0.0, 0.0, 0.0, 0, None
    mt_dev_ms, mt_kernel_ms, mt_wall = 0.0, 0.0, 0.0
    for _ in range(args.steps):
        res, dt = ba_step()
        s = res["summary"]
        ba_sum = s
        ba_dev_ms += s["time_device_ms"]
        ba_run_s += s["time_run_s"]
        ba_wall += dt
        ba_iters += s["iterations"]
        tot, ker = match_resident()
        mt_dev_ms += tot
        mt_kernel_ms += ker
        dte, matches = match_e2e()
        mt_wall += dte
    barrier()
    t_total = time.perf_counter() - t_begin
    clk = clocks.stop()
    launches = L.osfm_kernel_launch_count() - launches0
    if args.dump_outputs:
        matches = odist.gather_pair_results(matches, world)   # the pair list is sharded over the ranks
        if rank == 0:
            dump_outputs(args.dump_outputs, res, matches, pairs)

    # max over ranks
    vals = torch.tensor([t_total, ba_dev_ms, ba_wall, mt_dev_ms, mt_kernel_ms, mt_wall, ba_run_s], dtype=torch.float64, device="cuda")
    if world > 1:
        tdist.all_reduce(vals, op=tdist.ReduceOp.MAX)
    t_total, ba_dev_ms, ba_wall, mt_dev_ms, mt_kernel_ms, mt_wall, ba_run_s = vals.tolist()

    K = args.steps
    ba_value = nobs * ba_iters / (ba_dev_ms * 1e-3)
    ba_value_run = nobs * ba_iters / ba_run_s
    ba_e2e = nobs * ba_iters / ba_wall
    mt_value = pair_work_total * K / (mt_dev_ms * 1e-3)
    mt_e2e = pair_work_total * K / mt_wall

    # ---- rooflines (rank 0's kernels) ----
    s = ba_sum
    nloc = s["num_observations_local"]
    plane_bytes = s["jac_planes"] * 8
    kern = {}
    if s["schur_launches"]:
        # ba_schur reads the residual/Jacobian planes of every observation once + the 4-byte shot index; writes
        # V^-1 / g_p per point
        per_launch = nloc * (plane_bytes + 4) + len(pb.points) // world * 72
        dur = s["time_schur_ms"] / s["schur_launches"] * 1e-3
        kern["ba_schur"] = dict(bytes=per_launch, ms=dur * 1e3, share=s["time_schur_ms"] / s["time_device_ms"])
    if s["linearize_launches"]:
        # ba_linearize reads the 32-byte observation record + parameters, writes the planes
        per_launch = nloc * (32 + 8 + plane_bytes)
        dur = s["time_linearize_ms"] / s["linearize_launches"] * 1e-3
        kern["ba_linearize"] = dict(bytes=per_launch, ms=dur * 1e3, share=s["time_linearize_ms"] / s["time_device_ms"])
    kern["pcg"] = dict(ms=s["time_pcg_ms"], share=s["time_pcg_ms"] / s["time_device_ms"],
                       iterations=s["pcg_iterations"], reduced_dim=s["reduced_dim"])
    # DRAM traffic per launch from the committed `ncu --set full` capture of this command (scripts/extract_traffic.py)
    traffic = {}
    for tname in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath):
            traffic = json.load(open(tpath))
            break

    def dram(*names):
        vals = [traffic[n]["dram_bytes_per_launch"] for n in names if n in traffic]
        return float(sum(vals)) if vals else None

    if "ba_schur" in kern:
        # the Schur phase: its arithmetic intensity (~ 22 flop/B against the planes) is above the fp64 machine
        # balance (37.2 TFLOP/s / 6.57 TB/s = 5.7 flop/B): the fp64 tensor pipe is its roofline, the HBM figure
        # is reported next to it
        npts = len(pb.points) // world
        kk = nloc / max(npts, 1)
        wc_ = s["jac_planes"] / 2.0 - 4.0  # jac_planes = nres * (wc + 4), nres = 2
        fma = npts * (kk * wc_) ** 2 * 3
        tf = 2.0 * fma / (kern["ba_schur"]["ms"] * 1e-3) / 1e12
        kern["ba_schur"]["kernels"] = "ba_point_blocks + ba_schur_pipe<wc> (fp64 mma.m8n8k4, persistent producer / consumer CTAs)"
        kern["ba_schur"]["fp64_tflops"] = tf
        kern["ba_schur"]["fp64_peak_tflops"] = FP64_TENSOR_PEAK_TFLOPS
        kern["ba_schur"]["fp64_frac"] = tf / FP64_TENSOR_PEAK_TFLOPS
        kern["ba_schur"]["fp64_note"] = ("2*3*(k*wc)^2 flop per point, k = observations per point, wc = camera-side width "
                                         "(full square); peak = DMMA/DFMA rate measured by scripts/bench_dmma.cu")
    dom = max((k for k in kern if "bytes" in kern[k]), key=lambda k: kern[k]["share"])
    ach = kern[dom]["bytes"] / (kern[dom]["ms"] * 1e-3) / 1e9
    dom_traffic = dram("ba_point_blocks", "ba_schur_pipe<9, 0>", "ba_schur_pipe<0, 0>", "ba_schur_mma<9>", "ba_schur_mma<0>", "ba_schur") if dom == "ba_schur" else dram("ba_linearize<1, 5, 0>") or dram("ba_linearize<1, 3>") or dram("ba_linearize<1>")
    roofline = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": pk["hbm"], "unit": "GB/s",
                "frac": ach / pk["hbm"], "traffic": dom_traffic, "peak_source": pk["source"], "kernels": kern}
    flops = 2.0 * 128.0 * my_pair_work * K
    tc_ach = flops / (mt_kernel_ms * 1e-3) / 1e12
    mt_roof = {"kernel": "bf_top2_tc" if pm.last_kernel() == 2 else "bf_top2_f32_cv", "bound": "tensor",
               "achieved": tc_ach, "peak": pk["bf16_sustained"], "unit": "TFLOP/s", "frac": tc_ach / pk["bf16_sustained"],
               "traffic": dram("bf_top2_tc<0>") or dram("bf_top2_tc", "bf_top2_tc<false>"), "peak_source": pk["source"] + ", sustained bf16",
               "note": "2*128 flop per descriptor pair per direction (SURVEY 8d); kernel time = distance kernel only"}

    line = None
    if rank == 0:
        h2d_ba = sum(a.nbytes for a in (pb.obs_shot, pb.obs_point, pb.obs_xy, pb.obs_sigma, pb.points, pb.inst, pb.cam_params))
        d2h_ba = pb.points.nbytes + pb.inst.nbytes + pb.cam_params.nbytes + nobs * 24
        h2d_mt = sum(feats8[i].nbytes for i in needed)
        d2h_mt = sum(4 * sizes[a] for a, _ in my_pairs)
        conf = config_of(w, pb, pairs, feats, world)
        conf.update({"lm_iterations_per_step": ba_iters / K, "termination": s["message"],
                     "flush": "inputs larger than L2 (Jacobian planes %.0f MB, descriptor operands %.0f MB)" % (
                         nobs * plane_bytes / 1e6, sum(len(f) for f in feats) * 2 * 288 / 1e6),
                     "descriptor_upload": "uint8 (as stored by opensfm/features.py:526-534), widened on the device"})
        line = {
            "metric": "BA observations/sec", "value": ba_value, "unit": "observations/s", "n_gpus": world,
            "steps": K, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / K, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": conf, "value_run": ba_value_run,
            "ba_ms_per_step": ba_dev_ms / K, "ba_run_ms_per_step": 1e3 * ba_run_s / K, "match_ms_per_step": mt_dev_ms / K,
            "e2e": {"value": ba_e2e, "unit": "observations/s", "h2d_bytes_per_step": int(h2d_ba),
                    "d2h_bytes_per_step": int(d2h_ba)},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roofline,
            "match": {"metric": "descriptor-pairs/sec", "value": mt_value, "unit": "descriptor-pairs/s", "dtype": "bf16->f32",
                      "pairs": len(pairs), "descriptor_pairs_per_step": pair_work_total,
                      "images_resident_on_rank0": len(needed),
                      "e2e": {"value": mt_e2e, "unit": "descriptor-pairs/s", "h2d_bytes_per_step": int(h2d_mt),
                              "d2h_bytes_per_step": int(d2h_mt)},
                      "roofline": mt_roof},
        }
        if world == 1 and not args.no_extras:
            try:
                line["extras"] = run_extras(pk, clk.get("sm_mhz"), not args.no_cpu_baseline)
            except Exception as e:  # the extras never take the headline line down
                line["extras"] = {"error": repr(e)}
            try:
                line["extras"]["c5"] = run_c5()
            except Exception as e:
                line["extras"]["c5"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:
            its = CPU_BA_ITERATIONS.get(args.workload, 5)
            v, it, dt = cpu_ba_sample(pb, its)
            line["cpu_baseline"] = {"value": v, "unit": "observations/s", "cores": _CORES,
                                    "omp_threads": int(os.environ.get("OMP_NUM_THREADS", "0")), "kind": "port",
                                    "sample": "%d LM iterations of the same problem (%.1f s); restated Ceres path, OpenMP" % (it, dt)}
            npairs = min(len(pairs), max(_CORES // 2, 16))
            m, n, dtm = cpu_match_sample(feats, pairs, npairs, _CORES)
            line["match"]["cpu_baseline"] = {"value": m, "unit": "descriptor-pairs/s", "cores": _CORES, "kind": "reference",
                                             "sample": "%d symmetric pairs via cv2 BFMatcher, joblib threading (%.1f s)" % (n, dtm)}
        print(json.dumps(line))
    if world > 1:
        tdist.barrier()
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()
