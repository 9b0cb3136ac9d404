"""Seeded frame pairs for the SearchByProjection parity tests (SURVEY.md 8(f1)).  One definition shared by tools/make_golden_sbp.py
(which runs the REFERENCE's host code on them and commits its outputs) and by the tests (which run the oracle and the CUDA path on the
same inputs and compare with those outputs)."""
import zlib

import numpy as np

from jetson_slam_b200 import synth

F = np.float32
SF = np.cumprod(np.array([1.0] + [1.2] * 7, F)).astype(F)
MB = float(F(synth.SBP_MBF) / F(synth.SBP_K["fx"]))

# name -> (scene kwargs, th, which level window the poses ask for, bMono, mbCheckOrientation, fraction of last keypoints without map point,
#          fraction flagged outlier)
CASES = {
    "window_seed50": (dict(n_cur=1500, n_last=1200, seed=50), 7.0, 0, False, True, 0.2, 0.1),
    "forward_seed51": (dict(n_cur=1500, n_last=1200, seed=51), 15.0, 1, False, True, 0.2, 0.1),
    "backward_seed52": (dict(n_cur=1500, n_last=1200, seed=52), 7.0, 2, False, True, 0.2, 0.1),
    "mono_forward_pose_seed53": (dict(n_cur=1200, n_last=900, seed=53), 15.0, 1, True, True, 0.1, 0.0),
    "no_orientation_seed54": (dict(n_cur=1200, n_last=900, seed=54), 15.0, 0, False, False, 0.0, 0.0),
    "clustered_ties_seed55": (dict(n_cur=600, n_last=500, seed=55, clustered=True, dup_desc=True), 15.0, 0, False, True, 0.1, 0.05),
    "c4_size_seed56": (dict(n_cur=3412, n_last=3412, seed=56), 7.0, 0, False, True, 0.3, 0.05),
}
# more seeds, checked against the oracle only: one scene size, every level window
MORE_CASES = {f"more_seed{seed}": (dict(n_cur=1100, n_last=800, seed=seed), 7.0 if mode != 1 else 15.0, mode, False, True, 0.15, 0.05)
              for seed, mode in ((91, 0), (92, 1), (93, 2))}


def build(name):
    kw, th, want_mode, mono, check, p_nomp, p_out = CASES[name] if name in CASES else MORE_CASES[name]
    last, cur, R, t = synth.projection_scene(**kw)
    if kw.get("dup_desc"):
        last["desc"][:] = cur["desc"][0]            # every candidate ties: the arg-min is decided by the host's enumeration order
    n = last["P"].shape[1]
    rng = np.random.default_rng(kw["seed"] + 1000)
    has_mp = (rng.random(n) >= p_nomp).astype(np.uint8)
    outlier = (rng.random(n) < p_out).astype(np.uint8)
    frame_last = dict(P=last["P"], has_mp=has_mp, outlier=outlier, octave=last["octave"], angle=last["angle"], desc=last["desc"])
    # poses: the current one is the scene's; the last one is placed so that tlc = Rlw*twc + tlw = (0, 0, dz) selects the level window
    Rm = np.asarray(R, F).reshape(3, 3)
    twc = -(Rm.T.astype(np.float64) @ np.asarray(t, np.float64))
    dz = {0: 0.0, 1: 2.0, 2: -2.0}[want_mode]
    pose_cur = np.eye(4, dtype=F); pose_cur[:3, :3] = Rm; pose_cur[:3, 3] = t
    pose_last = np.eye(4, dtype=F); pose_last[:3, 3] = (np.array([0.0, 0.0, dz]) - twc).astype(F)
    camera = dict(**synth.SBP_K, **synth.SBP_BOUNDS, mbf=synth.SBP_MBF, mb=MB)
    keep = np.nonzero((has_mp != 0) & (outlier == 0))[0]
    kept = dict(P=np.ascontiguousarray(last["P"][:, keep]), octave=last["octave"][keep], angle=last["angle"][keep], desc=last["desc"][keep])
    expect_mode = 0 if mono else want_mode
    return dict(frame_last=frame_last, frame_cur=cur, pose_last=pose_last, pose_cur=pose_cur, camera=camera, th=th, mono=mono,
                check_orientation=check, keep=keep, kept_last=kept, R=np.asarray(R, F), t=np.asarray(t, F), expect_mode=expect_mode)


def checksum(c):
    h = 0
    for d in (c["frame_last"], c["frame_cur"]):
        for k in sorted(d):
            h = zlib.crc32(np.ascontiguousarray(d[k]).tobytes(), h)
    for k in ("pose_last", "pose_cur"):
        h = zlib.crc32(np.ascontiguousarray(c[k]).tobytes(), h)
    return h


def oracle_api_result_in_frame_indices(res, c, n_cur):
    """The oracle / CUDA API works on the kept last-frame points; map its cur_match back to last-frame keypoint indices."""
    cm = np.asarray(res["cur_match"]).copy()
    m = cm >= 0
    cm[m] = c["keep"][cm[m]]
    return cm
