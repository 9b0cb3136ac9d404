"""ctypes binding of oracle/_ref/libsbpref.so: the reference's OWN host code of ORBmatcher::SearchByProjection(Frame&, const Frame&,
th, bMono) (src/ORBmatcher.cpp:1647-1963) with Frame::AssignFeaturesToGrid / GetFeaturesInArea / PosInGrid (src/Frame.cpp:464-479,
569-639, 696-706), cut out of the reference checkout at build time and compiled unmodified (oracle/ref_build/sbp_slice/).
TEST INFRASTRUCTURE: used by tools/make_golden_sbp.py to produce tests/golden/sbpref_*.npz.  Never imported by the product."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "_ref", "libsbpref.so")
_lib = None


def available() -> bool:
    return os.path.exists(LIB)


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(LIB)
        vp, ci, f = C.c_void_p, C.c_int, C.c_float
        L.jsref_search_by_projection.restype = ci
        L.jsref_search_by_projection.argtypes = ([ci] + [vp] * 7 + [ci] + [vp] * 8 + [f] * 11 + [vp, ci, ci, ci, vp, vp])
        _lib = L
    return _lib


def pose_matrix(R9, t3):
    T = np.eye(4, dtype=np.float32)
    T[:3, :3] = np.asarray(R9, np.float32).reshape(3, 3)
    T[:3, 3] = np.asarray(t3, np.float32)
    return T


def search_by_projection(frame_last, frame_cur, pose_last, pose_cur, fx, fy, cx, cy, min_x, max_x, min_y, max_y, mbf, mb, th,
                         scale_factors, mono=False, check_orientation=True):
    """frame_last: dict(P[3,n], has_mp[n], outlier[n], octave, angle, desc[n,32]) over ALL keypoints of the last frame;
    frame_cur: dict(x, y, octave, angle, uright, occupied, desc[m,32]).  -> dict(nmatches, cur_match[m] (last-frame keypoint index
    or -1), level_mode)."""
    a = lambda v, t: np.ascontiguousarray(v, t)
    P = a(frame_last["P"], np.float32)
    n = P.shape[1]
    hm, ol = a(frame_last["has_mp"], np.uint8), a(frame_last["outlier"], np.uint8)
    lo, la, ld = a(frame_last["octave"], np.int32), a(frame_last["angle"], np.float32), a(frame_last["desc"], np.uint8)
    x, y = a(frame_cur["x"], np.float32), a(frame_cur["y"], np.float32)
    m = len(x)
    co, ca = a(frame_cur["octave"], np.int32), a(frame_cur["angle"], np.float32)
    cu, occ, cd = a(frame_cur["uright"], np.float32), a(frame_cur["occupied"], np.uint8), a(frame_cur["desc"], np.uint8)
    pl, pc = a(pose_last, np.float32), a(pose_cur, np.float32)
    sf = a(scale_factors, np.float32)
    cm = np.full(max(m, 1), -1, np.int32)
    mode = C.c_int(0)
    p = lambda arr: arr.ctypes.data
    nm = lib().jsref_search_by_projection(n, p(P), p(hm), p(ol), p(lo), p(la), p(ld), p(pl), m, p(x), p(y), p(co), p(ca), p(cu), p(occ),
                                          p(cd), p(pc), fx, fy, cx, cy, min_x, max_x, min_y, max_y, mbf, mb, th, p(sf), len(sf),
                                          int(mono), int(check_orientation), p(cm), C.addressof(mode))
    return dict(nmatches=int(nm), cur_match=cm[:m].copy(), level_mode=int(mode.value))
