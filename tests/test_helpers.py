"""Adjacent rows (SURVEY.md 8f): the three stateless helper kernels of the tracking thread.
CPU part: the oracle restatements against float64 math.  GPU part: the CUDA kernels (through the C ABI) bit-exact against
the oracle AND against the outputs of the reference's own kernels on the same inputs (tests/golden/helpersref_scene3.npz, written
by tools/make_golden_helpers.py on a B200)."""
import os
import zlib

import numpy as np
import pytest

from conftest import ROOT
from oracle import oracle as orc


def _scene(n=5000, seed=0):
    rng = np.random.default_rng(seed)
    P = rng.uniform(-20, 20, size=(3, n)).astype(np.float32)
    P[2] = rng.uniform(-5, 60, size=n)
    Pn = rng.normal(size=(3, n)).astype(np.float32)
    Pn /= np.linalg.norm(Pn, axis=0, keepdims=True)
    a = 0.1
    R = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]], np.float32).ravel()
    t = np.array([0.3, -0.2, 0.5], np.float32)
    Ow = (-(R.reshape(3, 3).T @ t)).astype(np.float32)
    maxd = rng.uniform(5, 80, size=n).astype(np.float32)
    return P, Pn, R, t, Ow, maxd, (maxd * 1.2).astype(np.float32), (maxd * 0.05).astype(np.float32)


K = dict(fx=718.856, fy=718.856, cx=607.19, cy=185.2)
BOX = dict(min_x=0.0, max_x=1241.0, min_y=0.0, max_y=376.0)
FRUSTUM = dict(min_x=0, max_x=1241, min_y=0, max_y=376, n_levels=8, log_scale_factor=float(np.log(np.float32(1.2))), view_cos_angle=0.5)
GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "helpersref_scene3.npz")


def gpu_case():
    """The inputs of the GPU test: a 20000-point scene and 50000 descriptor pairs."""
    rng = np.random.default_rng(5)
    dl, dr = rng.integers(0, 256, size=(3000, 32), dtype=np.uint8), rng.integers(0, 256, size=(3100, 32), dtype=np.uint8)
    il, ir = rng.integers(0, 3000, size=50000).astype(np.int32), rng.integers(0, 3100, size=50000).astype(np.int32)
    return _scene(20000, 3), (il, ir, dl, dr)


def checksum(scene, ham):
    h = 0
    for a in (*scene, *ham):
        h = zlib.crc32(np.ascontiguousarray(a).tobytes(), h)
    return h


def test_oracle_projection_matches_float64():
    P, Pn, R, t, Ow, *_ = _scene()
    u, v, iz, ok = orc.project_points(P, R, t, **K, min_x=0, max_x=1241, min_y=0, max_y=376)
    Pc = R.reshape(3, 3).astype(np.float64) @ P.astype(np.float64) + t[:, None]
    pos = Pc[2] > 1e-3
    assert np.allclose(u[pos], K["fx"] * Pc[0, pos] / Pc[2, pos] + K["cx"], rtol=1e-4, atol=1e-2)
    assert ((u[~(Pc[2] > 0)] == -1) & (ok[~(Pc[2] > 0)] == 0)).all()
    assert 0 < ok.sum() < len(ok)


def test_oracle_logf_and_hamming():
    L = orc.lib()
    for x in np.random.default_rng(1).uniform(1e-3, 1e3, size=500).astype(np.float32):
        assert abs(L.orc_logf(float(x)) - np.log(np.float64(x))) < 1e-6 * max(1.0, abs(np.log(x)))
    rng = np.random.default_rng(2)
    dl, dr = rng.integers(0, 256, size=(50, 32), dtype=np.uint8), rng.integers(0, 256, size=(60, 32), dtype=np.uint8)
    il, ir = rng.integers(0, 50, size=300), rng.integers(0, 60, size=300)
    want = np.unpackbits(dl[il] ^ dr[ir], axis=1).sum(1)
    assert np.array_equal(orc.hamming_pairs(il, ir, dl, dr), want)


def test_oracle_in_frustum_flags_are_consistent():
    P, Pn, R, t, Ow, maxd, ima, imi = _scene()
    iz, u, v, lvl, vc, ok = orc.in_frustum(P, Pn, maxd, ima, imi, R, t, Ow, **K, min_x=0, max_x=1241, min_y=0, max_y=376,
                                           n_levels=8, log_scale_factor=float(np.log(np.float32(1.2))), view_cos_angle=0.5)
    m = ok == 1
    assert 0 < m.sum() < len(m)
    assert (vc[m] >= 0.5).all() and (lvl[m] >= 0).all() and (lvl[m] < 8).all() and (iz[m] > 0).all()


@pytest.mark.gpu
def test_helpers_match_oracle_and_reference_kernels():
    import torch
    from jetson_slam_b200 import frontend
    dev = torch.device("cuda", 0)
    scene, (il, ir, dl, dr) = gpu_case()
    P, Pn, R, t, Ow, maxd, ima, imi = scene
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dP, dPn, dR, dt_, dOw, dmd, dima, dimi = map(tt, (P, Pn, R, t, Ow, maxd, ima, imi))
    # --- projection
    got = [x.cpu().numpy() for x in frontend.project_points(dP, dR, dt_, **K, **BOX)]
    want_proj = orc.project_points(P, R, t, **K, **BOX)
    for g, w in zip(got, want_proj):
        assert np.array_equal(g.view(np.uint8), w.view(np.uint8))
    # --- Hamming pairs
    d = frontend.hamming_pairs(tt(il), tt(ir), tt(dl), tt(dr)).cpu().numpy()
    assert np.array_equal(d, orc.hamming_pairs(il, ir, dl, dr))
    # --- frustum
    got = [x.cpu().numpy() for x in frontend.in_frustum(dP, dPn, dmd, dima, dimi, dR, dt_, dOw, **K, **FRUSTUM)]
    want = orc.in_frustum(P, Pn, maxd, ima, imi, R, t, Ow, **K, **FRUSTUM)
    m = want[5] == 1
    assert np.array_equal(got[5], want[5]) and m.sum() > 100
    for g, w in zip(got[:5], want[:5]):
        assert np.array_equal(g[m].view(np.uint8), w[m].view(np.uint8))
    # --- the reference's own kernels on the same inputs (their stored outputs)
    ref = np.load(GOLDEN_REF)
    assert int(ref["input_checksum"]) == checksum(scene, (il, ir, dl, dr)), "the seeded inputs changed: regenerate with tools/make_golden_helpers.py"
    for k, w in zip(("proj_u", "proj_v", "proj_iz", "proj_ok"), want_proj):
        assert np.array_equal(ref[k].view(np.uint8), w.view(np.uint8)), f"reference projection kernel != oracle ({k})"
    assert np.array_equal(ref["frustum_ok"], want[5]), "reference frustum kernel != oracle"
    for k, w in zip(("frustum_iz", "frustum_u", "frustum_v", "frustum_level", "frustum_view_cos"), want[:5]):
        assert np.array_equal(ref[k].view(np.uint8), w[m].view(np.uint8)), f"reference frustum outputs != oracle ({k})"
    assert np.array_equal(ref["hamming"], d)


@pytest.mark.gpu
def test_resident_map_pool_equals_the_stateless_frustum_kernel():
    """SURVEY.md 8(f2): the map-point SoA stays on the device (jsfe_mappool_*); a frame sends ids + pose.  Must equal jsfe_in_frustum /
    the oracle on the gathered arrays, before and after some map points move."""
    import torch
    from jetson_slam_b200 import frontend
    dev = torch.device("cuda", 0)
    N = 30000
    P, Pn, R, t, Ow, maxd, ima, imi = _scene(N, 11)
    pool = frontend.MapPool(N + 100)
    slots = np.random.default_rng(2).permutation(N + 100)[:N].astype(np.int32)     # map point k lives in slot slots[k]
    pool.update(slots, P, Pn, maxd, ima, imi)
    fr = dict(min_x=0, max_x=1241, min_y=0, max_y=376, n_levels=8, log_scale_factor=float(np.log(np.float32(1.2))), view_cos_angle=0.5)

    def check(query, Pq, Pnq, mdq, imaq, imiq):
        got = [x.cpu().numpy() for x in pool.in_frustum(torch.from_numpy(slots[query]).to(dev), R, t, Ow, **K, **fr)]
        want = orc.in_frustum(Pq, Pnq, mdq, imaq, imiq, R, t, Ow, **K, **fr)
        m = want[5] == 1
        assert np.array_equal(got[5], want[5]) and m.sum() > 50
        for g, w in zip(got[:5], want[:5]):
            assert np.array_equal(g[m].view(np.uint8), w[m].view(np.uint8))

    q = np.random.default_rng(3).permutation(N)[:12000]          # this frame's local map: a subset, in any order
    check(q, np.ascontiguousarray(P[:, q]), np.ascontiguousarray(Pn[:, q]), maxd[q], ima[q], imi[q])
    moved = q[:500]                                                # LocalMapping moves some points
    P2 = P.copy()
    P2[:, moved] += np.float32(0.25)
    pool.update(slots[moved], np.ascontiguousarray(P2[:, moved]), np.ascontiguousarray(Pn[:, moved]), maxd[moved], ima[moved], imi[moved])
    check(q, np.ascontiguousarray(P2[:, q]), np.ascontiguousarray(Pn[:, q]), maxd[q], ima[q], imi[q])
    with pytest.raises(frontend.JsfeError):
        pool.update(np.array([N + 100], np.int32), P[:, :1], Pn[:, :1], maxd[:1], ima[:1], imi[:1])
    pool.close()
