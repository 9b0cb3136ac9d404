"""SURVEY.md 8(f1): ORBmatcher::SearchByProjection(Frame&, const Frame&, th, bMono) fused on the device.

Pin      : tests/golden/sbpref_*.npz are outputs of the REFERENCE'S OWN host code -- src/ORBmatcher.cpp:1647-1963 and :2097-2138,
           src/Frame.cpp:464-479, 569-639 and 696-706, cut out of the reference checkout by line range at build time and compiled
           unmodified against minimal Frame / MapPoint / cv::Mat stand-ins (oracle/ref_build/sbp_slice/, `make -C oracle/ref_build
           sbp`); its two device calls run the oracle's restatements of those kernels, which are pinned against the reference's
           kernels on a B200 (tests/test_helpers.py).  tools/make_golden_sbp.py wrote the fixtures; tests/sbp_cases.py regenerates
           the inputs from seeds.
CPU part : the C oracle (oracle/jsfe_oracle.c: orc_search_by_projection) against those fixtures, against an independent pure-Python
           transliteration of the host loops in float32 arithmetic, plus the sequential-semantics corner cases.
GPU part : the CUDA path through the C ABI (jsfe_build_frame_grid + jsfe_search_by_projection) bit-exact against the oracle AND
           against the reference fixtures."""
import math

import numpy as np
import pytest

import sbp_cases
from jetson_slam_b200 import synth
from oracle import oracle as orc

F = np.float32
K, BOUNDS, MBF = synth.SBP_K, synth.SBP_BOUNDS, synth.SBP_MBF
SF = [F(1.2) ** 0]
for _ in range(7):
    SF.append(F(SF[-1] * F(1.2)))
SF = np.array(SF, F)


make_scene = synth.projection_scene


# ------------------------------------------------------------------------- literal transliteration (pure Python, float32)
def py_reference(last, cur, R, t, th, level_mode, th_high=100, check_orientation=True):
    COLS, ROWS, HL = 64, 48, 30
    mnx, mxx, mny, mxy = (F(BOUNDS[k]) for k in ("min_x", "max_x", "min_y", "max_y"))
    winv, hinv = F(COLS) / (mxx - mnx), F(ROWS) / (mxy - mny)

    def c_round(v):   # C round(): half away from zero
        return int(math.floor(float(v) + 0.5)) if v >= 0 else -int(math.floor(-float(v) + 0.5))

    grid = [[[] for _ in range(ROWS)] for _ in range(COLS)]
    for i in range(len(cur["x"])):
        px, py = c_round((cur["x"][i] - mnx) * winv), c_round((cur["y"][i] - mny) * hinv)
        if 0 <= px < COLS and 0 <= py < ROWS:
            grid[px][py].append(i)
    u, v, iz, ok = orc.project_points(last["P"], R, t, **K, **BOUNDS)    # the pinned kernel restatement
    n = last["P"].shape[1]
    nbr = [[] for _ in range(n)]
    fx_mbf = F(MBF)
    for i in range(n):
        if not ok[i]:
            continue
        lo = int(last["octave"][i])
        r = F(th) * SF[lo]
        mn, mx = (lo, -1) if level_mode == 1 else (0, lo) if level_mode == 2 else (lo - 1, lo + 1)
        x, y = u[i], v[i]
        cx0 = max(0, int(math.floor((x - mnx - r) * winv)))
        if cx0 >= COLS:
            continue
        cx1 = min(COLS - 1, int(math.ceil((x - mnx + r) * winv)))
        if cx1 < 0:
            continue
        cy0 = max(0, int(math.floor((y - mny - r) * hinv)))
        if cy0 >= ROWS:
            continue
        cy1 = min(ROWS - 1, int(math.ceil((y - mny + r) * hinv)))
        if cy1 < 0:
            continue
        check = mn > 0 or mx >= 0
        for ix in range(cx0, cx1 + 1):
            for iy in range(cy0, cy1 + 1):
                for idx in grid[ix][iy]:
                    if check:
                        if cur["octave"][idx] < mn:
                            continue
                        if mx >= 0 and cur["octave"][idx] > mx:
                            continue
                    dx, dy = cur["x"][idx] - x, cur["y"][idx] - y
                    if abs(dx) < r and abs(dy) < r:
                        if cur["occupied"][idx]:
                            continue
                        if cur["uright"][idx] > 0:
                            ur = x - fx_mbf * iz[i]
                            if abs(ur - cur["uright"][idx]) > r:
                                continue
                        nbr[i].append(idx)
    cur_match = [-1] * len(cur["x"])
    best_idx2, best_dist, rot_bin = [-1] * n, [256] * n, [-1] * n
    hist = [[] for _ in range(HL)]
    nmatches = 0
    factor = F(1.0) / F(HL)
    for i in range(n):
        bd, bi = 256, -1
        for idx in nbr[i]:
            d = int(np.unpackbits(last["desc"][i] ^ cur["desc"][idx]).sum())
            if d < bd:
                bd, bi = d, idx
        if bd <= th_high:
            cur_match[bi] = i
            best_idx2[i], best_dist[i] = bi, bd
            nmatches += 1
            if check_orientation:
                rot = last["angle"][i] - cur["angle"][bi]
                if rot < 0.0:
                    rot = rot + F(360.0)
                b = c_round(rot * factor)
                if b == HL:
                    b = 0
                rot_bin[i] = b
                hist[b].append(bi)
    sizes = [len(h) for h in hist]
    if check_orientation:
        m1 = m2 = m3 = 0
        i1 = i2 = i3 = -1
        for b, s in enumerate(sizes):
            if s > m1:
                m3, m2, m1, i3, i2, i1 = m2, m1, s, i2, i1, b
            elif s > m2:
                m3, m2, i3, i2 = m2, s, i2, b
            elif s > m3:
                m3, i3 = s, b
        if F(m2) < F(0.1) * F(m1):
            i2 = i3 = -1
        elif F(m3) < F(0.1) * F(m1):
            i3 = -1
        for b in range(HL):
            if b not in (i1, i2, i3):
                for idx in hist[b]:
                    cur_match[idx] = -1
                    nmatches -= 1
    return dict(nmatches=nmatches, best_idx2=np.array(best_idx2), best_dist=np.array(best_dist), rot_bin=np.array(rot_bin),
                cur_match=np.array(cur_match), hist=np.array(sizes))


def run_oracle(last, cur, R, t, th, level_mode, **kw):
    return orc.search_by_projection(last, cur, R, t, **K, **BOUNDS, mbf=MBF, th=th, scale_factors=SF, level_mode=level_mode, **kw)


def assert_same(a, b):
    assert a["nmatches"] == b["nmatches"]
    for k in ("best_idx2", "best_dist", "rot_bin", "cur_match", "hist"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k


# --------------------------------------------------------------------------------- reference fixtures (the parity pin of row f1)
def _fixture(name):
    import os
    from conftest import ROOT
    g = np.load(os.path.join(ROOT, "tests", "golden", f"sbpref_{name}.npz"))
    c = sbp_cases.build(name)
    assert int(g["input_checksum"]) == sbp_cases.checksum(c), "the seeded inputs changed: regenerate with tools/make_golden_sbp.py"
    assert int(g["level_mode"]) == c["expect_mode"], "bForward / bBackward of the reference's pose test"
    return c, int(g["nmatches"]), g["cur_match"]


def _api_kwargs(c):
    return dict(th=c["th"], level_mode=c["expect_mode"], check_orientation=c["check_orientation"])


@pytest.mark.parametrize("name", list(sbp_cases.CASES))
def test_oracle_equals_the_reference_host_code(name):
    c, want_n, want_cm = _fixture(name)
    r = run_oracle(c["kept_last"], c["frame_cur"], c["R"], c["t"], **_api_kwargs(c))
    assert r["nmatches"] == want_n and want_n > 100
    assert np.array_equal(sbp_cases.oracle_api_result_in_frame_indices(r, c, len(want_cm)), want_cm)


def test_oracle_equals_the_reference_host_code_on_more_seeds():
    """Three more seeds, one per level window, so that the fixtures above are not the only inputs the restatement is checked on."""
    for name in sbp_cases.MORE_CASES:
        c, want_n, want_cm = _fixture(name)
        r = run_oracle(c["kept_last"], c["frame_cur"], c["R"], c["t"], **_api_kwargs(c))
        assert r["nmatches"] == want_n > 100
        assert np.array_equal(sbp_cases.oracle_api_result_in_frame_indices(r, c, len(want_cm)), want_cm)


# ---------------------------------------------------------------------------------------------------------- CPU tests
def test_grid_matches_the_host_loops():
    _, cur, _, _ = make_scene(n_cur=2000, seed=3)
    cur["x"][:5] = [0.0, 1240.9, 1241.0, 9.7, 9.69]       # edge columns; round() may push one out of the grid
    start, items = orc.assign_features_to_grid(cur["x"], cur["y"], *(BOUNDS[k] for k in ("min_x", "max_x", "min_y", "max_y")))
    winv, hinv = F(64) / F(1241), F(48) / F(376)
    cells = {}
    for i in range(len(cur["x"])):
        px = int(math.floor(float(cur["x"][i] * winv) + 0.5)); py = int(math.floor(float(cur["y"][i] * hinv) + 0.5))
        if 0 <= px < 64 and 0 <= py < 48:
            cells.setdefault(px * 48 + py, []).append(i)
    assert start[0] == 0 and start[-1] == sum(len(v) for v in cells.values())
    for c in range(64 * 48):
        assert list(items[start[c]:start[c + 1]]) == cells.get(c, []), c


@pytest.mark.parametrize("level_mode,th,check", [(0, 7.0, True), (1, 15.0, True), (2, 7.0, True), (0, 15.0, False)])
def test_oracle_equals_literal_transliteration(level_mode, th, check):
    last, cur, R, t = make_scene(n_cur=500, n_last=300, seed=10 + level_mode)
    got = run_oracle(last, cur, R, t, th, level_mode, check_orientation=check)
    want = py_reference(last, cur, R, t, th, level_mode, check_orientation=check)
    assert_same(got, want)
    assert got["nmatches"] > 20


def test_oracle_ties_and_overwrites_follow_the_host_order():
    # identical descriptors everywhere: every candidate ties, so the arg-min is the first candidate in (ix, iy, insertion) order
    last, cur, R, t = make_scene(n_cur=400, n_last=300, seed=5, clustered=True, dup_desc=True)
    last["desc"][:] = cur["desc"][0]
    got = run_oracle(last, cur, R, t, 15.0, 0)
    want = py_reference(last, cur, R, t, 15.0, 0)
    assert_same(got, want)
    m = got["best_idx2"] >= 0
    assert m.sum() > 50 and (got["best_dist"][m] == 0).all()
    # several points claim the same keypoint: the highest point index (last assignment) survives unless any of them is culled
    claimed = {}
    for i in np.nonzero(m)[0]:
        claimed.setdefault(int(got["best_idx2"][i]), []).append(int(i))
    assert max(len(v) for v in claimed.values()) > 1
    kept_bins = set(np.argsort(-got["hist"], kind="stable")[:3].tolist())
    for idx, pts in claimed.items():
        if all(got["rot_bin"][p] in kept_bins for p in pts) and got["hist"][got["rot_bin"][pts]].min() >= 0.1 * got["hist"].max():
            assert got["cur_match"][idx] == max(pts)


def test_oracle_degenerate_inputs():
    last, cur, R, t = make_scene(n_cur=50, n_last=40, seed=8)
    empty_last = dict(P=np.zeros((3, 0), F), octave=np.zeros(0, np.int32), angle=np.zeros(0, F), desc=np.zeros((0, 32), np.uint8))
    r = run_oracle(empty_last, cur, R, t, 7.0, 0)
    assert r["nmatches"] == 0 and (r["cur_match"] == -1).all()
    empty_cur = {k: v[:0] for k, v in cur.items()}
    r = run_oracle(last, empty_cur, R, t, 7.0, 0)
    assert r["nmatches"] == 0 and (r["best_idx2"] == -1).all() and (r["best_dist"] == 256).all()


# ---------------------------------------------------------------------------------------------------------- GPU tests
def _to_dev(last, cur, R, t):
    import torch
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return ({k: d(v) for k, v in last.items()}, {k: (None if v is None else d(v)) for k, v in cur.items()}, d(R.astype(F)), d(t.astype(F)))


def run_cuda(last, cur, R, t, th, level_mode, **kw):
    import torch
    from jetson_slam_b200 import frontend
    keep = _to_dev(last, cur, R, t)          # keep every device tensor alive until the results are on the host
    out = frontend.search_by_projection(keep[0], keep[1], keep[2], keep[3], **K, **BOUNDS, mbf=MBF, th=th, scale_factors=SF,
                                        level_mode=level_mode, **kw)
    torch.cuda.synchronize()
    res = {k: out[k].cpu().numpy() for k in ("best_idx2", "best_dist", "rot_bin", "cur_match", "hist")}
    res["nmatches"] = int(out["n_matches"].cpu()[0])
    res["grid"] = (out["grid"][0].cpu().numpy(), out["grid"][1].cpu().numpy())
    del keep
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("level_mode,th,check", [(0, 7.0, True), (1, 15.0, True), (2, 7.0, True), (0, 15.0, False)])
def test_cuda_matches_oracle(level_mode, th, check):
    last, cur, R, t = make_scene(n_cur=3412, n_last=3000, seed=20 + level_mode)
    got = run_cuda(last, cur, R, t, th, level_mode, check_orientation=check)
    want = run_oracle(last, cur, R, t, th, level_mode, check_orientation=check)
    start, items = orc.assign_features_to_grid(cur["x"], cur["y"], *(BOUNDS[k] for k in ("min_x", "max_x", "min_y", "max_y")))
    assert np.array_equal(got["grid"][0], start) and np.array_equal(got["grid"][1][:len(items)], items)
    assert_same(got, want)
    assert want["nmatches"] > 500


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(sbp_cases.CASES))
def test_cuda_equals_the_reference_host_code(name):
    c, want_n, want_cm = _fixture(name)
    got = run_cuda(c["kept_last"], c["frame_cur"], c["R"], c["t"], **_api_kwargs(c))
    assert got["nmatches"] == want_n
    assert np.array_equal(sbp_cases.oracle_api_result_in_frame_indices(got, c, len(want_cm)), want_cm)


@pytest.mark.gpu
def test_cuda_ties_clusters_and_degenerate_inputs():
    last, cur, R, t = make_scene(n_cur=2000, n_last=1500, seed=31, clustered=True, dup_desc=True)
    last["desc"][:] = cur["desc"][0]
    assert_same(run_cuda(last, cur, R, t, 15.0, 0), run_oracle(last, cur, R, t, 15.0, 0))
    last, cur, R, t = make_scene(n_cur=64, n_last=40, seed=32)
    cur_none = dict(cur)
    cur_none["occupied"] = None
    want = run_oracle(last, dict(cur, occupied=np.zeros(64, np.uint8)), R, t, 7.0, 0)
    assert_same(run_cuda(last, cur_none, R, t, 7.0, 0), want)
    empty_last = dict(P=np.zeros((3, 0), F), octave=np.zeros(0, np.int32), angle=np.zeros(0, F), desc=np.zeros((0, 32), np.uint8))
    got = run_cuda(empty_last, cur, R, t, 7.0, 0)
    assert got["nmatches"] == 0 and (got["cur_match"] == -1).all()


@pytest.mark.gpu
def test_device_resident_chain_extract_stereo_view_grid_search():
    """Rows a12 / f1 / f4 end to end on the device: extract two stereo frames, stereo-match, unpack the current frame with
    jsfe_frame_view, and run the fused SearchByProjection on those device arrays (uRight and descriptors straight from the slot
    view) -- then check against the oracle fed with host copies of the same arrays."""
    import torch
    from jetson_slam_b200 import frontend
    from jetson_slam_b200.configs import CONFIGS
    cfg = CONFIGS["C1"]
    h, w = cfg.height, cfg.width
    la, ra = synth.stereo_pair(h, w, 77)
    shift = lambda im: np.roll(im, (1, 3), axis=(0, 1))      # the "current" frame: the same scene moved by (3, 1) pixels
    fe = frontend.Frontend(**cfg.extractor_kwargs(), max_images=4)
    fe.set_images(np.stack([la, ra, shift(la), shift(ra)]))
    fe.extract(0, 4)
    fe.stereo_match(cfg.mb, cfg.mbf, 0, 2)
    torch.cuda.synchronize()
    # last frame (pair 0) on the host: keypoints with depth become map points (that is SLAM-core work, done on the CPU)
    kA, dA = fe.get_keypoints(0)
    urA, depA, _, _ = fe.get_stereo(0)
    good = depA > 0
    fx = fy = cfg.fx
    cx, cy = w / 2.0, h / 2.0
    xA, yA = kA[0].astype(F), kA[1].astype(F)
    P = np.stack([(xA[good] - cx) * depA[good] / fx, (yA[good] - cy) * depA[good] / fy, depA[good]]).astype(F)
    last = dict(P=P, octave=kA[4][good].astype(np.int32), angle=kA[3][good].view(F).copy(), desc=dA[good].copy())
    R, t = np.eye(3, dtype=F).ravel(), np.zeros(3, F)
    # current frame (pair 1): device arrays only
    view = frontend.frame_view(fe, 2)
    sv = fe.slot_view(2)
    kB, dB = fe.get_keypoints(2)
    urB, _, _, _ = fe.get_stereo(1)
    n = kB.shape[1]
    keys = view["keys"].cpu().numpy().view(frontend.CV_KEYPOINT_DTYPE).reshape(-1)[:n]
    assert np.array_equal(keys["x"], kB[0].astype(F)) and np.array_equal(keys["y"], kB[1].astype(F))          # Frame.cpp:143-148
    assert np.array_equal(keys["response"], kB[2].astype(F)) and np.array_equal(keys["angle"].view(np.int32), kB[3])
    assert np.array_equal(keys["octave"], kB[4]) and np.array_equal(keys["size"], kB[5].astype(F)) and (keys["class_id"] == -1).all()
    cur_dev = dict(x=view["x"][:n], y=view["y"][:n], octave=view["octave"][:n], angle=view["angle"][:n],
                   uright=frontend.DevicePtr(sv.u_right), occupied=None, desc=frontend.DevicePtr(sv.desc))
    dl = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in last.items()}
    dR, dt = torch.from_numpy(R).cuda(), torch.from_numpy(t).cuda()
    bounds = dict(min_x=0.0, max_x=float(w), min_y=0.0, max_y=float(h))
    kw = dict(fx=fx, fy=fy, cx=cx, cy=cy, **bounds, mbf=cfg.mbf, th=7.0, scale_factors=fe.scale, level_mode=0)
    out = frontend.search_by_projection(dl, cur_dev, dR, dt, **kw)
    torch.cuda.synchronize()
    cur_host = dict(x=kB[0].astype(F), y=kB[1].astype(F), octave=kB[4].astype(np.int32), angle=kB[3].view(F).copy(), uright=urB,
                    occupied=np.zeros(n, np.uint8), desc=dB)
    want = orc.search_by_projection(last, cur_host, R, t, **kw)
    got = {k: out[k].cpu().numpy() for k in ("best_idx2", "best_dist", "rot_bin", "cur_match", "hist")}
    got["nmatches"] = int(out["n_matches"].cpu()[0])
    assert_same(got, want)
    assert want["nmatches"] > 30          # the shifted scene really is re-found
    fe.close()


def test_oracle_regression_pins():
    """The oracle restatement must not drift: fixed seeded scenes against tests/golden/adj_sbp_oracle.npz (tools/make_golden_adjacent.py)."""
    import os
    from conftest import ROOT
    g = np.load(os.path.join(ROOT, "tests", "golden", "adj_sbp_oracle.npz"))
    for mode in (0, 1, 2):
        last, cur, R, t = make_scene(n_cur=900, n_last=700, seed=40 + mode)
        r = run_oracle(last, cur, R, t, 7.0 if mode != 1 else 15.0, mode)
        assert r["nmatches"] == int(g[f"m{mode}_nmatches"]) and r["nmatches"] > 100
        for k in ("best_idx2", "best_dist", "rot_bin", "cur_match", "hist"):
            assert np.array_equal(np.asarray(r[k]), g[f"m{mode}_{k}"]), (mode, k)
