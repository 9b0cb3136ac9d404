#!/usr/bin/env python
"""Reference outputs for the helper kernels of SURVEY 8(f): runs the reference's OWN projection, frustum and Hamming kernels
(oracle/_ref/libjsref.so, its src/cuda compiled unmodified for sm_100a) on the inputs of tests/test_helpers.py's GPU test and stores
what they return in tests/golden/helpersref_scene3.npz, with a checksum of the inputs.  Frustum outputs other than the flag are
stored for the points the reference keeps (flag 1) only: the others are not defined.
usage: python tools/make_golden_helpers.py [--out DIR]        (needs a GPU and oracle/_ref/libjsref.so)"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ref  # noqa: E402
from test_helpers import BOX, FRUSTUM, K, checksum, gpu_case  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    args = ap.parse_args()
    if not ref.available():
        raise SystemExit("oracle/_ref/libjsref.so is missing: make -C oracle/ref_build")
    import torch
    dev = torch.device("cuda", 0)
    scene, (il, ir, dl, dr) = gpu_case()
    P, Pn, R, t, Ow, maxd, ima, imi = scene
    tt = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    dP, dPn, dR, dt_, dOw, dmd, dima, dimi = map(tt, (P, Pn, R, t, Ow, maxd, ima, imi))
    L = ref.lib()
    p = lambda x: C.c_void_p(x.data_ptr())
    n = P.shape[1]
    u, v, iz = (torch.empty(n, device=dev) for _ in range(3))
    ok = torch.empty(n, dtype=torch.uint8, device=dev)
    L.jsref_project_points(n, p(dP[0]), p(dP[1]), p(dP[2]), p(dR), p(dt_), K["fx"], K["fy"], K["cx"], K["cy"], BOX["min_x"], BOX["max_x"],
                           BOX["min_y"], BOX["max_y"], p(u), p(v), p(iz), p(ok))
    iz2, u2, v2, vc2 = (torch.zeros(n, device=dev) for _ in range(4))
    lv2 = torch.zeros(n, dtype=torch.int32, device=dev)
    ok2 = torch.empty(n, dtype=torch.uint8, device=dev)
    fr = FRUSTUM
    L.jsref_in_frustum(n, p(dP[0]), p(dP[1]), p(dP[2]), p(dPn[0]), p(dPn[1]), p(dPn[2]), p(dmd), p(dima), p(dimi), p(dR), p(dt_),
                       p(dOw), K["fx"], K["fy"], K["cx"], K["cy"], fr["min_x"], fr["max_x"], fr["min_y"], fr["max_y"], fr["n_levels"],
                       fr["log_scale_factor"], fr["view_cos_angle"], p(iz2), p(u2), p(v2), p(lv2), p(vc2), p(ok2))
    d2 = torch.empty(len(il), dtype=torch.int32, device=dev)
    t_il, t_ir, t_dl, t_dr = tt(il), tt(ir), tt(dl), tt(dr)   # keep the device buffers alive across the call
    L.jsref_hamming_pairs(len(il), p(t_il), p(t_ir), p(t_dl), p(t_dr), p(d2))
    torch.cuda.synchronize()
    h = lambda x: x.cpu().numpy()
    keep = h(ok2) == 1
    out = dict(proj_u=h(u), proj_v=h(v), proj_iz=h(iz), proj_ok=h(ok), frustum_ok=h(ok2),
               frustum_iz=h(iz2)[keep], frustum_u=h(u2)[keep], frustum_v=h(v2)[keep], frustum_level=h(lv2)[keep],
               frustum_view_cos=h(vc2)[keep], hamming=h(d2), input_checksum=np.array(checksum(scene, (il, ir, dl, dr)), np.uint64))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "helpersref_scene3.npz")
    np.savez_compressed(path, **out)
    print(f"{path}: {int(h(ok).sum())} projected, {int(keep.sum())} in the frustum, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
