"""Runs the fused SA-scale kernel on layer-1 / layer-2 shaped inputs (for timing and ncu captures).
usage: python tools/fused_probe.py [case-index ...] [hoist=1] [dyn=1]
  hoist=1 (default)  the hoisted form the model runs (first conv in the per-point table); hoist=0 the literal 3-conv stack
  dyn=1              developer build only (SSD3D_LIB=3dssd_b200/libssd3d_dev.so): force the run-time-shape kernel, for
                     A/B timing against the compile-time-shape kernels"""
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = importlib.import_module("3dssd_b200")
P = pkg.params
synth = importlib.import_module("3dssd_b200.synth")

CASES = [  # n, c, m, nsample, mlp, radius shell
    (16384, 1, 4096, 64, [32, 32, 64], (0.4, 0.8)),      # layer 1 scale 3
    (16384, 1, 4096, 32, [16, 16, 32], (0.0, 0.2)),      # layer 1 scale 1
    (4096, 64, 1024, 32, [64, 64, 128], (0.0, 0.4)),     # layer 2 scale 1
    (4096, 64, 1024, 64, [64, 96, 128], (0.8, 1.6)),     # layer 2 scale 3
]


def main():
    dev = torch.device("cuda:0")
    sel = [int(a) for a in sys.argv[1:] if "=" not in a] or range(len(CASES))
    kv = dict(a.split("=") for a in sys.argv[1:] if "=" in a)
    if "dyn" in kv:   # developer build only (nvcc -DSSD3D_DEV_HOOKS, loaded through SSD3D_LIB)
        import ctypes
        dl = ctypes.CDLL(pkg.LIB_PATH)
        dl.ssd3d_dev_set_fused_dynamic(int(kv["dyn"]))
    hoist = int(kv.get("hoist", 1))
    rng = np.random.default_rng(0)
    B = 8
    pts = torch.from_numpy(synth.kitti_like(B, 16384, seed=1000)).to(dev)
    for i in sel:
        n, c, m, k, mlp, (lo, hi) = CASES[i]
        xyz = pts[:, :n, :3].contiguous()
        feats = torch.randn((B, n, c), device=dev)
        fidx = pkg.farthest_point_sample(m, xyz)
        new_xyz = pkg.gather_point(xyz, fidx)
        idx, cnt = pkg.query_ball_point_dilated(lo, hi, k, xyz, new_xyz)
        prm, scopes, cin = {}, [], c + 3
        for j, cout in enumerate(mlp):
            P._conv_init(rng, prm, "s/conv0_%d" % j, cin, cout, True)
            scopes.append("s/conv0_%d" % j)
            cin = cout
        pp = P.prepare(prm, dev)
        if hoist:
            zconv, wxs, n1s = pp.hoisted([scopes[0]], True, c)
            hst = pp.fused_stack(scopes[1:], True, n1s[0], limit=0)
            p_hi, p_lo = pkg.split_rows(feats)
            z, _ = pkg.linear_tc(p_hi, p_lo, zconv, relu=False, want_f32=True, want_split=False)
            run = lambda: pkg.sa_mlp_fused_hoisted(xyz, z, 0, wxs[0], new_xyz, idx, cnt, hst)
        else:
            stack = pp.fused_stack(scopes, True, c + 3, limit=0)
            run = lambda: pkg.sa_mlp_fused(xyz, feats, new_xyz, idx, cnt, stack)
        for _ in range(3):
            run()
        torch.cuda.synchronize()
        ts = []
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); run(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        rows = B * m * k
        print("case %d n=%d c=%d m=%d k=%d mlp=%s rows=%d hoist=%d %s: %.1f us" % (i, n, c, m, k, mlp, rows, hoist, " ".join(sys.argv[1:]),
                                                                              1e3 * float(np.median(ts))), flush=True)


if __name__ == "__main__":
    main()
