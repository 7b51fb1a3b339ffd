"""
On-GPU diagnostic: per-layer comparison of the CUDA path against the CPU oracle.
Run under gpurun:  python scripts/gpu_diag.py [--quick]
Prints max|d| of every intermediate tensor for the CUDA-core validation kernels
(conv_impl=1) and the tcgen05 kernels (conv_impl=0) at several fp32-promotion periods.
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "dcscn-super-resolution_b200"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import dcscn_oracle as O  # noqa: E402
from helper import engine as E  # noqa: E402
from helper import tf_bundle  # noqa: E402


def run_case(name, cfg_kwargs, weights, n, h, w, seed=0, precision=E.PRECISION_F16X3, modes=((1, 1), (0, 1), (0, 0), (0, 3), (0, 4000))):
    ocfg = O.OracleConfig(**cfg_kwargs)
    if weights is None:
        weights = O.he_init_weights(ocfg, seed=seed)
    g = np.random.RandomState(seed)
    x = (g.rand(n, h, w, 1) * 255).astype(np.float32)
    s = ocfg.scale
    x2 = (g.rand(n, s * h, s * w, 1) * 255).astype(np.float32)
    o64 = O.Oracle(ocfg, weights, torch.float64)
    y64, inter = o64.forward(x.astype(np.float64), x2.astype(np.float64), return_intermediates=True)
    y32 = O.Oracle(ocfg, weights, torch.float32).forward(x, x2)
    print("== %s  n=%d h=%d w=%d  (fp32-oracle vs fp64-oracle max %.3e)" % (name, n, h, w, np.abs(y32 - y64).max()))
    eng = E.Engine(E.make_config(precision=precision, **{k: v for k, v in cfg_kwargs.items()}))
    eng.set_params(weights)
    xd, x2d = torch.from_numpy(x).cuda(), torch.from_numpy(x2).cuda()
    ok = True
    for impl, seg in modes:
        eng.set_option("seg_chunks", seg)
        eng.set_option("conv_impl", impl)
        t = time.time()
        y = eng.forward(xd, x2d)
        torch.cuda.synchronize()
        dt = time.time() - t
        y = y.cpu().numpy()
        line = "  impl=%s seg=%d  y max|d| vs fp64 %.3e  vs fp32 %.3e (%.1f ms)" % ("ref" if impl else "tc ", seg, np.abs(y - y64).max(), np.abs(y - y32).max(), dt * 1e3)
        bad = not np.isfinite(y).all() or np.abs(y - y64).max() > 2e-3
        print(line + ("   <-- MISMATCH" if bad else ""))
        if "-v" in sys.argv or (bad and "-q" not in sys.argv):
            for k in inter:
                key = "Up-PS" if k == "Up-PS" else k
                if k == "R-CNN":
                    continue
                a = eng.get_activation(key, inter[k].shape)
                d = np.abs(a - inter[k])
                print("      %-8s max|d| %.3e  (ref max %.2e)  nonfinite=%d" % (k, d.max(), np.abs(inter[k]).max(), (~np.isfinite(a)).sum()))
        ok = ok and not bad
    eng.close()
    return ok


def load_golden(name):
    r = tf_bundle.BundleReader(os.path.join(ROOT, "tests", "golden", "models", name + ".ckpt"))
    return {k: r.get_tensor(k) for k in r.keys()}


def main():
    print(torch.cuda.get_device_name(0))
    small = dict(scale=2, layers=4, filters=40, min_filters=24, filters_decay_gamma=1.5, nin_filters=24, nin_filters2=16)
    ok = run_case("small odd", small, None, 1, 20, 37, modes=((1, 1), (0, 1)))
    if "--first" in sys.argv:
        return
    ok &= run_case("small 48", small, None, 2, 48, 48)
    cd = dict(scale=2, layers=7, filters=32, min_filters=8, filters_decay_gamma=1.2, nin_filters=24, nin_filters2=8,
              reconstruct_layers=0, pixel_shuffler_filters=1)
    ok &= run_case("c-DCSCN x2 ckpt", cd, load_golden("dcscn_L7_F32to8_G1.20_NIN_A24_B8_PS_R1F32"), 1, 33, 50)
    ok &= run_case("L12 x2 ckpt", dict(), load_golden("dcscn_L12_F196to48_NIN_A64_PS_R1F32"), 2, 48, 48)
    ok &= run_case("L12 x4 ckpt", dict(scale=4), load_golden("dcscn_L12_F196to48_Sc4_NIN_A64_PS_R1F32"), 1, 24, 40,
                   modes=((1, 1), (0, 1)))
    ok &= run_case("L12 x2 ckpt fast(f16x1)", dict(), load_golden("dcscn_L12_F196to48_NIN_A64_PS_R1F32"), 1, 48, 48,
                   precision=E.PRECISION_F16X1, modes=((0, 1),))
    print("ALL OK" if ok else "SOME MISMATCH")


if __name__ == "__main__":
    main()
