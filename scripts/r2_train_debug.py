"""Debug of two round-2 findings: (A) full-width L12 x4 gradients at a small spatial size, (B) c-DCSCN training from random
weights diverging after ~50 steps.  Prints per-variable gradient errors / the loss curve under several engine options."""
import glob
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "dcscn-super-resolution_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import dcscn_oracle as O  # noqa: E402
from conftest import load_golden_weights, GOLDEN  # noqa: E402
from helper import engine as E  # noqa: E402
from helper import loader  # noqa: E402

which = sys.argv[1] if len(sys.argv) > 1 else "AB"

if "A" in which:
    for model, scale in (("dcscn_L12_F196to48_Sc4_NIN_A64_PS_R1F32", 4), ("dcscn_L12_F196to48_NIN_A64_PS_R1F32", 2)):
        cfg = O.OracleConfig(scale=scale)
        wts = {k: v.astype(np.float64) for k, v in load_golden_weights(model).items()}
        n, h, w = 2, 12, 10
        g = np.random.RandomState(21)
        x = (g.rand(n, h, w, 1) * 255).astype(np.float32)
        x2 = (g.rand(n, scale * h, scale * w, 1) * 255).astype(np.float32)
        y = np.clip(x2 + g.randn(n, scale * h, scale * w, 1) * 10, 0, 255).astype(np.float32)
        _, _, gref = O.Oracle(cfg, wts, torch.float64).loss_and_grads(x.astype(np.float64), x2.astype(np.float64), y.astype(np.float64), keep_prob=1.0)
        for opts in [{}, {"conv_impl": 1}]:
            eng = E.Engine(E.make_config(scale=scale, dropout_keep=1.0))
            eng.set_params({k: v.astype(np.float32) for k, v in wts.items()})
            for k, v in opts.items():
                eng.set_option(k, v)
            loss, mse = eng.train_step_host(x, x2, y, lr=0.002, seed=1, apply_update=False)
            print("A", model[6:20], "x%d" % scale, opts, "mse %.4f" % mse, "norm %.4e" % eng.last_grad_norm, flush=True)
            for name in reversed(list(gref.keys())):
                gr = gref[name]
                got = eng.get_grad(name)
                rel = float(np.abs(got - gr).max() / (np.abs(gr).max() + 1e-30))
                print("     %-34s max|ref| %.3e  max|got| %.3e  rel err %.2e %s" % (name, np.abs(gr).max(), np.abs(got).max(), rel, "BAD" if rel > 2e-3 else ""), flush=True)
            eng.close()

if "C" in which:
    model = "dcscn_L12_F196to48_NIN_A64_PS_R1F32"
    cfg = O.OracleConfig(scale=2)
    wts = {k: v.astype(np.float64) for k, v in load_golden_weights(model).items()}
    n, h, w = 2, 12, 10
    g = np.random.RandomState(21)
    x = (g.rand(n, h, w, 1) * 255).astype(np.float32)
    x2 = (g.rand(n, 2 * h, 2 * w, 1) * 255).astype(np.float32)
    y = np.clip(x2 + g.randn(n, 2 * h, 2 * w, 1) * 10, 0, 255).astype(np.float32)
    _, _, gref = O.Oracle(cfg, wts, torch.float64).loss_and_grads(x.astype(np.float64), x2.astype(np.float64), y.astype(np.float64), keep_prob=1.0)
    eng = E.Engine(E.make_config(scale=2, dropout_keep=1.0))
    eng.set_params({k: v.astype(np.float32) for k, v in wts.items()})
    eng.train_step_host(x, x2, y, lr=0.002, seed=1, apply_update=False)
    for name in ("CNN7/conv_B", "CNN7/prelu/CNN7_prelu", "CNN8/conv_B", "CNN6/conv_B"):
        got, ref = eng.get_grad(name), gref[name]
        d = np.abs(got - ref) / (np.abs(ref).max() + 1e-30)
        idx = np.argsort(-d)[:8]
        al = wts[name.split("/")[0] + "/prelu/" + name.split("/")[0] + "_prelu"]
        print("C", name, "worst channels:", [(int(i), "%.1e" % d[i], "ref %.3e got %.3e alpha %.3e" % (ref[i], got[i], al[i])) for i in idx], flush=True)
    eng.close()

if "B" in which:
    KW = dict(scale=2, layers=7, filters=32, min_filters=8, filters_decay_gamma=1.2, nin_filters=24, nin_filters2=8,
              reconstruct_layers=0, pixel_shuffler_filters=1)
    ds = loader.BatchDataSets(2, "unused", 32, stride_size=16)
    ds.build_batch(os.path.join(GOLDEN, "data", "set14"))
    cfgo = O.OracleConfig(**KW)
    rs = np.random.RandomState(0)
    w0 = {}
    for scope, k, cin, cout, bias, prelu in O.layer_table(cfgo):
        base = scope.split("/")[-1]
        std = np.sqrt(2.0 / (k * k * cin))
        w0[scope + "/conv_W"] = (np.clip(rs.randn(k, k, cin, cout), -2, 2) * std).astype(np.float32)
        if bias:
            w0[scope + "/conv_B"] = np.zeros(cout, np.float32)
        if prelu:
            w0["%s/prelu/%s_prelu" % (scope, base)] = np.full(cout, 0.1, np.float32)
    order = np.random.RandomState(1).permutation(ds.count)
    for opts in [{}, {"host": 1}, {"wgrad_impl": 1}, {"host_repack": 1}, {"conv_impl": 1}]:
        eng = E.Engine(E.make_config(dropout_keep=0.8, **KW))
        eng.set_params(w0)
        host = opts.pop("host", 0) if "host" in opts else 0
        for k, v in opts.items():
            eng.set_option(k, v)
        eng.set_patch_store(ds.input_images, ds.input_interpolated_images, ds.true_images)
        curve = []
        for step in range(160):
            idx = order[(np.arange(20) + step * 20) % ds.count]
            if host:
                xx, xx2, yy = eng.gather_patches(idx)
                loss, mse = eng.train_step_host(xx, xx2, yy, lr=0.002, seed=step)
            else:
                loss, mse = eng.train_step_indexed(idx, lr=0.002, seed=step)
            if step % 10 == 9:
                curve.append("%.0f(%.1f)" % (mse, eng.last_grad_norm))
        print("B", "host" if host else "indexed", opts, "mse(gradnorm) every 10 steps:", " ".join(curve), flush=True)
        eng.close()
