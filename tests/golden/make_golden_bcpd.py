#!/usr/bin/env python
"""Generate tests/golden/bcpd.npz by running the UNMODIFIED reference probreg/bcpd.py (v0.3.7).

Same loading trick as make_golden.py (a bare parent package, open3d stubbed, probreg._math replaced by float32 numpy
restatements) plus ``_math.inverse_multiquadric_kernel`` restated from cc/math_utils.cc:37-39 in float32.  Runs only in
the build container; the .npz is committed.   Usage:  python tests/golden/make_golden_bcpd.py
"""
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden as mg  # noqa: E402

from oracle import cpd_oracle as orc  # noqa: E402


def imq_f32(x, y, c=1.0):
    x32, y32 = np.asarray(x, dtype=np.float32), np.asarray(y, dtype=np.float32)
    d2 = ((x32[:, None, :] - y32[None, :, :]) ** 2).sum(-1, dtype=np.float32)
    return (np.float32(1.0) / np.sqrt(d2 + np.float32(c))).astype(np.float32)


def main():
    mg.load_reference()
    sys.modules["probreg._math"].inverse_multiquadric_kernel = imq_f32
    bcpd = importlib.import_module("probreg.bcpd")
    out = {}
    rng = np.random.default_rng(21)
    src, tgt = orc.synthetic_pair(700)
    tgt = tgt[:650]
    tgt_o = np.vstack([tgt, rng.uniform(-3.0, 3.0, (40, 3))])                 # far outliers
    m = src.shape[0]
    ts = orc.apply_rigid(src, orc.rot_z(27.0), np.array([0.1, -0.2, 0.3]), 1.02)
    obj = bcpd.CombinedBCPD(src)
    cases = {
        "a": (tgt, 1.0, np.full(m, 1.0 / m), np.ones(m), 0.05, 0.0),
        "b": (tgt, 1.02, rng.dirichlet(np.ones(m)), rng.uniform(0.0, 0.02, m), 0.004, 0.1),
        "c": (tgt_o, 0.97, rng.dirichlet(np.ones(m) * 0.3), rng.uniform(0.0, 1e-3, m), 3e-4, 0.3),
        "d": (tgt_o, 1.0, np.full(m, 1.0 / m), np.zeros(m), 3e-4, 0.0),      # w = 0 with dead columns
    }
    out["source"], out["t_source"], out["target"], out["target_outl"] = src, ts, tgt, tgt_o
    for tag, (x, scale, alpha, sdiag, s2, w) in cases.items():
        es = obj.expectation_step(ts, x, scale, alpha, np.diag(sdiag), s2, w)
        out[tag + "_target"] = np.array("target_outl" if x is tgt_o else "target")
        out[tag + "_scale"], out[tag + "_alpha"], out[tag + "_sdiag"], out[tag + "_sigma2"], out[tag + "_w"] = scale, alpha, sdiag, s2, w
        out[tag + "_nu_d"], out[tag + "_nu"], out[tag + "_np"], out[tag + "_px"], out[tag + "_xhat"] = es.nu_d, es.nu, es.n_p, es.px, es.x_hat
        mine = orc.bcpd_expectation_step(ts, x, scale, alpha, sdiag, s2, w)
        print(tag, "oracle vs reference: nu_d %.1e nu %.1e px %.1e dead %d" % (
            np.abs(mine.nu_d - es.nu_d).max(), np.abs(mine.nu - es.nu).max(), np.abs(mine.px - es.px).max(), int((es.nu_d == 0).sum())))
    # a short registration (5 iterations) of the reference's CombinedBCPD on a small pair: the end-to-end fixture
    s_small, t_small = orc.synthetic_pair(120)
    f = np.array([[1.0, 0.5, 0.0], [0.0, 1.0, 0.7], [0.3, 0.0, 1.0]])
    t_small = t_small + 0.01 * np.sin(2 * np.pi * t_small.dot(f))
    reg = bcpd.CombinedBCPD(s_small, lmd=2.0)
    tfm = reg.registration(t_small, w=0.05, maxiter=5, tol=-1.0)
    out["reg_source"], out["reg_target"] = s_small, t_small
    out["reg_rot"], out["reg_t"], out["reg_scale"], out["reg_v"] = tfm.rigid_trans.rot, tfm.rigid_trans.t, tfm.rigid_trans.scale, tfm.v
    np.savez_compressed(os.path.join(HERE, "bcpd.npz"), **out)
    # the float32 inverse of the kernel matrix that registration used (condition ~1e10: LAPACK's result depends on the CPU and the
    # thread count), so that the test can hand the same inverse to the package and compare the rest on any host
    np.savez_compressed(os.path.join(HERE, "bcpd_gmat_inv.npz"), gmat_inv=reg.gmat_inv)
    print("wrote bcpd.npz, bcpd_gmat_inv.npz")


if __name__ == "__main__":
    main()
