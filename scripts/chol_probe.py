"""Per-phase clock profile of the one-CTA Cholesky (csrc/chol.cuh) on the GPU.

    python scripts/chol_probe.py [--steps all|sample]

Shapes: (180, 17) is k_chol_w_solve on the 30-clone stress frame, (180, 22) k_chol_prior there, (210, 17) the
hybrid state (30 clones + 30 features), (202, 0) a whole 30-clone state, (64, 0) a small one.
"""
import argparse
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from orcvio_b200 import api

SHAPES = [(180, 17), (180, 22), (210, 17), (202, 0), (64, 0)]

ap = argparse.ArgumentParser()
ap.add_argument("--steps", default="all", choices=["all", "sample"])
args = ap.parse_args()

rng = np.random.default_rng(0)
for (m, nx) in SHAPES:
    B = rng.standard_normal((m, m + 20))
    A = B @ B.T + 1e-3 * np.eye(m)
    X = rng.standard_normal((nx, m)) if nx else None
    L, Xs, prof, us = api.chol_probe(A, X, reps=20)
    Lr = np.linalg.cholesky(A)
    err = np.abs(np.tril(L) - Lr).max() / np.abs(Lr).max()
    msg = f"m={m} nx={nx}: {us:.1f} us, rel err L {err:.2e}"
    if nx:
        Xr = np.linalg.solve(Lr, X.T).T
        msg += f", X {np.abs(Xs - Xr).max() / np.abs(Xr).max():.2e}"
    print(msg)
    npan = (m + 7) // 8
    p = prof[:npan].astype(np.int64)
    t0 = p[0, 0]
    print("  step: chain [factor  wait_tile  solve+diag_upd  step]   bulk warp 0 [seen_block  solve  col_q+1  bulk_q+2]   (cycles)")
    if args.steps == "all":
        ks = list(range(npan))
    else:
        ks = list(range(0, min(npan, 4))) + list(range(npan // 2, npan // 2 + 2)) + [npan - 2, npan - 1]
    cols = []
    for k in range(npan):
        r = p[k]
        nxt = p[k + 1, 0] if k + 1 < npan else r[3]
        c = (r[1] - r[0], max(r[2] - r[1], 0), r[3] - max(r[2], r[1]), nxt - r[0],
             r[4] - r[1], r[5] - r[4], r[6] - r[5], r[7] - r[6])
        cols.append(c)
        if k in ks:
            print(f"  {k:3d}: start {r[0]-t0:7d} | factor {c[0]:5d} wait {c[1]:5d} solve_upd {c[2]:5d} step {c[3]:5d}"
                  f" | seen {c[4]:5d} solve {c[5]:5d} col {c[6]:5d} bulk {c[7]:5d}")
    c = np.mean(np.array(cols[:-1], dtype=np.float64), axis=0)   # the last step has no tile below
    print(f"  mean of steps 0..{npan - 2}: factor {c[0]:5.0f} wait {c[1]:5.0f} solve_upd {c[2]:5.0f} step {c[3]:5.0f}"
          f" | seen {c[4]:5.0f} solve {c[5]:5.0f} col {c[6]:5.0f} bulk {c[7]:5.0f}")
    print(f"  total cycles {max(p[npan-1,3], p[npan-1,7])-t0}")
