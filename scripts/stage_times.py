"""Stage times (us) of the frozen stress frame.

    python scripts/stage_times.py [--features 4096] [--repeat 30] [--flush]

Prints one JSON line: the mean device time per frame, the per-stage times and those of k_syrk / k_chol_prior.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def one(n_feat, repeat, flush):
    import numpy as np
    import torch
    import bench
    from orcvio_b200 import api
    snap = bench.make_frame(0, n_feat)
    fr = api.Frame(bench.N_CLONES, 0, bench.NOISE_VAR, 0.95, -1.0, bench.TRI["cost_threshold"],
                   bench.TRI["init_final_dist_threshold"])
    out = fr.update(fr.prepare_inputs(snap))
    fr.load(snap)
    buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda") if flush else None
    for _ in range(3):
        fr.run(1)
    tot = 0.0
    for _ in range(repeat):
        if flush:
            buf.zero_()
            torch.cuda.synchronize()
        tot += fr.run(1)
    _, st = fr.run(10, stages=True)
    kt = fr.kernel_times()
    st = {k: round(v, 1) for k, v in st.items()}
    st.update(syrk=round(kt["syrk"], 1), chol_prior=round(kt["chol_prior"], 1))
    print(json.dumps(dict(features=n_feat, gated=int(((out["status"] & 2) != 0).sum()), us_per_frame=round(tot / repeat, 1),
                          stages=st, chk=float(np.abs(out["delta_x"]).sum()))), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--features", type=int, default=4096)
    ap.add_argument("--repeat", type=int, default=30)
    ap.add_argument("--flush", action="store_true")
    args = ap.parse_args()
    one(args.features, args.repeat, args.flush)


if __name__ == "__main__":
    main()
