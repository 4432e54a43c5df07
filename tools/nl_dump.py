"""Dump eng.neighbors() (CSR in the caller's order, within-row order included) of the bench workloads' first position
set, so that two builds of the library (SGPR_B200_LIB) can be compared byte for byte.

    python tools/nl_dump.py --workload c3 --out DIR      (writes DIR/nl_<workload>.npz)
"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    w = synth.WORKLOADS[args.workload]
    pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
    pos = pos + np.random.default_rng(123).normal(0, 0.03, pos.shape)   # bench.py's first position set
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"])
    eng = ab.SgprEngine(model, species=w["Zs"])
    first, J, S = eng.neighbors(pos, numbers, cell, True)
    eng.close()
    os.makedirs(args.out, exist_ok=True)
    np.savez(os.path.join(args.out, f"nl_{args.workload}.npz"), first=first, J=J, S=S)
    print(args.workload, "atoms", len(numbers), "pairs", len(J))


if __name__ == "__main__":
    main()
