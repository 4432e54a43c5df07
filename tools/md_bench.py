"""Molecular dynamics on the device (DeviceMD) against the host loop an ASE user runs today.

    python tools/md_bench.py [--out FILE] [--workloads c2,c3]

For each workload (bench.py's c2 / c3 cells and models) and each of NVE / Langevin, with and without covloss:
  device  DeviceMD.run(K, interval=100): positions, momenta and forces stay on the GPU, one host synchronisation per
          100 steps (thermo rows, write-back to the atoms);
  host    what ASE's VelocityVerlet / Langevin do around B200Calculator.calculate, restated in numpy (ASE is not a
          dependency): per step the calculator call (atoms.copy(), H2D of the positions, D2H of the forces, the results
          dict, max |F|), the integrator's N x 3 array work and, for Langevin, 2 x 3N normal deviates.
Steps/s are host clock around whole runs that end in a device synchronisation, after a warm-up run of each path.  The
covloss rows use a model with choli and an ediff that never trips.  The card's name and power limit are read in the
same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FS = 0.09822694788464063
KB = 8.617330337217213e-05
MASS = {3: 6.94, 8: 15.999, 15: 30.974, 16: 32.06, 29: 63.546}
STEPS = {"c2": (3000, 300), "c3": (400, 60)}   # device steps, host steps


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # pragma: no cover
        return {"gpu": None, "error": str(e)}


class Atoms:
    def __init__(self, positions, numbers, cell, momenta):
        self.positions, self.numbers, self.cell, self.pbc = positions.copy(), numbers, cell, np.array([True] * 3)
        self.momenta = momenta.copy()

    def copy(self):
        return Atoms(self.positions, self.numbers, self.cell, self.momenta)

    def get_masses(self):
        return np.array([MASS[int(z)] for z in self.numbers])

    def get_momenta(self):
        return self.momenta.copy()

    def set_momenta(self, p):
        self.momenta = np.array(p)

    def set_positions(self, r):
        self.positions = np.array(r)


def host_loop(calc, atoms, steps, dt_fs, T=None, friction=None, seed=0):
    """ASE's VelocityVerlet.step / Langevin.step around calculator.calculate, in numpy."""
    dt = dt_fs * FS
    m = atoms.get_masses()[:, None]
    rng = np.random.default_rng(seed)
    F = calc.calculate(atoms)["forces"]
    for _ in range(steps):
        p = atoms.get_momenta()
        p += 0.5 * dt * F
        if T is None:
            atoms.set_positions(atoms.positions + dt * p / m)
        else:
            g = friction / FS
            c1, c2 = np.exp(-g * dt), np.sqrt(1 - np.exp(-2 * g * dt))
            xi = rng.standard_normal(size=(2,) + p.shape)     # ASE's Langevin draws two N x 3 sets per step
            atoms.set_positions(atoms.positions + 0.5 * dt * p / m)
            p = c1 * p + c2 * np.sqrt(m * KB * T) * xi[0]
            atoms.set_positions(atoms.positions + 0.5 * dt * p / m)
        atoms.set_momenta(p)
        res = calc.calculate(atoms)
        F = res["forces"]
        calc.maximum_force = float(np.abs(F).max())
        atoms.set_momenta(atoms.get_momenta() + 0.5 * dt * F)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "md_bench.json"))
    ap.add_argument("--workloads", default="c2,c3")
    args = ap.parse_args()
    import torch

    import autoforce_b200 as ab
    from autoforce_b200 import synth

    info = gpu_info()
    results = []
    for name in args.workloads.split(","):
        w = synth.WORKLOADS[name]
        pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
        N = len(numbers)
        model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"], with_choli=True)
        m = np.array([MASS[int(z)] for z in numbers])[:, None]
        mom0 = np.random.default_rng(2).normal(size=(N, 3)) * np.sqrt(m * KB * 300.0)
        n_dev, n_host = STEPS[name]
        for covloss in (False, True):
            for T in (None, 300.0):
                kw = dict(temperature_K=T, friction=0.01) if T is not None else {}
                calc = ab.B200Calculator(model, covloss=covloss, ediff=1e300)
                md = ab.DeviceMD(calc, Atoms(pos, numbers, cell, mom0), timestep=1.0, seed=3, **kw)
                md.run(200, interval=100)   # warm-up: sizing step, graph capture
                t0 = time.perf_counter()
                md.run(n_dev, interval=100)
                t_dev = time.perf_counter() - t0
                hc = ab.B200Calculator(model, covloss=covloss, ediff=1e300)
                host_loop(hc, Atoms(pos, numbers, cell, mom0), 20, 1.0, T, 0.01)   # warm-up
                atoms = Atoms(pos, numbers, cell, mom0)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                host_loop(hc, atoms, n_host, 1.0, T, 0.01)
                t_host = time.perf_counter() - t0
                row = {"workload": name, "atoms": N, "inducing": model.M, "ensemble": "NVE" if T is None else "Langevin",
                       "covloss": covloss, "device_steps": n_dev, "device_steps_per_s": n_dev / t_dev,
                       "device_ms_per_step": 1e3 * t_dev / n_dev, "host_steps": n_host,
                       "host_steps_per_s": n_host / t_host, "host_ms_per_step": 1e3 * t_host / n_host,
                       "speedup": (n_dev / t_dev) / (n_host / t_host)}
                print(json.dumps(row), flush=True)
                results.append(row)
                for c in (calc, hc):
                    if c._engine is not None:
                        c._engine.close()
    out = {"tool": "tools/md_bench.py", **info, "interval": 100, "timestep_fs": 1.0, "results": results}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "results"}))


if __name__ == "__main__":
    main()
