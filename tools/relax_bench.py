"""Geometry relaxation on the device (DeviceRelax) against the host FIRE loop an ASE user runs today.

    python tools/relax_bench.py [--out FILE] [--workloads c2,c3]

For each workload (bench.py's c2 / c3 cells and models), with and without covloss, at fmax = 0 so that the number of
steps is fixed:
  device  DeviceRelax.run(fmax=0, steps=K, interval=100): positions, velocities and forces stay on the GPU, one host
          synchronisation per 100 steps (trace rows, write-back to the atoms);
  host    what ase.optimize.FIRE does around B200Calculator.calculate, restated in numpy (ASE is not a dependency): per
          step the calculator call (atoms.copy(), H2D of the positions, D2H of the forces, the results dict), the
          max |F_i| test and FIRE's N x 3 array work.
  frozen  a step enqueued after the converged step (move, place, commit and finish do nothing, the prediction still runs):
          what a run pays for each step of the interval in flight when it converges.
Then both paths relax the same rattled 256-atom cell on a lattice-well model (one inducing LCE cut from the perfect fcc
Cu cell, mu = -1) to fmax = 0.01: steps to convergence and wall time, the device path at interval 1, 7 and 100 with the
construction of DeviceRelax (its stream, the starting evaluation) timed apart.  Times are host clock around whole runs
that end in a device synchronisation, after a warm-up of each path.  The covloss rows use a model with choli and an ediff that never
trips.  The card's name and power limit are read in the same run.
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

STEPS = {"c2": (2000, 300), "c3": (300, 60)}   # device steps, host steps


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # pragma: no cover
        return {"gpu": None, "error": str(e)}


class Atoms:
    def __init__(self, positions, numbers, cell):
        self.positions, self.numbers, self.cell, self.pbc = positions.copy(), numbers, cell, np.array([True] * 3)

    def copy(self):
        return Atoms(self.positions, self.numbers, self.cell)

    def set_positions(self, r):
        self.positions = np.array(r)


def host_fire(calc, atoms, steps, fmax, dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1, fdec=0.5, astart=0.1,
              fa=0.99, a=0.1):
    """ase.optimize.FIRE.run(fmax, steps) around calculator.calculate, in numpy.  Returns (converged, steps done)."""
    v, Nsteps = None, 0
    for k in range(steps + 1):
        f = calc.calculate(atoms)["forces"]
        if (f ** 2).sum(axis=1).max() < fmax ** 2:
            return True, k
        if k == steps:
            return False, k
        if v is None:
            v = np.zeros((len(f), 3))
        else:
            vf = np.vdot(f, v)
            if vf > 0.0:
                v = (1.0 - a) * v + a * f / np.sqrt(np.vdot(f, f)) * np.sqrt(np.vdot(v, v))
                if Nsteps > Nmin:
                    dt = min(dt * finc, dtmax)
                    a *= fa
                Nsteps += 1
            else:
                v[:] *= 0.0
                a = astart
                dt *= fdec
                Nsteps = 0
        v += dt * f
        dr = dt * v
        normdr = np.sqrt(np.vdot(dr, dr))
        if normdr > maxstep:
            dr = maxstep * dr / normdr
        atoms.set_positions(atoms.positions + dr)


def lattice_well(rep=4, rattle=0.08):
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    pos, cell, numbers = synth.fcc(rep, [29], 0.0, 0)
    base = dict(lmax=3, nmax=3, xi=4.0, rc=6.0, kind="sesoap", radii={1: 0.5}, default_radius=1.0)
    probe = ab.SgprEngine(ab.SgprModel.from_envs([], **base), species=[29])
    try:
        first, J, S = probe.neighbors(pos, numbers, cell, True)
    finally:
        probe.close()
    envs = synth.cut_environments(pos, cell, True, numbers, 6.0, [0], first, J, S)
    model = ab.SgprModel.from_envs(envs, mu=np.array([-1.0]), mean_w={29: 0.0}, vscale={29: 1.0}, **base)
    return model, pos + np.random.default_rng(1).normal(0, rattle, pos.shape), cell, numbers


def frozen_ms(rx, n):
    """ms per step enqueued after convergence: the driver is made converged (any finite forces meet fmax = 1e300, so
    the call's first kernel sets the converged step) and n steps are timed after a warm-up that captures their graph."""
    import torch

    assert rx.run(fmax=1e300, steps=0) and rx.converged
    k = rx.nsteps
    with torch.cuda.device(rx._dev), torch.cuda.stream(rx._stream):
        rx._enqueue(5)
        t0 = time.perf_counter()
        rx._enqueue(n)
        t = time.perf_counter() - t0
    assert rx.nsteps == k
    return 1e3 * t / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_relax_bench.json"))
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
        n_dev, n_host = STEPS[name]
        for covloss in (False, True):
            calc = ab.B200Calculator(model, covloss=covloss, ediff=1e300)
            rx = ab.DeviceRelax(calc, Atoms(pos, numbers, cell))
            rx.run(fmax=0.0, steps=200, interval=100)   # warm-up: sizing step, graph capture
            t0 = time.perf_counter()
            rx.run(fmax=0.0, steps=n_dev, interval=100)
            t_dev = time.perf_counter() - t0
            assert rx.nsteps == 200 + n_dev
            t_frozen = frozen_ms(rx, 100 if name == "c2" else 30)
            hc = ab.B200Calculator(model, covloss=covloss, ediff=1e300)
            host_fire(hc, Atoms(pos, numbers, cell), 20, 0.0)   # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host_fire(hc, Atoms(pos, numbers, cell), n_host, 0.0)
            t_host = time.perf_counter() - t0
            row = {"workload": name, "atoms": N, "inducing": model.M, "covloss": covloss, "device_steps": n_dev,
                   "device_steps_per_s": n_dev / t_dev, "device_ms_per_step": 1e3 * t_dev / n_dev, "host_steps": n_host,
                   "host_steps_per_s": n_host / t_host, "host_ms_per_step": 1e3 * t_host / n_host,
                   "speedup": (n_dev / t_dev) / (n_host / t_host), "frozen_step_ms": t_frozen}
            print(json.dumps(row), flush=True)
            results.append(row)
            for c in (calc, hc):
                if c._engine is not None:
                    c._engine.close()

    model, pos, cell, numbers = lattice_well()
    conv = {"model": "lattice well: one inducing LCE of the perfect fcc Cu cell, mu = -1", "atoms": len(numbers),
            "rattle_A": 0.08, "fmax": 0.01}
    for interval in (100, 7, 1):
        calc = ab.B200Calculator(model)
        calc.calculate(Atoms(pos, numbers, cell))   # warm-up of the handle
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rx = ab.DeviceRelax(calc, Atoms(pos, numbers, cell))
        t1 = time.perf_counter()
        ok = rx.run(fmax=0.01, steps=5000, interval=interval)
        t2 = time.perf_counter()
        conv[f"device_interval_{interval}"] = {"converged": bool(ok), "steps": rx.nsteps, "construct_s": t1 - t0,
                                               "run_s": t2 - t1, "wall_s": t2 - t0,
                                               "steps_after_convergence": -rx.nsteps % interval}
        if interval == 100:
            conv["frozen_step_ms"] = frozen_ms(rx, 100)
        calc._engine.close()
    calc = ab.B200Calculator(model)
    calc.calculate(Atoms(pos, numbers, cell))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ok, k = host_fire(calc, Atoms(pos, numbers, cell), 5000, 0.01)
    conv["host"] = {"converged": bool(ok), "steps": int(k), "wall_s": time.perf_counter() - t0}
    calc._engine.close()
    print(json.dumps(conv), flush=True)
    out = {"tool": "tools/relax_bench.py", **info, "interval": 100, "results": results, "lattice_well": conv}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k not in ("results", "lattice_well")}))


if __name__ == "__main__":
    main()
