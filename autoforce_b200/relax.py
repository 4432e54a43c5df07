"""Geometry relaxation on the device: what ASE's ``FIRE`` optimiser does around ``B200Calculator`` in prediction mode,
with positions, velocities and forces kept in GPU memory between steps.

The algorithm is FIRE as ``ase/optimize/fire.py`` of ASE 3.22-3.23 states it with ``downhill_check=False`` (the
default), with ASE's parameter names and defaults; ``include/sgpr_b200.h`` (``sgpr_relax_params``) restates it.  It
differs from ASE in the order of the floating-point sums of the dot products and of |dr|: they are fixed-order device
reductions.  ``DeviceRelax(calc, atoms).run(fmax, steps, interval)`` enqueues ``interval`` steps at a time
(``sgpr_relax_steps``) and synchronises once per interval, to copy the per-step trace, write the positions back to
``atoms`` and call the observer.  The run ends at the first structure with max_i |F_i| < fmax (the starting one
included), like ``Optimizer.run``, or, with ``calc.covloss``, at the first step with max(beta) > ``calc.ediff``; neither
step depends on ``interval``.  The steps of the interval in flight after that step change nothing but still run their
prediction, so a short relaxation wants an ``interval`` near its expected number of steps.

``FixAtoms`` constraints act as in ASE: the forces of the fixed atoms are zero in every use, so those atoms never move.
Single GPU, one model handle: kernel sums, ``torch.distributed`` sharding and other constraints are refused.
Non-periodic and mixed-pbc structures work but size every step (one host synchronisation per step).
"""
from __future__ import annotations

import numpy as np

from .engine import sgpr_relax_params
from .md import SGPR_ERR_RETRY, check_driver, check_species


def fixed_mask(atoms, N):
    """uint8 [N] mask of the atoms that ``FixAtoms`` constraints fix (read duck-typed: class name ``FixAtoms`` and
    ``get_indices()``), or None when there are none; any other constraint is refused."""
    fixed = np.zeros(N, dtype=np.uint8)
    for c in getattr(atoms, "constraints", None) or ():
        if type(c).__name__ != "FixAtoms" or not hasattr(c, "get_indices"):
            raise NotImplementedError("DeviceRelax does not support ASE constraints other than FixAtoms")
        idx = np.asarray(c.get_indices(), dtype=np.int64).reshape(-1)
        if idx.size and (idx.min() < -N or idx.max() >= N):
            raise ValueError(f"FixAtoms index out of range for {N} atoms")
        fixed[idx] = 1
    return fixed if fixed.any() else None


class DeviceRelax:
    """FIRE relaxation of one structure on the GPU of ``calc`` (a ``B200Calculator``).

    ``trace`` holds, per step done so far, the potential energy, max_i |F_i|, FIRE's dt and a after the step's update,
    and the stress / virial of the step's structure."""

    def __init__(self, calc, atoms, dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1, fdec=0.5, astart=0.1, fa=0.99,
                 a=0.1):
        import torch

        check_driver(calc, "DeviceRelax")
        numbers = check_species(calc, atoms)
        N = len(numbers)
        fixed = fixed_mask(atoms, N)
        prm = dict(dt=dt, maxstep=maxstep, dtmax=dtmax, finc=finc, fdec=fdec)
        for k, v in prm.items():
            if not (np.isfinite(float(v)) and float(v) > 0):
                raise ValueError(f"{k} must be a positive number")
        for k, v in dict(astart=astart, fa=fa, a=a).items():
            if not np.isfinite(float(v)):
                raise ValueError(f"{k} must be finite")
        if int(Nmin) != Nmin or Nmin < 0 or Nmin >= 2 ** 31:
            raise ValueError("Nmin must be an integer >= 0")

        self.calc, self.atoms, self.N = calc, atoms, N
        self.cell = np.asarray(atoms.cell, dtype=np.float64).reshape(3, 3)
        self.pbc = np.broadcast_to(np.asarray(atoms.pbc), (3,)).copy()
        self.engine = eng = calc._get_engine(numbers)
        self.covloss = bool(calc.covloss)
        p = sgpr_relax_params()
        for k, v in prm.items():
            setattr(p, k, float(v))
        p.astart, p.fa, p.a = float(astart), float(fa), float(a)
        p.Nmin = int(Nmin)
        p.fmax = 0.0
        p.ediff = float(calc.ediff)
        p.stop_on_uncertain = 1 if self.covloss else 0
        self.params = p
        dev = torch.device("cuda", eng.device)
        self._dev = dev
        f64 = dict(dtype=torch.float64, device=dev)
        self.pos = torch.as_tensor(np.ascontiguousarray(atoms.positions, dtype=np.float64).reshape(N, 3)).to(dev)
        self.vel = torch.zeros((max(N, 1), 3), **f64)
        self.z = torch.as_tensor(np.ascontiguousarray(numbers, dtype=np.int32)).to(dev)
        self.fixed = torch.as_tensor(fixed).to(dev) if fixed is not None else None
        self.F = torch.zeros((max(N, 1), 3), **f64)
        self.beta_d = torch.zeros(max(N, 1), **f64) if self.covloss else None
        self.fire = torch.zeros(6, **f64)
        self.state = torch.zeros(6, dtype=torch.int64, device=dev)
        self._trace_d = None
        self._rows = []
        self.nsteps = 0
        self.repeats = 0          # steps enqueued again after they outgrew the neighbour buffers sized earlier
        self._notified = False
        # a stream of its own: warm steps are captured into CUDA graphs, which the legacy default stream does not allow
        self._stream = torch.cuda.Stream(device=dev)
        self._stream.wait_stream(torch.cuda.current_stream(dev))
        vol = abs(np.linalg.det(self.cell))
        self._vol = vol if vol != 0.0 else -2.0   # calculator/active.py:606-609, as B200Calculator
        with torch.cuda.device(dev), torch.cuda.stream(self._stream):
            for _ in range(2):     # a warm evaluation that outgrew the buffers sized earlier is repeated (it sizes)
                eng.relax_init(self.pos, self.z, self.fixed, self.cell, self.pbc, p, self.F, self.beta_d, self.fire,
                               self.state)
                self._stream.synchronize()
                status, msg = eng.check_status()
                if status != SGPR_ERR_RETRY:
                    break
                self.repeats += 1
            if status:
                raise RuntimeError(f"libsgpr_b200 error {status}: {msg}")
        self._state = self.state.cpu().numpy()

    # ------------------------------------------------------------------ results
    @property
    def converged(self):
        """True when the forces of the current structure met the ``fmax`` of the last ``run``."""
        return bool(self._state[4] >= 0)

    @property
    def stopped(self):
        """True once a step (0 = the starting structure) had max(beta) > ediff: the run cannot continue past it."""
        return bool(self._state[1] >= 0)

    @property
    def stop_step(self):
        return int(self._state[1]) if self.stopped else None

    @property
    def forces(self):
        """Forces of the current positions, zero on fixed atoms (what ASE's ``atoms.get_forces()`` returns)."""
        return self.F[: self.N].cpu().numpy()

    @property
    def velocities(self):
        """FIRE's velocities (ASE time units of FIRE's dt, not physical velocities)."""
        return self.vel[: self.N].cpu().numpy()

    @property
    def beta(self):
        return self.beta_d[: self.N].cpu().numpy() if self.beta_d is not None else None

    @property
    def trace(self):
        """Per step done so far: ``epot`` (eV), ``fmax`` (max_i |F_i|, eV/A), FIRE's ``dt`` and ``a``, ``stress`` [n,6]
        (Voigt xx,yy,zz,yz,xz,xy in eV/A^3, as ``B200Calculator``) and the raw virial ``W`` [n,3,3]."""
        rows = np.concatenate(self._rows) if self._rows else np.zeros((0, 13))
        W = rows[:, 4:].reshape(-1, 3, 3)
        return {
            "epot": rows[:, 0].copy(),
            "fmax": rows[:, 1].copy(),
            "dt": rows[:, 2].copy(),
            "a": rows[:, 3].copy(),
            "stress": (W / self._vol).reshape(-1, 9)[:, [0, 4, 8, 5, 2, 1]],
            "W": W,
        }

    # ------------------------------------------------------------------ driving
    def run(self, fmax=0.05, steps=100000, interval=100, observer=None):
        """Relax until max_i |F_i| < ``fmax`` or ``steps`` steps are done, synchronising every ``interval`` steps
        (write-back of the positions to ``atoms``, ``observer(atoms, step)``).  Returns True when converged, like ASE's
        ``Optimizer.run``.  When the uncertainty stop ends the run, ``calc.on_uncertain(atoms, beta)`` has been called
        once with the atoms at the stop step."""
        import torch

        fmax, steps, interval = float(fmax), int(steps), int(interval)
        if not (np.isfinite(fmax) and fmax >= 0) or steps < 0 or interval < 1:
            raise ValueError("fmax must be finite and >= 0, steps >= 0 and interval >= 1")
        self.params.fmax = fmax
        if self._trace_d is None or self._trace_d.shape[0] < interval:
            self._trace_d = torch.zeros((interval, 13), dtype=torch.float64, device=self._dev)
        with torch.cuda.device(self._dev), torch.cuda.stream(self._stream):
            self._enqueue(0)       # ASE tests the current forces against this fmax before the first step
            done = 0
            while done < steps and not self._frozen():
                n = min(interval, steps - done)
                chunk, retries = 0, 0
                while chunk < n and not self._frozen():
                    k, retry = self._enqueue(n - chunk)
                    chunk += k
                    if retry:
                        if retries >= 4:
                            raise RuntimeError(f"libsgpr_b200: relaxation step {self.nsteps + 1} kept outgrowing the "
                                               "neighbour buffers")
                        retries += 1   # the step outgrew the neighbour buffers and was not done: enqueue it again
                        self.repeats += 1
                done += chunk
                self._write_back()
                if observer is not None and not self.stopped:
                    observer(self.atoms, self.nsteps)
        if self.stopped:
            self._on_stop()
        return self.converged

    def _frozen(self):
        return self.stopped or self.converged

    def _enqueue(self, n):
        """n steps, one synchronisation; returns (steps done, whether the next step must be enqueued again)."""
        eng, start = self.engine, self.nsteps
        eng.relax_steps(self.pos, self.vel, self.z, self.fixed, self.cell, self.pbc, self.params, n, self.F,
                        self._trace_d, self.beta_d, self.fire, self.state)
        self._stream.synchronize()
        self._state = st = self.state.cpu().numpy()
        k = int(st[0]) - start
        if k > 0:
            self._rows.append(self._trace_d[:k].cpu().numpy())
        self.nsteps = int(st[0])
        status, msg = eng.check_status()
        if status == SGPR_ERR_RETRY and st[2]:
            return k, True
        if status and not (status == SGPR_ERR_RETRY and not st[2]):
            self._write_back()
            raise RuntimeError(f"libsgpr_b200 error {status}: relaxation step {int(st[0]) + 1}: {msg}")
        return k, False

    def _write_back(self):
        a = self.atoms
        pos = self.pos[: self.N].cpu().numpy()
        if hasattr(a, "set_positions"):
            a.set_positions(pos)
        else:
            a.positions = pos

    def _on_stop(self):
        if self._notified:
            return
        self._notified = True
        self._write_back()
        beta = self.beta
        c = self.calc
        c.beta = beta
        c.covlog = f"{float(np.max(beta)) if len(beta) else 0.0}"
        if c.on_uncertain is not None:
            c.on_uncertain(self.atoms, beta)
