"""Molecular dynamics on the device: what ASE's ``VelocityVerlet`` / ``Langevin`` do around ``B200Calculator`` in
prediction mode, with positions, momenta and forces kept in GPU memory between steps.

``DeviceMD(calc, atoms, ...).run(steps, interval)`` enqueues ``interval`` steps at a time (``sgpr_md_steps``,
include/sgpr_b200.h) and synchronises once per interval: to copy the per-step energies and virials, to write the positions
and momenta back to ``atoms`` and to call the observer.  With ``calc.covloss`` the covloss beta is evaluated every step
and the run ends at the first step with max(beta) > ``calc.ediff``; that step does not depend on ``interval``.

NVE is velocity Verlet in the operation order of ASE's ``VelocityVerlet.step``; NVT is Langevin with the BAOAB splitting
and Philox4x32-10 noise (keyed by ``seed``, counted by atom and step), without ASE's centre-of-mass correction
(``fixcm``).  Positions stay unwrapped, as in ASE.  Single GPU, one model handle: kernel sums, ``torch.distributed``
sharding and ASE constraints are refused.  Non-periodic and mixed-pbc structures work but size every step (one host
synchronisation per step, as ``sgpr_predict`` does for them).
"""
from __future__ import annotations

import numpy as np

from .engine import sgpr_md_params
from .model import MAX_SPECIES

FS = 0.09822694788464063      # ase.units.fs: one femtosecond in ASE time units
KB = 8.617330337217213e-05    # ase.units.kB: Boltzmann constant in eV/K
SGPR_ERR_RETRY = -7


def check_driver(calc, name):
    """What the device drivers (DeviceMD, DeviceRelax) refuse: kernel sums and torch.distributed sharding."""
    if len(getattr(calc, "models", ())) != 1:
        raise NotImplementedError(f"{name} runs a single model handle: kernel sums are not supported")
    _, _, world = calc._dist()
    if world > 1:
        raise NotImplementedError(f"{name} runs on one GPU: torch.distributed sharding is not supported")


def check_species(calc, atoms):
    """atoms.numbers as a flat array; unknown species are refused before any device work."""
    numbers = np.asarray(atoms.numbers).reshape(-1)
    species = set(int(z) for z in calc.model.species()) | set(int(z) for z in numbers)
    if any(z < 1 or z > 118 for z in species) or len(species) > MAX_SPECIES:
        raise ValueError(f"unknown species: atomic numbers {sorted(set(int(z) for z in numbers))} with the model's "
                         f"{sorted(calc.model.species())} (at most {MAX_SPECIES} species of Z 1..118)")
    return numbers


class DeviceMD:
    """MD of one structure on the GPU of ``calc`` (a ``B200Calculator``).

    ``timestep`` in fs; ``temperature_K=None`` means NVE, otherwise Langevin with ``friction`` in 1/fs.  ``masses`` (amu)
    default to ``atoms.get_masses()`` when ``atoms`` has it; momenta come from ``atoms.get_momenta()`` when present, else
    zero.  ``thermo`` holds the per-step potential and kinetic energy, temperature and stress of the steps done so far."""

    def __init__(self, calc, atoms, timestep=1.0, temperature_K=None, friction=None, seed=0, masses=None):
        import torch

        check_driver(calc, "DeviceMD")
        if getattr(atoms, "constraints", None):
            raise NotImplementedError("DeviceMD does not support ASE constraints")
        numbers = check_species(calc, atoms)
        N = len(numbers)
        if masses is None:
            if not hasattr(atoms, "get_masses"):
                raise ValueError("masses are required when atoms has no get_masses()")
            masses = atoms.get_masses()
        masses = np.asarray(masses, dtype=np.float64).reshape(-1)
        if masses.shape != (N,) or not (np.isfinite(masses).all() and (masses > 0).all()):
            raise ValueError(f"masses must be {N} positive finite numbers")
        mom = np.asarray(atoms.get_momenta(), dtype=np.float64).reshape(N, 3) if hasattr(atoms, "get_momenta") else np.zeros((N, 3))
        timestep = float(timestep)
        if not (np.isfinite(timestep) and timestep > 0):
            raise ValueError("timestep must be a positive number of fs")
        langevin = temperature_K is not None
        if langevin:
            temperature_K = float(temperature_K)
            if friction is None or not (np.isfinite(float(friction)) and float(friction) >= 0):
                raise ValueError("Langevin dynamics needs friction >= 0 (1/fs)")
            if not (np.isfinite(temperature_K) and temperature_K >= 0):
                raise ValueError("temperature_K must be >= 0")
        elif friction is not None:
            raise ValueError("friction without temperature_K: NVE has no friction")
        seed = int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must fit in 64 bits")

        self.calc, self.atoms, self.N = calc, atoms, N
        self.masses = masses
        self.cell = np.asarray(atoms.cell, dtype=np.float64).reshape(3, 3)
        self.pbc = np.broadcast_to(np.asarray(atoms.pbc), (3,)).copy()
        self.engine = eng = calc._get_engine(numbers)
        self.covloss = bool(calc.covloss)
        p = sgpr_md_params()
        p.dt = timestep * FS
        p.friction = float(friction) / FS if langevin else 0.0
        p.kT = KB * temperature_K if langevin else 0.0
        p.ediff = float(calc.ediff)
        p.seed = seed
        p.langevin = 1 if langevin else 0
        p.stop_on_uncertain = 1 if self.covloss else 0
        self.params = p
        dev = torch.device("cuda", eng.device)
        self._dev = dev
        f64 = dict(dtype=torch.float64, device=dev)
        self.pos = torch.as_tensor(np.ascontiguousarray(atoms.positions, dtype=np.float64).reshape(N, 3)).to(dev)
        self.mom = torch.as_tensor(np.ascontiguousarray(mom)).to(dev)
        self.z = torch.as_tensor(np.ascontiguousarray(numbers, dtype=np.int32)).to(dev)
        self.mass = torch.as_tensor(masses).to(dev)
        self.F = torch.zeros((max(N, 1), 3), **f64)
        self.beta_d = torch.zeros(max(N, 1), **f64) if self.covloss else None
        self.state = torch.zeros(4, dtype=torch.int64, device=dev)
        self._thermo_d = None
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
                eng.md_init(self.pos, self.z, self.cell, self.pbc, p, self.F, self.beta_d, self.state)
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
    def stopped(self):
        """True once a step (0 = the starting structure) had max(beta) > ediff: the run cannot continue past it."""
        return bool(self._state[1] >= 0)

    @property
    def stop_step(self):
        return int(self._state[1]) if self.stopped else None

    @property
    def forces(self):
        return self.F[: self.N].cpu().numpy()

    @property
    def beta(self):
        return self.beta_d[: self.N].cpu().numpy() if self.beta_d is not None else None

    @property
    def thermo(self):
        """Per step done so far: ``epot``, ``ekin`` (eV), ``temperature`` (K, 3N degrees of freedom), ``stress`` [n,6]
        (Voigt xx,yy,zz,yz,xz,xy in eV/A^3, the potential part, as ``B200Calculator``) and the raw virial ``W`` [n,3,3]."""
        rows = np.concatenate(self._rows) if self._rows else np.zeros((0, 11))
        W = rows[:, 2:].reshape(-1, 3, 3)
        return {
            "epot": rows[:, 0].copy(),
            "ekin": rows[:, 1].copy(),
            "temperature": 2.0 * rows[:, 1] / (3 * max(self.N, 1) * KB),
            "stress": (W / self._vol).reshape(-1, 9)[:, [0, 4, 8, 5, 2, 1]],
            "W": W,
        }

    # ------------------------------------------------------------------ driving
    def run(self, steps, interval=100, observer=None):
        """Advance by ``steps`` steps, synchronising every ``interval`` steps (write-back to ``atoms``, ``observer(atoms,
        step)``).  Returns the number of steps done: fewer than ``steps`` when the uncertainty stop ended the run, in
        which case ``calc.on_uncertain(atoms, beta)`` has been called once with the atoms at the stop step."""
        import torch

        steps, interval = int(steps), int(interval)
        if steps < 0 or interval < 1:
            raise ValueError("steps must be >= 0 and interval >= 1")
        if self.stopped:
            self._on_stop()
            return 0
        if self._thermo_d is None or self._thermo_d.shape[0] < interval:
            self._thermo_d = torch.zeros((interval, 11), dtype=torch.float64, device=self._dev)
        eng, done = self.engine, 0
        with torch.cuda.device(self._dev), torch.cuda.stream(self._stream):
            while done < steps and not self.stopped:
                n = min(interval, steps - done)
                chunk, retries = 0, 0
                while chunk < n and not self.stopped:
                    start = self.nsteps
                    eng.md_steps(self.pos, self.mom, self.z, self.mass, self.cell, self.pbc, self.params, n - chunk, self.F,
                                 self._thermo_d, self.beta_d, self.state)
                    self._stream.synchronize()
                    self._state = st = self.state.cpu().numpy()
                    k = int(st[0]) - start
                    if k > 0:
                        self._rows.append(self._thermo_d[:k].cpu().numpy())
                    chunk += k
                    self.nsteps = int(st[0])
                    status, msg = eng.check_status()
                    if status == SGPR_ERR_RETRY and st[2] and retries < 4:
                        retries += 1   # the step outgrew the neighbour buffers and was not integrated: enqueue it again
                        self.repeats += 1
                        continue
                    if status and not (status == SGPR_ERR_RETRY and not st[2]):
                        self._write_back()
                        raise RuntimeError(f"libsgpr_b200 error {status}: MD step {int(st[0]) + 1}: {msg}")
                done += chunk
                self._write_back()
                if observer is not None and not self.stopped:
                    observer(self.atoms, self.nsteps)
        if self.stopped:
            self._on_stop()
        return done

    def _write_back(self):
        a = self.atoms
        pos = self.pos.cpu().numpy()
        if hasattr(a, "set_positions"):
            a.set_positions(pos)
        else:
            a.positions = pos
        mom = self.mom.cpu().numpy()
        if hasattr(a, "set_momenta"):
            a.set_momenta(mom)
        elif hasattr(a, "set_velocities"):
            a.set_velocities(mom / self.masses[:, None])

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
