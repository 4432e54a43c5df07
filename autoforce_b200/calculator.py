"""Calculator facade: ActiveCalculator.calculate() in prediction mode on the GPU.

Mirrors what theforce.calculator.active.ActiveCalculator produces when
``calculator=None`` (calculator/active.py:425-611): ``results['energy']`` (0-d float64
ndarray), ``results['forces']`` [N,3], ``results['stress']`` Voigt (xx,yy,zz,yz,xz,xy) in
eV/A^3 = (W / V).flat[[0,4,8,5,2,1]] with V = -2 when there is no cell (active.py:604-611),
``results['free_energy']`` (active.py:527).  The on-the-fly training control flow, the
ab initio calls and the M x M algebra stay with the reference (INTEGRATION.md).

Works with any object exposing positions / cell / pbc / numbers (ase.Atoms does); when
ASE is importable the class is also a proper ase Calculator.
"""
from __future__ import annotations

import numpy as np

from .engine import SgprEngine
from .model import SgprModel

try:  # optional
    from ase.calculators.calculator import Calculator as _AseCalculator
    from ase.calculators.calculator import all_changes as _all_changes
except Exception:  # pragma: no cover
    _AseCalculator = object
    _all_changes = ["positions", "numbers", "cell", "pbc"]


def _as_models(covariance):
    """-> list of SgprModel whose energies / forces / virials add up (one entry unless the reference model sums
    similarity kernels with different hyper-parameters)."""
    if isinstance(covariance, (list, tuple)) and all(isinstance(m, SgprModel) for m in covariance):
        return list(covariance)
    if hasattr(covariance, "gp") and hasattr(covariance, "X"):
        return SgprModel.list_from_posterior_potential(covariance)
    if isinstance(covariance, str) and not covariance.endswith(".npz"):
        from theforce.regression.gppotential import PosteriorPotentialFromFolder

        return SgprModel.list_from_posterior_potential(PosteriorPotentialFromFolder(covariance, load_data=False, update_data=False))
    return [_as_model(covariance)]


def _as_model(covariance):
    if isinstance(covariance, SgprModel):
        return covariance
    if isinstance(covariance, str):
        if covariance.endswith(".npz"):
            return SgprModel.load(covariance)
        # a folder pickled by the reference (gppotential.py:1073-1119,1342-1368): needs theforce importable
        from theforce.regression.gppotential import PosteriorPotentialFromFolder

        return SgprModel.from_posterior_potential(PosteriorPotentialFromFolder(covariance, load_data=False, update_data=False))
    if hasattr(covariance, "gp") and hasattr(covariance, "X"):
        return SgprModel.from_posterior_potential(covariance)
    raise TypeError(f"cannot build an SGPR model from {type(covariance)}")


class B200Calculator(_AseCalculator):
    implemented_properties = ["energy", "forces", "stress", "free_energy"]

    def __init__(self, covariance, calculator=None, process_group=None, device=None, gather_forces=True, logfile=None,
                 covloss=False, ediff=0.04, on_uncertain=None, **kw):
        if _AseCalculator is not object:
            super().__init__()
        if calculator is not None:
            raise NotImplementedError(
                "on-the-fly training stays on the reference path: use theforce's ActiveCalculator with the "
                "GPU kernel plugged in (INTEGRATION.md); B200Calculator is the prediction-mode drop-in")
        self.models = _as_models(covariance)
        self.model = self.models[0]
        # prediction-mode uncertainty (calculator/active.py:492-499): covloss=True evaluates beta = get_covloss() every
        # step on the device, records its maximum in ``covlog`` and hands structures with max(beta) > ediff to
        # ``on_uncertain(atoms, beta)`` (the reference appends them to active_uncertain.traj)
        self.covloss = bool(covloss)
        if self.covloss and self.model.choli is None:
            raise ValueError("covloss=True needs a model with choli")
        if self.covloss and len(self.models) > 1:
            raise NotImplementedError("covloss of a model that sums kernels with different hyper-parameters")
        self.ediff = float(ediff)
        self.on_uncertain = on_uncertain
        self.covlog = ""
        self.beta = None
        self.process_group = process_group
        self.gather_forces = gather_forces
        self.results = {}
        self.step = 0
        self._engine = None
        self._more_engines = []      # handles of the 2nd, 3rd ... model of a kernel sum
        self._device = device
        self.atoms = None

    # ------------------------------------------------------------------ distributed
    def _dist(self):
        try:
            import torch.distributed as dist

            if dist.is_available() and dist.is_initialized():
                return dist, dist.get_rank(self.process_group), dist.get_world_size(self.process_group)
        except Exception:
            pass
        return None, 0, 1

    def _get_engine(self, numbers):
        import torch

        need = set(int(z) for z in np.unique(numbers))
        if self._engine is None or not need.issubset(self._engine.species):
            if self._engine is not None:
                self._engine.close()
            dev = self._device if self._device is not None else (torch.cuda.current_device() if torch.cuda.is_available() else 0)
            self._engine = SgprEngine(self.model, species=sorted(need), device=dev)
            for e in self._more_engines:
                e.close()
            self._more_engines = [SgprEngine(m, species=sorted(need), device=dev) for m in self.models[1:]]
        return self._engine

    def _reduce(self, dist, E, W, F, device_index):
        """The path's only exchange step: all-reduce of 10 doubles (energy + 3x3 virial),
        replacing the reference's all_reduce(energy), all_reduce(forces [N,3]) and
        all_reduce(cellgrad) (calculator/active.py:562,601-602).  Forces are owner-computed;
        ``gather_forces=True`` additionally sums them so that every rank sees all forces."""
        import torch

        backend = dist.get_backend(self.process_group)
        dev = torch.device("cuda", device_index) if backend == "nccl" else torch.device("cpu")
        ew = torch.tensor([E] + list(np.asarray(W).reshape(-1)), dtype=torch.float64, device=dev)
        dist.all_reduce(ew, group=self.process_group)
        ew = ew.cpu().numpy()
        E, W = float(ew[0]), ew[1:].reshape(3, 3)
        if self.gather_forces:
            ft = torch.as_tensor(np.ascontiguousarray(F), device=dev)
            dist.all_reduce(ft, group=self.process_group)
            F = ft.cpu().numpy()
        return E, W, F

    def _gather_beta(self, dist, beta, device_index):
        import torch

        backend = dist.get_backend(self.process_group)
        dev = torch.device("cuda", device_index) if backend == "nccl" else torch.device("cpu")
        b = torch.as_tensor(np.nan_to_num(beta, nan=0.0, posinf=0.0), device=dev)
        bad = torch.as_tensor((~np.isfinite(beta)).astype(np.float64) * np.where(np.isnan(beta), 1.0, 2.0), device=dev)
        dist.all_reduce(b, group=self.process_group)
        dist.all_reduce(bad, group=self.process_group)
        out = b.cpu().numpy()
        flag = bad.cpu().numpy()
        out[flag == 1.0] = np.nan
        out[flag == 2.0] = np.inf
        return out

    def get_covloss(self):
        """beta of the last structure (calculator/active.py:781-804); evaluates it if the step did not."""
        if self.beta is None:
            if self.atoms is None:
                raise RuntimeError("no structure has been calculated yet")
            prev, self.covloss = self.covloss, True
            try:
                self.calculate(self.atoms)
            finally:
                self.covloss = prev
        return self.beta

    # ------------------------------------------------------------------ the call
    def calculate(self, atoms=None, properties=("energy",), system_changes=_all_changes):
        if atoms is not None:
            self.atoms = atoms.copy() if hasattr(atoms, "copy") else atoms
        a = self.atoms
        pos = np.asarray(a.positions, dtype=np.float64)
        numbers = np.asarray(a.numbers)
        cell = np.asarray(a.cell, dtype=np.float64).reshape(3, 3)
        pbc = np.broadcast_to(np.asarray(a.pbc), (3,))
        eng = self._get_engine(numbers)
        dist, rank, world = self._dist()
        if world > 1 and self._more_engines and not self.gather_forces:
            raise NotImplementedError("a kernel sum shards every handle by its own cell order: use gather_forces=True")
        if self.covloss:
            E, F, W, owned, beta = eng.predict(pos, numbers, cell, pbc, rank=rank, world=world, want_beta=True)
        else:
            E, F, W, owned = eng.predict(pos, numbers, cell, pbc, rank=rank, world=world)
            for e in self._more_engines:   # kernels with different hyper-parameters: the contributions add up
                E2, F2, W2, _ = e.predict(pos, numbers, cell, pbc, rank=rank, world=world)
                E, F, W = E + E2, F + F2, W + W2
            beta = None
        if world > 1:
            E, W, F = self._reduce(dist, E, W, F, getattr(eng, "device", 0))
            if beta is not None:   # every rank filled the betas of the atoms it owns (zeros elsewhere)
                beta = self._gather_beta(dist, beta, getattr(eng, "device", 0))
        vol = abs(np.linalg.det(cell))
        if vol == 0.0:
            vol = -2.0  # calculator/active.py:606-609
        stress = (W / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]]
        self.results = {
            "energy": np.array(E, dtype=np.float64),
            "forces": F,
            "stress": stress,
            "free_energy": np.array(E, dtype=np.float64),
        }
        self.owned = owned
        self.beta = beta
        if beta is not None:
            covloss_max = float(np.max(beta)) if len(beta) else 0.0   # like torch.max: NaN / inf propagate
            self.covlog = f"{covloss_max}"
            if covloss_max > self.ediff and self.on_uncertain is not None and rank == 0:
                self.on_uncertain(a, beta)
        self.maximum_force = float(np.abs(F).max()) if F.size else 0.0
        self.step += 1
        return self.results

    def calculate_batch(self, images):
        """Many structures in one GPU call (``SgprEngine.predict_batch``): testing a model on a trajectory, the images of
        an NEB, scoring a data set.  Returns one results dict per image, with the keys, dtypes and stress convention of
        ``calculate``.  With ``covloss=True`` each image also gets ``beta`` and ``covlog``, and ``on_uncertain(image,
        beta)`` is called for each image whose max(beta) exceeds ``ediff``.  Under torch.distributed the images given
        are evaluated on the local device: splitting a data set over ranks is the caller's job.  Does not change
        ``self.atoms`` / ``self.results`` of the step-by-step interface."""
        images = list(images)
        if not images:
            return []
        numbers = np.concatenate([np.asarray(a.numbers).reshape(-1) for a in images])
        eng = self._get_engine(numbers)
        if self.covloss:
            E, F, W, beta = eng.predict_batch(images, want_beta=True)
        else:
            E, F, W = eng.predict_batch(images)
            for e in self._more_engines:   # kernels with different hyper-parameters: the contributions add up
                E2, F2, W2 = e.predict_batch(images)
                E, F, W = E + E2, F + F2, W + W2
            beta = None
        _, rank, _ = self._dist()
        out = []
        a0 = 0
        for b, a in enumerate(images):
            n = len(a.numbers)
            cell = np.asarray(a.cell, dtype=np.float64).reshape(3, 3)
            vol = abs(np.linalg.det(cell))
            if vol == 0.0:
                vol = -2.0  # calculator/active.py:606-609
            r = {
                "energy": np.array(E[b], dtype=np.float64),
                "forces": F[a0:a0 + n].copy(),
                "stress": (W[b] / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]],
                "free_energy": np.array(E[b], dtype=np.float64),
            }
            if beta is not None:
                bb = beta[a0:a0 + n].copy()
                covloss_max = float(np.max(bb)) if n else 0.0   # like torch.max: NaN / inf propagate
                r["beta"] = bb
                r["covlog"] = f"{covloss_max}"
                if covloss_max > self.ediff and self.on_uncertain is not None and rank == 0:
                    self.on_uncertain(a, bb)
            out.append(r)
            a0 += n
        return out

    # ------------------------------------------------------------------ getters (callers without ASE)
    def _same_state(self, atoms):
        a = self.atoms
        if a is None or not self.results:
            return False
        try:
            return (np.array_equal(np.asarray(a.positions), np.asarray(atoms.positions))
                    and np.array_equal(np.asarray(a.cell), np.asarray(atoms.cell))
                    and np.array_equal(np.asarray(a.numbers), np.asarray(atoms.numbers))
                    and np.array_equal(np.broadcast_to(np.asarray(a.pbc), (3,)), np.broadcast_to(np.asarray(atoms.pbc), (3,))))
        except Exception:
            return False

    def _property(self, name, atoms):
        """One evaluation per structure, like ase's Calculator.get_property: a second getter on an unchanged
        structure returns the cached result (no second GPU pass, no second ``step`` / ``on_uncertain``)."""
        if atoms is not None and not self._same_state(atoms):
            self.calculate(atoms)
        elif not self.results:
            if self.atoms is None and atoms is None:
                raise RuntimeError("no structure has been calculated yet")
            self.calculate(atoms)
        return self.results[name]


if _AseCalculator is object:
    # ase.calculators.calculator.Calculator provides these (with its own check_state caching) when ASE is there;
    # otherwise the same signatures, incl. the ``force_consistent`` keyword ASE optimisers pass
    def _get_potential_energy(self, atoms=None, force_consistent=False, **kw):
        return float(self._property("free_energy" if force_consistent else "energy", atoms))

    def _get_forces(self, atoms=None, **kw):
        return self._property("forces", atoms)

    def _get_stress(self, atoms=None, **kw):
        return self._property("stress", atoms)

    B200Calculator.get_potential_energy = _get_potential_energy
    B200Calculator.get_forces = _get_forces
    B200Calculator.get_stress = _get_stress
