"""Host-side mirror of the reference's similarity-kernel interface for the hot path.

Same constructor arguments, attribute names and eval-able ``state`` strings as
theforce.similarity.sesoap.SeSoapKernel (similarity/sesoap.py:10-24) and
theforce.similarity.universal.UniversalSoapKernel (similarity/universal.py:52-107);
``kern(atoms, inducing)`` returns the kernel matrix like
SimilarityKernel.forward(first, second, operation="func") (similarity/similarity.py:17-31)
-- evaluated on the GPU through libsgpr_b200 (no CPU path).
"""
from __future__ import annotations

import numpy as np

from .model import SgprModel


class DefaultRadii:
    """descriptor/sesoap.py:84-99: H -> 0.5, everything else -> 1.0."""

    def __init__(self, default=1.0, special=None):
        self.default = float(default)
        self.special = {1: 0.5} if special is None else {int(k): float(v) for k, v in special.items()}

    def get(self, number):
        return self.special.get(int(number), self.default)

    def __repr__(self):
        return f"DefaultRadii({self.default}, {self.special})"


class UniformRadii(DefaultRadii):
    def __init__(self, value=1.0):
        super().__init__(value, {})

    def __repr__(self):
        return f"UniformRadii({self.default})"


class EqAll:
    """util/util.py:113-124 / similarity/universal.py:44-49: equals everything but the exceptions."""

    def __init__(self, exceptions=()):
        self.exceptions = list(exceptions)

    def __eq__(self, val):
        return val not in self.exceptions


def _np(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def _is_structure(obj):
    return hasattr(obj, "positions") and hasattr(obj, "numbers") and hasattr(obj, "cell")


def _is_local(obj):
    return hasattr(obj, "number") and hasattr(obj, "_r") and hasattr(obj, "_b")


def _as_envs(obj):
    """Reference ``Local`` / ``LocalsData`` / list of ``Local`` (duck-typed: ``.number``, ``._r``, ``._b``;
    descriptor/atoms.py:36-52,802-847) or plain ``(Z, r[nn,3], b[nn])`` tuples -> (list of tuples, the objects)."""
    if _is_local(obj):
        objs = [obj]
    elif isinstance(obj, tuple) and len(obj) == 3 and np.ndim(obj[0]) == 0:
        objs = [obj]
    else:
        objs = list(obj)
    envs = []
    for o in objs:
        if _is_local(o):
            envs.append((int(o.number), _np(o._r).reshape(-1, 3), _np(o._b).reshape(-1)))
        else:
            envs.append((int(o[0]), np.asarray(o[1], dtype=np.float64).reshape(-1, 3), np.asarray(o[2]).reshape(-1)))
    return envs, objs


class _SoapKernelBase:
    kind = None
    max_cached_engines = 4

    def _base_model(self, envs=(), mu=None):
        return SgprModel.from_envs(
            list(envs), lmax=self.lmax, nmax=self.nmax, xi=float(self.exponent), rc=float(self.cutoff), kind=self.kind,
            normalize=self.normalize, radii=self._radii_dict(), default_radius=self._default_radius(),
            a_not=tuple(getattr(self._a, "exceptions", ())), a_only=tuple(getattr(self, "a_only", ())),
            b_only=tuple(getattr(self, "b", ())), mu=mu)

    @property
    def a(self):
        return self._a

    @property
    def state(self):
        return self.__class__.__name__ + "({})".format(self.state_args)

    def __repr__(self):
        return self.state

    # ------------------------------------------------------------------ one engine per inducing set, kept alive
    def _engine(self, envs, objs, species):
        """Engine whose inducing set is ``envs``.  Cached by the identity of the environment objects (strong references
        are kept, so ids cannot be recycled) and the species table; an inducing set that merely GREW is extended in
        place (``sgpr_append_inducing``) instead of being rebuilt."""
        from .engine import SgprEngine

        cache = self.__dict__.setdefault("_engines", [])      # [(ids, objs, engine)], most recent last
        ids = tuple(id(o) for o in objs)
        need = set(int(z) for z in species) | set(int(e[0]) for e in envs) | set(int(z) for e in envs for z in e[2])
        for k, (cid, cobjs, eng) in enumerate(cache):
            if not need.issubset(eng.species):
                continue
            if cid == ids:
                cache.append(cache.pop(k))
                return eng
            if len(cid) < len(ids) and ids[:len(cid)] == cid:
                eng.append_inducing(envs[len(cid):], np.zeros(len(envs)))
                cache.pop(k)
                cache.append((ids, list(objs), eng))
                return eng
        eng = SgprEngine(self._base_model(envs), species=sorted(need))
        cache.append((ids, list(objs), eng))
        while len(cache) > self.max_cached_engines:
            cache.pop(0)[2].close()
        return eng

    def close(self):
        for _, _, eng in self.__dict__.get("_engines", []):
            eng.close()
        self.__dict__["_engines"] = []

    def _cut_environments(self, atoms):
        """The local chemical environments of a structure given as ``second`` (``kern(atoms, atoms)``,
        calculator/active.py:655): neighbour list from ``sgpr_neighbors``."""
        from .engine import SgprEngine

        pos, numbers = np.asarray(atoms.positions, dtype=np.float64), np.asarray(atoms.numbers)
        cell = np.asarray(atoms.cell, dtype=np.float64).reshape(3, 3)
        probe = SgprEngine(self._base_model(()), species=np.unique(numbers))
        try:
            first, J, S = probe.neighbors(pos, numbers, cell, atoms.pbc)
        finally:
            probe.close()
        cc = cell.copy()
        return [(int(numbers[i]), pos[J[first[i]:first[i + 1]]] - pos[i] + S[first[i]:first[i + 1]].astype(np.float64) @ cc,
                 numbers[J[first[i]:first[i + 1]]].copy()) for i in range(len(numbers))]

    def __call__(self, first, second, operation="func"):
        """``SimilarityKernel.forward(first, second, operation)`` (similarity/similarity.py:17-31).

        first : a structure (``TorchAtoms`` / ``ase.Atoms`` / anything with positions, numbers, cell, pbc) -- every atom
                is a centre -- or ``Local`` / ``LocalsData`` / list of ``Local`` / ``(Z, r, b)`` tuples, or a list of
                structures: then "func" gives per-structure sums Ke [B, M] and "leftgrad" / "virial" the structures'
                rows stacked in order ([3 Ntot, M] / [6 B, M]), all from one batched call.
        second: the same kinds of object (a structure stands for all of its environments).
        operation: "func" -> K [len(first), len(second)];  with a structure as ``first`` also "leftgrad" ->
                d(sum_i K[i,m]) / d xyz  [3N, M] and "virial" -> [6, M] (similarity/universal.py:124-183; the true
                derivatives, see include/sgpr_b200.h sgpr_kernel_jacobian).
        Returns a torch tensor when the inputs are reference objects (carry torch tensors), else a numpy array."""
        if operation not in ("func", "leftgrad", "virial"):
            raise NotImplementedError(f"operation={operation!r}: only func / leftgrad / virial are implemented")
        as_torch = hasattr(first, "xyz") or any(hasattr(getattr(o, "_r", None), "detach")
                                                for o in ([first] if _is_local(first) else []))
        if _is_structure(second):
            envs2 = self._cut_environments(second)
            objs2 = envs2
        else:
            envs2, objs2 = _as_envs(second)
            as_torch = as_torch or any(hasattr(getattr(o, "_r", None), "detach") for o in objs2)
        if isinstance(first, (list, tuple)) and first and all(_is_structure(a) for a in first):
            # several structures: one sgpr_kernel_jacobian_batch call; "func" gives one row of Ke per structure, "leftgrad"
            # and "virial" the structures' rows stacked in order (regression/gppotential.py:63-77)
            eng = self._engine(envs2, objs2, np.unique(np.concatenate([np.asarray(a.numbers).reshape(-1) for a in first])))
            Ke, Kf, Kv = eng.training_kernels(list(first), want_jacobian=operation != "func")
            out = (Ke if operation == "func" else (-Kf if operation == "leftgrad" else Kv)).cpu()
        elif _is_structure(first):
            eng = self._engine(envs2, objs2, np.unique(first.numbers))
            args = (first.positions, first.numbers, np.asarray(first.cell, dtype=np.float64).reshape(3, 3), first.pbc)
            if operation == "func":
                out = eng.kernel_matrix(*args).cpu()
            else:
                _, Kf, Kv = eng.kernel_jacobian(*args)
                out = (-Kf).cpu() if operation == "leftgrad" else Kv.cpu()
        else:
            if operation != "func":
                raise NotImplementedError("leftgrad / virial need a structure as `first` (forces act on atoms)")
            envs1, objs1 = _as_envs(first)
            as_torch = as_torch or any(hasattr(getattr(o, "_r", None), "detach") for o in objs1)
            eng = self._engine(envs2, objs2, [e[0] for e in envs1] + [z for e in envs1 for z in e[2]])
            out = eng.kernel_envs(envs1).cpu()
        return out if as_torch else out.numpy()

    forward = __call__

    # ------------------------------------------------------------------ per-LCE descriptor cache of the reference
    def call_descriptor(self, loc, grad=False):
        """``kern.call_descriptor(loc, grad)`` (similarity/universal.py:97-98, similarity/sesoap.py:23-24): the normalised
        descriptor of one LCE as the reference's sparse COO tensor ``[120, 120, dim]`` indexed (Z_s2, Z_s1, :)
        (descriptor/sesoap.py:165-171,254-258; [119, 119, dim] for UniversalSoap, soap.py:749)."""
        if grad:
            raise NotImplementedError("descriptor Jacobians are not materialised on this path: use operation='leftgrad' / "
                                      "'virial' (sgpr_kernel_jacobian) for the training-time kernels")
        if hasattr(self, "b"):
            raise NotImplementedError("the dense per-kernel cache of SubSeSoapKernel / HeterogeneousSoapKernel is not exposed; "
                                      "kern(first, second) evaluates these kernels")
        import torch

        from .engine import SgprEngine

        (env,), _ = _as_envs(loc)
        species = sorted(set([env[0]]) | set(int(z) for z in env[2]))
        cache = self.__dict__.setdefault("_desc_engines", {})
        key = tuple(species)
        if key not in cache:
            cache[key] = SgprEngine(self._base_model(()), species=species)
        P = cache[key].kernel_envs([env], want_K=False, want_descriptors=True)[0]      # [S, S, nb, nb, L]
        size = 119 if self.kind == "universal" and type(self).__name__ == "UniversalSoapKernel" else 120
        present = sorted(set(int(z) for z in env[2]))    # blocks exist only for neighbour species that occur (sesoap.py:163)
        idx, vals = [], []
        for z1 in present:
            for z2 in present:
                blk = P[species.index(z1), species.index(z2)].reshape(-1)
                for d, v in enumerate(blk):
                    idx.append((z2, z1, d))
                    vals.append(v)
        if not idx:
            return torch.sparse_coo_tensor(torch.zeros((3, 0), dtype=torch.long), torch.zeros(0, dtype=torch.float64), (size, size, self.dim))
        return torch.sparse_coo_tensor(torch.tensor(idx, dtype=torch.long).t(), torch.tensor(vals, dtype=torch.float64),
                                       (size, size, self.dim))

    def precalculate(self, loc, dont_save_grads=True):
        """``kern.precalculate(loc)`` (similarity/universal.py:100-107): caches the descriptor on the LCE as
        ``loc.<name>_value`` -- ``None`` for an LCE without neighbours or with an excluded central species."""
        if not dont_save_grads:
            raise NotImplementedError("descriptor Jacobians are not materialised on this path (see call_descriptor)")
        (env,), _ = _as_envs(loc)
        ok = len(env[2]) > 0 and self._base_model(()).is_centre(env[0])
        value = self.call_descriptor(loc, grad=False) if ok else None
        if _is_local(loc):
            setattr(loc, self.name + "_value", value)
            setattr(loc, self.name + "_grad", None)
        return value


class SeSoapKernel(_SoapKernelBase):
    kind = "sesoap"

    def __init__(self, lmax, nmax, exponent, cutoff, a=None, radii=1.0, normalize=True):
        self.lmax, self.nmax, self.exponent, self.cutoff = int(lmax), int(nmax), exponent, float(cutoff)
        self.radii = UniformRadii(radii) if isinstance(radii, (int, float)) else radii
        self.normalize = bool(normalize)
        self.dim = (nmax + 1) ** 2 * (lmax + 1)
        self._a = EqAll() if a is None else a
        if not hasattr(self._a, "exceptions"):
            self.a_only = (int(a),)      # a fixed central species: loc.number == self.a (similarity/universal.py:101)
        self._args = f"{lmax}, {nmax}, {exponent}, {cutoff}, a={a}"
        self.name = "kern_0"
        self.params = []

    def _radii_dict(self):
        if isinstance(self.radii, dict):
            return dict(self.radii)
        return dict(getattr(self.radii, "special", {}))

    def _default_radius(self):
        return float(getattr(self.radii, "default", 1.0))

    @property
    def state_args(self):
        return f"{self._args}, radii={self.radii}, normalize={self.normalize}"


class SubSeSoapKernel(SeSoapKernel):
    """similarity/sesoap.py:27-43: fixed central species ``a`` and neighbour species list ``b`` (dense
    [S^2 * dim] descriptor); ``default_kernel(species=...)`` builds one per central species."""

    def __init__(self, lmax, nmax, exponent, cutoff, a, b, radii=1.0, normalize=True):
        super().__init__(lmax, nmax, exponent, cutoff, a=None, radii=radii, normalize=normalize)
        self.a_only = (int(a),)
        self.b = sorted(int(z) for z in (b if hasattr(b, "__iter__") else [b]))
        self._a = int(a)
        self.dim = len(self.b) ** 2 * (nmax + 1) ** 2 * (lmax + 1)
        self._args = f"{lmax}, {nmax}, {exponent}, {cutoff}, {a}, {b}"

    @property
    def a(self):
        return self._a


class HeterogeneousSoapKernel(_SoapKernelBase):
    """similarity/heterosoap.py:10-29 with the base kernel ``DotProd() ** exponent``: central species ``a``,
    neighbour species list ``b``, descriptor [NormalizedSoap(] HeteroSoap [)] with ONE length unit for all species
    (``atomic_unit`` or cutoff / 3, descriptor/soap.py:20-23)."""

    kind = "universal"

    def __init__(self, exponent, a, b, lmax, nmax, cutoff, atomic_unit=None, normalize=True):
        self.lmax, self.nmax, self.exponent, self.cutoff = int(lmax), int(nmax), exponent, float(cutoff)
        self.unit = float(atomic_unit) if atomic_unit else self.cutoff / 3
        self.normalize = bool(normalize)
        self.a_only = (int(a),)
        self._a = int(a)
        self.b = sorted(int(z) for z in (b if hasattr(b, "__iter__") else [b]))
        self.dim = len(self.b) ** 2 * (self.nmax + 1) ** 2 * (self.lmax + 1)
        self._args = "Pow(DotProd(), {}), {}, {}, {}, {}, PolyCut({}, n=2), atomic_unit={}, normalize={}".format(
            exponent, a, b, lmax, nmax, self.cutoff, atomic_unit, normalize)
        self.name = "kern_0"
        self.params = []

    def _radii_dict(self):
        return {}

    def _default_radius(self):
        return self.unit

    @property
    def state_args(self):
        return self._args


class UniversalSoapKernel(_SoapKernelBase):
    kind = "universal"

    def __init__(self, lmax, nmax, exponent, cutoff, atomic_unit=None, chemical=None, normalize=True, a=None, a_not=[]):
        if chemical is not None:
            raise NotImplementedError("only the Dirac-delta chemical kernel is supported")
        self.lmax, self.nmax, self.exponent, self.cutoff = int(lmax), int(nmax), exponent, float(cutoff)
        self.unit = float(atomic_unit) if atomic_unit else self.cutoff / 6  # descriptor/soap.py:724-728
        self.normalize = bool(normalize)
        self.dim = (nmax + 1) ** 2 * (lmax + 1)
        self._a = EqAll(a_not) if a is None else a
        if not hasattr(self._a, "exceptions"):
            self.a_only = (int(a),)      # a fixed central species (similarity/universal.py:85,101)
        self._args = "{}, {}, {}, PolyCut({}, n=2), atomic_unit={}, chemical=DiracDeltaChemical(), normalize={}, a={}, a_not={}".format(
            lmax, nmax, exponent, self.cutoff, atomic_unit, normalize, a, a_not)
        self.name = "kern_0"
        self.params = []

    def _radii_dict(self):
        return {}

    def _default_radius(self):
        return self.unit

    @property
    def state_args(self):
        return self._args
