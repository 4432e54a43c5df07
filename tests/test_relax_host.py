"""CPU: the FIRE restatement the GPU tests compare against (tests/relax_reference.py) on an analytic harmonic stand-in
for SgprEngine.predict; DeviceRelax's argument checks and refusals (they run before any device work); the layout of
sgpr_relax_params against include/sgpr_b200.h."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from relax_reference import host_fire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class Harmonic:
    """E = sum_i k_i |r_i - r0_i|^2 / 2: what host_fire reads of SgprEngine.predict (beta: |r_i - r0_i|)."""

    def __init__(self, r0, k):
        self.r0, self.k = np.asarray(r0, dtype=np.float64), np.asarray(k, dtype=np.float64)

    def predict(self, pos, numbers, cell, pbc, want_beta=False):
        d = np.asarray(pos) - self.r0
        F = -self.k[:, None] * d
        E = 0.5 * float(np.sum(self.k * (d ** 2).sum(axis=1)))
        W = -d.T @ F
        owned = np.ones(len(d), dtype=bool)
        if want_beta:
            return E, F, W, owned, np.sqrt((d ** 2).sum(axis=1))
        return E, F, W, owned


def _run(eng, pos, n, **kw):
    return host_fire(eng, pos, np.full(len(pos), 29), np.eye(3) * 10.0, True, n, **kw)


def test_reference_converges_on_harmonic_well():
    rng = np.random.default_rng(0)
    r0 = rng.uniform(0, 10, (16, 3))
    k = rng.uniform(1.0, 5.0, 16)
    out = _run(Harmonic(r0, k), r0 + rng.normal(0, 0.3, r0.shape), 2000, fmax=1e-4)
    assert out["converged"] is not None and out["converged"] == out["steps"] < 2000
    assert np.sqrt((out["F"] ** 2).sum(axis=1)).max() < 1e-4
    assert np.abs(out["pos"] - r0).max() < 1e-4
    assert out["rows"][-1, 1] < 1e-4 and out["rows"][0, 1] >= 1e-4
    # a second run from the converged structure does no step
    again = _run(Harmonic(r0, k), out["pos"], 10, fmax=1e-4)
    assert again["converged"] == 0 and again["steps"] == 0


def test_reference_follows_the_branch_rules():
    # one atom, 1 A from the minimum of a unit spring: the first step is v = dt F, dr = dt v
    eng = Harmonic(np.zeros((1, 3)), [1.0])
    assert _run(eng, [[1.0, 0.0, 0.0]], 1)["pos"][0, 0] == 1.0 + 0.1 * (0.1 * -1.0)     # 0.99
    out = _run(eng, [[1.0, 0.0, 0.0]], 2)
    # step 2: F = -0.99, F.v = 0.099 > 0: v = 0.9 (-0.1) + 0.1 (-0.99)/0.99 * 0.1 = -0.1, then v += 0.1 F
    v = (1.0 - 0.1) * -0.1 + 0.1 * -0.99 / 0.99 * 0.1 + 0.1 * -(1.0 + 0.1 * (0.1 * -1.0))
    assert out["vel"][0, 0] == v and out["pos"][0, 0] == 0.99 + 0.1 * v
    assert list(out["rows"][:, 2]) == [0.1, 0.1] and list(out["rows"][:, 3]) == [0.1, 0.1]
    # dt and a stay while Nsteps <= Nmin (steps 1..6 after the first), then grow by finc / shrink by fa
    out = _run(eng, [[1.0, 0.0, 0.0]], 200, fmax=1e-6)
    vf, dt, a = out["vf"], out["rows"][:, 2], out["rows"][:, 3]
    first_reset = next(k for k, x in enumerate(vf) if x <= 0.0) + 1      # vf[k] decides step k + 1
    assert first_reset > 8
    assert list(dt[:7]) == [0.1] * 7 and list(a[:7]) == [0.1] * 7
    assert dt[7] == 0.1 * 1.1 and a[7] == 0.1 * 0.99
    assert dt[8] == 0.1 * 1.1 * 1.1 and a[8] == 0.1 * 0.99 * 0.99
    # F.v <= 0 (overshoot): v = 0, a = astart, dt halves, Nsteps = 0
    assert dt[first_reset] == dt[first_reset - 1] * 0.5 and a[first_reset] == 0.1
    assert dt[first_reset + 1] == dt[first_reset] and a[first_reset + 1] == 0.1
    assert out["converged"] is not None
    # dt never exceeds dtmax
    assert dt.max() <= 1.0


def test_reference_caps_the_step_at_maxstep():
    eng = Harmonic(np.zeros((2, 3)), [1.0, 1.0])
    out = _run(eng, [[100.0, 0.0, 0.0], [0.0, 0.0, 0.0]], 1)
    # dr = dt^2 F = (-1, 0, 0) for the first atom: |dr| over all atoms is 1 > 0.2, so dr is scaled to 0.2
    assert out["pos"][0, 0] == 100.0 + 0.2 * -1.0 / 1.0 and out["pos"][1, 0] == 0.0


def test_reference_fixed_atoms_stay():
    rng = np.random.default_rng(1)
    r0 = rng.uniform(0, 10, (8, 3))
    start = r0 + rng.normal(0, 0.2, r0.shape)
    fixed = np.zeros(8, dtype=bool)
    fixed[[1, 5]] = True
    out = _run(Harmonic(r0, np.full(8, 2.0)), start, 500, fmax=1e-5, fixed=fixed)
    assert out["converged"] is not None
    assert np.array_equal(out["pos"][fixed], start[fixed]) and not out["F"][fixed].any()
    assert np.abs(out["pos"][~fixed] - r0[~fixed]).max() < 1e-5


def test_reference_uncertainty_stop():
    r0 = np.zeros((1, 3))
    out = _run(Harmonic(r0, [1.0]), [[1.0, 0.0, 0.0]], 50, covloss=True, ediff=0.95)
    # beta = |r - r0|: 1.0 at the start is already above ediff
    assert out["stop"] == 0 and out["steps"] == 0
    out = _run(Harmonic(r0, [1.0]), [[0.9, 0.0, 0.0]], 50, covloss=True, ediff=0.95)
    assert out["stop"] is None and out["steps"] == 50


class _Atoms:
    def __init__(self, n=4, numbers=None):
        self.positions = np.arange(3 * n, dtype=np.float64).reshape(n, 3)
        self.numbers = np.array(numbers if numbers is not None else [29] * n)
        self.cell = np.eye(3) * 10.0
        self.pbc = np.array([True] * 3)


class FixAtoms:
    def __init__(self, indices):
        self.indices = indices

    def get_indices(self):
        return np.asarray(self.indices)


class FixBondLength:
    def get_indices(self):
        return np.array([0, 1])


def _calc(**kw):
    import autoforce_b200 as ab
    from golden_util import b200_model, load_golden

    return ab.B200Calculator(b200_model(load_golden("cu108_sesoap")), **kw)


@pytest.mark.parametrize("kw,match", [
    (dict(dt=0.0), "dt must be a positive"),
    (dict(maxstep=-0.1), "maxstep must be a positive"),
    (dict(dtmax=np.inf), "dtmax must be a positive"),
    (dict(finc=np.nan), "finc must be a positive"),
    (dict(fdec=0.0), "fdec must be a positive"),
    (dict(a=np.nan), "a must be finite"),
    (dict(fa=np.inf), "fa must be finite"),
    (dict(Nmin=-1), "Nmin"),
    (dict(Nmin=2.5), "Nmin"),
])
def test_device_relax_argument_checks(kw, match):
    from autoforce_b200 import DeviceRelax

    calc = _calc()
    with pytest.raises(ValueError, match=match):
        DeviceRelax(calc, _Atoms(), **kw)
    assert calc._engine is None


def test_device_relax_refusals():
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax
    from golden_util import b200_model, load_golden

    calc = _calc()
    with pytest.raises(ValueError, match="unknown species"):
        DeviceRelax(calc, _Atoms(numbers=[29, 29, 29, 0]))
    model = b200_model(load_golden("cu108_sesoap"))
    with pytest.raises(NotImplementedError, match="DeviceRelax runs a single model handle: kernel sums"):
        DeviceRelax(ab.B200Calculator([model, model]), _Atoms())
    for bad in ([object()], [FixAtoms([0]), FixBondLength()]):
        atoms = _Atoms()
        atoms.constraints = bad
        with pytest.raises(NotImplementedError, match="constraints other than FixAtoms"):
            DeviceRelax(calc, atoms)
    atoms = _Atoms()
    atoms.constraints = [FixAtoms([0, 4])]
    with pytest.raises(ValueError, match="FixAtoms index out of range"):
        DeviceRelax(calc, atoms)
    assert calc._engine is None   # nothing was created on a device


def test_fixed_mask_reads_fixatoms():
    from autoforce_b200.relax import fixed_mask

    atoms = _Atoms(n=6)
    assert fixed_mask(atoms, 6) is None
    atoms.constraints = [FixAtoms([0, 2]), FixAtoms(np.array([-1]))]
    assert list(fixed_mask(atoms, 6)) == [1, 0, 1, 0, 0, 1]
    atoms.constraints = [FixAtoms([])]
    assert fixed_mask(atoms, 6) is None


def test_relax_params_layout_matches_header(tmp_path):
    from autoforce_b200.engine import sgpr_relax_params

    fields = [f for f, _ in sgpr_relax_params._fields_]
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "sgpr_b200.h"\nint main(void) {\n'
                   + "".join(f'  printf("%zu\\n", offsetof(sgpr_relax_params, {f}));\n' for f in fields)
                   + '  printf("%zu\\n", sizeof(sgpr_relax_params));\n  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    want = [getattr(sgpr_relax_params, f).offset for f in fields] + [ctypes.sizeof(sgpr_relax_params)]
    assert got == want
