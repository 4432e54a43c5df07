"""GPU: DeviceRelax (FIRE with positions, velocities and forces on the device) against the host FIRE loop around
SgprEngine.predict (tests/relax_reference.py), and on a lattice-well model whose minimum is known."""
import numpy as np
import pytest

from golden_util import b200_model, load_golden
from relax_reference import host_fire

pytestmark = pytest.mark.gpu

TOL = 1e-9


class Atoms:
    """What DeviceRelax reads and writes of an ase.Atoms."""

    def __init__(self, positions, numbers, cell, pbc, constraints=()):
        self.positions = np.array(positions, dtype=np.float64)
        self.numbers = np.asarray(numbers)
        self.cell = np.asarray(cell, dtype=np.float64)
        self.pbc = np.broadcast_to(np.asarray(pbc), (3,)).copy()
        self.constraints = list(constraints)

    def set_positions(self, r):
        self.positions = np.array(r)

    def copy(self):
        return Atoms(self.positions, self.numbers, self.cell, self.pbc, self.constraints)


class FixAtoms:
    def __init__(self, indices):
        self.indices = np.asarray(indices)

    def get_indices(self):
        return self.indices


def close(a, b, tol=TOL):
    return np.abs(np.asarray(a) - np.asarray(b)).max() <= tol * max(1.0, np.abs(np.asarray(b)).max())


def golden_case(name):
    g = load_golden(name)
    return g, Atoms(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])


def lattice_well(mu=-1.0, rattle=0.08, rep=3, seed=0, with_choli=False):
    """One inducing LCE cut from a perfect fcc Cu cell, mu = -1, mean 0: E = -sum_i k(env_i, lattice) >= -N, with
    equality exactly when every environment is the lattice's.  Returns (model, rattled atoms)."""
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    pos, cell, numbers = synth.fcc(rep, [29], 0.0, seed)
    base = dict(lmax=3, nmax=3, xi=4.0, rc=6.0, kind="sesoap", radii={1: 0.5}, default_radius=1.0)
    probe = ab.SgprEngine(ab.SgprModel.from_envs([], **base), species=[29])
    try:
        first, J, S = probe.neighbors(pos, numbers, cell, True)
    finally:
        probe.close()
    envs = synth.cut_environments(pos, cell, True, numbers, 6.0, [0], first, J, S)
    model = ab.SgprModel.from_envs(envs, mu=np.array([mu]), mean_w={29: 0.0}, vscale={29: 1.0},
                                   choli=0.5 * np.eye(1) if with_choli else None, **base)
    rng = np.random.default_rng(seed + 1)
    return model, Atoms(pos + rng.normal(0, rattle, pos.shape), numbers, cell, True)


@pytest.mark.parametrize("name", ["cu108_sesoap", "lipso108", "cluster_lone", "slab_ttf"])
def test_fire_matches_host_loop(name):
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax

    n = 100 if name in ("cu108_sesoap", "lipso108") else 60   # non-periodic / mixed pbc size every step
    g, atoms = golden_case(name)
    eng = ab.SgprEngine(b200_model(g), species=sorted(set(int(z) for z in g["numbers"])))
    ref = host_fire(eng, atoms.positions, atoms.numbers, atoms.cell, atoms.pbc, n)
    assert ref["min_cos"] > 1e-10, ref["min_cos"]     # every branch decision was far from a tie
    rx = DeviceRelax(ab.B200Calculator(b200_model(g)), atoms)
    assert rx.run(fmax=0.0, steps=n, interval=40) is False
    assert rx.nsteps == n and not rx.converged
    assert close(atoms.positions, ref["pos"]) and close(rx.velocities, ref["vel"]) and close(rx.forces, ref["F"])
    tr = rx.trace
    assert np.array_equal(tr["dt"], ref["rows"][:, 2]) and np.array_equal(tr["a"], ref["rows"][:, 3])
    assert close(tr["epot"], ref["rows"][:, 0], 1e-10) and close(tr["fmax"], ref["rows"][:, 1])
    assert close(tr["W"].reshape(-1, 9), ref["rows"][:, 4:])
    eng.close()


def test_converges_to_the_lattice_well_minimum():
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax

    model, start = lattice_well()
    N = len(start.numbers)
    calc = ab.B200Calculator(model)
    out = []
    for interval in (100, 7, 1):
        atoms = start.copy()
        rx = DeviceRelax(calc, atoms)
        seen = []
        assert rx.run(fmax=0.01, steps=3000, interval=interval, observer=lambda a, k: seen.append(k)) is True
        assert rx.converged and not rx.stopped and 0 < rx.nsteps < 3000
        assert seen[-1] == rx.nsteps
        assert rx.trace["fmax"][-1] < 0.01 and (rx.trace["fmax"][:-1] >= 0.01).all()
        # a second run at the same fmax does no step
        k = rx.nsteps
        assert rx.run(fmax=0.01, steps=100, interval=interval) is True and rx.nsteps == k == len(rx.trace["epot"])
        out.append((rx.nsteps, atoms.positions.copy(), rx.trace))
    # the step sequence does not depend on interval; the forces are summed with atomics, so the positions agree to
    # the last bits rather than bit for bit (as DeviceMD's)
    for k, pos, tr in out[1:]:
        assert k == out[0][0] and close(pos, out[0][1], 1e-12)
        assert close(tr["epot"], out[0][2]["epot"], 1e-12) and np.array_equal(tr["dt"], out[0][2]["dt"])
    # an independent evaluation of the written-back structure
    atoms = start.copy()
    atoms.positions = out[0][1]
    res = ab.B200Calculator(model).calculate(atoms)
    assert np.sqrt((res["forces"] ** 2).sum(axis=1)).max() < 0.01
    assert abs(float(res["energy"]) - (-N + 0.0)) < 1e-3 * N      # -N + N * mean, mean 0
    # the same relaxation in the host loop converges at the same step
    eng = ab.SgprEngine(model, species=[29])
    ref = host_fire(eng, start.positions, start.numbers, start.cell, start.pbc, 3000, fmax=0.01)
    assert ref["converged"] == out[0][0] and close(out[0][1], ref["pos"])
    eng.close()


def test_fixed_atoms_do_not_move():
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax

    model, start = lattice_well(rattle=0.1)
    fixed = [0, 5, 17, 60]
    atoms = start.copy()
    atoms.constraints = [FixAtoms(fixed[:2]), FixAtoms(fixed[2:])]
    rx = DeviceRelax(ab.B200Calculator(model), atoms)
    assert not rx.forces[fixed].any()
    n = 80
    rx.run(fmax=0.0, steps=n, interval=30)
    assert rx.nsteps == n
    assert np.array_equal(atoms.positions[fixed], start.positions[fixed])
    assert not rx.forces[fixed].any() and not rx.velocities[fixed].any()
    assert not np.array_equal(np.delete(atoms.positions, fixed, 0), np.delete(start.positions, fixed, 0))
    mask = np.zeros(len(start.numbers), dtype=bool)
    mask[fixed] = True
    eng = ab.SgprEngine(model, species=[29])
    ref = host_fire(eng, start.positions, start.numbers, start.cell, start.pbc, n, fixed=mask)
    assert close(atoms.positions, ref["pos"]) and close(rx.forces, ref["F"])
    assert np.array_equal(rx.trace["dt"], ref["rows"][:, 2])
    eng.close()


@pytest.mark.parametrize("interval", [1, 7, 100])
def test_uncertainty_stop_is_exact(interval):
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax

    # mu = +1: the relaxation drives every environment away from the inducing one, so max(beta) grows
    model, start = lattice_well(mu=1.0, with_choli=True)
    n = 60
    eng = ab.SgprEngine(model, species=[29])
    bmax = host_fire(eng, start.positions, start.numbers, start.cell, start.pbc, n, covloss=True)["bmax"]
    stop = next(s for s in range(n // 3, n + 1) if bmax[s] > max(bmax[:s]))
    ediff = 0.5 * (max(bmax[:stop]) + bmax[stop])
    ref = host_fire(eng, start.positions, start.numbers, start.cell, start.pbc, n, covloss=True, ediff=ediff)
    assert ref["stop"] == stop and ref["steps"] == stop
    calls = []
    calc = ab.B200Calculator(model, covloss=True, ediff=ediff,
                             on_uncertain=lambda a, b: calls.append((a.positions.copy(), b.copy())))
    atoms = start.copy()
    rx = DeviceRelax(calc, atoms)
    assert rx.run(fmax=0.0, steps=n, interval=interval) is False
    assert rx.stopped and rx.stop_step == stop and rx.nsteps == stop and len(rx.trace["epot"]) == stop
    assert close(atoms.positions, ref["pos"]) and close(rx.forces, ref["F"]) and close(rx.beta, ref["beta"], 1e-8)
    assert len(calls) == 1 and close(calls[0][0], ref["pos"]) and close(calls[0][1], ref["beta"], 1e-8)
    assert rx.run(fmax=0.0, steps=10, interval=interval) is False and rx.nsteps == stop and len(calls) == 1
    # stopped, but run(fmax) still answers for the fmax it is given: the current forces are tested against it
    assert rx.run(fmax=1e300, steps=10, interval=interval) is True and rx.nsteps == stop and len(calls) == 1
    eng.close()


def test_overflow_recovery():
    """A step (or the starting evaluation) whose pair list outgrows the capacity sized by an earlier step commits
    nothing: it is enqueued again after sizing, and the run equals one that never overflowed."""
    import torch

    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax

    g = load_golden("cu108_sesoap")
    # as tests/test_gpu_md.py: 2 x 2 x 2 copies of the cell, and the same atoms squeezed to 0.7 of it about the centre
    shifts = np.array([[i, j, k] for i in range(2) for j in range(2) for k in range(2)]) @ g["cell"]
    sparse = (g["pos"][None] + shifts[:, None]).reshape(-1, 3)
    numbers, cell = np.tile(g["numbers"], 8), 2 * g["cell"]
    centre = cell.sum(0) / 2
    dense = centre + 0.7 * (sparse - centre)

    def same(r1, r2):
        assert close(r1.pos.cpu().numpy(), r2.pos.cpu().numpy()) and close(r1.velocities, r2.velocities)
        assert close(r1.forces, r2.forces) and np.array_equal(r1.fire[:2].cpu().numpy(), r2.fire[:2].cpu().numpy())
        assert close(r1.trace["epot"], r2.trace["epot"], 1e-12) and np.array_equal(r1.trace["dt"], r2.trace["dt"])
        assert np.array_equal(r1.trace["a"], r2.trace["a"])

    # (1) a step overflows: a FIRE step moves at most maxstep and the capacity only grows, so the driver's structure is
    # carried from the sparse to the dense one between two runs; its next step predicts (nearly) the dense structure
    def run_across(calc):
        rx = DeviceRelax(calc, Atoms(sparse, numbers, cell, True))
        rx.run(fmax=0.0, steps=5, interval=5)
        rx.pos.copy_(torch.as_tensor(dense, device=rx.pos.device))
        torch.cuda.synchronize()
        rx.run(fmax=0.0, steps=15, interval=15)
        assert rx.nsteps == 20
        return rx

    rx1 = run_across(ab.B200Calculator(b200_model(g)))      # a handle that only ever sized the sparse structure
    assert rx1.repeats >= 1
    fresh = ab.B200Calculator(b200_model(g))
    fresh.calculate(Atoms(dense, numbers, cell, True))     # sized on the dense structure: never overflows
    rx2 = run_across(fresh)
    assert rx2.repeats == 0
    same(rx1, rx2)

    # (2) the starting evaluation overflows
    def run(calc):
        atoms = Atoms(dense, numbers, cell, True)
        rx = DeviceRelax(calc, atoms)
        rx.run(fmax=0.0, steps=20, interval=20)
        assert rx.nsteps == 20
        return atoms, rx

    calc = ab.B200Calculator(b200_model(g))
    calc.calculate(Atoms(sparse, numbers, cell, True))     # sized on the sparse structure
    a1, rx1 = run(calc)
    assert rx1.repeats >= 1
    a2, rx2 = run(ab.B200Calculator(b200_model(g)))
    assert rx2.repeats == 0
    assert close(a1.positions, a2.positions) and close(rx1.velocities, rx2.velocities)
    assert close(rx1.trace["epot"], rx2.trace["epot"], 1e-12) and np.array_equal(rx1.trace["dt"], rx2.trace["dt"])


def test_errors_name_the_step_and_leave_the_handle_usable():
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceRelax

    g, atoms = golden_case("cu108_sesoap")
    calc = ab.B200Calculator(b200_model(g))
    E0 = float(calc.calculate(atoms)["energy"])
    eng = calc._engine
    # the atom that moves furthest along a in step 3 of the host loop, 120 cells out, with the whole structure shifted
    # along a so that its fractional x crosses 121 (one more than the neighbour search accepts) in step 3
    inv = np.linalg.inv(atoms.cell)
    f2 = host_fire(eng, atoms.positions, atoms.numbers, atoms.cell, atoms.pbc, 2)["pos"] @ inv
    f3 = host_fire(eng, atoms.positions, atoms.numbers, atoms.cell, atoms.pbc, 3)["pos"] @ inv
    i = int(np.argmax(f3[:, 0] - f2[:, 0]))
    assert f3[i, 0] > f2[i, 0]
    t = 1.0 - 0.5 * (f2[i, 0] + f3[i, 0])
    pos = atoms.positions + t * atoms.cell[0]
    pos[i] += 120 * atoms.cell[0]
    far = Atoms(pos, atoms.numbers, atoms.cell, True)
    rx = DeviceRelax(calc, far)
    with pytest.raises(RuntimeError, match="relaxation step 3:.*120 cells"):
        rx.run(fmax=0.0, steps=10, interval=10)
    assert rx.nsteps == 2
    assert float(calc.calculate(atoms)["energy"]) == E0
    with pytest.raises(ValueError, match="fmax"):
        rx.run(fmax=-1.0)
    assert calc._engine is eng and float(calc.calculate(atoms)["energy"]) == E0


def test_md_and_relax_share_a_handle():
    """DeviceMD and DeviceRelax alternating on one handle give their solo results: the graph cache keeps their
    captured steps apart."""
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceMD, DeviceRelax

    g = load_golden("cu108_sesoap")
    rng = np.random.default_rng(4)
    mom = rng.normal(size=g["pos"].shape) * 0.3

    class MdAtoms(Atoms):
        def __init__(self):
            super().__init__(g["pos"], g["numbers"], g["cell"], True)
            self.momenta = mom.copy()

        def get_masses(self):
            return np.full(len(self.numbers), 63.546)

        def get_momenta(self):
            return self.momenta.copy()

        def set_momenta(self, p):
            self.momenta = np.array(p)

    def solo(kind):
        calc = ab.B200Calculator(b200_model(g))
        if kind == "md":
            atoms = MdAtoms()
            DeviceMD(calc, atoms, timestep=0.5).run(40, interval=10)
        else:
            atoms = Atoms(g["pos"], g["numbers"], g["cell"], True)
            DeviceRelax(calc, atoms).run(fmax=0.0, steps=40, interval=10)
        return atoms.positions

    md_solo, rx_solo = solo("md"), solo("relax")
    calc = ab.B200Calculator(b200_model(g))
    md_atoms, rx_atoms = MdAtoms(), Atoms(g["pos"], g["numbers"], g["cell"], True)
    md, rx = DeviceMD(calc, md_atoms, timestep=0.5), DeviceRelax(calc, rx_atoms)
    for _ in range(4):
        assert md.run(10, interval=10) == 10
        rx.run(fmax=0.0, steps=10, interval=10)
    assert md.nsteps == 40 and rx.nsteps == 40
    assert close(md_atoms.positions, md_solo, 1e-12) and close(rx_atoms.positions, rx_solo, 1e-12)
