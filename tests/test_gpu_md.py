"""GPU: DeviceMD (molecular dynamics with positions, momenta and forces on the device) against host loops around
SgprEngine.predict that use the same operation order and the same noise stream (tests/md_reference.py)."""
import numpy as np
import pytest

from golden_util import b200_model, load_golden
from md_reference import FS, KB, host_md

pytestmark = pytest.mark.gpu

MASS = {1: 1.008, 3: 6.94, 8: 15.999, 13: 26.98, 14: 28.085, 15: 30.974, 16: 32.06, 29: 63.546, 47: 107.87}
TOL = 1e-9


class Atoms:
    """What DeviceMD reads and writes of an ase.Atoms."""

    def __init__(self, positions, numbers, cell, pbc, momenta=None):
        self.positions = np.array(positions, dtype=np.float64)
        self.numbers = np.asarray(numbers)
        self.cell = np.asarray(cell, dtype=np.float64)
        self.pbc = np.broadcast_to(np.asarray(pbc), (3,)).copy()
        self.momenta = np.zeros_like(self.positions) if momenta is None else np.array(momenta, dtype=np.float64)

    def get_masses(self):
        return np.array([MASS[int(z)] for z in self.numbers])

    def get_momenta(self):
        return self.momenta.copy()

    def set_momenta(self, p):
        self.momenta = np.array(p)

    def set_positions(self, r):
        self.positions = np.array(r)


def thermal_momenta(numbers, T, seed):
    m = np.array([MASS[int(z)] for z in numbers])[:, None]
    return np.random.default_rng(seed).normal(size=(len(m), 3)) * np.sqrt(m * KB * T)


def case(name, T=300.0, seed=1):
    g = load_golden(name)
    return g, Atoms(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"], thermal_momenta(g["numbers"], T, seed))


def engine(g):
    import autoforce_b200 as ab

    return ab.SgprEngine(b200_model(g), species=sorted(set(int(z) for z in g["numbers"])))


def calculator(g, **kw):
    import autoforce_b200 as ab

    return ab.B200Calculator(b200_model(g), **kw)


def close(a, b, tol=TOL):
    return np.abs(np.asarray(a) - np.asarray(b)).max() <= tol * max(1.0, np.abs(np.asarray(b)).max())


@pytest.mark.parametrize("name", ["cu108_sesoap", "lipso108", "cluster_lone", "slab_ttf"])
def test_nve_matches_host_loop(name):
    from autoforce_b200 import DeviceMD

    n = 200 if name in ("cu108_sesoap", "lipso108") else 30   # non-periodic / mixed pbc size every step
    g, atoms = case(name)
    eng = engine(g)
    r, p, F, _, rows, _, _ = host_md(eng, atoms.positions, atoms.numbers, atoms.cell, atoms.pbc, atoms.get_masses(),
                                     atoms.momenta, n, timestep=0.5)
    md = DeviceMD(calculator(g), atoms, timestep=0.5)
    assert md.run(n, interval=50) == n
    assert close(atoms.positions, r) and close(atoms.momenta, p)
    assert close(md.forces, F, 1e-8)
    th = md.thermo
    assert close(th["epot"], rows[:, 0], 1e-10) and close(th["ekin"], rows[:, 1], 1e-10)
    assert close(th["W"].reshape(-1, 9), rows[:, 2:], 1e-9)
    eng.close()


@pytest.mark.parametrize("name", ["cu108_sesoap", "lipso108"])
def test_langevin_matches_host_loop(name):
    from autoforce_b200 import DeviceMD

    g, atoms = case(name)
    eng = engine(g)
    kw = dict(timestep=0.5, temperature_K=500.0, friction=0.02, seed=2 ** 40 + 3)
    r, p, F, _, rows, _, _ = host_md(eng, atoms.positions, atoms.numbers, atoms.cell, atoms.pbc, atoms.get_masses(),
                                     atoms.momenta, 100, **kw)
    md = DeviceMD(calculator(g), atoms, **kw)
    assert md.run(100, interval=30) == 100
    assert close(atoms.positions, r) and close(atoms.momenta, p)
    assert close(md.thermo["ekin"], rows[:, 1], 1e-10)
    eng.close()


@pytest.mark.parametrize("langevin", [False, True])
def test_interval_does_not_matter(langevin):
    from autoforce_b200 import DeviceMD

    g, _ = case("cu108_sesoap")
    kw = dict(timestep=0.5, temperature_K=400.0, friction=0.01, seed=7) if langevin else dict(timestep=0.5)
    calc = calculator(g)
    out = []
    for interval in (120, 10, 1):
        _, atoms = case("cu108_sesoap")
        md = DeviceMD(calc, atoms, **kw)
        seen = []
        assert md.run(120, interval=interval, observer=lambda a, k: seen.append(k)) == 120
        assert seen == list(range(interval, 121, interval))
        out.append((atoms.positions, atoms.momenta, md.forces, md.thermo))
    for r, p, F, th in out[1:]:
        assert close(r, out[0][0], 1e-12) and close(p, out[0][1], 1e-12) and close(F, out[0][2], 1e-10)
        assert close(th["epot"], out[0][3]["epot"], 1e-12) and close(th["ekin"], out[0][3]["ekin"], 1e-12)


def test_energy_error_is_second_order():
    from autoforce_b200 import DeviceMD

    g, _ = case("cu108_sesoap")
    calc = calculator(g)
    span = 40.0   # fs
    fluct = []
    for dt in (0.5, 0.25):
        _, atoms = case("cu108_sesoap", T=300.0)
        md = DeviceMD(calc, atoms, timestep=dt)
        md.run(int(round(span / dt)), interval=1000)
        th = md.thermo
        etot = th["epot"] + th["ekin"]
        fluct.append(np.std(etot))
    ratio = fluct[0] / fluct[1]
    assert 3.0 < ratio < 5.0, (fluct, ratio)


def test_thermostat_reaches_target_temperature():
    from autoforce_b200 import DeviceMD, synth

    w = synth.WORKLOADS["c2"]
    pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
    import autoforce_b200 as ab

    calc = ab.B200Calculator(synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"]))
    T = 300.0
    atoms = Atoms(pos, numbers, cell, True, thermal_momenta(numbers, T, 5))
    md = DeviceMD(calc, atoms, timestep=1.0, temperature_K=T, friction=0.05, seed=11)
    md.run(1500, interval=500)
    Tm = md.thermo["temperature"][500:].mean()
    assert abs(Tm / T - 1.0) < 0.02, Tm


def _beta_trace(eng, atoms, n):
    """max(beta) at steps 0..n of the host velocity-Verlet loop (dt 1 fs)."""
    dt = FS
    m = atoms.get_masses()[:, None]
    r, p = atoms.positions.copy(), atoms.momenta.copy()
    _, F, _, _, beta = eng.predict(r, atoms.numbers, atoms.cell, atoms.pbc, want_beta=True)
    out = [float(np.max(beta))]
    for _ in range(n):
        p = p + 0.5 * dt * F
        r = r + dt * p / m
        _, F, _, _, beta = eng.predict(r, atoms.numbers, atoms.cell, atoms.pbc, want_beta=True)
        p = p + 0.5 * dt * F
        out.append(float(np.max(beta)))
    return out


@pytest.mark.parametrize("interval", [1, 7, 100])
def test_uncertainty_stop_is_exact(interval):
    from autoforce_b200 import DeviceMD

    g, atoms0 = case("cu108_sesoap", T=2000.0, seed=3)
    n = 60
    eng = engine(g)
    # ediff half-way between the running maximum of max(beta) and the first later step above it
    bmax = _beta_trace(eng, atoms0, n)
    stop = next(s for s in range(n // 3, n + 1) if bmax[s] > max(bmax[:s]))
    ediff = 0.5 * (max(bmax[:stop]) + bmax[stop])
    r, p, F, beta, _, done, host_stop = host_md(eng, atoms0.positions, atoms0.numbers, atoms0.cell, atoms0.pbc,
                                                atoms0.get_masses(), atoms0.momenta, n, timestep=1.0, covloss=True,
                                                ediff=ediff)
    assert host_stop == stop and done == stop
    calls = []
    calc = calculator(g, covloss=True, ediff=ediff, on_uncertain=lambda a, b: calls.append((a.positions.copy(), b.copy())))
    _, atoms = case("cu108_sesoap", T=2000.0, seed=3)
    md = DeviceMD(calc, atoms, timestep=1.0)
    assert md.run(n, interval=interval) == stop
    assert md.stop_step == stop and md.nsteps == stop and len(md.thermo["epot"]) == stop
    assert close(atoms.positions, r) and close(atoms.momenta, p) and close(md.forces, F, 1e-8)
    assert close(md.beta, beta, 1e-8)
    assert len(calls) == 1 and close(calls[0][0], r) and close(calls[0][1], beta, 1e-8)
    assert md.run(10, interval=interval) == 0 and len(calls) == 1   # stopped: nothing more, no second call
    eng.close()


def test_overflow_recovery():
    """A step whose pair list outgrows the capacity sized by an earlier step is not integrated: it is enqueued again
    after sizing, and the run equals one that never overflowed."""
    from autoforce_b200 import DeviceMD

    g = load_golden("cu108_sesoap")
    # 2 x 2 x 2 copies of the cell, and the same atoms squeezed to 0.7 of it about the centre: more than the head room
    # of the capacity sized on the original (sgpr_neighbors: 1.25 x + 4096 pairs)
    shifts = np.array([[i, j, k] for i in range(2) for j in range(2) for k in range(2)]) @ g["cell"]
    sparse = (g["pos"][None] + shifts[:, None]).reshape(-1, 3)
    numbers, cell = np.tile(g["numbers"], 8), 2 * g["cell"]
    centre = cell.sum(0) / 2
    dense = centre + 0.7 * (sparse - centre)
    m = np.array([MASS[int(z)] for z in numbers])[:, None]
    dt = 0.5
    # momenta that carry the sparse structure into the dense one in the first step
    p_in = m * (dense - sparse) / (dt * FS)

    def run(calc, pos, mom, steps):
        atoms = Atoms(pos, numbers, cell, True, mom)
        md = DeviceMD(calc, atoms, timestep=dt)
        assert md.run(steps, interval=steps) == steps
        return atoms, md

    # (1) the first step overflows: the handle was sized on the sparse structure
    calc = calculator(g)
    calc.calculate(Atoms(sparse, numbers, cell, True))
    a1, md1 = run(calc, sparse, p_in, 1)
    assert md1.repeats >= 1
    fresh = calculator(g)
    fresh.calculate(Atoms(dense, numbers, cell, True))     # sized on the dense structure: never overflows
    a2, md2 = run(fresh, sparse, p_in, 1)
    assert md2.repeats == 0
    assert close(a1.positions, a2.positions, 1e-12) and close(a1.momenta, a2.momenta, 1e-10)
    assert close(md1.thermo["epot"], md2.thermo["epot"], 1e-12)
    # (2) the starting evaluation overflows: a driver started from the dense structure on a handle sized sparse
    calc = calculator(g)
    calc.calculate(Atoms(sparse, numbers, cell, True))
    a3, md3 = run(calc, dense, np.zeros_like(dense), 20)
    assert md3.repeats >= 1
    a4, md4 = run(calculator(g), dense, np.zeros_like(dense), 20)
    assert md4.repeats == 0
    assert close(a3.positions, a4.positions) and close(a3.momenta, a4.momenta)
    assert close(md3.thermo["epot"], md4.thermo["epot"], 1e-12)


def test_errors_name_the_step_and_leave_the_handle_usable():
    from autoforce_b200 import DeviceMD

    g, atoms = case("cu108_sesoap", T=0.0)
    calc = calculator(g)
    E0 = float(calc.calculate(atoms)["energy"])
    eng = calc._engine
    # the atom with the largest fractional x, moved 120 cells along a and pushed outward so that floor(frac) reaches
    # 121 (one more than the neighbour search accepts) half-way through step 3
    frac = atoms.positions @ np.linalg.inv(atoms.cell)
    i = int(np.argmax(frac[:, 0]))
    pos = atoms.positions.copy()
    pos[i] += 120 * atoms.cell[0]
    mom = np.zeros_like(pos)
    dt = 1.0
    mom[i] = MASS[29] * (1.0 - frac[i, 0] % 1.0) / 2.5 * atoms.cell[0] / (dt * FS)
    far = Atoms(pos, atoms.numbers, atoms.cell, True, mom)
    md = DeviceMD(calc, far, timestep=dt)
    with pytest.raises(RuntimeError, match="MD step 3:.*120 cells"):
        md.run(10, interval=10)
    assert md.nsteps == 2
    assert float(calc.calculate(atoms)["energy"]) == E0
    # unknown species: refused at construction, before the handle is touched
    bad = Atoms(atoms.positions, np.where(np.arange(len(atoms.numbers)) == 0, 0, atoms.numbers), atoms.cell, True)
    with pytest.raises(ValueError, match="unknown species"):
        DeviceMD(calc, bad, masses=np.full(len(bad.numbers), 63.5))
    assert calc._engine is eng and float(calc.calculate(atoms)["energy"]) == E0
