"""GPU parity tests proper: the CUDA path, called through the C ABI (ctypes), against
(a) the golden vectors produced by the unmodified reference (tests/golden/*.npz) and
(b) the oracle on the same seeded inputs.

Bars (BASELINE.json north_star): neighbour lists bit-exact; energies within 1e-6 eV/atom,
forces within 1e-5 eV/A, stress within 1e-6 eV/A^3 of the reference's float64 path.
Everything on this path computes in float64, so the asserts below are far tighter.
"""
import numpy as np
import pytest

from golden_util import golden_cases, golden_radii, load_golden, load_train, oracle_model, train_cases
from oracle import sgpr_oracle as o

pytestmark = pytest.mark.gpu

TOL_E_PER_ATOM = 1e-9   # north_star: 1e-6 eV/atom
TOL_F = 1e-8            # north_star: 1e-5 eV/A
TOL_S = 1e-9            # north_star: 1e-6 eV/A^3


def model_from_golden(g, big=False):
    from golden_util import b200_model

    return b200_model(g, big)


def sorted_rows(first, J, S):
    I = np.repeat(np.arange(len(first) - 1), np.diff(first))
    order = np.lexsort((S[:, 2], S[:, 1], S[:, 0], J, I))
    return I[order], J[order].astype(np.int64), S[order].astype(np.int64)


def stress_of(W, cell):
    vol = abs(np.linalg.det(np.asarray(cell, dtype=float).reshape(3, 3))) or -2.0
    return (W / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]]


def golden_engine(name):
    import autoforce_b200 as ab

    g = load_golden(name)
    if g["meta"]["kernel"]["kind"] == "multi":
        pytest.skip("kernel sums run through one handle per kernel: test_kernel_sum_with_different_hyperparameters")
    return g, ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])


@pytest.fixture(params=golden_cases())
def case(request):
    g, eng = golden_engine(request.param)
    yield g, eng
    eng.close()


# The golden cells have 1-9 bins (cluster_lone: 1,700), so the automatic choice runs them through the warp-per-atom
# neighbour kernel; "<name>-bins" runs the same case through the block-per-bin kernel (SGPR_NL is read when the handle
# is created).  Tests that depend on the neighbour list take this fixture instead of `case`.
@pytest.fixture(params=golden_cases() + [n + "-bins" for n in golden_cases()])
def nl_case(request, monkeypatch):
    name, _, mode = request.param.partition("-")
    if mode:
        monkeypatch.setenv("SGPR_NL", mode)
    g, eng = golden_engine(name)
    yield g, eng
    eng.close()


def assert_golden_efs(g, E, F, W):
    N = len(g["numbers"])
    assert abs(E - float(g["energy"])) / N < TOL_E_PER_ATOM
    assert np.abs(F - g["forces"]).max() < TOL_F
    assert np.abs(stress_of(W, g["cell"]) - g["stress"]).max() < TOL_S


def test_neighbor_list_bit_exact(nl_case):
    g, eng = nl_case
    first, J, S = eng.neighbors(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    assert len(J) == len(g["nl_j"])
    a, b = sorted_rows(first, J, S), sorted_rows(g["nl_first"], g["nl_j"], g["nl_S"])
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_descriptors_match_reference_cache(case):
    g, eng = case
    if g["meta"]["kernel"]["kind"] in ("subsesoap", "heterosoap", "multi"):
        pytest.skip("dense per-kernel caches are not stored for SubSeSoapKernel lists")
    species = np.array(g["meta"]["species"])
    Zh = eng.inducing_descriptors()
    keep = ~oracle_model(g).excluded_centres(g["ind_Z"])
    ref = g["ind_desc"].reshape(Zh.shape)
    assert np.abs(Zh[keep] - ref[keep]).max() < 1e-13
    Zo, _ = o.inducing_descriptors(oracle_model(g), species)
    assert np.abs(Zh - Zo).max() < 1e-13
    P = eng.descriptors(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    om = oracle_model(g)
    for key in [k for k in g if k.startswith("desc_")]:
        a = int(key.split("_")[1])
        if om.excluded_centres(g["numbers"][a:a + 1])[0]:
            continue
        assert np.abs(P[a] - g[key].reshape(P[a].shape)).max() < 1e-13


def test_kernel_matrix(case):
    g, eng = case
    K = eng.kernel_matrix(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"]).cpu().numpy()
    assert K.shape == g["K"].shape
    assert np.abs(K - g["K"]).max() < 1e-12


def test_energy_forces_stress(nl_case):
    g, eng = nl_case
    N = len(g["numbers"])
    E, F, W, owned = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    assert owned.all()
    assert abs(E - float(g["energy"])) / N < TOL_E_PER_ATOM
    assert np.abs(F - g["forces"]).max() < TOL_F
    assert np.abs(stress_of(W, g["cell"]) - g["stress"]).max() < TOL_S
    # same through the oracle (independent derivative formulation)
    ref = o.predict(oracle_model(g), g["pos"], g["cell"], g["meta"]["pbc"], g["numbers"])
    assert abs(E - ref["energy"]) / N < TOL_E_PER_ATOM
    assert np.abs(F - ref["forces"]).max() < TOL_F
    assert np.abs(W - ref["virial"]).max() < 1e-8
    # weights x1000 through sgpr_set_weights: same K, amplified E/F/stress (relative bars)
    eng.set_weights(mu=g["mu_big"])
    E, F, W, _ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    assert abs(E - float(g["energy_big"])) / N < 1e-9 * max(1.0, abs(float(g["energy_big"])) / N)
    assert np.abs(F - g["forces_big"]).max() < 1e-10 * max(1.0, np.abs(g["forces_big"]).max())
    assert np.abs(stress_of(W, g["cell"]) - g["stress_big"]).max() < 1e-10 * max(1.0, np.abs(g["stress_big"]).max())


def test_device_pointer_api_matches_host_api(case):
    import torch

    g, eng = case
    E0, F0, W0, _ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    pos_t = torch.as_tensor(g["pos"], device="cuda")
    z_t = torch.as_tensor(g["numbers"].astype(np.int32), device="cuda")
    E, F, W = eng.predict_device(pos_t, z_t, g["cell"], g["meta"]["pbc"])
    torch.cuda.synchronize()
    assert float(E.cpu()[0]) == E0  # deterministic reductions: bit-identical energy
    assert np.abs(F.cpu().numpy() - F0).max() < 1e-12
    assert np.array_equal(W.cpu().numpy().reshape(3, 3), W0)


def test_calculator_results_mirror_reference(case):
    import autoforce_b200 as ab

    g, eng = case

    class A:  # anything with positions / cell / pbc / numbers
        positions, cell, pbc, numbers = g["pos"], g["cell"], g["meta"]["pbc"], g["numbers"]

    calc = ab.B200Calculator(model_from_golden(g))
    res = calc.calculate(A())
    assert res["energy"].shape == () and res["energy"].dtype == np.float64      # active.py:572
    assert res["stress"].shape == (6,)                                             # active.py:574
    assert abs(float(res["energy"]) - float(g["energy"])) / len(g["numbers"]) < TOL_E_PER_ATOM
    assert np.abs(res["forces"] - g["forces"]).max() < TOL_F
    assert np.abs(res["stress"] - g["stress"]).max() < TOL_S
    assert float(res["free_energy"]) == float(res["energy"])                      # active.py:527


def test_unknown_species_is_an_error():
    import autoforce_b200 as ab

    g = load_golden("cu108_sesoap")
    eng = ab.SgprEngine(model_from_golden(g))
    numbers = g["numbers"].copy()
    numbers[3] = 47
    with pytest.raises(RuntimeError, match="species"):
        eng.predict(g["pos"], numbers, g["cell"], True)
    eng.close()


def test_empty_structure():
    import autoforce_b200 as ab

    g = load_golden("cu108_sesoap")
    eng = ab.SgprEngine(model_from_golden(g))
    E, F, W, owned = eng.predict(np.zeros((0, 3)), np.zeros(0, np.int32), g["cell"], True)
    assert E == 0.0 and F.shape == (0, 3) and np.all(W == 0)
    eng.close()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_atom_sharding_sums_to_single_rank_result(nl_case, world):
    """SURVEY 8e: every rank evaluates its owned environments + the one-cutoff halo and
    returns E/W partial sums and the forces of its owned atoms; summing the ranks (what
    the 10-double all-reduce does for E and W) must reproduce the unsharded result."""
    g, eng = nl_case
    args = (g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    E0, F0, W0, own0 = eng.predict(*args)
    E, F, W = 0.0, np.zeros_like(F0), np.zeros_like(W0)
    count = np.zeros(len(F0), dtype=int)
    for rank in range(world):
        e, f, w, owned = eng.predict(*args, rank=rank, world=world)
        assert np.all(f[~owned] == 0.0)
        E, F, W = E + e, F + f, W + w
        count += owned
    assert np.all(count == 1)                       # disjoint and complete ownership
    N = len(F0)
    assert abs(E - E0) / N < 1e-12
    assert np.abs(F - F0).max() < 1e-11
    assert np.abs(W - W0).max() < 1e-10
    assert_golden_efs(g, E, F, W)                   # both sides run the same neighbour kernel: check the list itself


def test_covloss_matches_reference(nl_case):
    """beta = get_covloss() (calculator/active.py:781-804), incl. sqrt(vscale), inf for species
    without variance scale and NaN for centres excluded via a/a_not."""
    g, eng = nl_case
    E, F, W, owned, beta = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"], want_beta=True)
    ref = g["covloss"]
    fin = np.isfinite(ref)
    assert np.array_equal(np.isfinite(beta), fin)
    assert np.array_equal(np.isnan(beta), np.isnan(ref))
    # the sqrt next to the clamp amplifies rounding: compare beta^2
    assert np.abs(beta[fin] ** 2 - ref[fin] ** 2).max() < 1e-9
    # asking for beta must not change E/F/W (same tcgen05 GEMMs; the covloss GEMM is an extra launch)
    E0, F0, W0, _ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    assert abs(E - E0) < 1e-10 * max(1.0, abs(E0)) and np.abs(W - W0).max() < 1e-9 and np.abs(F - F0).max() < 1e-10
    # sharded: each rank fills the betas of the atoms it owns
    parts = np.zeros_like(beta)
    for rank in range(3):
        _, _, _, own, b = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"], rank=rank, world=3, want_beta=True)
        parts[own] = b[own]
    assert np.array_equal(np.isnan(parts), np.isnan(beta))
    assert np.abs(parts[fin] ** 2 - beta[fin] ** 2).max() < 1e-12


def test_differentiable_cov_matches_reference_autograd(case):
    """Compat mode (SURVEY 8f-2): cov[N,M] as a differentiable torch tensor.  With E = (cov @ mu).sum(), autograd
    through sgpr_kernel_forward / sgpr_kernel_backward must reproduce the reference's forces and stress
    (calculator/active.py:587-611: F = -dE/dxyz, stress = (-sum F (x) x + sum cellgrad (x) lll) / V)."""
    import torch

    g, eng = case
    xyz = torch.tensor(g["pos"], dtype=torch.float64, requires_grad=True)
    lll = torch.tensor(g["cell"], dtype=torch.float64, requires_grad=True)
    cov = eng.cov(xyz, lll, g["numbers"], g["meta"]["pbc"])
    assert cov.shape == g["K"].shape and np.abs(cov.detach().numpy() - g["K"]).max() < 1e-12
    mu = torch.tensor(g["mu"], dtype=torch.float64)
    E = (cov @ mu).sum()
    gx, gl = torch.autograd.grad(E, [xyz, lll])
    forces = -gx.numpy()
    assert np.abs(forces - g["forces"]).max() < TOL_F
    stress1 = -(forces[:, None, :] * g["pos"][:, :, None]).sum(axis=0)
    stress2 = (gl.numpy()[:, None, :] * g["cell"][:, :, None]).sum(axis=0)
    vol = abs(np.linalg.det(g["cell"])) or -2.0
    stress = ((stress1 + stress2) / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]]
    assert np.abs(stress - g["stress"]).max() < TOL_S
    # a random cotangent: forces of L = sum_im w_im K_im against finite differences of the forward hook
    rng = np.random.default_rng(0)
    w = torch.tensor(rng.normal(size=g["K"].shape))
    cov = eng.cov(xyz, lll, g["numbers"], g["meta"]["pbc"])
    (gx,) = torch.autograd.grad((cov * w).sum(), [xyz])
    i, k, d = len(g["pos"]) // 2, 1, 1e-5
    p = g["pos"].copy()
    p[i, k] += d
    Lp = float((eng.kernel_matrix(p, g["numbers"], g["cell"], g["meta"]["pbc"]).cpu() * w).sum())
    p[i, k] -= 2 * d
    Lm = float((eng.kernel_matrix(p, g["numbers"], g["cell"], g["meta"]["pbc"]).cpu() * w).sum())
    assert abs((Lp - Lm) / (2 * d) - float(gx[i, k])) < 1e-6 * max(1.0, abs(float(gx[i, k])))


@pytest.mark.gpu
def test_pinned_host_buffers_take_the_direct_dma_path():
    """sgpr_predict_host copies page-locked caller buffers without staging: same results as pageable ones."""
    import autoforce_b200 as ab

    g = load_golden("lipso108")
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    E0, F0, W0, own0 = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    pos = ab.SgprEngine.pinned(g["pos"].shape)
    pos[...] = g["pos"]
    Z = ab.SgprEngine.pinned((len(g["numbers"]),), np.int32)
    Z[...] = g["numbers"]
    F = ab.SgprEngine.pinned(g["pos"].shape)
    F[...] = np.nan
    E1, F1, W1, own1 = eng.predict(pos, Z, g["cell"], g["meta"]["pbc"], out_forces=F)
    # (forces are scattered with atomics: equal to rounding, not bitwise)
    assert F1 is F and abs(E1 - E0) < 1e-10 and np.abs(F - F0).max() < 1e-11 and np.abs(W1 - W0).max() < 1e-9
    assert np.array_equal(own0, own1)
    with pytest.raises(ValueError):
        eng.predict(pos, Z, g["cell"], g["meta"]["pbc"], out_forces=np.zeros((3, 3)))


@pytest.mark.parametrize("name", ["lipso108", "cu108_sesoap"])
def test_append_inducing_matches_a_model_built_in_one_go(name):
    """sgpr_append_inducing (add_inducing + make_munu, regression/gppotential.py:888-940): a handle built from the
    first inducing LCEs and then extended gives the golden E/F/stress/beta of the full model."""
    import dataclasses

    import autoforce_b200 as ab

    g = load_golden(name)
    full = model_from_golden(g)
    M = full.M
    k = max(1, M // 3)
    f = full.ind_first
    part = dataclasses.replace(full, ind_Z=full.ind_Z[:k], ind_first=f[: k + 1], ind_r=full.ind_r[: f[k]], ind_b=full.ind_b[: f[k]],
                               mu=full.mu[:k], choli=None)
    eng = ab.SgprEngine(part, species=g["meta"]["species"])
    envs = [(int(full.ind_Z[m]), full.ind_r[f[m] : f[m + 1]], full.ind_b[f[m] : f[m + 1]]) for m in range(k, M)]
    # an unknown species is refused and leaves the old model in place
    E_part, *_ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    with pytest.raises(RuntimeError):
        eng.append_inducing([(99, np.zeros((0, 3)), np.zeros(0, dtype=np.int32))], np.zeros(k + 1))
    assert abs(eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])[0] - E_part) < 1e-9 * max(1.0, abs(E_part))
    # two appends: one LCE, then the rest (intermediate weights are placeholders)
    eng.append_inducing(envs[:1], np.zeros(k + 1))
    eng.append_inducing(envs[1:], full.mu, full.choli)
    assert eng.model.M == M and np.array_equal(eng.model.ind_first, full.ind_first)
    E, F, W, owned, beta = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"], want_beta=True)
    N = len(g["numbers"])
    assert abs(E - float(g["energy"])) < TOL_E_PER_ATOM * N
    assert np.abs(F - g["forces"]).max() < TOL_F
    assert np.abs(stress_of(W, g["cell"]) - g["stress"]).max() < TOL_S
    ref = o.predict(oracle_model(g), g["pos"], g["cell"], g["meta"]["pbc"], g["numbers"], want_beta=True)["beta"]
    fin = np.isfinite(ref)
    assert np.abs(beta[fin] ** 2 - ref[fin] ** 2).max() < 1e-9
    Kmat = eng.kernel_matrix(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"]).cpu().numpy()
    assert np.abs(Kmat - g["K"]).max() < 1e-12
    eng.close()


@pytest.mark.parametrize("name", train_cases())
def test_training_kernels_match_reference_autograd(name):
    """sgpr_kernel_jacobian: Kf = forces_energy, Kv = virial_energy of the structure against the inducing set
    (regression/gppotential.py:66-77) equal the derivatives torch.autograd takes through the reference's own
    forward pass (tests/golden/make_golden_train.py), and the oracle's."""
    import autoforce_b200 as ab

    g, t = load_golden(name), load_train(name)
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    K, Kf, Kv = eng.kernel_jacobian(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    K, Kf, Kv = K.cpu().numpy(), Kf.cpu().numpy(), Kv.cpu().numpy()
    N, M = len(g["numbers"]), len(g["mu"])
    assert Kf.shape == (3 * N, M) and Kv.shape == (6, M)
    assert np.abs(K.sum(axis=0) - t["Ke"]).max() < 1e-11
    assert np.abs(Kf - t["Kf_autograd"]).max() < 1e-9
    assert np.abs(Kv - t["Kv_autograd"]).max() < 1e-8
    assert np.abs(Kv - t["Kv_analytic"]).max() < 1e-6
    # a sub-range of inducing LCEs gives the same columns; forces = Kf @ mu
    _, Kf2, Kv2 = eng.kernel_jacobian(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"], m0=1, m1=min(M, 4))
    assert np.abs(Kf2.cpu().numpy() - Kf[:, 1 : min(M, 4)]).max() < 1e-12 and np.abs(Kv2.cpu().numpy() - Kv[:, 1 : min(M, 4)]).max() < 1e-11
    assert np.abs(Kf @ g["mu"] - g["forces"].reshape(-1)).max() < TOL_F
    eng.close()


def test_similarity_kernel_operations():
    """kern(atoms, X, operation=...) of similarity/similarity.py:17-31 for func / leftgrad / virial."""
    import types

    import autoforce_b200 as ab

    g, t = load_golden("cu108_sesoap"), load_train("cu108_sesoap")
    k = g["meta"]["kernel"]
    kern = ab.SeSoapKernel(k["lmax"], k["nmax"], k["xi"], k["rc"], radii=ab.DefaultRadii())
    atoms = types.SimpleNamespace(positions=g["pos"], numbers=g["numbers"], cell=g["cell"], pbc=g["meta"]["pbc"])
    X = [(int(z), r, b) for z, r, b in zip(g["ind_Z"], g["envs_r"], g["envs_b"])]
    assert np.abs(kern(atoms, X) - g["K"]).max() < 1e-12
    assert np.abs(-kern(atoms, X, operation="leftgrad") - t["Kf_autograd"]).max() < 1e-9
    assert np.abs(kern(atoms, X, operation="virial") - t["Kv_autograd"]).max() < 1e-8
    with pytest.raises(NotImplementedError):
        kern(atoms, X, operation="gradgrad")


def test_lammps_fix_external_callback_drives_the_gpu_path():
    """cl/lmp.py:42-71 with the B200 calculator: forces by tag, global energy and virial handed to the fix."""
    import autoforce_b200 as ab
    from autoforce_b200 import lammps_driver as ld
    from test_lammps_driver import FakeLammps

    g = load_golden("cu108_sesoap")
    cell = np.asarray(g["cell"], dtype=float)
    assert np.allclose(cell, np.triu(cell))          # LAMMPS box convention
    lmp = FakeLammps(cell, g["pos"], [1] * len(g["numbers"]))
    calc = ab.B200Calculator(model_from_golden(g))
    cb = ld.FixExternalCallback(lmp, calc, "metal", {1: int(g["numbers"][0])})
    tag = np.random.default_rng(0).permutation(len(g["numbers"])) + 1
    fext = np.zeros((len(tag), 3))
    cb(None, 0, len(tag), tag, None, fext)
    assert np.abs(fext - g["forces"][tag - 1]).max() < TOL_F
    assert abs(lmp.energy[1] - float(g["energy"])) < TOL_E_PER_ATOM * len(tag)
    vol = abs(np.linalg.det(cell))
    assert np.allclose(lmp.virial[1], -g["stress"][[0, 1, 2, 5, 4, 3]] * vol, rtol=1e-6, atol=1e-9)


def test_calculator_prediction_mode_uncertainty():
    """calculator/active.py:492-499: in prediction mode the covloss is evaluated every step, its maximum logged
    (covlog) and uncertain structures handed on."""
    import types

    import autoforce_b200 as ab

    g = load_golden("lipso108")
    atoms = types.SimpleNamespace(positions=g["pos"], numbers=g["numbers"], cell=g["cell"], pbc=g["meta"]["pbc"])
    seen = []
    calc = ab.B200Calculator(model_from_golden(g), covloss=True, ediff=0.0, on_uncertain=lambda a, b: seen.append(b.copy()))
    res = calc.calculate(atoms, properties=("energy", "forces", "stress"))
    assert abs(float(res["energy"]) - float(g["energy"])) / len(g["numbers"]) < TOL_E_PER_ATOM
    ref = g["covloss"]
    assert np.abs(calc.beta ** 2 - ref ** 2).max() < 1e-9 and len(seen) == 1
    assert abs(float(calc.covlog) - float(ref.max())) < 1e-6
    # without the option nothing is evaluated until asked for
    calc2 = ab.B200Calculator(model_from_golden(g))
    calc2.calculate(atoms)
    assert calc2.beta is None and calc2.covlog == ""
    assert np.abs(calc2.get_covloss() ** 2 - ref ** 2).max() < 1e-9
    with pytest.raises(ValueError):
        import dataclasses

        ab.B200Calculator(dataclasses.replace(model_from_golden(g), choli=None), covloss=True)


@pytest.mark.parametrize("mode", ["bins", "warp"])
def test_neighbor_list_far_from_the_origin(mode, monkeypatch):
    """Unwrapped trajectories: atoms up to ~100 cells away from the unit cell (the library's limit is 120 and is
    reported as an error).  The accept/reject decision must still be the reference's (distance from the given
    positions in its rounding sequence), for both neighbour kernels."""
    import autoforce_b200 as ab

    monkeypatch.setenv("SGPR_NL", mode)
    g = load_golden("cu108_perfect")    # perfect lattice: many pairs at exactly equal distances
    rc = g["meta"]["kernel"]["rc"]
    a0 = g["cell"][0, 0] / 3
    # scale so that a shell of neighbours sits (numerically) at the cutoff, then move everything far away
    scale = rc / (a0 * np.sqrt(2.5))
    cell = g["cell"] * scale
    pos = g["pos"] * scale + 100.0 * cell[0] - 97.0 * cell[1] + 64.0 * cell[2] + np.array([0.3, -0.2, 0.1])
    pos[::7] -= 15.0 * cell[0]
    pos[3::5] += 20.0 * cell[2]
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    first, J, S = eng.neighbors(pos, g["numbers"], cell, True)
    f0, J0, S0 = o.neighbor_list(pos, cell, True, rc)
    assert np.array_equal(first, f0)
    a, b = sorted_rows(first, J, S), sorted_rows(f0, J0, S0)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    with pytest.raises(RuntimeError, match="120 cells"):
        eng.neighbors(pos + 400.0 * cell[1], g["numbers"], cell, True)
    eng.close()
    # opposite wraps: half the atoms 70 cells out, half -70, so neighbours are ~140 cells apart.  Prediction (int shifts)
    # must equal the oracle's on the same atoms at home (the oracle's image search over +-140 cells would take hours);
    # the exported list cannot hold such a shift in int8 and must refuse instead of wrapping it.
    g = load_golden("lipso108")
    pos = np.array(g["pos"], dtype=float)
    out = 70.0 * g["cell"].sum(axis=0)
    pos[0::2] += out
    pos[1::2] -= out
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    E, F, W, _ = eng.predict(pos, g["numbers"], g["cell"], g["meta"]["pbc"])
    ref = o.predict(oracle_model(g), g["pos"], g["cell"], g["meta"]["pbc"], g["numbers"])
    N = len(g["numbers"])
    assert abs(E - ref["energy"]) / N < TOL_E_PER_ATOM
    assert np.abs(F - ref["forces"]).max() < TOL_F
    assert np.abs(W - ref["virial"]).max() < 1e-8
    with pytest.raises(RuntimeError, match="int8 range"):
        eng.neighbors(pos, g["numbers"], g["cell"], g["meta"]["pbc"])
    eng.close()


@pytest.mark.parametrize("name", ["lipso108", "tric_oh"])
def test_many_kernel_front_end_of_very_large_systems(name, monkeypatch):
    """Above 2^18 bin x species keys / 2^16 rows the cell sort and the row scan use cub scans and separate kernels instead
    of the one-block versions; SGPR_NL_LEAN=0 forces that path on a small case.  Same lists, same results, also on
    sync-free (warm) steps, and for a batch (structure-major keys of many structures): the same E and W, bit for bit,
    as the one-block path."""
    import autoforce_b200 as ab
    from test_gpu_batch import golden_batch, run_batch

    g = load_golden(name)
    structs = golden_batch(g)
    monkeypatch.delenv("SGPR_NL_LEAN", raising=False)
    lean = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])   # reads SGPR_NL_LEAN when created
    E0, F0, W0 = run_batch(lean, structs)
    lean.close()
    monkeypatch.setenv("SGPR_NL_LEAN", "0")
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    first, J, S = eng.neighbors(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    f0, J0, S0 = o.neighbor_list(g["pos"], g["cell"], g["meta"]["pbc"], g["meta"]["kernel"]["rc"])
    assert np.array_equal(first, f0)
    assert all(np.array_equal(x, y) for x, y in zip(sorted_rows(first, J, S), sorted_rows(f0, J0, S0)))
    for _ in range(3):    # sizing step, then warm steps
        E, F, W, _ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
        assert abs(E - float(g["energy"])) / len(g["numbers"]) < TOL_E_PER_ATOM
        assert np.abs(F - g["forces"]).max() < TOL_F
    E, F, W = run_batch(eng, structs)
    assert np.array_equal(E, E0) and np.array_equal(W, W0)
    assert np.abs(F - F0).max() < 1e-12
    eng.close()


@pytest.mark.parametrize("mode", ["bins", "warp"])
def test_neighbor_list_with_crowded_bins(mode, monkeypatch):
    """More than 32 atoms of one species in one bin (the warp-per-bin ordering of the cell sort falls back to an insertion
    sort there) and candidate tiles that span several batches: a dense droplet in a large periodic box, and the same
    droplet in an open box.  Rows and their order-independent content must equal the oracle's."""
    import autoforce_b200 as ab

    monkeypatch.setenv("SGPR_NL", mode)
    g = load_golden("lipso108")
    rc = g["meta"]["kernel"]["rc"]
    rng = np.random.default_rng(11)
    n = 2400                                    # > 2048 candidates per atom: beyond the accept-bit words of the count pass
    pos = rng.uniform(0.0, 1.6 * rc, size=(n, 3)) + np.array([7.0, 9.0, 5.0])
    sp = np.asarray(g["meta"]["species"])
    Z = sp[rng.integers(0, 2, size=n)]          # two species: hundreds of atoms per (bin, species) key
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    for cell, pbc in ((np.diag([41.0, 39.0, 43.0]), True), (np.diag([41.0, 39.0, 43.0]), False)):
        first, J, S = eng.neighbors(pos, Z, cell, pbc)
        f0, J0, S0 = o.neighbor_list(pos, cell, pbc, rc)
        assert np.array_equal(first, f0)
        a, b = sorted_rows(first, J, S), sorted_rows(f0, J0, S0)
        assert all(np.array_equal(x, y) for x, y in zip(a, b))
    eng.close()


def test_kernel_sum_with_different_hyperparameters():
    """EnergyForceKernel sums similarity kernels (regression/gppotential.py:81-84); kernels with different lmax / nmax /
    exponent / cutoff run as one handle each and add up.  The golden structure has an isolated atom and a pair whose
    distance lies between the two cutoffs ("neighbour-less" refers to the largest cutoff in the reference)."""
    import types

    import autoforce_b200 as ab

    g = load_golden("two_kernels")
    models = model_from_golden(g)
    assert len(models) == 2
    lead = max(range(2), key=lambda i: models[i].rc)
    for i, m in enumerate(models):      # what SgprModel.list_from_posterior_potential sets up
        m.lone_weight = 2.0 if i == lead else -1.0
        if i != lead:
            m.mean_w = {}
    atoms = types.SimpleNamespace(positions=g["pos"], numbers=g["numbers"], cell=g["cell"], pbc=g["meta"]["pbc"])
    calc = ab.B200Calculator(models)
    res = calc.calculate(atoms, properties=("energy", "forces", "stress"))
    N = len(g["numbers"])
    assert abs(float(res["energy"]) - float(g["energy"])) / N < TOL_E_PER_ATOM
    assert np.abs(res["forces"] - g["forces"]).max() < TOL_F
    assert np.abs(res["stress"] - g["stress"]).max() < TOL_S
    # the kernel matrices add up as well
    K = sum(e.kernel_matrix(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"]).cpu().numpy()
            for e in [calc._engine] + calc._more_engines)
    assert np.abs(K - g["K"]).max() < 1e-12
    with pytest.raises(NotImplementedError):
        ab.B200Calculator([dataclasses_replace(m, choli=g["choli"]) for m in models], covloss=True)


def dataclasses_replace(obj, **kw):
    import dataclasses

    return dataclasses.replace(obj, **kw)


def test_one_handle_survives_growing_structures():
    """ADVICE r1 (high): the pinned staging area of sgpr_predict_host grows with the structure; the fixed-size
    tensor-map staging of the tcgen05 path must survive that (it was freed and reused).  One handle sees N, 8N (grow)
    and N again; every result must equal a fresh handle's."""
    import autoforce_b200 as ab

    g = load_golden("lipso108")
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    pos, Z, cell = np.asarray(g["pos"]), np.asarray(g["numbers"]), np.asarray(g["cell"]).reshape(3, 3)
    reps = [(1, 1, 1), (2, 2, 2), (1, 1, 1), (3, 2, 2)]
    for rep in reps:
        shifts = np.array([[i, j, k] for i in range(rep[0]) for j in range(rep[1]) for k in range(rep[2])], dtype=float)
        P = (pos[None, :, :] + (shifts @ cell)[:, None, :]).reshape(-1, 3)
        Zr = np.tile(Z, len(shifts))
        C = cell * np.array(rep)[:, None]
        E, F, W, _ = eng.predict(P, Zr, C, g["meta"]["pbc"])
        n = len(shifts)
        # a periodic supercell repeats the primitive result
        assert abs(E - n * float(g["energy"])) / len(Zr) < TOL_E_PER_ATOM
        assert np.abs(F.reshape(n, len(Z), 3) - g["forces"][None]).max() < TOL_F
        assert np.abs(stress_of(W, C) - g["stress"]).max() < TOL_S
    eng.close()


def test_similarity_interface_on_environments_and_cached_engine():
    """VERDICT r1 item 9: the kernel mirrors take environments (reference ``Local``-like objects or tuples) on either
    side, keep ONE engine per inducing set, and expose precalculate / call_descriptor (similarity/universal.py:97-107)."""
    import types

    import autoforce_b200 as ab
    from autoforce_b200 import engine as eng_mod

    g = load_golden("lipso108")
    k = g["meta"]["kernel"]
    kern = ab.SeSoapKernel(k["lmax"], k["nmax"], k["xi"], k["rc"], radii=ab.DefaultRadii())
    atoms = types.SimpleNamespace(positions=g["pos"], numbers=g["numbers"], cell=g["cell"], pbc=g["meta"]["pbc"])
    X = [types.SimpleNamespace(number=int(z), _r=r, _b=b) for z, r, b in zip(g["ind_Z"], g["envs_r"], g["envs_b"])]
    created = []
    orig = eng_mod.SgprEngine.__init__

    def counting(self, *a, **kw):
        created.append(1)
        orig(self, *a, **kw)

    eng_mod.SgprEngine.__init__ = counting
    try:
        K1 = kern(atoms, X)
        K2 = kern(atoms, X)
        assert len(created) == 1, "the engine of an inducing set must be cached"
        assert np.abs(K1 - g["K"]).max() < 1e-12 and np.array_equal(K1, K2)
        # a grown inducing set extends the cached engine in place
        extra = types.SimpleNamespace(number=int(g["ind_Z"][0]), _r=g["envs_r"][0] * 1.01, _b=g["envs_b"][0])
        K3 = kern(atoms, X + [extra])
        assert len(created) == 1 and K3.shape[1] == len(X) + 1 and np.abs(K3[:, :-1] - g["K"]).max() < 1e-12
    finally:
        eng_mod.SgprEngine.__init__ = orig
    # environments on the left: kern(X, X) is the M x M matrix; it equals the oracle's and has a unit diagonal
    KXX = kern(X, X)
    om = oracle_model(g)
    species = np.array(g["meta"]["species"])
    Zh, lone = o.inducing_descriptors(om, species)
    Ko, _, _ = o.kernel_from_descriptors(om, Zh, np.asarray(g["ind_Z"], dtype=np.int64), lone, Zh, lone)
    assert KXX.shape == (len(X), len(X)) and np.abs(KXX - Ko).max() < 1e-12
    assert np.abs(np.diag(KXX) - 1.0).max() < 1e-12
    # one environment against the set: a row of the same matrix
    assert np.abs(kern(X[3], X) - KXX[3:4]).max() < 1e-13
    # a structure on the right stands for all of its environments: kern(atoms, atoms) (calculator/active.py:655)
    Kaa = kern(atoms, atoms)
    assert Kaa.shape == (len(g["numbers"]), len(g["numbers"])) and np.abs(np.diag(Kaa) - 1.0).max() < 1e-12
    assert np.abs(Kaa - Kaa.T).max() < 1e-12
    # call_descriptor / precalculate: the reference's sparse [120, 120, dim] cache (loc.kern_0_value)
    d = kern.call_descriptor(X[0]).to_dense().numpy()
    ref = g["ind_desc"][0].reshape(len(species), len(species), -1)
    for a, z1 in enumerate(species):
        for b, z2 in enumerate(species):
            assert np.abs(d[z2, z1] - ref[a, b]).max() < 1e-13
    assert kern.precalculate(X[0]) is not None and X[0].kern_0_value is not None
    lone_loc = types.SimpleNamespace(number=3, _r=np.zeros((0, 3)), _b=np.zeros(0, dtype=np.int64))
    assert kern.precalculate(lone_loc) is None and lone_loc.kern_0_value is None
    kern.close()


def test_fixed_central_species_kernel():
    """ADVICE r1: a kernel with a fixed central species (a=Z) must only produce rows for that species."""
    import types

    import autoforce_b200 as ab

    g = load_golden("afixed_2sp")
    k = g["meta"]["kernel"]
    kern = ab.SeSoapKernel(k["lmax"], k["nmax"], k["xi"], k["rc"], a=k["a"], radii=ab.DefaultRadii())
    atoms = types.SimpleNamespace(positions=g["pos"], numbers=g["numbers"], cell=g["cell"], pbc=g["meta"]["pbc"])
    X = [(int(z), r, b) for z, r, b in zip(g["ind_Z"], g["envs_r"], g["envs_b"])]
    K = kern(atoms, X)
    assert np.abs(K - g["K"]).max() < 1e-12
    assert np.abs(K[np.asarray(g["numbers"]) != k["a"]]).max() == 0.0
    kern.close()


@pytest.mark.parametrize("world", [2, 3, 8])
def test_peer_memory_exchange_emulated_on_one_gpu(nl_case, world):
    """The force exchange bench.py --gpus N uses (sgpr_predict_p2p + sgpr_p2p_collect): every emulated rank evaluates
    only the environments it owns and adds neighbour forces into the OWNER's accumulation buffer.  Here the peer table
    points at ``world`` local buffers of one GPU (one handle per emulated rank); the assembled result must equal the
    unsharded one.  (tools/p2p_check.py runs the same comparison over real NVLink peers under torchrun.)"""
    import torch

    import autoforce_b200 as ab

    g, eng0 = nl_case
    N = len(g["numbers"])
    E0, F0, W0, _ = eng0.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    dev = torch.device("cuda", 0)
    pos_t = torch.as_tensor(np.asarray(g["pos"], dtype=np.float64), device=dev)
    z_t = torch.as_tensor(np.asarray(g["numbers"], dtype=np.int32), device=dev)
    bufs = torch.zeros((world, 3 * N + 8), dtype=torch.float64, device=dev)
    ews = torch.zeros((world, 10), dtype=torch.float64, device=dev)
    engines = [ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"]) for _ in range(world)]
    try:
        ptrs = [bufs[r].data_ptr() for r in range(world)]
        for r, e in enumerate(engines):
            e.predict_p2p(pos_t, z_t, g["cell"], g["meta"]["pbc"], r, world, ptrs, ews[r])
        torch.cuda.synchronize()
        F = torch.zeros((N, 3), dtype=torch.float64, device=dev)
        covered = torch.zeros(N, dtype=torch.int32, device=dev)
        for r, e in enumerate(engines):
            Fr = torch.zeros((N, 3), dtype=torch.float64, device=dev)
            own = torch.zeros(N, dtype=torch.uint8, device=dev)
            e.p2p_collect(bufs[r], Fr, own)
            torch.cuda.synchronize()
            F += Fr * own.to(torch.float64)[:, None]
            covered += own.to(torch.int32)
        assert bool((covered == 1).all()), "every atom is owned by exactly one rank"
        ew = ews.sum(dim=0).cpu().numpy()
        assert abs(ew[0] - E0) / N < 1e-12
        assert np.abs(F.cpu().numpy() - F0).max() < 1e-10
        assert np.abs(ew[1:].reshape(3, 3) - W0).max() < 1e-9
        assert_golden_efs(g, ew[0], F.cpu().numpy(), ew[1:].reshape(3, 3))
    finally:
        for e in engines:
            e.close()


def test_sync_free_steps_and_overflow_recovery():
    """Steps after the first one of a shape run without host synchronisation (pair count, species row ranges and error
    flags stay on the device).  (1) warm steps reproduce the sizing step bit for bit; (2) a warm step whose pair list
    outgrows the capacity sized earlier is repeated transparently by the host entry point; (3) the asynchronous
    device-pointer entry point reports it through check() and never corrupts memory; (4) species per atom may change
    between warm steps (row ranges are re-derived on the device)."""
    import torch

    import autoforce_b200 as ab
    from autoforce_b200 import synth

    Zs = [3, 8]
    model = synth.synth_model(Zs, 40, 5, lmax=3, nmax=3, rc=6.0)
    pos, cell, numbers = synth.fcc(6, Zs, 0.1, 1)
    N = len(numbers)
    ref_eng = ab.SgprEngine(model, species=Zs)
    E_ref, F_ref, W_ref, _ = ref_eng.predict(pos, numbers, cell, True)
    n_pairs_dense = ref_eng.stats()["n_pairs"]
    eng = ab.SgprEngine(model, species=Zs)
    # (1) sizing step then warm steps: identical results
    E0, F0, W0, _ = eng.predict(pos, numbers, cell, True)
    for _ in range(3):
        E1, F1, W1, _ = eng.predict(pos, numbers, cell, True)
        assert E1 == E0 and np.array_equal(W1, W0) and np.abs(F1 - F0).max() < 1e-11
    assert E0 == E_ref
    # (4) another species assignment of the same atoms, still warm
    numbers2 = numbers.copy()
    numbers2[::3] = np.where(numbers2[::3] == 3, 8, 3)
    E2, F2, W2, _ = eng.predict(pos, numbers2, cell, True)
    E2r, F2r, W2r, _ = ref_eng.predict(pos, numbers2, cell, True)
    assert abs(E2 - E2r) / N < 1e-13 and np.abs(F2 - F2r).max() < 1e-11
    eng.close()
    # (2) capacity sized on an expanded (sparse) structure, then the dense one: transparent repeat
    eng = ab.SgprEngine(model, species=Zs)
    Es, Fs, Ws, _ = eng.predict(pos * 1.5, numbers, cell * 1.5, True)
    assert eng.stats()["n_pairs"] * 2 < n_pairs_dense
    Ed, Fd, Wd, _ = eng.predict(pos, numbers, cell, True)
    assert Ed == E_ref and np.abs(Fd - F_ref).max() < 1e-11 and np.array_equal(Wd, W_ref)
    assert eng.stats()["n_pairs"] == n_pairs_dense
    Ed2, Fd2, _, _ = eng.predict(pos, numbers, cell, True)     # warm again, now with enough room
    assert Ed2 == E_ref
    eng.close()
    # (3) asynchronous device-pointer API
    eng = ab.SgprEngine(model, species=Zs)
    eng.set_async(True)
    dev = torch.device("cuda", 0)
    z_t = torch.as_tensor(numbers.astype(np.int32), device=dev)
    p_sparse, p_dense = torch.as_tensor(pos * 1.5, device=dev), torch.as_tensor(pos, device=dev)
    eng.predict_device(p_sparse, z_t, cell * 1.5, True)      # sizing step
    torch.cuda.synchronize()
    eng.check()
    E, F, W = eng.predict_device(p_dense, z_t, cell, True)   # warm: overflows
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="exceed the capacity"):
        eng.check()
    E, F, W = eng.predict_device(p_dense, z_t, cell, True)   # sizes again
    torch.cuda.synchronize()
    assert eng.check() == n_pairs_dense
    assert float(E.item()) == E_ref and np.abs(F.cpu().numpy() - F_ref).max() < 1e-11
    E, F, W = eng.predict_device(p_dense, z_t, cell, True)   # warm and valid
    torch.cuda.synchronize()
    assert eng.check() == n_pairs_dense and float(E.item()) == E_ref
    # an unknown species in a warm step is reported, not silently evaluated
    z_bad = z_t.clone()
    z_bad[5] = 47
    eng.predict_device(p_dense, z_bad, cell, True)
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="species table"):
        eng.check()
    eng.close()
    ref_eng.close()


@pytest.mark.parametrize("world,mode", [(2, None), (4, None), (2, "bins"), (4, "bins")], ids=["2", "4", "2-bins", "4-bins"])
def test_fused_exchange_step_emulated_on_one_gpu(world, mode, monkeypatch):
    """sgpr_p2p_step (no NCCL: mailboxes + stamped flags) with ``world`` ranks emulated on ONE GPU: one handle and one
    stream per rank, the ranks' symmetric blocks are plain device buffers.  Several steps (sizing, warm, CUDA-graph
    replay, both buffer parities, moving atoms) must reproduce the unsharded result on every rank, and the oracle's.
    The cell has 27 bins, so the ranks run the warp-per-atom neighbour kernel unless "bins" forces the block-per-bin one
    (the unsharded reference then keeps the warp kernel)."""
    import torch

    import autoforce_b200 as ab
    from autoforce_b200 import synth
    from oracle_engine import to_oracle

    Zs = [3, 8]
    model = synth.synth_model(Zs, 40, 5, lmax=3, nmax=3, rc=6.0)
    om = to_oracle(model)
    pos0, cell, numbers = synth.fcc(6, Zs, 0.1, 1)
    N = len(numbers)
    dev = torch.device("cuda", 0)
    ref = ab.SgprEngine(model, species=Zs)
    if mode:
        monkeypatch.setenv("SGPR_NL", mode)
    engines = [ab.SgprEngine(model, species=Zs) for _ in range(world)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    stride = 3 * N + 8
    blocks = torch.zeros((world, 2 * stride + 2 * world * 16), dtype=torch.float64, device=dev)
    bases = np.array([blocks[r].data_ptr() for r in range(world)], dtype=np.uint64)
    ews = [torch.zeros(10, dtype=torch.float64, device=dev) for _ in range(world)]
    Fs = [torch.zeros((N, 3), dtype=torch.float64, device=dev) for _ in range(world)]
    owns = [torch.zeros(N, dtype=torch.uint8, device=dev) for _ in range(world)]
    z_t = torch.as_tensor(numbers.astype(np.int32), device=dev)
    torch.cuda.synchronize()
    rng = np.random.default_rng(5)
    try:
        for e in engines:
            e.set_async(True)
        for step in range(6):
            pos = pos0 + rng.normal(0, 0.02, pos0.shape) if step % 2 else pos0   # steps 0, 2, 4 repeat: graph replay
            pos_t = torch.as_tensor(pos, device=dev)
            torch.cuda.synchronize()
            for r in range(world):
                with torch.cuda.stream(streams[r]):
                    engines[r].p2p_step(pos_t, z_t, cell, True, r, world, bases, ews[r], Fs[r], owns[r])
            torch.cuda.synchronize()
            for e in engines:
                e.check()
            E0, F0, W0, _ = ref.predict(pos, numbers, cell, True)
            F = torch.zeros((N, 3), dtype=torch.float64, device=dev)
            covered = torch.zeros(N, dtype=torch.int32, device=dev)
            for r in range(world):
                ew = ews[r].cpu().numpy()
                assert abs(ew[0] - E0) / N < 1e-12, (step, r)
                assert np.abs(ew[1:].reshape(3, 3) - W0).max() < 1e-9
                assert np.array_equal(ew, ews[0].cpu().numpy()), "the reduction is bit-identical on every rank"
                F += Fs[r] * owns[r].to(torch.float64)[:, None]
                covered += owns[r].to(torch.int32)
            assert bool((covered == 1).all())
            assert np.abs(F.cpu().numpy() - F0).max() < 1e-10, step
            out = o.predict(om, pos, cell, True, numbers)
            assert abs(ew[0] - out["energy"]) / N < TOL_E_PER_ATOM, step
            assert np.abs(F.cpu().numpy() - out["forces"]).max() < TOL_F, step
            assert np.abs(ew[1:].reshape(3, 3) - out["virial"]).max() < 1e-8, step
    finally:
        for e in engines + [ref]:
            e.close()


def test_more_than_eight_species_is_refused_loudly():
    """The dense species table holds at most SGPR_MAX_SPECIES = 8 species (the reference's sparse [120,120] layout has no
    such limit): a ninth species must be an error at construction, never a silent truncation."""
    import autoforce_b200 as ab

    g = load_golden("lipso108")
    with pytest.raises(ValueError, match="at most 8 species"):
        ab.SgprEngine(model_from_golden(g), species=[1, 3, 6, 7, 8, 9, 15, 16, 17])
    # ... and an atom of a species the handle does not know is an error of the call, not a wrong number
    eng = ab.SgprEngine(model_from_golden(g), species=g["meta"]["species"])
    Z = np.asarray(g["numbers"]).copy()
    Z[0] = 79
    with pytest.raises(RuntimeError, match="species table"):
        eng.predict(g["pos"], Z, g["cell"], g["meta"]["pbc"])
    E, F, W, _ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])     # the handle stays usable
    assert abs(E - float(g["energy"])) / len(Z) < TOL_E_PER_ATOM
    # the same in a WARM step (the error flag is read with the results)
    with pytest.raises(RuntimeError, match="species table"):
        eng.predict(g["pos"], Z, g["cell"], g["meta"]["pbc"])
    E2, _, _, _ = eng.predict(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    assert E2 == E
    eng.close()
