"""GPU: BASELINE.json's full-size configurations.

C2 (4,000-atom Cu, M=500) is compared with the oracle atom by atom.  C3 (97,556 atoms,
4 species, M=2000) is checked through size-independent properties: permutation and
translation invariance, Newton's third law, forces as finite differences of the energy,
the virial as the strain derivative of the energy, run-to-run reproducibility, and the
kernel-matrix rows / local environments of a random sample of atoms against the oracle.
"""
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from oracle import sgpr_oracle as o

pytestmark = pytest.mark.gpu


def to_oracle(model):
    first = model.ind_first
    return o.OracleModel(
        lmax=model.lmax, nmax=model.nmax, xi=model.xi, rc=model.rc, radii=model.radii, default_radius=model.default_radius,
        ind_Z=model.ind_Z.astype(np.int64), ind_r=[model.ind_r[first[m]:first[m + 1]] for m in range(model.M)],
        ind_b=[model.ind_b[first[m]:first[m + 1]].astype(np.int64) for m in range(model.M)], mu=model.mu,
        mean_w=model.mean_w, choli=model.choli, vscale=model.vscale, a_not=model.a_not)


def test_c2_matches_oracle_full_size():
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    w = synth.WORKLOADS["c2"]
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"])
    pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
    eng = ab.SgprEngine(model, species=w["Zs"])
    E, F, W, _ = eng.predict(pos, numbers, cell, True)
    first, J, S = eng.neighbors(pos, numbers, cell, True)
    eng.close()
    ref = o.predict(to_oracle(model), pos, cell, True, numbers)
    N = len(pos)
    assert len(J) == len(ref["j"])
    I = np.repeat(np.arange(N), np.diff(first))
    order = np.lexsort((S[:, 2], S[:, 1], S[:, 0], J, I))
    assert np.array_equal(J[order], ref["j"]) and np.array_equal(S[order].astype(np.int64), ref["S"])
    assert abs(E - ref["energy"]) / N < 1e-9
    assert np.abs(F - ref["forces"]).max() < 1e-8
    vol = abs(np.linalg.det(cell))
    assert np.abs(W - ref["virial"]).max() / vol < 1e-9


@pytest.fixture(scope="module")
def c3():
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    w = synth.WORKLOADS["c3"]
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"])
    pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
    eng = ab.SgprEngine(model, species=w["Zs"])
    yield model, pos, cell, numbers, eng
    eng.close()


def test_c3_invariances_and_reproducibility(c3):
    model, pos, cell, numbers, eng = c3
    N = len(pos)
    E0, F0, W0, _ = eng.predict(pos, numbers, cell, True)
    E1, F1, W1, _ = eng.predict(pos, numbers, cell, True)
    assert E1 == E0 and np.array_equal(W1, W0)            # fixed-order reductions
    assert np.abs(F1 - F0).max() < 1e-11                  # forces: atomic accumulation order only
    assert np.abs(F0.sum(axis=0)).max() < 1e-8            # Newton's third law
    # permutation of the atom order
    perm = np.random.default_rng(0).permutation(N)
    E2, F2, W2, _ = eng.predict(pos[perm], numbers[perm], cell, True)
    assert abs(E2 - E0) / N < 1e-12
    assert np.abs(F2 - F0[perm]).max() < 1e-10
    assert np.abs(W2 - W0).max() < 1e-7
    # rigid translation + lattice-vector shifts of some atoms (positions outside the cell)
    shift = np.array([1.2345, -0.777, 3.21])
    pos3 = pos + shift
    pos3[::7] += cell[0] * 2 - cell[2]
    E3, F3, W3, _ = eng.predict(pos3, numbers, cell, True)
    assert abs(E3 - E0) / N < 1e-12
    assert np.abs(F3 - F0).max() < 1e-9


def test_c3_forces_and_virial_are_energy_derivatives(c3):
    model, pos, cell, numbers, eng = c3
    E0, F0, W0, _ = eng.predict(pos, numbers, cell, True)
    rng = np.random.default_rng(1)
    d = 1e-4
    for i in rng.choice(len(pos), 3, replace=False):
        for k in range(3):
            p = pos.copy()
            p[i, k] += d
            Ep = eng.predict(p, numbers, cell, True)[0]
            p[i, k] -= 2 * d
            Em = eng.predict(p, numbers, cell, True)[0]
            assert abs(-(Ep - Em) / (2 * d) - F0[i, k]) < 1e-5
    # dE/d(strain) = W  (stress = W/V, calculator/active.py:604-611)
    eps = 1e-6
    for (a, b) in [(0, 0), (1, 2)]:
        strain = np.eye(3)
        strain[a, b] += eps
        Ep = eng.predict(pos @ strain, numbers, cell @ strain, True)[0]
        strain[a, b] -= 2 * eps
        Em = eng.predict(pos @ strain, numbers, cell @ strain, True)[0]
        assert abs((Ep - Em) / (2 * eps) - W0[a, b]) < 1e-4 * max(1.0, abs(W0[a, b]))


def test_c3_sampled_rows_match_oracle(c3):
    """Kernel-matrix rows of a random sample of atoms vs the oracle evaluated on the
    environments the GPU neighbour list produced (exact displacements recomputed on
    the host from j and S)."""
    import torch

    model, pos, cell, numbers, eng = c3
    om = to_oracle(model)
    species = np.array(sorted(set(int(z) for z in numbers)))
    first, J, S = eng.neighbors(pos, numbers, cell, True)
    K = eng.kernel_matrix(pos, numbers, cell, True)
    sample = np.random.default_rng(2).choice(len(pos), 64, replace=False)
    Ks = K[torch.as_tensor(sample, device=K.device)].cpu().numpy()
    del K
    envs_r, envs_b = [], []
    for i in sample:
        sl = slice(first[i], first[i + 1])
        # brute-force check of this atom's neighbour set against all atoms, minimum image
        dv = pos - pos[i]
        dv -= np.round(dv / np.diag(cell)) * np.diag(cell)
        dist = np.sqrt((dv * dv).sum(axis=1))
        expect = np.nonzero((dist < model.rc) & (np.arange(len(pos)) != i))[0]
        assert np.array_equal(np.sort(J[sl]), expect)
        envs_r.append(o.displacements(pos, cell, i, J[sl].astype(np.int64), S[sl].astype(np.int64)))
        envs_b.append(numbers[J[sl]].astype(np.int64))
    R, Zb, mask = o.pad_environments(envs_r, envs_b)
    P = o.descriptor_batch(om, species, R, Zb, mask)
    Zh, lone_m = o.inducing_descriptors(om, species)
    Ko, _, _ = o.kernel_from_descriptors(om, P, numbers[sample].astype(np.int64), ~mask.any(axis=1), Zh, lone_m)
    assert np.abs(Ks - Ko).max() < 1e-12


def test_c3_sharded_over_8_ranks_matches_unsharded(c3):
    model, pos, cell, numbers, eng = c3
    E0, F0, W0, _ = eng.predict(pos, numbers, cell, True)
    E, F, W = 0.0, np.zeros_like(F0), np.zeros_like(W0)
    n_active = []
    for rank in range(8):
        e, f, w, owned = eng.predict(pos, numbers, cell, True, rank=rank, world=8)
        assert abs(int(owned.sum()) - len(pos) / 8) <= 1
        n_active.append(eng.stats()["n_active"])
        E, F, W = E + e, F + f, W + w
    assert abs(E - E0) / len(pos) < 1e-12
    assert np.abs(F - F0).max() < 1e-10
    assert np.abs(W - W0).max() < 1e-7
    # halo = one cutoff on each side of an x-slab: redundant work stays bounded
    assert max(n_active) < 2.6 * len(pos) / 8


# ------------------------------------------------------------------------------------------------------------------
# VERDICT r1 items 2c / 2d: c4 and c5 at full size; c3 with 1000x larger weights, tcgen05 int8 slices vs FP64 DMMA
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", params=["c4", "c5"])
def big(request):
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    w = synth.WORKLOADS[request.param]
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"])
    pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
    eng = ab.SgprEngine(model, species=w["Zs"])
    yield request.param, model, pos, cell, numbers, eng
    eng.close()


def test_c4_c5_full_size_against_oracle_and_derivatives(big):
    """BASELINE.json configs 4 (lmax 6 / nmax 8 / rc 7, 19,652 atoms) and 5 (1,000,188 atoms, M = 4000) at full size:
    neighbour rows and complete forces of probe atoms against the oracle, kernel rows of sampled environments,
    Newton's third law, forces = -dE/dx and virial = dE/d(strain) by finite differences, run-to-run reproducibility."""
    import sys

    sys.path.insert(0, ROOT)
    from bench import parity_full_size

    name, model, pos, cell, numbers, eng = big
    N = len(pos)
    E0, F0, W0, _ = eng.predict(pos, numbers, cell, True)
    E1, F1, W1, _ = eng.predict(pos, numbers, cell, True)
    assert E1 == E0 and np.array_equal(W1, W0) and np.abs(F1 - F0).max() < 1e-10
    assert np.abs(F0.sum(axis=0)).max() < 1e-7
    par = parity_full_size(eng, model, pos, cell, numbers, F0, n_probe=2)
    assert par["neighbour_rows_identical"] and par["max_abs_dF"] < 1e-8, par
    # kernel rows of sampled environments (sgpr_kernel_envs) vs the oracle on the same displacements
    om = to_oracle(model)
    species = np.array(sorted(set(int(z) for z in numbers)))
    first, J, S = eng.neighbors(pos, numbers, cell, True)
    sample = np.random.default_rng(3).choice(N, 24, replace=False)
    envs = [(int(numbers[i]), o.displacements(pos, cell, int(i), J[first[i]:first[i + 1]].astype(np.int64),
                                              S[first[i]:first[i + 1]].astype(np.int64)),
             numbers[J[first[i]:first[i + 1]]].astype(np.int64)) for i in sample]
    Ks = eng.kernel_envs(envs).cpu().numpy()
    R, Zb, mask = o.pad_environments([e[1] for e in envs], [e[2] for e in envs])
    P = o.descriptor_batch(om, species, R, Zb, mask)
    Zh, lone_m = o.inducing_descriptors(om, species)
    Ko, _, _ = o.kernel_from_descriptors(om, P, numbers[sample].astype(np.int64), ~mask.any(axis=1), Zh, lone_m)
    assert np.abs(Ks - Ko).max() < 1e-12
    # finite differences
    d = 1e-4
    for i in np.random.default_rng(4).choice(N, 2, replace=False):
        for k in (0, 2):
            p = pos.copy()
            p[i, k] += d
            Ep = eng.predict(p, numbers, cell, True)[0]
            p[i, k] -= 2 * d
            Em = eng.predict(p, numbers, cell, True)[0]
            assert abs(-(Ep - Em) / (2 * d) - F0[i, k]) < 2e-5
    eps = 1e-6
    strain = np.eye(3)
    strain[0, 0] += eps
    Ep = eng.predict(pos @ strain, numbers, cell @ strain, True)[0]
    strain[0, 0] -= 2 * eps
    Em = eng.predict(pos @ strain, numbers, cell @ strain, True)[0]
    assert abs((Ep - Em) / (2 * eps) - W0[0, 0]) < 2e-4 * max(1.0, abs(W0[0, 0]))


def test_c3_large_weights_int8_slices_vs_fp64_dmma(c3, monkeypatch):
    """SURVEY 8d stress variant: mu ~ N(0,1) * 100 (1000x the default).  The tcgen05 path (46-bit fixed-point operands,
    21 of 36 slice products) against the plain FP64 DMMA GEMMs (SGPR_GEMM=dmma) at c3 size."""
    import autoforce_b200 as ab
    from autoforce_b200 import synth

    _, pos, cell, numbers, _ = c3
    w = synth.WORKLOADS["c3"]
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"], mu_scale=100.0)
    N = len(pos)
    eng_i8 = ab.SgprEngine(model, species=w["Zs"])
    Ei, Fi, Wi, _ = eng_i8.predict(pos, numbers, cell, True)
    assert eng_i8.stats()["i8_ops"] > 0
    eng_i8.close()
    monkeypatch.setenv("SGPR_GEMM", "dmma")
    eng_d = ab.SgprEngine(model, species=w["Zs"])
    Ed, Fd, Wd, _ = eng_d.predict(pos, numbers, cell, True)
    assert eng_d.stats()["i8_ops"] == 0
    eng_d.close()
    assert abs(Ei - Ed) / N < 1e-7, (Ei, Ed)
    assert np.abs(Fi - Fd).max() < 1e-6
    vol = abs(np.linalg.det(cell))
    assert np.abs(Wi - Wd).max() / vol < 1e-7


def test_bench_dumps_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs DIR: energy, forces and virial of the last timed step as float64 .npy files, equal to a
    prediction of the same seeded inputs through the host API.  Run from another directory: bench.py needs none."""
    import subprocess
    import sys

    import autoforce_b200 as ab
    from autoforce_b200 import synth

    sys.path.insert(0, ROOT)
    from bench import workload_inputs

    steps, variants = 3, 2
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c2", "--steps", str(steps), "--warmup", "1",
           "--variants", str(variants), "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {name: np.load(out / f"{name}.npy") for name in ("energy", "forces", "virial")}
    w, pos_variants, cell, numbers = workload_inputs("c2", variants)
    N = len(numbers)
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["energy"].shape == (1,) and got["forces"].shape == (N, 3) and got["virial"].shape == (3, 3)
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"])
    eng = ab.SgprEngine(model, species=w["Zs"])
    E, F, W, _ = eng.predict(pos_variants[(steps - 1) % variants], numbers, cell, True)
    eng.close()
    assert abs(got["energy"][0] - E) / N < 1e-12
    assert np.abs(got["forces"] - F).max() < 1e-10
    assert np.abs(got["virial"] - W).max() < 1e-9
