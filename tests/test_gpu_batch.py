"""Batched prediction (sgpr_predict_batch / SgprEngine.predict_batch / B200Calculator.calculate_batch): many structures,
each with its own atom count, cell and pbc, in one call -- the same results as one call per structure."""
import ctypes
import types

import numpy as np
import pytest

from golden_util import b200_model, golden_cases, load_golden, oracle_model
from oracle import sgpr_oracle as o

pytestmark = pytest.mark.gpu

TOL_E_PER_ATOM = 1e-9   # against the reference / the oracle (test_gpu_parity.py)
TOL_F = 1e-8
TOL_S = 1e-9


def stress_of(W, cell):
    vol = abs(np.linalg.det(np.asarray(cell, dtype=float).reshape(3, 3))) or -2.0
    return (W / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]]


def run_batch(eng, structs, want_beta=False):
    first = np.concatenate([[0], np.cumsum([len(s[1]) for s in structs])])
    pos = np.concatenate([np.asarray(s[0], dtype=float).reshape(-1, 3) for s in structs])
    Z = np.concatenate([np.asarray(s[1]).reshape(-1) for s in structs]).astype(np.int32)
    return eng.predict_batch(pos, Z, first, [np.asarray(s[2], dtype=float).reshape(3, 3) for s in structs],
                             [np.broadcast_to(np.asarray(s[3]), (3,)) for s in structs], want_beta=want_beta)


def assert_same_as_single(eng, structs, out, rel=False):
    """Each structure of the batch against SgprEngine.predict of that structure alone."""
    E, F, W = out[:3]
    beta = out[3] if len(out) > 3 else None
    a0 = 0
    for b, (pos, Z, cell, pbc) in enumerate(structs):
        n = len(Z)
        if beta is not None:
            e1, f1, w1, _, b1 = eng.predict(pos, Z, cell, pbc, want_beta=True)
        else:
            e1, f1, w1, _ = eng.predict(pos, Z, cell, pbc)
        se = max(1.0, abs(e1) / max(n, 1)) if rel else 1.0
        sf = max(1.0, np.abs(f1).max() if n else 0.0) if rel else 1.0
        sw = max(1.0, np.abs(w1).max()) if rel else 1.0
        assert abs(E[b] - e1) / max(n, 1) <= 1e-12 * se, (b, E[b], e1)
        assert np.abs(F[a0:a0 + n] - f1).max(initial=0.0) <= 1e-12 * sf, b
        assert np.abs(W[b] - w1).max() <= 1e-11 * sw, b
        if beta is not None:
            bb = beta[a0:a0 + n]
            assert np.array_equal(np.isnan(bb), np.isnan(b1)) and np.array_equal(np.isposinf(bb), np.isposinf(b1)), b
            fin = np.isfinite(b1)
            assert np.abs(bb[fin] - b1[fin]).max(initial=0.0) <= 1e-12, b
        a0 += n


def golden_batch(g):
    """The golden structure, a rattled copy, a 2x1x1 supercell (periodic x), a permuted copy and an empty structure."""
    pos, Z = np.asarray(g["pos"], dtype=float), np.asarray(g["numbers"]).astype(np.int32)
    cell, pbc = np.asarray(g["cell"], dtype=float).reshape(3, 3), tuple(bool(p) for p in g["meta"]["pbc"])
    rng = np.random.default_rng(7)
    perm = rng.permutation(len(Z))
    structs = [(pos, Z, cell, pbc), (pos + rng.normal(0, 0.05, pos.shape), Z, cell, pbc),
               (pos[perm], Z[perm], cell, pbc), (np.zeros((0, 3)), np.zeros(0, dtype=np.int32), cell, pbc)]
    if pbc[0]:
        sup = np.concatenate([pos, pos + cell[0]])
        structs.append((sup, np.concatenate([Z, Z]), cell * np.array([[2.0], [1.0], [1.0]]), pbc))
    return structs


@pytest.fixture(params=golden_cases())
def case(request):
    import autoforce_b200 as ab

    g = load_golden(request.param)
    if g["meta"]["kernel"]["kind"] == "multi":
        pytest.skip("kernel sums: test_calculator_batch_kernel_sum")
    eng = ab.SgprEngine(b200_model(g), species=g["meta"]["species"])
    yield g, eng
    eng.close()


def test_golden_cases_batched(case):
    g, eng = case
    structs = golden_batch(g)
    N = len(g["numbers"])
    want_beta = eng.model.choli is not None
    out = run_batch(eng, structs, want_beta=want_beta)
    E, F, W = out[:3]
    assert_same_as_single(eng, structs, out)
    # the golden structure against the unmodified reference
    assert abs(E[0] - float(g["energy"])) / N < TOL_E_PER_ATOM
    assert np.abs(F[:N] - g["forces"]).max() < TOL_F
    assert np.abs(stress_of(W[0], g["cell"]) - g["stress"]).max() < TOL_S
    assert E[3] == 0.0 and not W[3].any()
    if len(structs) == 5:   # the supercell repeats the primitive result
        o0 = 3 * N
        assert abs(E[4] - 2 * E[0]) / (2 * N) < 1e-12
        assert np.abs(F[o0:o0 + N] - F[:N]).max() < 1e-12 and np.abs(F[o0 + N:o0 + 2 * N] - F[:N]).max() < 1e-12
        assert np.abs(W[4] - 2 * W[0]).max() < 1e-10
    # amplified weights (relative bars); unnorm_2sp runs on the FP64 DMMA path
    eng.set_weights(mu=g["mu_big"])
    out = run_batch(eng, structs)
    assert_same_as_single(eng, structs, out, rel=True)
    E, F, W = out
    assert abs(E[0] - float(g["energy_big"])) / N < 1e-9 * max(1.0, abs(float(g["energy_big"])) / N)
    assert np.abs(F[:N] - g["forces_big"]).max() < 1e-10 * max(1.0, np.abs(g["forces_big"]).max())


# ---------------------------------------------------------------------------------- one 4-species model
@pytest.fixture(scope="module")
def model4():
    from autoforce_b200.synth import synth_model

    return synth_model([3, 8, 15, 16], 240, seed=11, with_choli="tril")


@pytest.fixture
def eng4(model4):
    import autoforce_b200 as ab

    eng = ab.SgprEngine(model4, species=[3, 8, 15, 16])
    yield eng
    eng.close()


def mixed_structures(seed=3):
    from autoforce_b200.synth import fcc

    rng = np.random.default_rng(seed)
    Zs = [3, 8, 15, 16]
    out = []
    pos, cell, Z = fcc(2, Zs, 0.1, seed)                                    # cubic
    out.append((pos, Z, cell, (True, True, True)))
    tri = np.array([[7.2, 0.0, 0.0], [2.1, 6.9, 0.0], [1.3, 1.7, 7.4]])     # triclinic
    f = rng.random((40, 3))
    out.append((f @ tri, rng.choice(Zs, 40).astype(np.int32), tri, (True, True, True)))
    pos, cell, Z = fcc((3, 3, 2), Zs, 0.1, seed + 1)                        # slab
    out.append((pos, Z, cell, (True, True, False)))
    pos, _, Z = fcc(2, Zs, 0.1, seed + 2)                                   # cluster with a neighbour-less atom
    pos = np.concatenate([pos, [[40.0, 40.0, 40.0]]])
    out.append((pos, np.concatenate([Z, [8]]).astype(np.int32), np.zeros((3, 3)), (False, False, False)))
    pos, cell, Z = fcc(1, Zs, 0.1, seed + 3)                                # cell < 2 rc: many images of a neighbour
    out.append((pos, Z, cell, (True, True, True)))
    pos, cell, Z = fcc(2, Zs, 0.1, seed + 4)                                # atoms far outside their cell
    pos = pos + rng.integers(-5, 6, (len(pos), 3)) @ cell
    out.append((pos, Z, cell, (True, True, True)))
    out.append((np.array([[0.3, 0.2, 0.1]]), np.array([15], dtype=np.int32), np.eye(3) * 4.0, (True, True, True)))   # one atom
    pos, cell, _ = fcc(2, Zs, 0.1, seed + 5)                                # missing species
    out.append((pos, rng.choice([3, 16], len(pos)).astype(np.int32), cell, (True, True, True)))
    return out


def test_mixed_geometries_one_model(eng4, model4):
    from oracle_engine import to_oracle

    structs = mixed_structures()
    out = run_batch(eng4, structs, want_beta=True)
    assert_same_as_single(eng4, structs, out)
    E, F, W, beta = out
    om = to_oracle(model4)
    a0 = 0
    for b, (pos, Z, cell, pbc) in enumerate(structs):
        n = len(Z)
        ref = o.predict(om, pos, cell, pbc, Z, want_beta=True)
        assert abs(E[b] - ref["energy"]) / n < TOL_E_PER_ATOM, b
        assert np.abs(F[a0:a0 + n] - ref["forces"]).max() < TOL_F, b
        assert np.abs(W[b] - ref["virial"]).max() < 1e-8, b
        assert np.allclose(beta[a0:a0 + n], ref["beta"], rtol=0, atol=1e-10, equal_nan=True), b
        a0 += n


def test_results_do_not_depend_on_the_rest_of_the_batch(eng4):
    structs = mixed_structures()
    fixed = structs[1]
    n = len(fixed[1])
    ref = None
    for others in ([], structs[:1], structs[2:], structs[::-1][:5], structs * 2):
        batch = others[: len(others) // 2] + [fixed] + others[len(others) // 2:]
        k = len(others) // 2
        E, F, W, beta = run_batch(eng4, batch, want_beta=True)
        a0 = sum(len(s[1]) for s in batch[:k])
        got = (E[k], F[a0:a0 + n], W[k], beta[a0:a0 + n])
        if ref is None:
            ref = got
            continue
        assert got[0] == ref[0]
        assert np.array_equal(got[2], ref[2])
        assert np.array_equal(got[3], ref[3], equal_nan=True)
        assert np.abs(got[1] - ref[1]).max() <= 1e-13


# ---------------------------------------------------------------------------------- calculator
def as_atoms(s):
    return types.SimpleNamespace(positions=s[0], numbers=s[1], cell=s[2], pbc=s[3])


def assert_results_match(rs, ref, n):
    assert set(rs) >= set(ref)
    for k in ref:
        a, b = np.asarray(rs[k]), np.asarray(ref[k])
        assert a.shape == b.shape and a.dtype == b.dtype, k
    assert abs(float(rs["energy"]) - float(ref["energy"])) / max(n, 1) <= 1e-12
    assert np.abs(rs["forces"] - ref["forces"]).max(initial=0.0) <= 1e-12
    assert np.abs(rs["stress"] - ref["stress"]).max() <= 1e-11


def test_calculator_batch(model4):
    import autoforce_b200 as ab

    structs = mixed_structures()
    images = [as_atoms(s) for s in structs]
    seen_b, seen_1 = [], []
    calc_b = ab.B200Calculator(model4, covloss=True, ediff=0.0, on_uncertain=lambda a, b: seen_b.append((a, b.copy())))
    calc_1 = ab.B200Calculator(model4, covloss=True, ediff=0.0, on_uncertain=lambda a, b: seen_1.append((a, b.copy())))
    res = calc_b.calculate_batch(images)
    assert len(res) == len(images)
    for a, r in zip(images, res):
        ref = dict(calc_1.calculate(a))
        assert_results_match(r, ref, len(a.numbers))
        assert r["covlog"] == calc_1.covlog or abs(float(r["covlog"]) - float(calc_1.covlog)) <= 1e-12
        assert np.allclose(r["beta"], calc_1.beta, rtol=0, atol=1e-12, equal_nan=True)
    assert [a for a, _ in seen_b] == [a for a, _ in seen_1] == images
    assert calc_b.calculate_batch([]) == []
    # no cell: V = -2 (calculator/active.py:606-609)
    cl = res[3]
    assert np.array_equal(cl["stress"], (calc_b._engine.predict_batch([images[3]])[2][0] / -2.0).reshape(-1)[[0, 4, 8, 5, 2, 1]])


def test_calculator_batch_kernel_sum():
    import autoforce_b200 as ab

    g = load_golden("two_kernels")
    models = b200_model(g)
    lead = max(range(2), key=lambda i: models[i].rc)
    for i, m in enumerate(models):      # what SgprModel.list_from_posterior_potential sets up
        m.lone_weight = 2.0 if i == lead else -1.0
        if i != lead:
            m.mean_w = {}
    s0 = (np.asarray(g["pos"]), np.asarray(g["numbers"]), np.asarray(g["cell"]), g["meta"]["pbc"])
    rng = np.random.default_rng(5)
    images = [as_atoms(s0), as_atoms((s0[0] + rng.normal(0, 0.05, s0[0].shape),) + s0[1:])]
    calc = ab.B200Calculator(models)
    res = calc.calculate_batch(images)
    N = len(g["numbers"])
    assert abs(float(res[0]["energy"]) - float(g["energy"])) / N < TOL_E_PER_ATOM
    assert np.abs(res[0]["forces"] - g["forces"]).max() < TOL_F
    assert np.abs(res[0]["stress"] - g["stress"]).max() < TOL_S
    for a, r in zip(images, res):
        assert_results_match(r, dict(ab.B200Calculator(models).calculate(a)), N)


# ---------------------------------------------------------------------------------- handle interplay
def device_steps(eng, s, n):
    import torch

    pos_t = torch.as_tensor(np.asarray(s[0], dtype=float), device="cuda")
    z_t = torch.as_tensor(np.asarray(s[1]).astype(np.int32), device="cuda")
    out = None
    for _ in range(n):
        out = eng.predict_device(pos_t, z_t, s[2], s[3])
    torch.cuda.synchronize()
    eng.check()
    return float(out[0].cpu()[0]), out[1].cpu().numpy().copy(), out[2].cpu().numpy().copy()


def assert_step_equal(a, b):
    assert a[0] == b[0]
    assert np.array_equal(a[2], b[2])
    assert np.abs(a[1] - b[1]).max() <= 1e-13


def test_warm_steps_around_a_growing_batch(model4):
    import autoforce_b200 as ab

    from autoforce_b200.synth import fcc

    pos, cell, Z = fcc(3, [3, 8, 15, 16], 0.1, 21)
    A = (pos, Z, cell, (True, True, True))
    fresh = ab.SgprEngine(model4, species=[3, 8, 15, 16])
    ref = device_steps(fresh, A, 3)
    fresh.close()
    eng = ab.SgprEngine(model4, species=[3, 8, 15, 16])
    eng.set_async(True)
    assert_step_equal(device_steps(eng, A, 4), ref)          # sizing, capture, replays
    big = mixed_structures() * 40                            # grows every per-step workspace
    run_batch(eng, big, want_beta=True)
    assert_step_equal(device_steps(eng, A, 1), ref)          # sizing step after the batch
    assert_step_equal(device_steps(eng, A, 3), ref)          # warm again: new graph on the new workspaces
    eng.close()


def test_warm_steps_after_a_larger_structure(model4):
    """A, A (graph captured), a larger B (workspaces reallocated), A, A: the last steps must not replay the graph
    that points at the freed workspaces."""
    import autoforce_b200 as ab

    from autoforce_b200.synth import fcc

    pos, cell, Z = fcc(3, [3, 8, 15, 16], 0.1, 22)
    A = (pos, Z, cell, (True, True, True))
    pos, cell, Z = fcc(6, [3, 8, 15, 16], 0.1, 23)
    Bs = (pos, Z, cell, (True, True, True))
    fresh = ab.SgprEngine(model4, species=[3, 8, 15, 16])
    ref_a, ref_b = device_steps(fresh, A, 3), None
    fresh.close()
    fresh = ab.SgprEngine(model4, species=[3, 8, 15, 16])
    ref_b = device_steps(fresh, Bs, 1)
    fresh.close()
    eng = ab.SgprEngine(model4, species=[3, 8, 15, 16])
    eng.set_async(True)
    assert_step_equal(device_steps(eng, A, 2), ref_a)
    assert_step_equal(device_steps(eng, Bs, 1), ref_b)
    assert_step_equal(device_steps(eng, A, 1), ref_a)
    assert_step_equal(device_steps(eng, A, 2), ref_a)
    eng.close()


# ---------------------------------------------------------------------------------- errors
def test_errors_name_the_structure_and_leave_the_handle_usable(eng4):
    structs = mixed_structures()
    good = run_batch(eng4, structs)
    bad = list(structs)
    bad[2] = (bad[2][0], np.where(np.arange(len(bad[2][1])) == 5, 99, bad[2][1]).astype(np.int32), bad[2][2], bad[2][3])
    with pytest.raises(RuntimeError, match=r"error -3: structure 2: atomic number 99"):
        run_batch(eng4, bad)
    bad = list(structs)
    bad[4] = (bad[4][0], bad[4][1], np.array([[3.0, 0, 0], [3.0, 0, 0], [0, 0, 3.0]]), bad[4][3])
    with pytest.raises(RuntimeError, match=r"error -4: structure 4: singular cell"):
        run_batch(eng4, bad)
    bad = list(structs)
    bad[6] = (bad[6][0] + 1000.0, bad[6][1], bad[6][2], bad[6][3])
    with pytest.raises(RuntimeError, match=r"error -4: structure 6: an atom lies more than 120 cells"):
        run_batch(eng4, bad)
    lib, h = eng4.lib, eng4._h
    import torch

    pos = torch.tensor([[0.0, 0, 0], [1.5, 0, 0], [0, 0, 0], [0, 1.5, 0]], dtype=torch.float64, device="cuda")
    Z = torch.full((4,), 3, dtype=torch.int32, device="cuda")
    E = torch.zeros(2, dtype=torch.float64, device="cuda")
    F = torch.zeros((4, 3), dtype=torch.float64, device="cuda")
    W = torch.zeros((2, 9), dtype=torch.float64, device="cuda")
    cells = np.tile(np.eye(3).reshape(9) * 8.0, 2)
    pbcs = np.ones(6, dtype=np.int32)
    p = ctypes.c_void_p

    def call(first, E_=E, F_=F, B=2):
        first = np.asarray(first, dtype=np.int64)
        return lib.sgpr_predict_batch(h, B, p(first.ctypes.data), p(pos.data_ptr()), p(Z.data_ptr()), p(cells.ctypes.data),
                                      p(pbcs.ctypes.data), None, p(E_.data_ptr()) if E_ is not None else None,
                                      p(F_.data_ptr()) if F_ is not None else None, p(W.data_ptr()), None)

    assert call([1, 2, 4]) == -1 and b"first_h[0]" in lib.sgpr_last_error()
    assert call([0, 3, 2]) == -1 and b"structure 1" in lib.sgpr_last_error()
    assert call([0, 2, 4], E_=None) == -1
    assert call([0, 2, 4], F_=None) == -1
    assert call([0], B=0) == 0
    assert call([0, 2, 4]) == 0
    torch.cuda.synchronize()
    again = run_batch(eng4, structs)
    for x, y in zip(good, again):
        assert np.array_equal(x, y) or np.abs(x - y).max() <= 1e-13
    E0, F0, W0 = eng4.predict_batch([])
    assert E0.shape == (0,) and F0.shape == (0, 3) and W0.shape == (0, 3, 3)
