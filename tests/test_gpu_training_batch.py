"""Training-time kernels of many structures in one call (sgpr_kernel_jacobian_batch / SgprEngine.training_kernels):
Ke, Kf and Kv of every structure against every inducing LCE -- the same as kernel_jacobian on each structure alone."""
import ctypes
import types

import numpy as np
import pytest

from golden_util import b200_model, load_golden, load_train, oracle_model, train_cases
from oracle import sgpr_oracle as o

pytestmark = pytest.mark.gpu

TOL_F = 1e-8


def as_atoms(pos, Z, cell, pbc):
    return types.SimpleNamespace(positions=np.asarray(pos, dtype=float).reshape(-1, 3), numbers=np.asarray(Z).astype(np.int32),
                                 cell=np.asarray(cell, dtype=float).reshape(3, 3), pbc=np.broadcast_to(np.asarray(pbc), (3,)))


def golden_structs(g):
    """The golden structure, a rattled copy, a non-periodic cut-out, an empty structure and (periodic along x) a 2x1x1
    supercell."""
    pos, Z = np.asarray(g["pos"], dtype=float), np.asarray(g["numbers"]).astype(np.int32)
    cell, pbc = np.asarray(g["cell"], dtype=float).reshape(3, 3), tuple(bool(p) for p in g["meta"]["pbc"])
    rng = np.random.default_rng(5)
    near = np.linalg.norm(pos - pos[0], axis=1) < 0.6 * float(g["meta"]["kernel"].get("rc", 5.0))
    out = [as_atoms(pos, Z, cell, pbc), as_atoms(pos + rng.normal(0, 0.04, pos.shape), Z, cell, pbc),
           as_atoms(pos[near], Z[near], cell, (False, False, False)), as_atoms(np.zeros((0, 3)), np.zeros(0), cell, pbc)]
    if pbc[0]:
        out.append(as_atoms(np.concatenate([pos, pos + cell[0]]), np.concatenate([Z, Z]), cell * np.array([[2.0], [1.0], [1.0]]), pbc))
    return out


def single(eng, a):
    """kernel_jacobian of one structure: (Ke in atom order, Kf, Kv) as host arrays (zeros for an empty structure, which
    kernel_jacobian does not take)."""
    if len(a.numbers) == 0:
        M = eng.model.M
        return np.zeros(M), np.zeros((0, M)), np.zeros((6, M))
    K, Kf, Kv = eng.kernel_jacobian(a.positions, a.numbers, a.cell, a.pbc)
    K = K.cpu().numpy()
    return K.sum(axis=0), Kf.cpu().numpy(), Kv.cpu().numpy()


def rel(x, y):
    return np.abs(x - y).max(initial=0.0) / max(1.0, np.abs(y).max(initial=0.0))


def assert_slices_match_single(eng, structs, Ke, Kf, Kv):
    a0 = 0
    for b, a in enumerate(structs):
        n = len(a.numbers)
        ke1, kf1, kv1 = single(eng, a)
        # numpy's axis-0 sum adds the rows in order, like the library's per-structure reduction
        assert np.array_equal(Ke[b], ke1), b
        assert rel(Kf[3 * a0:3 * (a0 + n)], kf1) <= 1e-13, b
        assert rel(Kv[6 * b:6 * b + 6], kv1) <= 1e-13, b
        a0 += n


def engine_for(name):
    import autoforce_b200 as ab

    g = load_golden(name)
    return g, ab.SgprEngine(b200_model(g), species=g["meta"]["species"])


@pytest.mark.parametrize("name", train_cases())
def test_train_golden_as_batch_of_one(name):
    g, eng = engine_for(name)
    t = load_train(name)
    a = as_atoms(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    Ke, Kf, Kv = (x.cpu().numpy() for x in eng.training_kernels([a]))
    N, M = len(g["numbers"]), len(g["mu"])
    assert Ke.shape == (1, M) and Kf.shape == (3 * N, M) and Kv.shape == (6, M)
    assert np.abs(Ke[0] - t["Ke"]).max() < 1e-11
    assert np.abs(Kf - t["Kf_autograd"]).max() < 1e-9
    assert np.abs(Kv - t["Kv_autograd"]).max() < 1e-8
    assert np.abs(Kf @ g["mu"] - g["forces"].reshape(-1)).max() < TOL_F
    # B = 1 is kernel_jacobian
    ke1, kf1, kv1 = single(eng, a)
    assert np.array_equal(Ke[0], ke1) and rel(Kf, kf1) <= 1e-13 and rel(Kv, kv1) <= 1e-13
    eng.close()


# lone atoms and LCEs, triclinic and narrow cells with several images, excluded centres, xi = 2, the (6,8) descriptor,
# neighbour species left out, normalize=False
SPECIAL = ["cluster_lone", "tric_oh", "cu108_sesoap", "afixed_2sp", "anot_xi2", "highres_l6n8", "subse_3sp", "unnorm_2sp"]


@pytest.mark.parametrize("name", SPECIAL)
def test_batch_slices_match_single_structure(name):
    g, eng = engine_for(name)
    structs = golden_structs(g)
    Ke, Kf, Kv = (x.cpu().numpy() for x in eng.training_kernels(structs))
    M = len(g["mu"])
    Ntot = sum(len(a.numbers) for a in structs)
    assert Ke.shape == (len(structs), M) and Kf.shape == (3 * Ntot, M) and Kv.shape == (6 * len(structs), M)
    assert_slices_match_single(eng, structs, Ke, Kf, Kv)
    assert not Ke[3].any() and not Kv[18:24].any()
    # the float64 oracle (true derivative, not the reference's scatter_quirk) on the small members
    om = oracle_model(g)
    for b in (0, 2):
        a = structs[b]
        if len(a.numbers) == 0 or len(a.numbers) > 64:
            continue
        a0 = sum(len(s.numbers) for s in structs[:b])
        ke, kf, kv = o.kernel_jacobian(om, a.positions, a.cell, a.pbc, a.numbers)
        assert np.abs(Ke[b] - ke).max() < 1e-11 * max(1.0, np.abs(ke).max())
        assert np.abs(Kf[3 * a0:3 * (a0 + len(a.numbers))] - kf).max() < 1e-9
        assert np.abs(Kv[6 * b:6 * b + 6] - kv).max() < 1e-8
    eng.close()


def test_structure_is_independent_of_its_batch():
    g, eng = engine_for("tric_oh")
    s = golden_structs(g)
    n0, n1 = len(s[0].numbers), len(s[1].numbers)
    Ke_a, Kf_a, Kv_a = (x.cpu().numpy() for x in eng.training_kernels([s[1], s[2]]))
    Ke_b, Kf_b, Kv_b = (x.cpu().numpy() for x in eng.training_kernels([s[0], s[3], s[1]]))
    assert np.array_equal(Ke_a[0], Ke_b[2])
    assert rel(Kf_a[:3 * n1], Kf_b[3 * n0:3 * (n0 + n1)]) <= 1e-13
    assert rel(Kv_a[:6], Kv_b[12:18]) <= 1e-13
    eng.close()


def test_subranges_and_ke_only():
    g, eng = engine_for("cu108_sesoap")
    structs = golden_structs(g)
    M = len(g["mu"])
    Ke, Kf, Kv = (x.cpu().numpy() for x in eng.training_kernels(structs))
    for m0, m1 in [(1, 4), (0, 1), (M - 3, M), (5, 5)]:
        k2, f2, v2 = (x.cpu().numpy() for x in eng.training_kernels(structs, m0=m0, m1=m1))
        assert np.array_equal(k2, Ke[:, m0:m1])
        assert rel(f2, Kf[:, m0:m1]) <= 1e-13 and rel(v2, Kv[:, m0:m1]) <= 1e-13
    k3, f3, v3 = eng.training_kernels(structs, want_jacobian=False)
    assert f3 is None and v3 is None and np.array_equal(k3.cpu().numpy(), Ke)
    eng.close()


def test_invalid_arguments_and_unknown_species():
    import torch

    g, eng = engine_for("cu108_sesoap")
    lib, M = eng.lib, len(g["mu"])
    a = as_atoms(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    N = len(a.numbers)
    pos = torch.as_tensor(a.positions).cuda()
    Z = torch.as_tensor(a.numbers).cuda()
    cells = np.ascontiguousarray(np.stack([a.cell.reshape(9)] * 2))
    pbcs = np.ascontiguousarray(np.stack([a.pbc.astype(np.int32)] * 2))
    Ke = torch.zeros(2 * M, dtype=torch.float64, device="cuda")
    J = torch.zeros(M * N * 3, dtype=torch.float64, device="cuda")
    W = torch.zeros(2 * M * 9, dtype=torch.float64, device="cuda")
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None   # noqa: E731

    def call(first, m0=0, m1=M, J_=J, W_=W):
        f = np.ascontiguousarray(first, dtype=np.int64)
        return lib.sgpr_kernel_jacobian_batch(eng._h, len(f) - 1, ctypes.c_void_p(f.ctypes.data), p(pos), p(Z),
                                              ctypes.c_void_p(cells.ctypes.data), ctypes.c_void_p(pbcs.ctypes.data),
                                              m0, m1, stream, p(Ke), p(J_), p(W_))

    assert call([0, N]) == 0
    assert call([0, N], J_=None) == -1 and b"both" in lib.sgpr_last_error()
    assert call([0, N], W_=None) == -1
    assert call([0, N, N - 1]) == -1 and b"structure 1" in lib.sgpr_last_error()
    assert call([1, N]) == -1
    assert call([0, N], m1=M + 1) == -1 and call([0, N], m0=-1) == -1 and call([0, N], m0=3, m1=2) == -1
    assert call([0, N], J_=None, W_=None) == 0
    # an unknown species names its structure and leaves the handle usable
    bad = as_atoms(a.positions[:4], np.array([29, 29, 99, 29]), a.cell, a.pbc)
    with pytest.raises(RuntimeError, match=r"error -3: structure 1: atomic number 99"):
        eng.training_kernels([a, bad])
    E, F, Wv, _ = eng.predict(a.positions, a.numbers, a.cell, a.pbc)
    assert abs(E - float(g["energy"])) / N < 1e-9 and np.abs(F - g["forces"]).max() < TOL_F
    eng.close()


def test_four_species_against_prediction():
    """B = 32 frames of 128 atoms, 4 species, M = 2000: Kf @ mu, Kv @ mu and Ke @ mu + means are the batch prediction."""
    import autoforce_b200 as ab
    from autoforce_b200.synth import fcc, synth_model

    Zs = [3, 8, 15, 16]
    model = synth_model(Zs, 2000, seed=17)
    eng = ab.SgprEngine(model, species=Zs)
    frames = []
    for f in range(32):
        pos, cell, Z = fcc((4, 4, 2), Zs, 0.1, 100 + f)
        frames.append(as_atoms(pos, Z, cell, (True, True, True)))
    Ke, Kf, Kv = eng.training_kernels(frames)
    E, F, W = eng.predict_batch(frames)
    mu = np.asarray(model.mu, dtype=float)
    Ke, Kf, Kv = Ke.cpu().numpy(), Kf.cpu().numpy(), Kv.cpu().numpy()
    assert np.abs(Kf @ mu - F.reshape(-1)).max() < 1e-9 * max(1.0, np.abs(F).max())
    Wsel = W.reshape(len(frames), 9)[:, [0, 4, 8, 5, 2, 1]].reshape(-1)
    assert np.abs(Kv @ mu - Wsel).max() < 1e-8 * max(1.0, np.abs(Wsel).max())
    means = np.array([sum(model.mean_w.get(int(z), 0.0) for z in a.numbers) for a in frames])
    assert np.abs(Ke @ mu + means - E).max() < 1e-9 * max(1.0, np.abs(E).max())
    eng.close()


def test_similarity_kernel_with_a_list_of_structures():
    import autoforce_b200 as ab

    g = load_golden("cu108_sesoap")
    k = g["meta"]["kernel"]
    kern = ab.SeSoapKernel(k["lmax"], k["nmax"], k["xi"], k["rc"], radii=ab.DefaultRadii())
    X = [(int(z), r, b) for z, r, b in zip(g["ind_Z"], g["envs_r"], g["envs_b"])]
    a1 = as_atoms(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"])
    a2 = as_atoms(g["pos"] + np.random.default_rng(2).normal(0, 0.03, g["pos"].shape), g["numbers"], g["cell"], g["meta"]["pbc"])
    for op in ("leftgrad", "virial"):
        both = kern([a1, a2], X, operation=op)
        stacked = np.concatenate([kern(a1, X, operation=op), kern(a2, X, operation=op)])
        assert both.shape == stacked.shape and rel(both, stacked) <= 1e-13
    Ke = kern([a1, a2], X)
    assert Ke.shape == (2, len(X))
    assert np.abs(Ke[0] - kern(a1, X).sum(axis=0)).max() < 1e-11 * max(1.0, np.abs(Ke).max())
    kern.close()
