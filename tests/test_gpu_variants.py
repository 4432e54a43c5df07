"""Every descriptor-kernel instantiation and the tile edges of the tcgen05 int8 GEMMs against the float64 oracle.

descriptor.cu picks a template instantiation of the forward, backward and Jacobian kernels from (lmax, nmax+1) and the
shared-memory plan from S*(nmax+1); the golden cases and bench workloads reach only three of them.  CASES below names a
model for every other one, together with the instantiation it is meant to reach; test_case_table_matches_dispatch checks
the names of the kernels actually launched, so the table cannot go stale.  The GEMM cases cross the 128-row / 64-column
tiles and the 64-byte K chunks of i8gemm.cu at and around every edge, on both GEMM engines.

The oracle references of every case are also built in the CPU suite (test_*_reference_*), so a broken case shows up
before any GPU run.
"""
import functools
import re
from dataclasses import dataclass

import numpy as np
import pytest

from autoforce_b200.model import SgprModel
from autoforce_b200.synth import cut_environments, fcc
from oracle import sgpr_oracle as o
from oracle_engine import to_oracle

RC = 4.5   # fcc Cu, a0 = 3.61: three shells (12 + 6 + 24 neighbours)

# DESIGN.md section 2
TOL_DESC, TOL_K, TOL_E, TOL_F, TOL_SIGMA, TOL_BETA2 = 1e-13, 1e-12, 1e-9, 1e-8, 1e-9, 1e-9


@dataclass(frozen=True)
class Case:
    name: str
    lmax: int
    nmax: int
    Zs: tuple
    fwd: tuple      # desc_forward_kernel<LMAX, TN, TL, ENV, EXNB, BATCH>: (LMAX, TN, TL, EXNB)
    bwd: tuple      # desc_backward_kernel<LMAX, NB, EXACT, BATCH> and jacobian_kernel<LMAX, NB, EXACT, MM>: (LMAX, NB, EXACT)
    rep: tuple = (2, 2, 2)
    pbc: tuple = (True, True, True)
    tric: bool = False

    @property
    def A(self):
        return len(self.Zs) * (self.nmax + 1)

    @property
    def D(self):
        return self.A * (self.A + 1) // 2 * (self.lmax + 1)


F, T = False, True
CASES = [
    Case("l0n0", 0, 0, (29,), (3, 2, 1, 0), (3, 4, F)),                                       # L2 = 1, D = 1
    Case("l1n5_2sp", 1, 5, (29, 47), (3, 4, 1, 0), (3, 8, F), tric=T),
    Case("l2n7", 2, 7, (29,), (3, 4, 1, 0), (3, 8, F), pbc=(T, F, T)),
    Case("l3n9", 3, 9, (29,), (3, 6, 1, 0), (6, 12, F)),
    Case("l4n4_2sp", 4, 4, (13, 29), (6, 2, 5, 0), (6, 6, F), pbc=(T, T, F), tric=T),
    Case("l5n2", 5, 2, (29,), (6, 2, 5, 0), (6, 6, F)),
    Case("l5n7", 5, 7, (29,), (6, 3, 5, 0), (6, 9, F), tric=T),
    Case("l6n11", 6, 11, (29,), (6, 4, 5, 0), (6, 12, F)),
    Case("l7n3_2sp", 7, 3, (29, 47), (8, 6, 6, 0), (8, 12, F), pbc=(F, T, T)),
    Case("l8n11", 8, 11, (29,), (8, 6, 6, 0), (8, 12, F)),
    # A = 20 > 16: the per-species runs of the forward contraction, the generic dE/dc product (exact (3, 4) kernels)
    Case("l3n3_5sp", 3, 3, (3, 8, 15, 16, 29), (3, 2, 1, 4), (3, 4, T), rep=(2, 2, 3), tric=T),
    Case("l2n5_3sp", 2, 5, (8, 16, 29), (3, 4, 1, 0), (3, 8, F), rep=(2, 2, 3), pbc=(T, T, F)),
    # A = 96, D = 9312: the packed row does not fit the chunk buffer (pspec_entry), one warp per block in the force kernel
    Case("l1n11_8sp", 1, 11, (3, 6, 8, 13, 15, 16, 29, 47), (3, 6, 1, 0), (6, 12, F), rep=(2, 2, 4)),
]
CASE = {c.name: c for c in CASES}


def structure(rep, Zs, seed, counts=None, pbc=(True, True, True), tric=False, sigma=0.08):
    """Rattled fcc cell; every species present (round-robin, or `counts` atoms of each), optionally sheared."""
    pos, cell, _ = fcc(rep, Zs, 0.0, seed)
    rng = np.random.default_rng(seed)
    n = len(pos)
    numbers = np.repeat(np.asarray(Zs), counts) if counts is not None else np.asarray(Zs)[np.arange(n) % len(Zs)]
    assert len(numbers) == n
    numbers = rng.permutation(numbers).astype(np.int32)
    if tric:
        frac = pos @ np.linalg.inv(cell)
        a, b, c = np.diag(cell)
        cell = np.array([[a, 0.0, 0.0], [0.3 * a, b, 0.0], [-0.2 * a, 0.15 * b, c]])
        pos = frac @ cell
    pos = pos + rng.normal(0, sigma, pos.shape)
    return pos, cell, numbers, tuple(bool(p) for p in pbc)


def make_model(Zs, Ms, lmax, nmax, xi=4.0, seed=0, mu=None, rc=RC):
    """Ms[k] inducing LCEs of species Zs[k], grouped by species (caller's order = the engine's sorted order), cut out of a
    rattled 500-atom fcc cell; dense lower-triangular choli."""
    pos, cell, numbers = fcc(5, Zs, 0.15, seed + 100)
    first, J, S = o.neighbor_list(pos, cell, True, rc)
    rng = np.random.default_rng(seed)
    sel = []
    for z, m in zip(Zs, Ms):
        idx = np.nonzero(numbers == z)[0]
        sel += list(rng.choice(idx, m, replace=len(idx) < m))
    envs = cut_environments(pos, cell, True, numbers, rc, sel, first, J, S)
    M = len(envs)
    if mu is None:
        mu = rng.normal(0, 0.1, M)
    choli = 0.5 * np.eye(M) + np.tril(np.random.default_rng(seed + 7).normal(0, 0.02 / np.sqrt(M), (M, M)), -1)
    return SgprModel.from_envs(envs, mu=np.asarray(mu, dtype=float), mean_w={z: -3.0 for z in Zs}, vscale={z: 1.0 for z in Zs},
                               choli=choli, lmax=lmax, nmax=nmax, xi=float(xi), rc=rc, kind="sesoap", radii={1: 0.5},
                               default_radius=1.0)


# ------------------------------------------------------------------------------------------------------------------
# descriptor cases: model, two structures and their oracle references (built once per case)
# ------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def case_data(name):
    c = CASE[name]
    model = make_model(list(c.Zs), [3] * len(c.Zs), c.lmax, c.nmax, seed=11)
    s1 = structure(c.rep, c.Zs, 1, pbc=c.pbc, tric=c.tric)
    rep2 = (c.rep[0], c.rep[1], c.rep[2] + 1)
    s2 = structure(rep2, c.Zs, 2, pbc=(True, True, True) if c.pbc != (True, True, True) else (True, False, True),
                   tric=not c.tric)
    om = to_oracle(model)
    species = np.asarray(sorted(c.Zs), dtype=np.int64)
    ref = []
    for pos, cell, Z, pbc in (s1, s2):
        first, J, S = o.neighbor_list(pos, cell, pbc, om.rc)
        envs_r = [o.displacements(pos, cell, i, J[first[i]:first[i + 1]], S[first[i]:first[i + 1]]) for i in range(len(Z))]
        R, Zb, mask = o.pad_environments(envs_r, [Z[J[first[i]:first[i + 1]]] for i in range(len(Z))])
        ref.append(dict(P=o.descriptor_batch(om, species, R, Zb, mask),
                        out=o.predict(om, pos, cell, pbc, Z, want_beta=True)))
    Zh, _ = o.inducing_descriptors(om, species)
    Ke, Kf, Kv = o.kernel_jacobian(om, *s1[:2], s1[3], s1[2], scatter_quirk=False)
    return model, (s1, s2), ref, Zh, (Ke, Kf, Kv)


def vol(cell):
    return abs(np.linalg.det(cell))


@pytest.mark.parametrize("name", list(CASE))
def test_descriptor_case_reference(name):
    """CPU: the oracle references of the case are finite, every species block of the descriptors is non-zero (every
    species has neighbours) and the case reaches the shape the table says."""
    c = CASE[name]
    model, structs, ref, Zh, (Ke, Kf, Kv) = case_data(name)
    S = len(c.Zs)
    for r in ref:
        P, out = r["P"], r["out"]
        assert P.shape[1:] == (S, S, c.nmax + 1, c.nmax + 1, c.lmax + 1)
        blocks = np.abs(P).sum(axis=(0, 3, 4, 5))
        assert (blocks > 0).all(), blocks
        for k in ("energy", "forces", "virial", "beta"):
            assert np.isfinite(out[k]).all(), k
        assert np.abs(out["forces"]).max() > 0
    assert np.isfinite(Zh).all() and (np.abs(Zh).sum(axis=(0, 3, 4, 5)) > 0).any()
    assert np.isfinite(Ke).all() and np.isfinite(Kf).all() and np.isfinite(Kv).all() and np.abs(Kf).max() > 0
    assert 32 <= len(structs[0][2]) <= 64 and len(structs[1][2]) != len(structs[0][2])
    if name == "l1n11_8sp":
        assert c.D == 9312


def engine_for(model, species):
    import autoforce_b200 as ab

    return ab.SgprEngine(model, species=list(species))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASE))
def test_descriptor_case(name):
    c = CASE[name]
    print(f"\n[variants] {name}", flush=True)
    model, structs, ref, Zh_ref, (Ke_ref, Kf_ref, Kv_ref) = case_data(name)
    eng = engine_for(model, c.Zs)
    try:
        # inducing LCEs: the ENV instantiation
        Zh = eng.inducing_descriptors()
        assert np.abs(Zh - Zh_ref).max() < TOL_DESC
        # atoms: descriptors, E / F / virial / covloss
        for (pos, cell, Z, pbc), r in zip(structs, ref):
            N = len(Z)
            P = eng.descriptors(pos, Z, cell, pbc)
            assert np.abs(P - r["P"]).max() < TOL_DESC
            E, Fo, W, _, beta = eng.predict(pos, Z, cell, pbc, want_beta=True)
            out = r["out"]
            assert abs(E - out["energy"]) / N < TOL_E
            assert np.abs(Fo - out["forces"]).max() < TOL_F
            assert np.abs(W - out["virial"]).max() / vol(cell) < TOL_SIGMA
            assert np.abs(beta ** 2 - out["beta"] ** 2).max() < TOL_BETA2
        # the BATCH instantiations: both structures in one call
        import types

        atoms = [types.SimpleNamespace(positions=p, numbers=Z, cell=cell, pbc=pbc) for p, cell, Z, pbc in structs]
        Eb, Fb, Wb, bb = eng.predict_batch(atoms, want_beta=True)
        a0 = 0
        for b, ((pos, cell, Z, pbc), r) in enumerate(zip(structs, ref)):
            N, out = len(Z), r["out"]
            assert abs(Eb[b] - out["energy"]) / N < TOL_E
            assert np.abs(Fb[a0:a0 + N] - out["forces"]).max() < TOL_F
            assert np.abs(Wb[b] - out["virial"]).max() / vol(cell) < TOL_SIGMA
            assert np.abs(bb[a0:a0 + N] ** 2 - out["beta"] ** 2).max() < TOL_BETA2
            a0 += N
        # training-time kernels (the Jacobian kernel): Ke sums N kernel entries, each within TOL_K
        Ke, Kf, Kv = (x.cpu().numpy() for x in eng.training_kernels(atoms[:1]))
        pos, cell, Z, pbc = structs[0]
        assert np.abs(Ke[0] - Ke_ref).max() < TOL_K * len(Z)
        assert np.abs(Kf - Kf_ref).max() < TOL_F
        assert np.abs(Kv - Kv_ref).max() / vol(cell) < TOL_SIGMA
    finally:
        eng.close()


def launched_templates(fn):
    """Template argument lists of the descriptor kernels launched by fn(), from the demangled kernel names that
    torch.profiler records."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = {"desc_forward_kernel": set(), "desc_backward_kernel": set(), "jacobian_kernel": set()}
    for e in prof.events():
        for k in found:
            m = re.search(k + r"<([^<>]*)>", e.name)
            if m:
                found[k].add(tuple(x.strip() for x in m.group(1).split(",")))
    return found


def expected_templates(c):
    b = lambda v: "true" if v else "false"   # noqa: E731
    LM, TN, TL, EX = (str(v) for v in c.fwd)
    BL, NB, EXACT = str(c.bwd[0]), str(c.bwd[1]), b(c.bwd[2])
    MM = "4" if c.bwd[1] <= 4 else "2"
    return {
        "desc_forward_kernel": {(LM, TN, TL, "false", EX, "false"), (LM, TN, TL, "true", EX, "false"),
                                (LM, TN, TL, "false", EX, "true")},
        "desc_backward_kernel": {(BL, NB, EXACT, "false"), (BL, NB, EXACT, "true")},
        "jacobian_kernel": {(BL, NB, EXACT, MM)},
    }


@pytest.mark.gpu
def test_case_table_matches_dispatch():
    """Every row of CASES launches the forward (plain, ENV, BATCH), backward (plain, BATCH) and Jacobian kernels the
    table names, and no other descriptor kernel."""
    import types

    for c in CASES:
        print(f"\n[variants] profile {c.name}", flush=True)
        model, structs, _, _, _ = case_data(c.name)
        atoms = [types.SimpleNamespace(positions=p, numbers=Z, cell=cell, pbc=pbc) for p, cell, Z, pbc in structs]
        box = {}

        def run():
            box["eng"] = eng = engine_for(model, c.Zs)
            pos, cell, Z, pbc = structs[0]
            eng.predict(pos, Z, cell, pbc)
            eng.predict_batch(atoms)
            eng.training_kernels(atoms[:1])

        try:
            found = launched_templates(run)
        finally:
            if "eng" in box:
                box["eng"].close()
        want = expected_templates(c)
        for k in want:
            # all three forms launched, and every launch of the kernel is this row's instantiation
            assert want[k] <= found[k], (c.name, k, found[k])
            assert {t[:3] for t in found[k]} == {t[:3] for t in want[k]}, (c.name, k, found[k])


@pytest.mark.gpu
def test_too_large_descriptor_is_refused_at_create():
    """lmax 2, nmax 11, 8 species (D = 13,968): the force kernel's per-warp rows (2 D + 2 csize doubles) exceed the
    shared memory of a block; the model is refused when the engine is created, not at its first prediction."""
    Zs = [3, 6, 8, 13, 15, 16, 29, 47]
    base = dict(lmax=2, nmax=11, xi=4.0, rc=RC, kind="sesoap", radii={1: 0.5}, default_radius=1.0)
    with pytest.raises(RuntimeError, match=r"too large for shared memory \(S=8 nmax=11 lmax=2\)"):
        engine_for(SgprModel.from_envs([], **base), Zs)
    # the largest row of the table is accepted
    engine_for(SgprModel.from_envs([], **dict(base, lmax=1)), Zs).close()


# ------------------------------------------------------------------------------------------------------------------
# GEMM tile edges: BM = 128 rows, BN = 64 columns, K chunks of 64 bytes (i8gemm.cu); tcgen05 and FP64 DMMA engines
# ------------------------------------------------------------------------------------------------------------------
@dataclass(frozen=True)
class GemmCase:
    name: str
    Zs: tuple
    Ms: tuple            # inducing LCEs per species
    lmax: int = 3
    nmax: int = 3
    xi: float = 4.0
    rep: tuple = (3, 3, 3)
    counts: tuple = None  # atoms per species (None: round-robin)
    hot: tuple = None    # (species k, column c): mu is zero except at the c-th LCE of species k


def gemm_cases():
    cs = []
    # rows of a central species around the 128-row tiles (the next species' block starts mid-tile)
    for counts, rep in (((1, 255), (4, 4, 4)), ((127, 129), (4, 4, 4)), ((128, 128), (4, 4, 4)), ((257, 63), (4, 4, 5))):
        cs.append(GemmCase(f"rows_{counts[0]}_{counts[1]}", (29, 47), (9, 7), rep=rep, counts=counts))
    # LCEs of a species around the 64-column tiles; one-hot weights on an edge column
    for Ms, hot in (((1, 129), (1, 64)), ((63, 65), (1, 63)), ((63, 65), (1, 64)), ((64, 128), (1, 64)),
                    ((64, 128), (0, 63)), ((129, 1), (0, 128))):
        cs.append(GemmCase(f"ms_{Ms[0]}_{Ms[1]}_hot{hot[0]}_{hot[1]}", (29, 47), Ms, hot=hot))
    # D around one K chunk: 40, 60, 63 take the single-chunk kernel; 66, 84 two chunks; 544 nine
    for lmax, nmax, Zs in ((3, 3, (29,)), (3, 4, (29,)), (2, 5, (29,)), (0, 10, (29,)), (3, 2, (29, 47)),
                           (3, 3, (3, 8, 15, 16))):
        D = (len(Zs) * (nmax + 1)) * (len(Zs) * (nmax + 1) + 1) // 2 * (lmax + 1)
        cs.append(GemmCase(f"D{D}", Zs, (24,) * len(Zs), lmax=lmax, nmax=nmax))
    # epilogue exponents, on the single-chunk (D = 40) and the multi-chunk (D = 84) kernel
    for xi in (1, 2, 3, 4, 5):
        cs.append(GemmCase(f"xi{xi}_D40", (29,), (70,), xi=xi))
        cs.append(GemmCase(f"xi{xi}_D84", (29, 47), (40, 30), nmax=2, xi=xi))
    # covloss: M not a multiple of 64 (the zero K chunks of the triangular choli are skipped)
    for Ms in ((30, 35), (64, 65), (100, 93)):
        cs.append(GemmCase(f"cov_M{sum(Ms)}", (29, 47), Ms))
    return cs


GEMM = {c.name: c for c in gemm_cases()}


def gemm_mu(c, scale):
    M = sum(c.Ms)
    if c.hot is None:
        return np.random.default_rng(3).normal(0, 0.1, M) * scale
    mu = np.zeros(M)
    mu[sum(c.Ms[:c.hot[0]]) + c.hot[1]] = scale
    return mu


@functools.lru_cache(maxsize=None)
def gemm_data(name, scale):
    c = GEMM[name]
    model = make_model(list(c.Zs), list(c.Ms), c.lmax, c.nmax, xi=c.xi, seed=23, mu=gemm_mu(c, scale))
    pos, cell, Z, pbc = structure(c.rep, c.Zs, 5, counts=c.counts)
    out = o.predict(to_oracle(model), pos, cell, pbc, Z, want_K=True, want_beta=True)
    return model, (pos, cell, Z, pbc), out


def gemm_params():
    ps = []
    for n, c in GEMM.items():
        for scale in ((1.0, 1000.0) if c.hot is not None else (1.0,)):
            ps.append((n, scale))
    return ps


@pytest.mark.parametrize("name,scale", gemm_params())
def test_gemm_case_reference(name, scale):
    """CPU: the case has the shape it is named for and a finite oracle reference."""
    c = GEMM[name]
    model, (pos, cell, Z, pbc), out = gemm_data(name, scale)
    for z, n in zip(c.Zs, c.counts or ()):
        assert (Z == z).sum() == n
    assert [int((model.ind_Z == z).sum()) for z in c.Zs] == list(c.Ms)
    assert np.isfinite(out["energy"]) and np.isfinite(out["forces"]).all() and np.isfinite(out["beta"]).all()
    assert np.abs(out["forces"]).max() > 0
    if c.hot is not None:
        m = sum(c.Ms[:c.hot[0]]) + c.hot[1]
        assert model.ind_Z[m] == c.Zs[c.hot[0]] and np.abs(out["K"][:, m]).max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["i8", "dmma"])
@pytest.mark.parametrize("name,scale", gemm_params())
def test_gemm_case(name, scale, engine, monkeypatch):
    c = GEMM[name]
    print(f"\n[variants] gemm {name} x{scale:g} {engine}", flush=True)
    if engine == "dmma":
        monkeypatch.setenv("SGPR_GEMM", "dmma")
    else:
        monkeypatch.delenv("SGPR_GEMM", raising=False)
    model, (pos, cell, Z, pbc), out = gemm_data(name, scale)
    N = len(Z)
    eng = engine_for(model, c.Zs)
    try:
        E, Fo, W, _, beta = eng.predict(pos, Z, cell, pbc, want_beta=True)
        i8_ops = eng.stats()["i8_ops"]
    finally:
        eng.close()
    assert (i8_ops > 0) if engine == "i8" else (i8_ops == 0)
    # the GEMMs' error is relative to the largest weight (the back projection is scaled by max |xi mu|)
    s = max(1.0, scale)
    assert abs(E - out["energy"]) / N < TOL_E * s
    assert np.abs(Fo - out["forces"]).max() < TOL_F * s
    assert np.abs(W - out["virial"]).max() / vol(cell) < TOL_SIGMA * s
    assert np.abs(beta ** 2 - out["beta"] ** 2).max() < TOL_BETA2
    if c.hot is not None:
        # E minus the means is the hot column's sum of k^xi times its weight: a dropped or repeated column shows
        m = sum(c.Ms[:c.hot[0]]) + c.hot[1]
        means = sum(model.mean_w[int(z)] for z in Z)
        assert abs((E - means) / scale - out["K"][:, m].sum()) / N < TOL_E
