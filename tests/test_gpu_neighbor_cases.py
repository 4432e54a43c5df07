"""Both neighbour kernels against the float64 oracle on every geometry they branch on.

nl.cu has two searches: one warp per atom (neighbor_kernel) and one block per bin (neighbor_bin_kernel<NS>), which the
automatic mode picks from 64 bins on.  The golden cells have 1-9 bins, so most of the bin kernel's branches are reached
only by the geometries below: stencil reaches of 2 and 3 (a periodic axis thinner than rc), more stencil runs than one
shared-memory chunk holds, candidate tiles and accept-bit slots past the 64-slot word, several rounds of atoms per bin,
5-8 species (NS = 8), triclinic and mixed-pbc cells, merged bins, lone atoms and atoms exactly on cell faces.

bin_plan() restates nl.cu's binning (geom_cell, geom_bins, frac_bin and the stencil walk of neighbor_bin_kernel) in numpy
and derives what each structure reaches; test_case_reaches_its_branch checks every row of CASES against it on the CPU,
and test_case_table_matches_dispatch checks the kernel the GPU actually launches (and its grid) against it, so the table
and the restatement cannot go stale.
"""
import functools
import json
import os
import re
import tempfile
import types
from dataclasses import dataclass

import numpy as np
import pytest

from oracle import sgpr_oracle as o
from oracle_engine import to_oracle
from test_gpu_variants import make_model, structure

# nl.cu constants
K_BIN_ATOMS = 32          # kBinAtoms: atoms of a bin per round of neighbor_bin_kernel (one row reservation each)
K_BIN_CAP = 1024          # kBinCap: candidates per shared-memory tile
K_RUN_CHUNK = 128         # kRunChunk: stencil runs staged at once (stage_runs)
K_MASK_SLOTS = 64         # kMaskSlots: 32-candidate slots covered by the accept-bit word; later slots are retested
MIN_BINS_BIN_KERNEL = 64  # use_bin_kernels: the automatic mode runs neighbor_bin_kernel from this many bins on
RC_SLACK = 1.0 + 1e-7     # geom_bins: bins are sized for rc * (1 + 1e-7)

# DESIGN.md section 2
TOL_E, TOL_F, TOL_SIGMA, TOL_BETA2 = 1e-9, 1e-8, 1e-9, 1e-9

A0 = 3.61
EIGHT = (3, 6, 8, 13, 15, 16, 29, 47)


def bin_plan(pos, cell, pbc, rc, S):
    """The bins, stencil and work split nl.cu derives for a structure (host geometry and the bin kernel's walk)."""
    pos = np.asarray(pos, dtype=float).reshape(-1, 3)
    pbc = np.broadcast_to(np.asarray(pbc, dtype=bool), (3,))
    cell = o.complete_cell(np.asarray(cell, dtype=float).reshape(3, 3))
    inv = np.linalg.inv(cell)
    hface = 1.0 / np.linalg.norm(inv, axis=0)            # geom_cell: distances between opposite faces
    frac = pos @ inv
    N = len(pos)
    lo, hi = np.zeros(3), np.ones(3)
    if not pbc.all() and N:
        lo, hi = frac.min(axis=0), frac.max(axis=0)
    rcs = rc * RC_SLACK
    nb, reach, flo, fscale = [0] * 3, [0] * 3, [0.0] * 3, [0.0] * 3
    for c in range(3):                                   # geom_bins
        if pbc[c]:
            nb[c] = max(1, int(np.floor(hface[c] / rcs)))
            reach[c] = int(np.ceil(rcs / (hface[c] / nb[c])))
            fscale[c] = float(nb[c])
        else:
            nb[c] = max(1, int(np.floor((hi[c] - lo[c]) * hface[c] / rcs)))
            reach[c] = 1
            flo[c] = lo[c]
            fscale[c] = nb[c] / (hi[c] - lo[c]) if hi[c] > lo[c] else 0.0
    merges = 0
    while float(nb[0]) * nb[1] * nb[2] > max(4096.0, 4.0 * N):   # keep the cell table small relative to N
        c = int(np.argmax(nb))                           # first axis of the largest count
        n2 = (nb[c] + 1) // 2
        if pbc[c]:
            fscale[c] = float(n2)
            reach[c] = int(np.ceil(rcs / (hface[c] / n2)))
        else:
            fscale[c] *= n2 / nb[c]
        nb[c] = n2
        merges += 1
    # frac_bin: periodic axes wrap (w = floor), the bin index is truncated and clamped
    b3 = np.zeros((N, 3), dtype=np.int64)
    wrapped = clamped = False
    for c in range(3):
        f = frac[:, c].copy()
        if pbc[c]:
            w = np.floor(f)
            f = f - w
            wrapped |= bool((w != 0).any())
        else:
            f = f - flo[c]
        raw = (f * fscale[c]).astype(np.int64)
        clamped |= bool(((raw < 0) | (raw > nb[c] - 1)).any())
        b3[:, c] = np.clip(raw, 0, nb[c] - 1)
    cnt = np.zeros(nb, dtype=np.int64)
    np.add.at(cnt, (b3[:, 0], b3[:, 1], b3[:, 2]), 1)
    # neighbor_bin_kernel's stencil of every occupied bin: runs (z merged into one run per column when the z stencil
    # neither wraps nor leaves the box), chunks of runs, tiles of candidates per chunk, 32-candidate slots
    plan = dict(N=N, nb=tuple(nb), ncell=int(np.prod(nb)), reach=tuple(reach), merges=merges, wrapped=wrapped,
                clamped=clamped, max_bin=int(cnt.max()) if N else 0, runs=0, run_chunks=0, max_cand=0, tiles=0, slots=0,
                z_merged=False, z_unmerged=False)

    def wrap(n, c):
        if pbc[c]:
            return n % nb[c], True
        return n, 0 <= n < nb[c]

    for bx, by, bz in zip(*np.nonzero(cnt)):
        zlo, zhi = bz - reach[2], bz + reach[2]
        merged = zlo >= 0 and zhi < nb[2]
        plan["z_merged" if merged else "z_unmerged"] = True
        lens = []
        for dx in range(-reach[0], reach[0] + 1):
            for dy in range(-reach[1], reach[1] + 1):
                for dz in ([0] if merged else range(-reach[2], reach[2] + 1)):
                    nx, okx = wrap(bx + dx, 0)
                    ny, oky = wrap(by + dy, 1)
                    if merged:
                        zs, okz = range(zlo, zhi + 1), True
                    else:
                        nz, okz = wrap(bz + dz, 2)
                        zs = [nz]
                    lens.append(int(cnt[nx, ny, list(zs)].sum()) if okx and oky and okz else 0)
        tiles = slots = 0
        for r0 in range(0, len(lens), K_RUN_CHUNK):
            total = sum(lens[r0:r0 + K_RUN_CHUNK])
            for t0 in range(0, total, K_BIN_CAP):
                tiles += 1
                slots += -(-min(K_BIN_CAP, total - t0) // 32)
        plan["runs"] = max(plan["runs"], len(lens))
        plan["run_chunks"] = max(plan["run_chunks"], -(-len(lens) // K_RUN_CHUNK))
        plan["max_cand"] = max(plan["max_cand"], sum(lens))
        plan["tiles"] = max(plan["tiles"], tiles)
        plan["slots"] = max(plan["slots"], slots)
    plan["rounds"] = -(-plan["max_bin"] // K_BIN_ATOMS)
    plan["slots_past_word"] = plan["slots"] > K_MASK_SLOTS
    plan["kernel"] = "bins" if plan["ncell"] >= MIN_BINS_BIN_KERNEL else "warp"
    plan["NS"] = 1 if S <= 1 else 2 if S <= 2 else 4 if S <= 4 else 8     # launch_neighbor_bins / launch_neighbor
    return plan


# ------------------------------------------------------------------------------------------------------------------
# geometries
# ------------------------------------------------------------------------------------------------------------------
def conventional(rep, Zs, seed, pbc=(True, True, True), sigma=0.05):
    return structure(rep, Zs, seed, pbc=pbc, sigma=sigma)


def primitive(Zs, seed):
    cell = 0.5 * A0 * np.array([[0.0, 1.0, 1.0], [1.0, 0.0, 1.0], [1.0, 1.0, 0.0]])
    return np.array([[0.4, -0.3, 0.2]]), cell, np.asarray(Zs[:1], dtype=np.int32), (True, True, True)


def sparse_gas(Zs, seed, n=500, box=150.0):
    rng = np.random.default_rng(seed)
    pos = rng.uniform(0.0, box, (n, 3))
    return pos, np.eye(3) * box, np.asarray(Zs)[rng.integers(0, len(Zs), n)].astype(np.int32), (True, True, True)


def faces(Zs, seed):
    """Simple cubic lattice (2 A) in a 16 A box; atoms of the x = 0, y = 0 and z = 0 planes are stored at exact face
    values: 16 (fractional 1: wraps to 0), -0.0, 16 (1 - 2^-53) (just inside), and -2^-56 (fractional -2^-60: wraps to
    1 - 2^-60, which rounds to 1, so the bin index reaches nb and is clamped).  Interior atoms are rattled lightly."""
    L, a = 16.0, 2.0
    g = np.arange(0.0, L, a)
    pos = np.stack(np.meshgrid(g, g, g, indexing="ij"), axis=-1).reshape(-1, 3)
    rng = np.random.default_rng(seed)
    interior = (pos > 0).all(axis=1)
    pos[interior] += rng.normal(0.0, 0.03, (int(interior.sum()), 3))
    edge = [L, -0.0, L * (1.0 - 2.0 ** -53), -(2.0 ** -56)]
    for c in range(3):
        on = np.nonzero(pos[:, c] == 0.0)[0]
        for k, i in enumerate(on):
            pos[i, c] = edge[(k + c) % 4]
    numbers = np.asarray(Zs)[rng.integers(0, len(Zs), len(pos))].astype(np.int32)
    return pos, np.eye(3) * L, numbers, (True, True, True)


@dataclass(frozen=True)
class Case:
    name: str
    reaches: str       # what the row is there for
    Zs: tuple
    rc: float
    make: object       # (Zs, seed) -> pos, cell, numbers, pbc
    expect: tuple      # (bin_plan key, value) pairs the geometry must have


T, F = True, False
CASES = [
    Case("prim", "reach 3 on every axis: 343 runs in 3 run chunks, the atom's own images", (29,), 4.5, primitive,
         (("ncell", 1), ("reach", (3, 3, 3)), ("runs", 343), ("run_chunks", 3), ("kernel", "warp"), ("NS", 1))),
    Case("thin_221", "reach (2,2,3), 175 runs in 2 chunks, 2,800 candidates: 3 tiles, slots past the word across chunks",
         (3, 8), 7.5, lambda Zs, s: conventional((2, 2, 1), Zs, s),
         (("ncell", 1), ("reach", (2, 2, 3)), ("runs", 175), ("run_chunks", 2), ("max_cand", 2800), ("tiles", 3),
          ("slots_past_word", T), ("kernel", "warp"), ("NS", 2))),
    Case("monolayer", "64 bins: the bin kernel by default, reach 2 in z, unmerged z stencil", (3, 8), 6.0,
         lambda Zs, s: conventional((14, 14, 1), Zs, s),
         (("ncell", 64), ("nb", (8, 8, 1)), ("reach", (1, 1, 2)), ("z_unmerged", T), ("z_merged", F), ("runs", 45),
          ("kernel", "bins"), ("NS", 2))),
    Case("wire", "open x and y, reach 2 along the periodic z", (29,), 6.0,
         lambda Zs, s: conventional((3, 3, 1), Zs, s, pbc=(False, False, True)),
         (("nb", (1, 1, 1)), ("reach", (1, 1, 2)), ("runs", 45), ("kernel", "warp"), ("NS", 1))),
    Case("eight_sp", "64 bins, 8 species: neighbor_bin_kernel<8> by default, merged z stencil", EIGHT, 4.5,
         lambda Zs, s: conventional((5, 5, 5), Zs, s),
         (("ncell", 64), ("reach", (1, 1, 1)), ("z_merged", T), ("z_unmerged", T), ("kernel", "bins"), ("NS", 8))),
    Case("five_sp_tric", "sheared cell, 5 species (NS = 8 with S = 5), 125 bins", (3, 8, 15, 16, 29), 4.0,
         lambda Zs, s: structure((6, 6, 6), Zs, s, tric=True, sigma=0.05),
         (("ncell", 125), ("reach", (1, 1, 1)), ("wrapped", T), ("kernel", "bins"), ("NS", 8))),
    Case("sparse_gas", "500 atoms in a 150 A box: bins merged by the max(4096, 4N) rule, empty bins, lone atoms", EIGHT,
         6.0, sparse_gas,
         (("nb", (12, 12, 24)), ("merges", 2), ("reach", (1, 1, 1)), ("kernel", "bins"), ("NS", 8))),
    Case("faces", "atoms exactly on cell faces: wrap at fractional 1, -0.0, 1 - 2^-53, clamp at -2^-60", (3, 8, 15, 29),
         4.5, faces,
         (("nb", (3, 3, 3)), ("reach", (1, 1, 1)), ("wrapped", T), ("clamped", T), ("kernel", "warp"), ("NS", 4))),
]
CASE = {c.name: c for c in CASES}
BIG = [c.name for c in CASES if dict(c.expect).get("kernel") == "bins"]   # at least 64 bins: sharding, fused step


def rows_sorted(first, J, S):
    I = np.repeat(np.arange(len(first) - 1), np.diff(first))
    order = np.lexsort((S[:, 2], S[:, 1], S[:, 0], J, I))
    return I[order], J[order].astype(np.int64), S[order].astype(np.int64)


@functools.lru_cache(maxsize=None)
def case_data(name):
    """Model, structure, bin plan and oracle references of a case."""
    c = CASE[name]
    Zs = tuple(sorted(c.Zs))
    model = make_model(list(Zs), [3] * len(Zs), 2, 2, rc=c.rc, seed=31)
    pos, cell, Z, pbc = c.make(Zs, 7)
    nl = o.neighbor_list(pos, cell, pbc, c.rc)
    out = o.predict(to_oracle(model), pos, cell, pbc, Z, want_beta=True, nl=nl)
    return model, (pos, cell, Z, pbc), bin_plan(pos, cell, pbc, c.rc, len(Zs)), nl, out


@functools.lru_cache(maxsize=None)
def table_data():
    """One 8-species model (rc 6) for the whole table, for one predict_batch over every structure."""
    model = make_model(list(EIGHT), [2] * len(EIGHT), 2, 2, rc=6.0, seed=37)
    structs = [case_data(c.name)[1] for c in CASES]
    om = to_oracle(model)
    return model, structs, [o.predict(om, pos, cell, pbc, Z, want_beta=True) for pos, cell, Z, pbc in structs]


def vol(cell):
    return abs(np.linalg.det(cell))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the table reaches what it names; references build
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CASE))
def test_case_reaches_its_branch(name):
    c = CASE[name]
    _, (pos, cell, Z, pbc), plan, (first, J, S), out = case_data(name)
    for key, want in c.expect:
        assert plan[key] == want, (name, key, plan[key], want)
    assert len(pos) <= 1000 and set(np.unique(Z)) == set(c.Zs)
    assert len(J) > 0 and np.isfinite(out["energy"]) and np.isfinite(out["forces"]).all()
    assert np.isfinite(out["beta"]).all() and np.abs(out["forces"]).max() > 0
    if name == "sparse_gas":
        assert (np.diff(first) == 0).sum() > len(Z) // 2           # mostly lone atoms
    if len(Z) < 300:
        fb, Jb, Sb = o.neighbor_list_bruteforce(pos, cell, pbc, c.rc)
        assert np.array_equal(first, fb)
        assert all(np.array_equal(x, y) for x, y in zip(rows_sorted(first, J, S), rows_sorted(fb, Jb, Sb)))


def test_table_covers_the_bin_kernel_branches():
    """Across the table: every NS of the bin kernel, reaches 1-3, several run chunks, several tiles, slots past the
    word, several rounds, merged and unmerged z stencils, merged bins, wraps and clamps."""
    plans = [case_data(c.name)[2] for c in CASES]
    assert {p["NS"] for p in plans} == {1, 2, 4, 8}
    assert {max(p["reach"]) for p in plans} == {1, 2, 3}
    assert max(p["run_chunks"] for p in plans) >= 2 and max(p["tiles"] for p in plans) >= 3
    assert any(p["slots_past_word"] for p in plans) and max(p["rounds"] for p in plans) >= 2
    assert any(p["z_merged"] for p in plans) and any(p["z_unmerged"] for p in plans)
    assert any(p["merges"] for p in plans) and any(p["clamped"] for p in plans) and any(p["wrapped"] for p in plans)


def test_bin_plan_of_the_golden_cells():
    """The restatement reproduces the bin counts the golden cells are known to have (1-9 bins; cluster_lone 1,700)."""
    from golden_util import golden_cases, load_golden

    for n in golden_cases():
        g = load_golden(n)
        k = g["meta"]["kernel"]
        rc = max(kk["rc"] for kk in k["kernels"]) if k["kind"] == "multi" else k["rc"]
        p = bin_plan(g["pos"], g["cell"], g["meta"]["pbc"], rc, len(g["meta"]["species"]))
        assert (p["ncell"] == 1700) if n == "cluster_lone" else (1 <= p["ncell"] <= 9), (n, p["ncell"])


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def engine(model, Zs):
    import autoforce_b200 as ab

    return ab.SgprEngine(model, species=sorted(Zs))


def assert_matches(out, E, Fo, W, cell, N, beta=None, tag=""):
    assert abs(E - out["energy"]) / N < TOL_E, tag
    assert np.abs(Fo - out["forces"]).max() < TOL_F, tag
    assert np.abs(W - out["virial"]).max() / vol(cell) < TOL_SIGMA, tag
    if beta is not None:
        assert np.abs(beta ** 2 - out["beta"] ** 2).max() < TOL_BETA2, tag


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["warp", "bins"])
@pytest.mark.parametrize("name", list(CASE))
def test_neighbor_case(name, mode, monkeypatch):
    """The list (first, rows as sorted sets, species order inside rows) and E / F / W / beta^2 against the oracle."""
    monkeypatch.setenv("SGPR_NL", mode)
    c = CASE[name]
    model, (pos, cell, Z, pbc), _, (f0, J0, S0), out = case_data(name)
    eng = engine(model, c.Zs)
    try:
        first, J, S = eng.neighbors(pos, Z, cell, pbc)
        assert np.array_equal(first, f0)
        assert all(np.array_equal(x, y) for x, y in zip(rows_sorted(first, J, S), rows_sorted(f0, J0, S0)))
        # rows are species-contiguous in ascending species order (the descriptor kernels' per-species runs)
        zj = Z[J].astype(np.int64)
        inner = np.ones(len(J), dtype=bool)
        inner[first[:-1][np.diff(first) > 0]] = False              # first pair of a row may start anywhere
        assert (np.diff(zj, prepend=0)[inner] >= 0).all()
        for _ in range(2):                                         # sizing step, then a warm one
            E, Fo, W, owned, beta = eng.predict(pos, Z, cell, pbc, want_beta=True)
            assert owned.all()
            assert_matches(out, E, Fo, W, cell, len(Z), beta, name)
    finally:
        eng.close()


@pytest.mark.gpu
def test_whole_table_in_one_batch():
    model, structs, refs = table_data()
    atoms = [types.SimpleNamespace(positions=p, numbers=Z, cell=cell, pbc=pbc) for p, cell, Z, pbc in structs]
    eng = engine(model, EIGHT)
    try:
        Eb, Fb, Wb, bb = eng.predict_batch(atoms, want_beta=True)
    finally:
        eng.close()
    a0 = 0
    for b, ((pos, cell, Z, pbc), out) in enumerate(zip(structs, refs)):
        N = len(Z)
        assert_matches(out, Eb[b], Fb[a0:a0 + N], Wb[b], cell, N, bb[a0:a0 + N], CASES[b].name)
        a0 += N


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["warp", "bins"])
@pytest.mark.parametrize("name", BIG)
def test_sharded_case(name, mode, monkeypatch):
    """Halo sharding at world 3 (rank sum) and the fused exchange step at world 2 against the oracle: a shard's first
    and last atoms cut through bins, its halo is marked by the count pass."""
    import torch

    monkeypatch.setenv("SGPR_NL", mode)
    c = CASE[name]
    model, (pos, cell, Z, pbc), _, _, out = case_data(name)
    N = len(Z)
    eng = engine(model, c.Zs)
    try:
        E, Fo, W = 0.0, np.zeros((N, 3)), np.zeros((3, 3))
        count = np.zeros(N, dtype=int)
        for rank in range(3):
            e, f, w, owned = eng.predict(pos, Z, cell, pbc, rank=rank, world=3)
            E, Fo, W = E + e, Fo + f, W + w
            count += owned
        assert np.all(count == 1)
        assert_matches(out, E, Fo, W, cell, N, tag=f"{name} halo")
    finally:
        eng.close()
    world = 2
    dev = torch.device("cuda", 0)
    engines = [engine(model, c.Zs) for _ in range(world)]
    streams = [torch.cuda.Stream(device=dev) for _ in range(world)]
    stride = 3 * N + 8
    blocks = torch.zeros((world, 2 * stride + 2 * world * 16), dtype=torch.float64, device=dev)
    bases = np.array([blocks[r].data_ptr() for r in range(world)], dtype=np.uint64)
    ews = [torch.zeros(10, dtype=torch.float64, device=dev) for _ in range(world)]
    Fs = [torch.zeros((N, 3), dtype=torch.float64, device=dev) for _ in range(world)]
    owns = [torch.zeros(N, dtype=torch.uint8, device=dev) for _ in range(world)]
    pos_t = torch.as_tensor(pos, device=dev)
    z_t = torch.as_tensor(Z.astype(np.int32), device=dev)
    torch.cuda.synchronize()
    try:
        for e in engines:
            e.set_async(True)
        for step in range(2):                                      # sizing step, then a warm one
            for r in range(world):
                with torch.cuda.stream(streams[r]):
                    engines[r].p2p_step(pos_t, z_t, cell, pbc, r, world, bases, ews[r], Fs[r], owns[r])
            torch.cuda.synchronize()
            for e in engines:
                e.check()
            Fsum = sum((Fs[r] * owns[r].to(torch.float64)[:, None] for r in range(world))).cpu().numpy()
            assert bool((sum(o_.to(torch.int32) for o_ in owns) == 1).all())
            ew = ews[0].cpu().numpy()
            assert_matches(out, ew[0], Fsum, ew[1:].reshape(3, 3), cell, N, tag=f"{name} fused step {step}")
    finally:
        for e in engines:
            e.close()


def trajectory(pos0, cell, steps, seed):
    """Positions of a warm trajectory: every atom displaced by up to ~0.35 A around its start, and the layer at x = 0
    moved back and forth across the cell face (its wrap counts change between steps)."""
    rng = np.random.default_rng(seed)
    layer = np.abs((pos0 @ np.linalg.inv(cell))[:, 0]) < 0.02
    out = []
    for k in range(steps):
        p = pos0 + rng.uniform(-0.2, 0.2, pos0.shape)
        p[layer, 0] += 0.3 if k % 2 else -0.4
        out.append(p)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["monolayer", "eight_sp"])
def test_warm_trajectory_through_the_bin_kernel(name, monkeypatch):
    """Sync-free steps (set_async, same buffers: CUDA-graph replay after the first warm step) under the bin kernel while
    atoms move and cross a cell face: every step's E / F against the oracle, check() clean."""
    import torch

    monkeypatch.setenv("SGPR_NL", "bins")
    c = CASE[name]
    model, (pos0, cell, Z, pbc), _, _, _ = case_data(name)
    om = to_oracle(model)
    N = len(Z)
    dev = torch.device("cuda", 0)
    eng = engine(model, c.Zs)
    eng.set_async(True)
    pos_t = torch.empty((N, 3), dtype=torch.float64, device=dev)
    z_t = torch.as_tensor(Z.astype(np.int32), device=dev)
    res = (torch.empty(1, dtype=torch.float64, device=dev), torch.empty((N, 3), dtype=torch.float64, device=dev),
           torch.empty(9, dtype=torch.float64, device=dev))
    outside = set()
    try:
        for k, p in enumerate(trajectory(pos0, cell, 10, 3)):
            outside.add(int((p[:, 0] < 0).sum()))
            pos_t.copy_(torch.as_tensor(p))
            E, Fo, W = eng.predict_device(pos_t, z_t, cell, pbc, out=res)
            torch.cuda.synchronize()
            eng.check()
            out = o.predict(om, p, cell, pbc, Z)
            assert_matches(out, float(E.item()), Fo.cpu().numpy(), W.cpu().numpy().reshape(3, 3), cell, N, tag=f"{name} {k}")
    finally:
        eng.close()
    assert len(outside) > 1                                        # wrap counts changed between warm steps


def launched_neighbor_kernels(fn):
    """(kernel, NS) of every neighbour-search launch recorded by torch.profiler while fn() runs, and the grids of the
    block-per-bin launches when the trace records them."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    found = set()
    for e in prof.events():
        m = re.search(r"neighbor_bin_kernel<(\d+)>", e.name)
        if m:
            found.add(("bins", int(m.group(1))))
        m = re.search(r"neighbor_kernel<\s*(true|false)\s*,\s*(\d+)\s*,\s*(true|false)\s*>", e.name)
        if m:
            found.add(("warp" if m.group(3) == "false" else "warp-batch", int(m.group(2))))
    grids = set()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as fh:
            trace = json.load(fh)
    for ev in trace.get("traceEvents", []):
        if "neighbor_bin_kernel" in str(ev.get("name", "")) and "grid" in ev.get("args", {}):
            grids.add(tuple(ev["args"]["grid"]))
    return found, grids


@pytest.mark.gpu
def test_case_table_matches_dispatch(monkeypatch):
    """Every row launches the kernel bin_plan names in the automatic mode, with its NS; forced modes launch theirs; the
    bin kernel's grid is bin_plan's bin count."""
    seen = set()
    for c in CASES:
        model, (pos, cell, Z, pbc), plan, _, _ = case_data(c.name)
        for mode in (None, "warp", "bins"):
            if mode is None:
                monkeypatch.delenv("SGPR_NL", raising=False)
            else:
                monkeypatch.setenv("SGPR_NL", mode)
            box = {}

            def run():
                box["eng"] = eng = engine(model, c.Zs)
                eng.predict(pos, Z, cell, pbc)

            try:
                found, grids = launched_neighbor_kernels(run)
            finally:
                if "eng" in box:
                    box["eng"].close()
            want = mode or plan["kernel"]
            assert found == {(want, plan["NS"])}, (c.name, mode, found)
            if want == "bins":
                seen.add(plan["NS"])
                if grids:
                    assert grids == {(plan["ncell"], 1, 1)}, (c.name, grids)
    assert seen == {1, 2, 4, 8}
