"""Covloss (beta, calculator/active.py:781-804) against the float64 oracle where the int8 path can lose accuracy.

beta decides what the on-the-fly learner samples and stops DeviceMD / DeviceRelax.  On tcgen05 it runs through int8
digit slicing (i8gemm.cu): Epi1T writes the digits of K = k^xi, the covloss GEMM multiplies them with the digits of the
choli rows (each row divided by its power-of-two bound, row_pow2_kernel), Epi3 sums squares of 16 columns and
beta_finish_kernel (api.cu) adds the partials and divides by the self kernel.  The synthetic models elsewhere have
choli = 0.5 I + noise, one row scale and no cancellation; ROWS below name what each row reaches instead.

The digits of q_hat and K are absolute steps of 2^-46, while c / alpha needs K relative to |q_hat|^xi: an environment
whose every neighbour sits close to rc has |p| ~ eps, |q_hat| = |p| / (|p| + eps) << 1 and alpha << 1.  beta_finish_kernel
therefore hands normalised rows with |p| < 2^-40 to beta_fp64_rows_kernel, which finishes them in float64 from the
descriptor rows (fp64_rows() restates the rule).

emulate_beta2() restates that arithmetic with exact integers from a float64 K, and emulation_bound() bounds its distance
from exact arithmetic per row (see there).  The CPU tests check, for every row, that the emulation is within that bound
of the oracle and that the bound is below the suite's 1e-9.  On the GPU every row must match the oracle at 1e-9 on
tcgen05 and at 1e-12 on the FP64 DMMA path; the tcgen05 beta^2 must also match the emulation within the same bound
taken with one whole digit step per K entry (plus the kernel-matrix GEMM's error on K).
"""
import functools
import types
from dataclasses import dataclass
from fractions import Fraction

import numpy as np
import pytest

from autoforce_b200.model import SgprModel
from autoforce_b200.synth import cut_environments, fcc
from oracle import sgpr_oracle as o
from oracle_engine import to_oracle
from test_gpu_neighbor_cases import case_data as neighbor_case
from test_gpu_variants import make_model, structure

# DESIGN.md section 2
TOL_E, TOL_F, TOL_BETA2, TOL_BETA2_DMMA = 1e-9, 1e-8, 1e-9, 1e-12

# i8gemm.cu
NS, TR, BN = 6, 8, 64           # digits per operand, covloss slice pairs t + u <= TR, output tile columns
DIGIT = 2.0 ** -46              # step of rint(x 2^(8 NS - 2)) (digit_bytes<6>)
EPS = np.finfo(float).eps       # the descriptors' q = p / (|p| + eps)
TOL_K1 = 1e-12                  # kernel-matrix GEMM (TR = 7) on q_hat . z_hat (i8gemm_kernel.cuh header)
COV_FP64_NORM = 2.0 ** -40      # api.cu kCovFp64Norm: normalised rows with |p| below it are finished in float64


# ------------------------------------------------------------------------------------------------------------------
# the int8 covloss arithmetic in exact integers
# ------------------------------------------------------------------------------------------------------------------
def digits(x):
    """digit_bytes<6>: balanced base-256 digits of v = rint(x 2^46) (round half to even), most significant first:
    v = sum_t d[t] 256^(5 - t), d in [-128, 127]."""
    v = np.rint(np.asarray(x, dtype=float) * 2.0 ** 46).astype(np.int64)
    d = np.zeros((NS,) + v.shape, dtype=np.int64)
    for t in range(NS - 1, -1, -1):
        r = ((v + 128) & 255) - 128
        d[t] = r
        v = (v - r) >> 8
    assert not v.any()
    return d


def row_pow2(X):
    """row_pow2_kernel: the power of two >= max |row| (frexp exponent), 1 for an all-zero row."""
    m = np.abs(X).max(axis=1) if X.shape[1] else np.zeros(len(X))
    _, e = np.frexp(m)
    return np.where(m > 0, np.ldexp(1.0, e), 1.0)


def sliced_product(Kd, Cd):
    """Slice products with t + u <= TR (t, u = 1..NS) combined exactly and rounded once (combine_groups):
    T = sum_g acc_g 256^(NG - 1 - g), result T 2^-(8 (NG - 1) + 12), NG = TR - 1."""
    NG = TR - 1
    T = np.zeros((Kd.shape[1], Cd.shape[1]), dtype=object)
    for g in range(NG):
        acc = np.zeros(T.shape, dtype=np.int64)
        for t in range(1, NS + 1):
            u = g + 2 - t
            if 1 <= u <= NS:
                acc += Kd[t - 1] @ Cd[u - 1].T
        T = T + acc.astype(object) * 256 ** (NG - 1 - g)
    sc = 2.0 ** -(8 * (NG - 1) + 12)
    return np.array([float(x) for x in T.ravel()], dtype=float).reshape(T.shape) * sc


def fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def sorted_blocks(model, species):
    """The engine's inducing order: grouped by central species (species table order), caller's order inside."""
    sp = np.array([species.index(int(z)) for z in model.ind_Z], dtype=np.int64)
    perm = np.argsort(sp, kind="stable")
    first = np.searchsorted(sp[perm], np.arange(len(species) + 1))
    return perm, first


def emulate_c(model, species, K, numbers, lone_c):
    """c_i = sum_k b_ik^2 of the tcgen05 path before the division by the self kernel, from the float64 K [N, M] (caller's
    column order); NaN marks rows the GEMM does not produce (lone atoms, species without usable inducing LCEs)."""
    M = model.M
    choli = np.asarray(model.choli, dtype=float)
    perm, mf = sorted_blocks(model, species)
    n_part = -(-M // BN) * (BN // 16)
    c = np.full(len(numbers), np.nan)
    for s, z in enumerate(species):
        cols = perm[mf[s]:mf[s + 1]]
        rows = np.nonzero((numbers == z) & ~lone_c)[0]
        if len(cols) == 0 or len(rows) == 0 or not model.is_centre(z):
            continue
        Ct = choli[:, cols]                                   # choli_t of species s: rows k, columns p
        rs = row_pow2(Ct)
        v = sliced_product(digits(K[np.ix_(rows, cols)]), digits(Ct / rs[:, None]))
        t = v * rs[None, :]                                   # Epi3: times the row scale of output column k (exact)
        part = np.zeros((len(rows), n_part))
        for r in range(len(rows)):
            for p in range(n_part):
                acc = 0.0
                for k in range(16 * p, min(16 * p + 16, M)):
                    acc = fma(t[r, k], t[r, k], acc)
                part[r, p] = acc
        cc = np.zeros(len(rows))
        for p in range(n_part):                               # beta_finish_kernel: partials in order
            cc = cc + part[:, p]
        c[rows] = cc
    return c


def fp64_rows(model, lone_c, alpha):
    """Rows beta_finish_kernel hands to beta_fp64_rows_kernel: normalised, not lone, |p| < 2^-40, with |p| from the
    self kernel alpha = |q_hat|^(2 xi), |q_hat| = |p| / (|p| + eps)."""
    q = np.asarray(alpha, dtype=float) ** (1.0 / (2.0 * float(model.xi)))
    with np.errstate(divide="ignore", invalid="ignore"):
        p = np.where(q < 1.0, EPS * q / (1.0 - q), np.inf)
    return bool(model.normalize) & ~np.asarray(lone_c) & (p < COV_FP64_NORM)


def emulate_beta2(model, species, K, numbers, lone_c, alpha):
    """beta^2 of the tcgen05 path (beta_finish_kernel): c / alpha, the lone atoms' constant, NaN for excluded centres;
    the rows of fp64_rows() in float64 (beta_fp64_rows_kernel)."""
    numbers = np.asarray(numbers)
    c = emulate_c(model, species, K, numbers, lone_c)
    fp64 = fp64_rows(model, lone_c, alpha)
    c64 = ((np.asarray(model.choli, dtype=float) @ K.T) ** 2).sum(axis=0)
    perm, mf = sorted_blocks(model, species)
    lone_m = np.array([model.ind_first[m + 1] == model.ind_first[m] for m in range(model.M)], dtype=bool)
    choli = np.asarray(model.choli, dtype=float)
    lw = max(model.lone_weight, 0.0)
    out = np.zeros(len(numbers))
    for i, z in enumerate(numbers):
        s = species.index(int(z))
        if lone_c[i]:
            cols = [m for m in perm[mf[s]:mf[s + 1]] if lone_m[m]]
            cc = sum(lw * float(choli[k, cols].sum()) ** 2 for k in range(model.M)) if cols else 0.0
        elif not model.is_centre(z):
            out[i] = np.nan
            continue
        elif np.isnan(c[i]):
            cc = 0.0                                          # sp_on = 0: no inducing LCE of this species
        elif fp64[i]:
            cc = c64[i] / alpha[i]
        else:
            cc = c[i] / alpha[i]
        out[i] = max(1.0 - cc, 0.0) * model.vscale.get(int(z), np.inf)
    return out


def emulation_bound(model, species, K, numbers, lone_c, alpha, dK=None):
    """Per-row bound on |beta^2 of the int8 scheme - exact beta^2|.  With b_k = sum_p L_kp K_p:
      K digits   : rint(K 2^46) moves an entry by at most half a step, and by no more than |K| (dK given: that per entry)
      choli      : rint(L_kp / rs_k 2^46) moves L_kp by at most rs_k 2^-47
      dropped    : the pairs t + u > 8 weigh at most 2^-52 rs_k |K_p| per term (none where K's digits are all zero);
                   the single rounding of v at most |b_k| 2^-53
    so |db_k| <= sum_p |L_kp| dK_p + rs_k (2^-47 + 2^-52) |K_p| + |b_k| 2^-53, |dc| <= sum_k 2 |b_k| db_k + db_k^2 plus the
    float64 sums of squares ((M + parts) 2^-53 c), and beta^2 = 1 - c / alpha adds the rounding of alpha (2 xi 2^-51
    relative, and 2 xi 2^-105 / |p| from recovering |p| = (|p| + eps) - eps, at most 2 xi 2^-65 above 2^-40).  The rows of
    fp64_rows() are float64 evaluations of the oracle's own formula: their bound is the FP64 bar, 1e-12."""
    numbers = np.asarray(numbers)
    choli = np.asarray(model.choli, dtype=float)
    perm, mf = sorted_blocks(model, species)
    M = model.M
    xi = float(model.xi)
    bound = np.zeros(len(numbers))
    for s, z in enumerate(species):
        cols = perm[mf[s]:mf[s + 1]]
        rows = np.nonzero((numbers == z) & ~lone_c)[0]
        if len(cols) == 0 or len(rows) == 0 or not model.is_centre(z):
            continue
        Ct = choli[:, cols]
        rs = row_pow2(Ct)
        Kr = np.abs(K[np.ix_(rows, cols)])
        dKr = np.minimum(Kr, DIGIT / 2) if dK is None else dK[np.ix_(rows, cols)]
        b = np.abs(K[np.ix_(rows, cols)] @ Ct.T)
        db = dKr @ np.abs(Ct).T + Kr.sum(axis=1)[:, None] * rs[None, :] * (2.0 ** -47 + 2.0 ** -52) + b * 2.0 ** -53
        c = (b * b).sum(axis=1)
        dc = (2 * b * db + db * db).sum(axis=1) + c * (M + -(-M // BN) * 4) * 2.0 ** -53
        a = alpha[rows]
        q = a ** (1.0 / (2 * xi))                             # |q_hat|
        with np.errstate(divide="ignore"):
            p = np.where(q < 1.0, EPS * q / np.maximum(1.0 - q, 1e-300), np.inf)
        rel_alpha = 2 * xi * (2.0 ** -51 + 2.0 ** -105 / p) if model.normalize else 0.0
        bound[rows] = (dc / a + c / a * rel_alpha) * model.vscale.get(int(z), 1.0)
    return np.where(fp64_rows(model, lone_c, alpha), TOL_BETA2_DMMA, bound)


# ------------------------------------------------------------------------------------------------------------------
# models and structures
# ------------------------------------------------------------------------------------------------------------------
def model_like(model, envs=None, **kw):
    """A copy of `model` with other inducing LCEs / weights / flags."""
    base = dict(mu=model.mu, mean_w=model.mean_w, vscale=model.vscale, choli=model.choli, lmax=model.lmax, nmax=model.nmax,
                xi=model.xi, rc=model.rc, kind=model.kind, radii=model.radii, default_radius=model.default_radius,
                normalize=model.normalize, a_not=model.a_not)
    base.update(kw)
    if envs is None:
        f = model.ind_first
        envs = [(int(model.ind_Z[m]), model.ind_r[f[m]:f[m + 1]], model.ind_b[f[m]:f[m + 1]]) for m in range(model.M)]
    return SgprModel.from_envs(envs, **base)


def real_choli(model, jitter, species):
    """choli = inv(cholesky(Kmm + jitter I)) with Kmm the oracle's kernel of the model's own inducing LCEs
    (regression/gppotential.py:588)."""
    om = to_oracle(model_like(model, choli=np.eye(model.M)))
    Zh, lone_m = o.inducing_descriptors(om, np.asarray(species))
    Kmm, _, _ = o.kernel_from_descriptors(om, Zh, np.asarray(model.ind_Z, dtype=np.int64), lone_m, Zh, lone_m)
    L = np.linalg.cholesky(Kmm + jitter * np.eye(model.M))
    return np.linalg.inv(L)


def dimers(Zs, rc, seed, n=12, box=60.0):
    """Isolated pairs at separations stepped towards rc (down to rc (1 - 1e-4)): each atom has one neighbour, whose
    cutoff weight and hence |p| fall by orders of magnitude along the table, and K falls past 2^-47."""
    rng = np.random.default_rng(seed)
    gaps = rc * (1.0 - np.geomspace(0.6, 1e-4, n))
    pos, Z = [], []
    g = int(np.ceil(n ** (1 / 3)))
    for k, d in enumerate(gaps):
        c0 = (np.array([k % g, (k // g) % g, k // (g * g)]) + 0.5) * box / g
        u = rng.normal(size=3)
        u /= np.linalg.norm(u)
        pos += [c0 - 0.5 * d * u, c0 + 0.5 * d * u]
        Z += [Zs[k % len(Zs)], Zs[(k + 1) % len(Zs)]]
    return np.array(pos), np.eye(3) * box, np.array(Z, dtype=np.int32), (True, True, True)


def with_lone_atoms(s, Zs, gap=30.0):
    """Structure s plus one isolated atom per species of Zs, stacked `gap` apart beyond the cell along an open z."""
    pos, cell, Z, pbc = s
    cell = np.array(cell, dtype=float)
    extra = np.array([[1.0, 1.0, pos[:, 2].max() + gap * (k + 1)] for k in range(len(Zs))])
    return np.vstack([pos, extra]), cell, np.concatenate([Z, np.asarray(Zs, dtype=np.int32)]), (True, True, False)


@dataclass(frozen=True)
class Row:
    name: str
    reaches: str
    build: object          # () -> (model, [structures], species)


def _sparse_gas():
    model, s, _, _, _ = neighbor_case("sparse_gas")
    return model, [s], sorted(set(int(z) for z in model.ind_Z) | set(int(z) for z in s[2]))


def _real(jitter):
    def b():
        Zs = [29, 47]
        m = make_model(Zs, [24, 20], 2, 2, seed=41)
        m = model_like(m, choli=real_choli(m, jitter, Zs))
        return m, [structure((2, 2, 2), Zs, 3)], Zs
    return b


def _c_to_1():
    Zs = [29, 47]
    m = make_model(Zs, [36, 28], 2, 2, seed=43)
    m = model_like(m, choli=real_choli(m, 1e-8, Zs))
    pos, cell, numbers = fcc(5, Zs, 0.15, 43 + 100)          # make_model's source cell: the inducing LCEs are its atoms
    return m, [(pos, cell, numbers.astype(np.int32), (True, True, True))], Zs


def _clamp():
    """c_to_1 with choli scaled by 1.001: c / alpha = 1.002 on the atoms that coincide with inducing LCEs."""
    m, structs, Zs = _c_to_1()
    return model_like(m, choli=1.001 * np.asarray(m.choli)), structs, Zs


def _dimers(xi):
    def b():
        Zs = [29, 47]
        m = make_model(Zs, [10, 8], 2, 2, xi=xi, seed=47)
        m = model_like(m, choli=real_choli(m, 1e-5, Zs))
        return m, [dimers(Zs, m.rc, 5), structure((2, 2, 2), Zs, 6)], Zs
    return b


def _species_edges():
    """Two species interleaved in the caller's order (64 of species 8 first, then 8 / 29 alternating), M = 131: after
    the species sort species 8 has 74 columns (crossing the 64-column tile) and species 29's first 64 output columns
    are identically zero (cov_nk = 0).  Species 47's only inducing LCE is lone (the clone path); 13 has no inducing
    LCEs (sp_on = 0); 15 is an excluded centre (a_not: NaN, as the reference).  Lone atoms of 8 (a lone inducing LCE
    of 8 exists), 29 (none) and 47 (its clone)."""
    rc = 4.5
    Zsrc = [8, 29]
    pos, cell, numbers = fcc(5, Zsrc, 0.15, 149)
    first, J, S = o.neighbor_list(pos, cell, True, rc)
    rng = np.random.default_rng(149)
    i8 = rng.choice(np.nonzero(numbers == 8)[0], 73, replace=False)
    i29 = rng.choice(np.nonzero(numbers == 29)[0], 56, replace=False)
    order = list(i8[:64]) + [x for pair in zip(i29[:9], i8[64:73]) for x in pair] + list(i29[9:])
    envs = cut_environments(pos, cell, True, numbers, rc, order, first, J, S)
    envs.insert(70, (8, np.zeros((0, 3)), np.zeros(0, np.int32)))
    envs.append((47, np.zeros((0, 3)), np.zeros(0, np.int32)))
    M = len(envs)
    Zs = [8, 13, 15, 29, 47]
    base = make_model([29], [3], 2, 2, seed=0)
    m = model_like(base, envs=envs, mu=np.random.default_rng(5).normal(0, 0.1, M), mean_w={z: -3.0 for z in Zs},
                   vscale={z: 1.0 + 0.25 * k for k, z in enumerate(Zs)}, choli=np.eye(M), a_not=(15,), rc=rc)
    m = model_like(m, choli=real_choli(m, 1e-5, Zs))
    s = with_lone_atoms(structure((2, 2, 2), Zs[:4], 8, counts=(10, 6, 6, 10)), [8, 29, 47])
    return m, [s], Zs


def _unnormalised():
    Zs = [29, 47]
    m = make_model(Zs, [12, 12], 2, 2, seed=53)
    m = model_like(m, normalize=False)
    m = model_like(m, choli=real_choli(m, 1e-5, Zs))
    return m, [structure((2, 2, 2), Zs, 7), dimers(Zs, m.rc, 9, n=8)], Zs


ROWS = [
    Row("sparse_gas", "the neighbour table's row: single neighbours near rc, |p| ~ eps, self kernels alpha << 1",
        _sparse_gas),
    Row("real_1e-2", "choli = L^-1 of Kmm + 1e-2 I: per-row scales, entries > 1", _real(1e-2)),
    Row("real_1e-5", "choli = L^-1 of Kmm + 1e-5 I: row scales over many powers of two, cancellation in b", _real(1e-5)),
    Row("real_1e-8", "choli = L^-1 of Kmm + 1e-8 I: entries >> 1, the largest cancellation", _real(1e-8)),
    Row("c_to_1", "atoms = inducing LCEs under a real choli: c -> 1, cancellation in 1 - c down to the jitter", _c_to_1),
    Row("clamp", "c_to_1 with choli x 1.001: c / alpha > 1, the fmax(1 - c, 0) clamp", _clamp),
] + [
    Row(f"dimers_xi{xi:g}", "one neighbour stepped towards rc, unlike the inducing set: K from 1e-1 past 2^-47"
        + (", pow() branch of Epi1T<0>" if xi != int(xi) else ""), _dimers(xi)) for xi in (1, 2, 3, 4, 5, 2.5)
] + [
    Row("species_edges", "interleaved species, M = 131, cov_nk = 0 tile, clone path, sp_on = 0, a_not, lone atoms",
        _species_edges),
    Row("unnormalised", "un-normalised model (DMMA only): c / (p.p)^xi with rows of small norm", _unnormalised),
]
ROW = {r.name: r for r in ROWS}


@functools.lru_cache(maxsize=None)
def row_data(name):
    """Model, species, structures and, per structure, the oracle output (with K and alpha) and the lone mask."""
    model, structs, species = ROW[name].build()
    om = to_oracle(model)
    refs = []
    for pos, cell, Z, pbc in structs:
        out = o.predict(om, pos, cell, pbc, Z, want_K=True, want_beta=True)
        out["lone"] = np.diff(out["first"]) == 0
        refs.append(out)
    return model, list(species), structs, refs


def beta2_oracle(out):
    return out["beta"] ** 2


def q_hat(model, out):
    """|q_hat| per atom from the oracle's self kernel alpha = (q_hat . q_hat)^xi (1 for lone atoms)."""
    return out["alpha"] ** (1.0 / (2.0 * float(model.xi)))


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(ROW))
def test_emulation_within_its_bound_of_the_oracle(name):
    """The int8 scheme restated in exact integers is within its derived per-row bound of the float64 oracle, and the
    bound is below the suite's beta^2 bar on every row."""
    model, species, structs, refs = row_data(name)
    for (pos, cell, Z, pbc), out in zip(structs, refs):
        b2 = emulate_beta2(model, species, out["K"], Z, out["lone"], out["alpha"])
        ref = beta2_oracle(out)
        assert np.array_equal(np.isnan(b2), np.isnan(ref)), name
        ok = ~np.isnan(ref)
        bound = emulation_bound(model, species, out["K"], Z, out["lone"], out["alpha"])[ok]
        err = np.abs(b2[ok] - ref[ok])
        assert (err <= bound + 4 * EPS).all(), (name, float(err.max()), float(bound[np.argmax(err - bound)]))
        if model.normalize:
            assert bound.max(initial=0.0) < TOL_BETA2, (name, float(bound.max(initial=0.0)))


@pytest.mark.parametrize("name", list(ROW))
def test_row_reaches_what_it_names(name):
    model, species, structs, refs = row_data(name)
    K = np.concatenate([r["K"] for r in refs])
    alpha = np.concatenate([r["alpha"] for r in refs])
    b2 = np.concatenate([beta2_oracle(r) for r in refs])
    lone = np.concatenate([r["lone"] for r in refs])
    if name.startswith("real_") or name in ("c_to_1", "clamp"):
        rs = row_pow2(np.asarray(model.choli))
        assert np.log2(rs).max() - np.log2(rs).min() >= 2 and np.abs(model.choli).max() > 1.0
    if name == "c_to_1":
        assert 0.0 < np.nanmin(b2) < 1e-7                                    # 1 - c cancels down to the jitter
    if name == "clamp":
        c = np.concatenate([((np.asarray(model.choli) @ r["K"].T) ** 2).sum(axis=0) / r["alpha"] for r in refs])
        assert c.max() > 1.0 + 1e-4 and (b2 == 0.0).any() and (b2 > 1e-3).any()
    if name == "sparse_gas":
        assert alpha[~lone].min() < 1e-20
    if name.startswith("dimers"):
        k = np.abs(K[K != 0])
        assert k.max() > 1e-1 and k.min() < (2.0 ** -47 if model.xi > 1 else 1e-7), (k.max(), k.min())
        q = np.concatenate([q_hat(model, r) for r in refs])
        fp64 = fp64_rows(model, lone, alpha)
        assert q.min() < 1e-5 and fp64.any() and (~fp64 & ~lone & (q < 1.0 - 1e-12)).any()
    if name == "species_edges":
        perm, mf = sorted_blocks(model, species)
        Ct = np.asarray(model.choli)[:, perm[mf[3]:mf[4]]]                   # species 29
        assert model.M > 64 and mf[1] - mf[0] > 64 and not Ct[:64].any()
        Z = np.concatenate([s[2] for s in structs])
        assert np.isnan(b2[Z == 15]).all() and np.allclose(b2[(Z == 13) & ~lone], model.vscale[13], rtol=1e-15)
        assert lone[Z == 8].any() and lone[Z == 29].any() and lone[Z == 47].any()
    if name == "unnormalised":
        assert not model.normalize and alpha[~lone].min() < 1e-6


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def set_engine(monkeypatch, engine):
    if engine == "dmma":
        monkeypatch.setenv("SGPR_GEMM", "dmma")
    else:
        monkeypatch.delenv("SGPR_GEMM", raising=False)


def check_beta2(beta, out, model, species, Z, engine, tag, owned=None):
    b2 = beta ** 2
    ref = beta2_oracle(out)
    sel = np.ones(len(Z), bool) if owned is None else owned
    assert np.array_equal(np.isnan(b2[sel]), np.isnan(ref[sel])), tag
    ok = sel & ~np.isnan(ref)
    tol = TOL_BETA2_DMMA if (engine == "dmma" or not model.normalize) else TOL_BETA2
    err = np.abs(b2[ok] - ref[ok])
    assert err.max(initial=0.0) < tol, (tag, float(err.max(initial=0.0)))
    if engine == "i8" and model.normalize:
        # the tcgen05 path against its own restatement: one digit step per K entry plus the kernel-matrix GEMM's error
        K = out["K"]
        xi = float(model.xi)
        kk = np.abs(K) ** (1.0 / xi)
        dK = DIGIT + xi * kk ** (xi - 1) * TOL_K1
        emu = emulate_beta2(model, species, K, Z, out["lone"], out["alpha"])
        bound = emulation_bound(model, species, K, Z, out["lone"], out["alpha"], dK=dK)
        bound = bound + emulation_bound(model, species, K, Z, out["lone"], out["alpha"])
        d = np.abs(b2[ok] - emu[ok])
        assert (d <= bound[ok] + 4 * EPS).all(), (tag, float(d.max()))


def gpu_engine(model, species):
    import autoforce_b200 as ab

    return ab.SgprEngine(model, species=list(species))


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["i8", "dmma"])
@pytest.mark.parametrize("name", list(ROW))
def test_covloss_row(name, engine, monkeypatch):
    """predict (sizing step, then a warm one) and one predict_batch over the row's structures: beta^2 and NaN placement
    against the oracle (tcgen05 also against the emulation, DMMA at 1e-12); E and F at the usual bars."""
    set_engine(monkeypatch, engine)
    model, species, structs, refs = row_data(name)
    eng = gpu_engine(model, species)
    try:
        for k, ((pos, cell, Z, pbc), out) in enumerate(zip(structs, refs)):
            for step in range(2):
                E, Fo, W, owned, beta = eng.predict(pos, Z, cell, pbc, want_beta=True)
                assert owned.all()
                assert abs(E - out["energy"]) / len(Z) < TOL_E and np.abs(Fo - out["forces"]).max() < TOL_F
                check_beta2(beta, out, model, species, Z, engine, f"{name} {engine} structure {k} step {step}")
        atoms = [types.SimpleNamespace(positions=p, numbers=Z, cell=cell, pbc=pbc) for p, cell, Z, pbc in structs]
        _, _, _, bb = eng.predict_batch(atoms, want_beta=True)
        a0 = 0
        for k, ((pos, cell, Z, pbc), out) in enumerate(zip(structs, refs)):
            check_beta2(bb[a0:a0 + len(Z)], out, model, species, Z, engine, f"{name} {engine} batch {k}")
            a0 += len(Z)
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["i8", "dmma"])
def test_covloss_halo_sharded(engine, monkeypatch):
    """sparse_gas (bins merged, 3,456 of them) sharded at world 3: beta_finish of the owned rows only (active / owned)."""
    set_engine(monkeypatch, engine)
    model, species, structs, refs = row_data("sparse_gas")
    (pos, cell, Z, pbc), out = structs[0], refs[0]
    eng = gpu_engine(model, species)
    try:
        count = np.zeros(len(Z), dtype=int)
        for rank in range(3):
            _, _, _, owned, beta = eng.predict(pos, Z, cell, pbc, rank=rank, world=3, want_beta=True)
            count += owned
            check_beta2(beta, out, model, species, Z, engine, f"sparse_gas {engine} rank {rank}", owned=owned)
        assert (count == 1).all()
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["i8", "dmma"])
def test_covloss_live_updates(engine, monkeypatch):
    """A warm engine (graph replay) under choli 0.5 I, then set_weights(choli = L^-1), then append_inducing with a new
    choli: each against the oracle of the updated model.  Changing choli reruns i8_prepare_covloss, cov_nk and the
    cached problem descriptors."""
    import torch

    set_engine(monkeypatch, engine)
    Zs = [29, 47]
    model = make_model(Zs, [24, 20], 2, 2, seed=59)
    pos, cell, Z, pbc = structure((2, 2, 2), Zs, 4)
    eng = gpu_engine(model, Zs)

    def check(m, tag):
        out = o.predict(to_oracle(m), pos, cell, pbc, Z, want_K=True, want_beta=True)
        out["lone"] = np.diff(out["first"]) == 0
        for step in range(3):                                       # sizing step, then warm ones (graph replay)
            _, _, _, _, beta = eng.predict(pos, Z, cell, pbc, want_beta=True)
            check_beta2(beta, out, m, Zs, Z, engine, f"{tag} {engine} step {step}")

    try:
        check(model, "choli 0.5 I")
        eng.set_weights(choli=real_choli(model, 1e-5, Zs))
        check(eng.model, "set_weights(L^-1)")
        src, scell, snum = fcc(5, Zs, 0.15, 61)
        first, J, S = o.neighbor_list(src, scell, True, model.rc)
        new = cut_environments(src, scell, True, snum, model.rc, [0, 1, 2, 3, 4], first, J, S)
        f = model.ind_first
        old = [(int(model.ind_Z[m]), model.ind_r[f[m]:f[m + 1]], model.ind_b[f[m]:f[m + 1]]) for m in range(model.M)]
        mu = np.concatenate([model.mu, np.full(len(new), 0.05)])
        grown = model_like(model, envs=old + new, mu=mu, choli=np.eye(model.M + len(new)))
        eng.append_inducing(new, mu, choli=real_choli(grown, 1e-5, Zs))
        assert eng.model.M == grown.M
        check(eng.model, "append_inducing")
    finally:
        eng.close()
