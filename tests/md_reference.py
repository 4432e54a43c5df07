"""Host restatements used by the MD tests: the Langevin noise stream of sgpr_math.cuh (Philox4x32-10 + Box-Muller) in
numpy, and the velocity-Verlet / BAOAB loops around ``SgprEngine.predict`` in the operation order of the device
integrators (ASE's ``VelocityVerlet.step`` for NVE)."""
import numpy as np

FS = 0.09822694788464063
KB = 8.617330337217213e-05
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, k0, k1):
    """ctr: 4 arrays of uint32 counters (broadcast together); returns the 4 output words as uint64 arrays."""
    c = [np.asarray(x, dtype=np.uint64) for x in ctr]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(0x9E3779B9)) & _MASK
            k1 = (k1 + np.uint64(0xBB67AE85)) & _MASK
        p0, p1 = m0 * c[0], m1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
    return c


def _uniform(lo, hi):
    x = (hi << np.uint64(32)) | lo
    return ((x >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def langevin_normals(seed, n_atoms, step):
    """[n_atoms, 3] standard normals of the O step of global step ``step`` (steps done before it)."""
    seed, step = int(seed), int(step)
    atom = np.arange(n_atoms, dtype=np.uint64)
    xi = np.empty((n_atoms, 3))
    for call in (0, 1):
        c = philox4x32_10([atom, call, step & 0xFFFFFFFF, step >> 32], seed & 0xFFFFFFFF, seed >> 32)
        u0, u1 = _uniform(c[0], c[1]), _uniform(c[2], c[3])
        rad = np.sqrt(-2.0 * np.log(u0))
        if call == 0:
            xi[:, 0] = rad * np.cos(2.0 * np.pi * u1)
            xi[:, 1] = rad * np.sin(2.0 * np.pi * u1)
        else:
            xi[:, 2] = rad * np.cos(2.0 * np.pi * u1)
    return xi


def host_md(eng, pos, numbers, cell, pbc, masses, mom, n_steps, timestep, temperature_K=None, friction=None, seed=0,
            covloss=False, ediff=np.inf):
    """Host loop: returns (pos, mom, F, beta, thermo rows [n, 11], steps done, stop step or None).  Stops after the
    first step (0 = the starting structure) with max(beta) > ediff, like the device driver."""
    dt = timestep * FS
    h = 0.5 * dt
    m = np.asarray(masses, dtype=np.float64)[:, None]
    r, p = np.array(pos, dtype=np.float64), np.array(mom, dtype=np.float64)

    def evaluate(x):
        if covloss:
            E, F, W, _, beta = eng.predict(x, numbers, cell, pbc, want_beta=True)
            return E, F.copy(), W, beta.copy()
        E, F, W, _ = eng.predict(x, numbers, cell, pbc)
        return E, F.copy(), W, None

    E, F, W, beta = evaluate(r)
    if covloss and np.max(beta) > ediff:
        return r, p, F, beta, np.zeros((0, 11)), 0, 0
    langevin = temperature_K is not None
    if langevin:
        gamma = friction / FS
        c1 = np.exp(-gamma * dt)
        c2 = np.sqrt(1.0 - c1 * c1)
        kT = KB * temperature_K
    rows = []
    for step in range(n_steps):
        p = p + h * F
        if not langevin:
            r = r + dt * p / m
        else:
            r = r + h * p / m
            p = c1 * p + (c2 * np.sqrt(m * kT)) * langevin_normals(seed, len(r), step)
            r = r + h * p / m
        E, F, W, beta = evaluate(r)
        p = p + h * F
        rows.append(np.concatenate([[E, 0.5 * np.sum(p * p / m)], np.asarray(W).reshape(9)]))
        if covloss and np.max(beta) > ediff:
            return r, p, F, beta, np.array(rows), step + 1, step + 1
    return r, p, F, beta, np.array(rows).reshape(-1, 11), n_steps, None
