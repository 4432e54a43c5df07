"""Host restatement used by the relaxation tests: ASE's FIRE (ase/optimize/fire.py, downhill_check=False) around
``SgprEngine.predict``, in the operation order of the device kernels (relax.cu), with ASE's convergence test and the
forces of fixed atoms zeroed before every use (FixAtoms through get_forces())."""
import numpy as np

FIRE_DEFAULTS = dict(dt=0.1, maxstep=0.2, dtmax=1.0, Nmin=5, finc=1.1, fdec=0.5, astart=0.1, fa=0.99, a=0.1)


def host_fire(eng, pos, numbers, cell, pbc, n_steps, fmax=0.0, fixed=None, covloss=False, ediff=np.inf, **fire):
    """Up to ``n_steps`` FIRE steps; stops at the first structure (0 = the start) with max_i |F_i| < fmax or, with
    covloss, max(beta) > ediff.  Returns a dict: pos, vel, F, beta, rows [n, 13] {E, max |F_i|, dt, a, W[9]}, steps,
    converged (step or None), stop (step or None), vf (F.v of every step after the first), bmax (max(beta) of every
    structure, with covloss) and min_cos, the smallest |F.v| / (|F| |v|) met by a branch decision (how far the run
    stayed from a tie)."""
    prm = dict(FIRE_DEFAULTS, **fire)
    dt, a, Nsteps = prm["dt"], prm["a"], 0
    maxstep = prm["maxstep"]
    fixed = None if fixed is None else np.asarray(fixed, dtype=bool)
    r = np.array(pos, dtype=np.float64)

    def evaluate(x):
        if covloss:
            E, F, W, _, beta = eng.predict(x, numbers, cell, pbc, want_beta=True)
        else:
            (E, F, W, _), beta = eng.predict(x, numbers, cell, pbc), None
        F = np.array(F, dtype=np.float64)
        if fixed is not None:
            F[fixed] = 0.0
        return E, F, W, None if beta is None else np.array(beta)

    def fmax2(F):
        return (F ** 2).sum(axis=1).max() if len(F) else -np.inf

    E, F, W, beta = evaluate(r)
    out = dict(converged=None, stop=None, vf=[], min_cos=np.inf, bmax=[np.max(beta)] if covloss else [])
    if covloss and np.max(beta) > ediff:
        out["stop"] = 0
    if fmax2(F) < fmax ** 2:
        out["converged"] = 0
    v, rows, step = None, [], 0
    while step < n_steps and out["converged"] is None and out["stop"] is None:
        if v is None:
            v = np.zeros_like(r)
        else:
            vf = np.vdot(F, v)
            out["vf"].append(vf)
            nF, nv = np.sqrt(np.vdot(F, F)), np.sqrt(np.vdot(v, v))
            if nF > 0 and nv > 0:
                out["min_cos"] = min(out["min_cos"], abs(vf) / (nF * nv))
            if vf > 0.0:
                v = (1.0 - a) * v + a * F / np.sqrt(np.vdot(F, F)) * np.sqrt(np.vdot(v, v))
                if Nsteps > prm["Nmin"]:
                    dt = min(dt * prm["finc"], prm["dtmax"])
                    a *= prm["fa"]
                Nsteps += 1
            else:
                v[:] *= 0.0
                a = prm["astart"]
                dt *= prm["fdec"]
                Nsteps = 0
        v = v + dt * F
        dr = dt * v
        normdr = np.sqrt(np.vdot(dr, dr))
        if normdr > maxstep:
            dr = maxstep * dr / normdr
        r = r + dr
        E, F, W, beta = evaluate(r)
        step += 1
        rows.append(np.concatenate([[E, np.sqrt(fmax2(F)), dt, a], np.asarray(W).reshape(9)]))
        if covloss:
            out["bmax"].append(np.max(beta))
            if np.max(beta) > ediff:
                out["stop"] = step
        if fmax2(F) < fmax ** 2:
            out["converged"] = step
    out.update(pos=r, vel=np.zeros_like(r) if v is None else v, F=F, beta=beta, rows=np.array(rows).reshape(-1, 13),
               steps=step)
    return out
