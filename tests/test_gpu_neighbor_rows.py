"""Neighbour rows as (begin, end) ranges: the block-per-bin kernel reserves each bin's rows with one atomic on a device
pair cursor, so rows land in the pair list in whatever order the atomics return.  What callers see must not depend on
that placement, and a warm step whose pair list outgrows the capacity must be caught on the device and recovered."""
import numpy as np
import pytest

from golden_util import b200_model, load_golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("mode", ["bins", "warp"])
def test_neighbor_rows_repeat_in_order(mode, monkeypatch):
    """The CSR list in the caller's order, within-row order included, is the same on the sizing call that grows the
    capacity (the block-per-bin kernel then runs twice) and on later calls: on a golden cell and on a crowded droplet
    (several rounds of atoms per bin, candidate tiles beyond the accept-bit words)."""
    import autoforce_b200 as ab

    monkeypatch.setenv("SGPR_NL", mode)
    g = load_golden("lipso108")
    rc = g["meta"]["kernel"]["rc"]
    rng = np.random.default_rng(11)
    n = 2400
    drop = rng.uniform(0.0, 1.6 * rc, size=(n, 3)) + np.array([7.0, 9.0, 5.0])
    sp = np.asarray(g["meta"]["species"])
    cases = [(g["pos"], g["numbers"], g["cell"], g["meta"]["pbc"]),
             (drop, sp[rng.integers(0, 2, size=n)], np.diag([41.0, 39.0, 43.0]), True)]
    for pos, Z, cell, pbc in cases:
        eng = ab.SgprEngine(b200_model(g), species=g["meta"]["species"])
        a = eng.neighbors(pos, Z, cell, pbc)
        b = eng.neighbors(pos, Z, cell, pbc)
        eng.close()
        assert len(a[1]) > 0
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


@pytest.mark.parametrize("mode", ["bins", "warp"])
def test_warm_pair_overflow_recovered_on_the_device(mode, monkeypatch):
    """Capacity sized on an expanded structure, then warm steps on the dense one: the first overflows on the device
    (reported by check(), no memory touched beyond the list), the next one sizes again, and the warm step after it
    gives energy and virial bit for bit, and forces to rounding, of an engine that never overflowed."""
    import torch

    import autoforce_b200 as ab
    from autoforce_b200 import synth

    monkeypatch.setenv("SGPR_NL", mode)
    Zs = [3, 8]
    model = synth.synth_model(Zs, 40, 5, lmax=3, nmax=3, rc=6.0)
    pos, cell, numbers = synth.fcc(10, Zs, 0.1, 1)    # 4,000 atoms, 216 bins
    dev = torch.device("cuda", 0)
    z_t = torch.as_tensor(numbers.astype(np.int32), device=dev)
    p_sparse, p_dense = torch.as_tensor(pos * 1.5, device=dev), torch.as_tensor(pos, device=dev)

    ref = ab.SgprEngine(model, species=Zs)
    ref.set_async(True)
    ref.predict_device(p_dense, z_t, cell, True)                  # sizing step
    torch.cuda.synchronize()
    n_dense = ref.check()
    E0, F0, W0 = (t.cpu().numpy().copy() for t in ref.predict_device(p_dense, z_t, cell, True))   # warm, fits
    torch.cuda.synchronize()
    assert ref.check() == n_dense
    ref.close()

    eng = ab.SgprEngine(model, species=Zs)
    eng.set_async(True)
    eng.predict_device(p_sparse, z_t, cell * 1.5, True)          # sizing step on the sparse structure
    torch.cuda.synchronize()
    assert eng.check() * 2 < n_dense
    eng.predict_device(p_dense, z_t, cell, True)                 # warm: overflows
    torch.cuda.synchronize()
    with pytest.raises(RuntimeError, match="exceed the capacity"):
        eng.check()
    eng.predict_device(p_dense, z_t, cell, True)                 # sizes again
    torch.cuda.synchronize()
    assert eng.check() == n_dense
    E, F, W = (t.cpu().numpy() for t in eng.predict_device(p_dense, z_t, cell, True))   # warm and valid
    torch.cuda.synchronize()
    assert eng.check() == n_dense
    eng.close()
    assert np.array_equal(E, E0) and np.array_equal(W, W0)
    assert np.abs(F - F0).max() < 1e-11
