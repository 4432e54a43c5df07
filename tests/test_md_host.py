"""CPU: the Langevin noise generator of sgpr_math.cuh (compiled with g++, the code md.cu runs) against the published
Philox4x32-10 known answers and the numpy restatement the GPU tests use; DeviceMD's argument checks (no GPU needed:
they run before any device work)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from md_reference import langevin_normals, philox4x32_10

HERE = os.path.dirname(os.path.abspath(__file__))
KNOWN = [   # Random123 kat_vectors, philox4x32 10 rounds: counter, key -> output
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("philox") / "libphilox_harness.so")
    src = os.path.join(HERE, "cpu_harness", "philox_harness.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", out])
    lib = ctypes.CDLL(out)
    lib.harness_philox.argtypes = [ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p]
    lib.harness_langevin_normals.argtypes = [ctypes.c_uint64, ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p]
    return lib


@pytest.mark.parametrize("ctr,key,want", KNOWN)
def test_philox_known_answers(harness, ctr, key, want):
    c = np.array(ctr, dtype=np.uint32)
    out = np.zeros(4, dtype=np.uint32)
    harness.harness_philox(c.ctypes.data, key[0], key[1], out.ctypes.data)
    assert [int(x) for x in out] == list(want)
    assert [int(x) for x in philox4x32_10([np.uint32(x) for x in ctr], *key)] == list(want)


@pytest.mark.parametrize("seed,step", [(0, 0), (12345, 7), (2 ** 63 + 11, 2 ** 33 + 5), (2 ** 64 - 1, 2 ** 64 - 1)])
def test_langevin_normals_match_numpy(harness, seed, step):
    n = 4000
    xi = np.zeros((n, 3))
    harness.harness_langevin_normals(seed, n, step, xi.ctypes.data)
    ref = langevin_normals(seed, n, step)
    assert np.abs(xi - ref).max() < 1e-13
    # a standard normal stream: mean 0, variance 1, independent components
    assert abs(xi.mean()) < 0.05 and abs(xi.var() - 1.0) < 0.05
    assert np.abs(np.corrcoef(xi.T) - np.eye(3)).max() < 0.06


def test_noise_streams_differ_by_step_atom_and_seed():
    a = langevin_normals(1, 64, 0)
    assert not np.array_equal(a, langevin_normals(1, 64, 1))
    assert not np.array_equal(a, langevin_normals(2, 64, 0))
    assert len(np.unique(a[:, 0])) == 64
    assert np.array_equal(a, langevin_normals(1, 64, 0))


class _Atoms:
    def __init__(self, n=4, numbers=None):
        self.positions = np.arange(3 * n, dtype=np.float64).reshape(n, 3)
        self.numbers = np.array(numbers if numbers is not None else [29] * n)
        self.cell = np.eye(3) * 10.0
        self.pbc = np.array([True] * 3)


def _model():
    from golden_util import b200_model, load_golden

    return b200_model(load_golden("cu108_sesoap"))


def _calc(**kw):
    import autoforce_b200 as ab

    return ab.B200Calculator(_model(), **kw)


@pytest.mark.parametrize("kw,err,match", [
    (dict(), ValueError, "masses are required"),
    (dict(masses=[1.0, 1.0, 1.0]), ValueError, "masses must be 4"),
    (dict(masses=[1.0, 1.0, -1.0, 1.0]), ValueError, "masses must be 4"),
    (dict(masses=[63.5] * 4, timestep=0.0), ValueError, "timestep"),
    (dict(masses=[63.5] * 4, friction=0.01), ValueError, "friction without temperature_K"),
    (dict(masses=[63.5] * 4, temperature_K=300.0), ValueError, "friction"),
    (dict(masses=[63.5] * 4, temperature_K=-1.0, friction=0.01), ValueError, "temperature_K"),
    (dict(masses=[63.5] * 4, seed=-1), ValueError, "seed"),
])
def test_device_md_argument_checks(kw, err, match):
    from autoforce_b200 import DeviceMD

    with pytest.raises(err, match=match):
        DeviceMD(_calc(), _Atoms(), **kw)


def test_device_md_refusals():
    import autoforce_b200 as ab
    from autoforce_b200 import DeviceMD

    calc = _calc()
    with pytest.raises(ValueError, match="unknown species"):
        DeviceMD(calc, _Atoms(numbers=[29, 29, 29, 0]), masses=[1.0] * 4)
    with pytest.raises(ValueError, match="unknown species"):
        DeviceMD(calc, _Atoms(n=9, numbers=[1, 2, 3, 4, 5, 6, 7, 8, 9]), masses=[1.0] * 9)
    two = ab.B200Calculator([_model(), _model()])
    with pytest.raises(NotImplementedError, match="kernel sums"):
        DeviceMD(two, _Atoms(), masses=[63.5] * 4)
    atoms = _Atoms()
    atoms.constraints = [object()]
    with pytest.raises(NotImplementedError, match="constraints"):
        DeviceMD(calc, atoms, masses=[63.5] * 4)
    assert calc._engine is None   # nothing was created on a device
