"""ctypes binding of libsgpr_b200.so (include/sgpr_b200.h) + a thin engine object.

PyTorch is used only for device memory and streams.  No CPU fallback: a missing
library or a missing CUDA device raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int8, c_int32, c_int64, c_uint8, c_void_p

import numpy as np

from .model import MAX_SPECIES, SgprModel

_LIB = None


def library_path():
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libsgpr_b200.so")


class sgpr_model_desc(ctypes.Structure):
    _fields_ = [
        ("lmax", c_int32), ("nmax", c_int32), ("xi", c_double), ("rc", c_double), ("normalize", c_int32),
        ("n_species", c_int32), ("species_Z", c_int32 * MAX_SPECIES), ("radii", c_double * MAX_SPECIES),
        ("central_enabled", c_int32 * MAX_SPECIES), ("neighbor_enabled", c_int32 * MAX_SPECIES), ("M", c_int32), ("ind_first_h", c_void_p), ("ind_r_h", c_void_p),
        ("ind_b_h", c_void_p), ("ind_Z_h", c_void_p), ("mu_h", c_void_p), ("mean_w_h", c_void_p),
        ("choli_h", c_void_p), ("vscale_h", c_void_p), ("device", c_int32), ("lone_weight", c_double),
    ]


class sgpr_stats(ctypes.Structure):
    _fields_ = [
        ("n_atoms", c_int64), ("n_active", c_int64), ("n_pairs", c_int64), ("d_packed", c_int32), ("d_full", c_int32),
        ("kernel_launches", c_int64), ("gemm_flops", c_double), ("covloss_flops", c_double), ("i8_ops", c_double), ("ms_nl", c_float),
        ("ms_desc", c_float), ("ms_gemm", c_float), ("ms_force", c_float), ("ms_beta", c_float), ("ms_total", c_float),
    ]


class sgpr_md_params(ctypes.Structure):
    _fields_ = [
        ("dt", c_double), ("friction", c_double), ("kT", c_double), ("ediff", c_double), ("seed", ctypes.c_uint64),
        ("langevin", c_int32), ("stop_on_uncertain", c_int32),
    ]


class sgpr_relax_params(ctypes.Structure):
    _fields_ = [
        ("dt", c_double), ("maxstep", c_double), ("dtmax", c_double), ("finc", c_double), ("fdec", c_double),
        ("astart", c_double), ("fa", c_double), ("a", c_double), ("fmax", c_double), ("ediff", c_double),
        ("Nmin", c_int32), ("stop_on_uncertain", c_int32),
    ]


EXPORTS = {
    # name: (restype, argtypes)       -- every symbol include/sgpr_b200.h declares
    "sgpr_create": (c_int32, [POINTER(sgpr_model_desc), POINTER(c_void_p)]),
    "sgpr_destroy": (None, [c_void_p]),
    "sgpr_last_error": (c_char_p, []),
    "sgpr_abi_version": (c_int32, []),
    "sgpr_set_weights": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_append_inducing": (c_int32, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_predict": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_predict_host": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_predict_batch": (c_int32, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_predict_p2p": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                                   c_void_p, c_void_p, c_void_p]),
    "sgpr_p2p_collect": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_p2p_step": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_kernel_forward": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_kernel_backward": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_kernel_jacobian": (c_int32, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "sgpr_kernel_jacobian_batch": (c_int32, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                             c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_neighbors": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_int64, POINTER(c_int64)]),
    "sgpr_descriptors": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_inducing_descriptors": (c_int32, [c_void_p, c_void_p, c_void_p]),
    "sgpr_kernel_envs": (c_int32, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_md_init": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, POINTER(sgpr_md_params), c_void_p,
                               c_void_p, c_void_p, c_void_p]),
    "sgpr_md_steps": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                POINTER(sgpr_md_params), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_relax_init": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  POINTER(sgpr_relax_params), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "sgpr_relax_steps": (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   POINTER(sgpr_relax_params), c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p]),
    "sgpr_set_async": (c_int32, [c_void_p, c_int32]),
    "sgpr_check": (c_int32, [c_void_p, POINTER(c_int64)]),
    "sgpr_get_stats": (c_int32, [c_void_p, POINTER(sgpr_stats)]),
    "sgpr_enable_timing": (c_int32, [c_void_p, c_int32]),
}


def load_library(path=None):
    """dlopen libsgpr_b200.so and declare every exported symbol.  Raises if missing."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    path = path or os.environ.get("SGPR_B200_LIB") or library_path()   # env override: A/B builds of the library
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(autoforce_b200 has no CPU fallback)")
    import torch  # noqa: F401  (loads libcudart.so.12 into the process before our dlopen)

    lib = ctypes.CDLL(path)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.sgpr_abi_version() != 1:
        raise RuntimeError("libsgpr_b200.so: ABI version mismatch")
    _LIB = lib
    return lib


def _check(lib, status):
    if status != 0:
        msg = lib.sgpr_last_error().decode(errors="replace")
        raise RuntimeError(f"libsgpr_b200 error {status}: {msg}")


def _ptr(a):
    return c_void_p(a.ctypes.data)


class PeerForceExchange:
    """Atom-sharded prediction without halo recompute: every rank evaluates the environments it owns and adds
    the forces on atoms of other ranks straight into their accumulation buffers over NVLink (peer-mapped
    symmetric memory).  ``fused=True`` (default): the whole step is ONE library call, ``sgpr_p2p_step`` -- E and the
    virial travel through peer-mapped mailboxes with stamped flags that double as the barrier, so there is no NCCL call,
    no torch kernel and no host synchronisation in a warm step (it replays as one CUDA graph).  ``fused=False``:
    ``sgpr_predict_p2p`` + an NCCL all-reduce of the 10 doubles (the barrier) + ``sgpr_p2p_collect``.
    Two accumulation buffers alternate between steps so that zeroing never races with remote adds."""

    def __init__(self, engine, N, group=None, fused=True):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        self.engine, self.N, self.fused = engine, int(N), bool(fused)
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        dev = torch.device("cuda", engine.device)
        self.stride = 3 * self.N + 8
        self.buf = symm.empty(2 * self.stride + 2 * self.world * 16, dtype=torch.float64, device=dev)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, self.group)
        self.ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self._bases = np.array(self.ptrs, dtype=np.uint64)
        self.parity = 0
        self.ew = torch.zeros(10, dtype=torch.float64, device=dev)
        self.F = torch.zeros((self.N, 3), dtype=torch.float64, device=dev)
        self.owned = torch.zeros(self.N, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        dist.barrier(self.group)

    def step(self, pos_t, z_t, cell, pbc):
        """Device tensors in; returns (E, F_owned [N,3], W [3,3] tensor, owned mask) with E and W already summed
        over the ranks."""
        eng = self.engine
        p = self.parity
        if self.fused:
            eng.p2p_step(pos_t, z_t, cell, pbc, self.rank, self.world, self._bases, self.ew, self.F, self.owned)
        else:
            import torch.distributed as dist

            # the other buffer was collected at the end of the previous step: clear it for the next one
            self.buf[(1 - p) * self.stride:(2 - p) * self.stride].zero_()
            eng.predict_p2p(pos_t, z_t, cell, pbc, self.rank, self.world, [ptr + 8 * p * self.stride for ptr in self.ptrs], self.ew)
            dist.all_reduce(self.ew, group=self.group)   # E + virial; also: every rank's force kernel has finished
            eng.p2p_collect(self.buf[p * self.stride:(p + 1) * self.stride], self.F, self.owned)
        self.parity = 1 - p
        return self.ew[0], self.F, self.ew[1:].view(3, 3), self.owned


def _make_cov_function():
    import torch

    class _CovFn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, xyz, lll, engine, numbers, pbc):
            K = engine.kernel_matrix(xyz.detach(), numbers, lll.detach().cpu().numpy(), pbc)
            ctx.engine = engine
            ctx.xyz_dev, ctx.lll_dev = xyz.device, lll.device
            return K.to(xyz.device)

        @staticmethod
        def backward(ctx, gK):
            gpos, gcell = ctx.engine.kernel_matrix_vjp(gK)
            import torch as _t

            return gpos.to(ctx.xyz_dev), _t.as_tensor(gcell).to(ctx.lll_dev), None, None, None

    return _CovFn


class _CovProxy:
    """Lazy holder so that importing the module does not import torch."""

    _fn = None

    @classmethod
    def apply(cls, *args):
        if cls._fn is None:
            cls._fn = _make_cov_function()
        return cls._fn.apply(*args)


_Cov = _CovProxy


_PINNED_KEEPALIVE = []


class SgprEngine:
    """One handle on one CUDA device.  Host-side mirror of the C ABI."""

    def __init__(self, model: SgprModel, species=None, device=0):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: autoforce_b200 has no CPU fallback")
        self.lib = load_library()
        self.model = model
        self.device = int(device)
        self.species = sorted(set(model.species()) | set(int(z) for z in (species if species is not None else [])))
        if len(self.species) > MAX_SPECIES:
            raise ValueError(f"at most {MAX_SPECIES} species are supported, got {self.species}")
        self._h = c_void_p()
        d = sgpr_model_desc()
        d.lmax, d.nmax, d.xi, d.rc = model.lmax, model.nmax, float(model.xi), float(model.rc)
        d.normalize = 1 if model.normalize else 0
        d.n_species = len(self.species)
        mean_w = np.zeros(MAX_SPECIES)
        vscale = np.full(MAX_SPECIES, np.inf)
        for s, z in enumerate(self.species):
            d.species_Z[s] = z
            d.radii[s] = model.unit_of(z)
            d.central_enabled[s] = 1 if model.is_centre(z) else 0
            d.neighbor_enabled[s] = 1 if model.is_neighbour(z) else 0
            mean_w[s] = model.mean_w.get(z, 0.0)
            vscale[s] = model.vscale.get(z, np.inf)
        d.lone_weight = float(getattr(model, "lone_weight", 1.0))
        d.M = model.M
        self._keep = (model.ind_first, model.ind_r, model.ind_b, model.ind_Z, model.mu, mean_w, vscale, model.choli)
        d.ind_first_h, d.ind_r_h, d.ind_b_h = _ptr(model.ind_first), _ptr(model.ind_r), _ptr(model.ind_b)
        d.ind_Z_h, d.mu_h, d.mean_w_h, d.vscale_h = _ptr(model.ind_Z), _ptr(model.mu), _ptr(mean_w), _ptr(vscale)
        d.choli_h = _ptr(model.choli) if model.choli is not None else None
        d.device = self.device
        _check(self.lib, self.lib.sgpr_create(ctypes.byref(d), ctypes.byref(self._h)))
        self.d_full = len(self.species) ** 2 * (model.nmax + 1) ** 2 * (model.lmax + 1)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.sgpr_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def _geom(cell, pbc):
        cell_h = np.ascontiguousarray(np.asarray(cell, dtype=np.float64).reshape(9))
        pbc_h = np.ascontiguousarray(np.broadcast_to(np.asarray(pbc), (3,)).astype(np.int32))
        return cell_h, pbc_h

    def _dev(self, pos, numbers):
        import torch

        dev = torch.device("cuda", self.device)
        pos_t = torch.as_tensor(np.ascontiguousarray(pos, dtype=np.float64)).to(dev) if not torch.is_tensor(pos) else pos.to(dev, torch.float64).contiguous()
        z_t = torch.as_tensor(np.ascontiguousarray(numbers, dtype=np.int32)).to(dev) if not torch.is_tensor(numbers) else numbers.to(dev, torch.int32).contiguous()
        return pos_t.reshape(-1, 3), z_t.reshape(-1)

    def _batch(self, pos, numbers, first, cells, pbcs):
        """Inputs of the batched entry points (``predict_batch``, ``training_kernels``): a list of structures, or
        concatenated ``pos`` / ``numbers`` with ``first`` [B+1] and ``cells`` / ``pbcs`` (one value for all, or one per
        structure).  Returns first_h int64 [B+1], B, N, cell_h [B,9], pbc_h int32 [B,3] (host) and pos_t, z_t (device)."""
        if first is None:
            images = list(pos)
            if numbers is not None or cells is not None or pbcs is not None:
                raise ValueError("pass either a list of structures or pos, numbers, first, cells, pbcs")
            counts = [len(a.numbers) for a in images]
            pos = np.concatenate([np.asarray(a.positions, dtype=np.float64).reshape(-1, 3) for a in images]) if images else np.zeros((0, 3))
            numbers = np.concatenate([np.asarray(a.numbers).reshape(-1) for a in images]) if images else np.zeros(0, dtype=np.int32)
            first = np.concatenate([[0], np.cumsum(counts)])
            cells = [np.asarray(a.cell, dtype=np.float64).reshape(3, 3) for a in images]
            pbcs = [np.broadcast_to(np.asarray(a.pbc), (3,)) for a in images]
        first_h = np.ascontiguousarray(first, dtype=np.int64).reshape(-1)
        B = len(first_h) - 1
        if B < 0:
            raise ValueError("first must have B+1 >= 1 entries")
        cell_h = np.ascontiguousarray(np.broadcast_to(np.asarray(cells, dtype=np.float64).reshape(-1, 9), (B, 9)))
        pb = np.asarray(pbcs).astype(np.int32)
        pbc_h = np.ascontiguousarray(np.broadcast_to(pb.reshape(-1, 3) if pb.size and pb.size % 3 == 0 else pb.reshape(-1, 1), (B, 3)))
        pos_t, z_t = self._dev(pos, numbers)
        N = z_t.numel()
        if pos_t.shape[0] != N or first_h[-1] != N:
            raise ValueError(f"first[-1] = {first_h[-1]} does not match {N} atoms")
        return first_h, B, N, cell_h, pbc_h, pos_t, z_t

    @staticmethod
    def _stream():
        import torch

        return c_void_p(torch.cuda.current_stream().cuda_stream)

    # ------------------------------------------------------------------ hot path
    @staticmethod
    def pinned(shape, dtype=np.float64):
        """Page-locked host array (numpy view of a pinned torch tensor).  predict() copies such buffers with the
        DMA engine directly; ordinary (pageable) arrays take one extra host memcpy each way."""
        import torch

        t = torch.empty(shape, dtype=getattr(torch, np.dtype(dtype).name)).pin_memory()
        a = t.numpy()
        _PINNED_KEEPALIVE.append(t)
        return a

    def predict(self, pos, numbers, cell, pbc, rank=0, world=1, want_beta=False, out_forces=None):
        """Host numpy in, host numpy out (H2D/D2H inside): E, F[N,3], W[3,3], owned[N]
        (+ beta[N], the covloss of calculator/active.py:781-804, when want_beta).  ``out_forces`` may be a
        caller-owned (ideally pinned()) float64 [N,3] array that receives F."""
        pos = np.ascontiguousarray(pos, dtype=np.float64).reshape(-1, 3)
        Z = np.ascontiguousarray(numbers, dtype=np.int32).reshape(-1)
        N = len(Z)
        cell_h, pbc_h = self._geom(cell, pbc)
        E = np.zeros(1)
        if out_forces is not None:
            if out_forces.dtype != np.float64 or out_forces.shape != (N, 3) or not out_forces.flags.c_contiguous:
                raise ValueError("out_forces must be a C-contiguous float64 [N,3] array")
            F = out_forces
        else:
            F = np.empty((N, 3))
        W = np.zeros(9)
        owned = np.zeros(N, dtype=np.uint8)
        beta = np.zeros(N) if want_beta else None
        _check(self.lib, self.lib.sgpr_predict_host(self._h, N, _ptr(pos), _ptr(Z), _ptr(cell_h), _ptr(pbc_h), rank, world,
                                                    _ptr(E), _ptr(F), _ptr(W), _ptr(beta) if want_beta else None, _ptr(owned)))
        if want_beta:
            return float(E[0]), F, W.reshape(3, 3), owned.astype(bool), beta
        return float(E[0]), F, W.reshape(3, 3), owned.astype(bool)

    def predict_device(self, pos_t, z_t, cell, pbc, rank=0, world=1, out=None):
        """Device tensors in, device tensors out, on torch's current stream."""
        import torch

        N = z_t.numel()
        cell_h, pbc_h = self._geom(cell, pbc)
        if out is None:
            dev = pos_t.device
            out = (torch.empty(1, dtype=torch.float64, device=dev), torch.empty((N, 3), dtype=torch.float64, device=dev),
                   torch.empty(9, dtype=torch.float64, device=dev))
        E, F, W = out
        _check(self.lib, self.lib.sgpr_predict(self._h, N, c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()), _ptr(cell_h),
                                               _ptr(pbc_h), rank, world, self._stream(), c_void_p(E.data_ptr()),
                                               c_void_p(F.data_ptr()), c_void_p(W.data_ptr()), None, None))
        return E, F, W

    def predict_batch(self, pos, numbers=None, first=None, cells=None, pbcs=None, want_beta=False):
        """B structures in one call (``sgpr_predict_batch``): the same E, F, W (and beta) as ``predict`` on each structure
        alone, at a fraction of the cost when the structures are small.

        ``pos`` [Ntot,3] and ``numbers`` [Ntot] hold the structures one after the other (host arrays or CUDA tensors),
        ``first`` [B+1] their atom offsets, ``cells`` [B,3,3] and ``pbcs`` [B,3] (or one value for all) their cells.
        Alternatively ``pos`` may be a list of structures (anything with positions / cell / pbc / numbers, like
        ase.Atoms) and the other arguments are left out.  Returns host numpy E [B], F [Ntot,3], W [B,3,3] (+ beta [Ntot]
        when ``want_beta``)."""
        import torch

        first_h, B, N, cell_h, pbc_h, pos_t, z_t = self._batch(pos, numbers, first, cells, pbcs)
        dev = pos_t.device
        E = torch.zeros(max(B, 1), dtype=torch.float64, device=dev)
        F = torch.zeros((N, 3), dtype=torch.float64, device=dev)
        W = torch.zeros((max(B, 1), 9), dtype=torch.float64, device=dev)
        beta = torch.zeros(max(N, 1), dtype=torch.float64, device=dev) if want_beta else None
        _check(self.lib, self.lib.sgpr_predict_batch(self._h, B, _ptr(first_h), c_void_p(pos_t.data_ptr()),
                                                     c_void_p(z_t.data_ptr()), _ptr(cell_h), _ptr(pbc_h), self._stream(),
                                                     c_void_p(E.data_ptr()), c_void_p(F.data_ptr()), c_void_p(W.data_ptr()),
                                                     c_void_p(beta.data_ptr()) if want_beta else None))
        E, F, W = E[:B].cpu().numpy(), F.cpu().numpy(), W[:B].cpu().numpy().reshape(B, 3, 3)
        if want_beta:
            return E, F, W, beta[:N].cpu().numpy()
        return E, F, W

    def training_kernels(self, pos, numbers=None, first=None, cells=None, pbcs=None, m0=0, m1=None, want_jacobian=True):
        """Training-time kernels of B structures against the inducing LCEs m0 <= m < m1 in one call
        (``sgpr_kernel_jacobian_batch``): the blocks of ``EnergyForceKernel(first=[...], X, cov=...)``
        (regression/gppotential.py:63-77) that make_munu stacks.

        Inputs as in ``predict_batch``: concatenated arrays or CUDA tensors with ``first`` [B+1], ``cells`` and ``pbcs``,
        or a list of structures.  Returns device tensors ``(Ke [B, m], Kf [3 Ntot, m], Kv [6 B, m])``: energy_energy,
        forces_energy (= -d Ke / d xyz, rows 3i..3i+2 of atom i) and virial_energy (rows 6b..6b+5 of structure b:
        xx, yy, zz, yz, xz, xy, not divided by the volume), structures stacked in order.  ``want_jacobian=False`` skips
        the Jacobian and returns ``(Ke, None, None)``.  For B = 1 this is ``kernel_jacobian`` (Ke = K.sum(0))."""
        import torch

        first_h, B, N, cell_h, pbc_h, pos_t, z_t = self._batch(pos, numbers, first, cells, pbcs)
        m1 = self.model.M if m1 is None else int(m1)
        m0 = int(m0)
        if not 0 <= m0 <= m1 <= self.model.M:
            raise ValueError(f"inducing range [{m0}, {m1}) outside [0, {self.model.M})")
        nm = m1 - m0
        dev = pos_t.device
        # flat buffers of at least one element: empty outputs still get valid (non-NULL) device pointers
        buf = lambda n: torch.zeros(max(n, 1), dtype=torch.float64, device=dev)   # noqa: E731
        Ke = buf(B * nm)
        J = buf(nm * N * 3) if want_jacobian else None
        W = buf(B * nm * 9) if want_jacobian else None
        _check(self.lib, self.lib.sgpr_kernel_jacobian_batch(self._h, B, _ptr(first_h), c_void_p(pos_t.data_ptr()),
                                                             c_void_p(z_t.data_ptr()), _ptr(cell_h), _ptr(pbc_h), m0, m1,
                                                             self._stream(), c_void_p(Ke.data_ptr()),
                                                             c_void_p(J.data_ptr()) if want_jacobian else None,
                                                             c_void_p(W.data_ptr()) if want_jacobian else None))
        Ke = Ke[:B * nm].reshape(B, nm)
        if not want_jacobian:
            return Ke, None, None
        Kf = -J[:nm * N * 3].reshape(nm, 3 * N).t().contiguous()
        Kv = W[:B * nm * 9].reshape(B, nm, 9)[:, :, [0, 4, 8, 5, 2, 1]].permute(0, 2, 1).reshape(6 * B, nm).contiguous()
        return Ke, Kf, Kv

    def predict_p2p(self, pos_t, z_t, cell, pbc, rank, world, peer_ptrs, ew):
        """``sgpr_predict_p2p``: this rank's environments only; forces on every atom are ADDED into the accumulation
        buffer of the atom's owner, ``peer_ptrs[r]`` (device addresses valid on this GPU: peer-mapped over NVLink, or plain
        local buffers when several ranks are emulated on one GPU).  ``ew`` [10] receives this rank's E and 3x3 virial."""
        cell_h, pbc_h = self._geom(cell, pbc)
        peers = np.array([int(p) for p in peer_ptrs], dtype=np.uint64)
        _check(self.lib, self.lib.sgpr_predict_p2p(self._h, z_t.numel(), c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()),
                                                   _ptr(cell_h), _ptr(pbc_h), int(rank), int(world), self._stream(), _ptr(peers),
                                                   c_void_p(ew.data_ptr()), c_void_p(ew.data_ptr() + 8)))

    def p2p_step(self, pos_t, z_t, cell, pbc, rank, world, bases, ew, F, owned):
        """``sgpr_p2p_step``: the fused exchange step (include/sgpr_b200.h).  ``bases`` uint64 [world]: every rank's
        symmetric block as mapped on this device; ``ew`` [10] receives the reduced E and 3x3 virial."""
        cell_h, pbc_h = self._geom(cell, pbc)
        bases = np.ascontiguousarray(bases, dtype=np.uint64)
        _check(self.lib, self.lib.sgpr_p2p_step(self._h, z_t.numel(), c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()),
                                                _ptr(cell_h), _ptr(pbc_h), int(rank), int(world), self._stream(), _ptr(bases),
                                                c_void_p(ew.data_ptr()), c_void_p(F.data_ptr()),
                                                c_void_p(ew.data_ptr() + 8), c_void_p(owned.data_ptr())))

    def p2p_collect(self, own_buf, F, owned):
        """``sgpr_p2p_collect``: after every rank's ``predict_p2p`` has finished, copy this rank's accumulated forces
        (cell order) into ``F`` [N,3] (caller's order, rows of owned atoms) and fill the ``owned`` mask."""
        _check(self.lib, self.lib.sgpr_p2p_collect(self._h, self._stream(), c_void_p(own_buf.data_ptr()), c_void_p(F.data_ptr()),
                                                   c_void_p(owned.data_ptr())))

    def peer_exchange(self, N, group=None, fused=True):
        """Set up the peer-memory (NVLink) force exchange for structures of N atoms (torch symmetric memory)."""
        return PeerForceExchange(self, N, group, fused)

    def kernel_matrix(self, pos, numbers, cell, pbc):
        import torch

        pos_t, z_t = self._dev(pos, numbers)
        N = z_t.numel()
        cell_h, pbc_h = self._geom(cell, pbc)
        K = torch.empty((N, self.model.M), dtype=torch.float64, device=pos_t.device)
        _check(self.lib, self.lib.sgpr_kernel_forward(self._h, N, c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()),
                                                      _ptr(cell_h), _ptr(pbc_h), self._stream(), c_void_p(K.data_ptr())))
        return K

    def kernel_matrix_vjp(self, gK):
        """Vector-Jacobian product of the LAST kernel_matrix() call: given gK = dL/dK [N, M] returns
        (dL/dxyz [N,3] device tensor, dL/dcell [3,3] numpy) -- what torch.autograd.grad does in the
        reference (calculator/active.py:587-599, regression/gppotential.py:905-911)."""
        import torch

        dev = torch.device("cuda", self.device)
        gK = gK.to(dev, torch.float64).contiguous()
        N = gK.shape[0]
        gpos = torch.empty((N, 3), dtype=torch.float64, device=dev)
        gcell = np.zeros(9)
        _check(self.lib, self.lib.sgpr_kernel_backward(self._h, c_void_p(gK.data_ptr()), self._stream(), c_void_p(gpos.data_ptr()),
                                                       _ptr(gcell)))
        return gpos, gcell.reshape(3, 3)

    def kernel_jacobian(self, pos, numbers, cell, pbc, m0=0, m1=None):
        """Training-time kernels of one structure against the inducing set (regression/gppotential.py:63-77):
        returns (K [N,M] device tensor, Kf [3N, m1-m0], Kv [6, m1-m0]) with Kf = forces_energy = -leftgrad and
        Kv = virial_energy (xx,yy,zz,yz,xz,xy; not divided by the volume); Ke = K.sum(0)."""
        import torch

        K = self.kernel_matrix(pos, numbers, cell, pbc)
        N = K.shape[0]
        m1 = self.model.M if m1 is None else m1
        J = torch.zeros((m1 - m0, N, 3), dtype=torch.float64, device=K.device)
        W = torch.zeros((m1 - m0, 9), dtype=torch.float64, device=K.device)
        _check(self.lib, self.lib.sgpr_kernel_jacobian(self._h, m0, m1, self._stream(), c_void_p(J.data_ptr()),
                                                       c_void_p(W.data_ptr())))
        Kf = -J.reshape(m1 - m0, 3 * N).t().contiguous()
        Kv = W[:, [0, 4, 8, 5, 2, 1]].t().contiguous()
        return K, Kf, Kv

    def cov(self, xyz, lll, numbers, pbc):
        """Differentiable kernel matrix: ``cov = model.gp.kern(atoms, model.X)`` (calculator/active.py:464) as a
        torch tensor [N, M] on xyz's device that back-propagates into ``xyz`` (positions) and ``lll`` (cell) --
        the seam the on-the-fly training control flow needs (SURVEY.md 3.2)."""
        return _Cov.apply(xyz, lll, self, np.asarray(numbers), tuple(bool(b) for b in np.broadcast_to(np.asarray(pbc), (3,))))

    # ------------------------------------------------------------------ parity hooks
    def neighbors(self, pos, numbers, cell, pbc):
        """CSR (first[N+1], j[nnz], S[nnz,3]) in the caller's atom order."""
        import torch

        pos_t, z_t = self._dev(pos, numbers)
        N = z_t.numel()
        cell_h, pbc_h = self._geom(cell, pbc)
        first = torch.empty(N + 1, dtype=torch.int64, device=pos_t.device)
        nnz = c_int64(0)
        cap = max(1, 128 * N)
        for _ in range(2):
            j = torch.empty(cap, dtype=torch.int32, device=pos_t.device)
            S = torch.empty((cap, 3), dtype=torch.int8, device=pos_t.device)
            _check(self.lib, self.lib.sgpr_neighbors(self._h, N, c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()), _ptr(cell_h),
                                                     _ptr(pbc_h), self._stream(), c_void_p(first.data_ptr()),
                                                     c_void_p(j.data_ptr()), c_void_p(S.data_ptr()), cap, ctypes.byref(nnz)))
            if nnz.value <= cap:
                break
            cap = nnz.value
        n = nnz.value
        return first.cpu().numpy(), j[:n].cpu().numpy(), S[:n].cpu().numpy()

    def descriptors(self, pos, numbers, cell, pbc):
        """[N, S, S, nmax+1, nmax+1, lmax+1] normalised descriptors (reference layout)."""
        import torch

        pos_t, z_t = self._dev(pos, numbers)
        N = z_t.numel()
        cell_h, pbc_h = self._geom(cell, pbc)
        P = torch.empty((N, self.d_full), dtype=torch.float64, device=pos_t.device)
        _check(self.lib, self.lib.sgpr_descriptors(self._h, N, c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()), _ptr(cell_h),
                                                   _ptr(pbc_h), self._stream(), c_void_p(P.data_ptr())))
        S, n, L = len(self.species), self.model.nmax + 1, self.model.lmax + 1
        return P.cpu().numpy().reshape(N, S, S, n, n, L)

    def inducing_descriptors(self):
        import torch

        dev = torch.device("cuda", self.device)
        Zh = torch.empty((self.model.M, self.d_full), dtype=torch.float64, device=dev)
        _check(self.lib, self.lib.sgpr_inducing_descriptors(self._h, self._stream(), c_void_p(Zh.data_ptr())))
        S, n, L = len(self.species), self.model.nmax + 1, self.model.lmax + 1
        return Zh.cpu().numpy().reshape(self.model.M, S, S, n, n, L)

    def kernel_envs(self, envs, want_K=True, want_descriptors=False):
        """Explicit environments ``[(Z, r[nn,3], b[nn]), ...]`` (reference ``Local``s) against the inducing set:
        ``K [n, M]`` = ``kern(locs, X)`` (device tensor) and / or their descriptors ``[n, S, S, nmax+1, nmax+1, lmax+1]``
        (numpy) = ``kern.call_descriptor(loc, grad=False)`` (similarity/universal.py:97-122)."""
        import torch

        n = len(envs)
        Z = np.ascontiguousarray([int(e[0]) for e in envs], dtype=np.int32)
        rs = [np.asarray(e[1], dtype=np.float64).reshape(-1, 3) for e in envs]
        bs = [np.asarray(e[2], dtype=np.int32).reshape(-1) for e in envs]
        first = np.zeros(n + 1, dtype=np.int64)
        first[1:] = np.cumsum([len(b) for b in bs])
        r = np.ascontiguousarray(np.concatenate(rs) if n else np.zeros((0, 3)))
        b = np.ascontiguousarray(np.concatenate(bs) if n else np.zeros(0, dtype=np.int32))
        dev = torch.device("cuda", self.device)
        K = torch.zeros((n, self.model.M), dtype=torch.float64, device=dev) if want_K else None
        P = torch.zeros((n, self.d_full), dtype=torch.float64, device=dev) if want_descriptors else None
        if n:
            _check(self.lib, self.lib.sgpr_kernel_envs(self._h, n, _ptr(Z), _ptr(first), _ptr(r), _ptr(b), self._stream(),
                                                       c_void_p(K.data_ptr()) if want_K else None,
                                                       c_void_p(P.data_ptr()) if want_descriptors else None))
        S, nb, L = len(self.species), self.model.nmax + 1, self.model.lmax + 1
        Pn = P.cpu().numpy().reshape(n, S, S, nb, nb, L) if want_descriptors else None
        return (K, Pn) if (want_K and want_descriptors) else (K if want_K else Pn)

    # ------------------------------------------------------------------ misc
    def set_weights(self, mu=None, mean_w=None, choli=None, vscale=None):
        def arr(x, n):
            if x is None:
                return None, None
            a = np.ascontiguousarray(x, dtype=np.float64)
            assert a.size == n
            return a, _ptr(a)

        M = self.model.M
        mw = None if mean_w is None else np.array([mean_w.get(z, 0.0) for z in self.species])
        vs = None if vscale is None else np.array([vscale.get(z, np.inf) for z in self.species])
        a1, p1 = arr(mu, M)
        a2, p2 = arr(mw, len(self.species))
        a3, p3 = arr(choli, M * M)
        a4, p4 = arr(vs, len(self.species))
        _check(self.lib, self.lib.sgpr_set_weights(self._h, p1, p2, p3, p4))
        # keep the host-side model in step with the device (save(), `model.choli is None` checks)
        m = self.model
        if a1 is not None:
            m.mu = a1.reshape(-1).copy()
        if mean_w is not None:
            m.mean_w = {int(z): float(w) for z, w in mean_w.items()}
        if a3 is not None:
            m.choli = a3.reshape(M, M).copy()
        if vscale is not None:
            m.vscale = {int(z): float(v) for z, v in vscale.items()}

    def append_inducing(self, envs, mu, choli=None):
        """Add inducing LCEs ``[(Z, r[nn,3], b[nn]), ...]`` after the existing ones and install the refitted
        weights ``mu [M+n]`` (and ``choli [M+n, M+n]``): what ``model.add_inducing(loc)`` + ``make_munu`` do in
        the reference (regression/gppotential.py:888-940, 548-601).  All new species must already be in the
        engine's species table (pass ``species=`` when constructing the engine)."""
        n = len(envs)
        Z = np.ascontiguousarray([int(e[0]) for e in envs], dtype=np.int32)
        rs = [np.asarray(e[1], dtype=np.float64).reshape(-1, 3) for e in envs]
        bs = [np.asarray(e[2], dtype=np.int32).reshape(-1) for e in envs]
        for r, b in zip(rs, bs):
            if len(r) != len(b):
                raise ValueError("environment with mismatched r / b lengths")
        first = np.zeros(n + 1, dtype=np.int64)
        first[1:] = np.cumsum([len(b) for b in bs])
        r = np.ascontiguousarray(np.concatenate(rs) if n else np.zeros((0, 3)))
        b = np.ascontiguousarray(np.concatenate(bs) if n else np.zeros(0, dtype=np.int32))
        M1 = self.model.M + n
        mu = np.ascontiguousarray(mu, dtype=np.float64).reshape(-1)
        if mu.size != M1:
            raise ValueError(f"mu must have {M1} entries")
        ch = None
        if choli is not None:
            ch = np.ascontiguousarray(choli, dtype=np.float64)
            if ch.shape != (M1, M1):
                raise ValueError(f"choli must be [{M1},{M1}]")
        _check(self.lib, self.lib.sgpr_append_inducing(self._h, n, _ptr(Z), _ptr(first), _ptr(r), _ptr(b), _ptr(mu),
                                                       _ptr(ch) if ch is not None else None))
        m = self.model
        m.ind_first = np.concatenate([m.ind_first, m.ind_first[-1] + first[1:]])
        m.ind_Z = np.concatenate([m.ind_Z, Z])
        m.ind_r = np.concatenate([m.ind_r, r])
        m.ind_b = np.concatenate([m.ind_b, b])
        m.mu = mu
        m.choli = ch

    # ------------------------------------------------------------------ molecular dynamics (md.DeviceMD drives these)
    def md_init(self, pos_t, z_t, cell, pbc, params, F, beta, state):
        """``sgpr_md_init``: F [N,3] (and beta [N] when ``params.stop_on_uncertain``) of pos_t, state reset; enqueued on
        torch's current stream, validated by ``sgpr_check`` after synchronising."""
        cell_h, pbc_h = self._geom(cell, pbc)
        _check(self.lib, self.lib.sgpr_md_init(self._h, z_t.numel(), c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()),
                                               _ptr(cell_h), _ptr(pbc_h), ctypes.byref(params), self._stream(),
                                               c_void_p(F.data_ptr()), c_void_p(beta.data_ptr()) if beta is not None else None,
                                               c_void_p(state.data_ptr())))

    def md_steps(self, pos_t, mom_t, z_t, mass_t, cell, pbc, params, n_steps, F, thermo, beta, state):
        """``sgpr_md_steps``: enqueue n_steps MD steps on torch's current stream (include/sgpr_b200.h)."""
        cell_h, pbc_h = self._geom(cell, pbc)
        _check(self.lib, self.lib.sgpr_md_steps(self._h, z_t.numel(), c_void_p(pos_t.data_ptr()), c_void_p(mom_t.data_ptr()),
                                                c_void_p(z_t.data_ptr()), c_void_p(mass_t.data_ptr()), _ptr(cell_h), _ptr(pbc_h),
                                                ctypes.byref(params), int(n_steps), self._stream(), c_void_p(F.data_ptr()),
                                                c_void_p(thermo.data_ptr()),
                                                c_void_p(beta.data_ptr()) if beta is not None else None,
                                                c_void_p(state.data_ptr())))

    # ------------------------------------------------------------------ geometry relaxation (relax.DeviceRelax drives these)
    def relax_init(self, pos_t, z_t, fixed, cell, pbc, params, F, beta, fire, state):
        """``sgpr_relax_init``: F [N,3] (and beta [N] when ``params.stop_on_uncertain``) of pos_t with the rows of
        ``fixed`` (uint8 [N] or None) zeroed, FIRE scalars and state reset; validated by ``sgpr_check`` after
        synchronising."""
        cell_h, pbc_h = self._geom(cell, pbc)
        _check(self.lib, self.lib.sgpr_relax_init(self._h, z_t.numel(), c_void_p(pos_t.data_ptr()), c_void_p(z_t.data_ptr()),
                                                  c_void_p(fixed.data_ptr()) if fixed is not None else None, _ptr(cell_h),
                                                  _ptr(pbc_h), ctypes.byref(params), self._stream(), c_void_p(F.data_ptr()),
                                                  c_void_p(beta.data_ptr()) if beta is not None else None,
                                                  c_void_p(fire.data_ptr()), c_void_p(state.data_ptr())))

    def relax_steps(self, pos_t, vel_t, z_t, fixed, cell, pbc, params, n_steps, F, trace, beta, fire, state):
        """``sgpr_relax_steps``: enqueue n_steps FIRE steps on torch's current stream (include/sgpr_b200.h)."""
        cell_h, pbc_h = self._geom(cell, pbc)
        _check(self.lib, self.lib.sgpr_relax_steps(self._h, z_t.numel(), c_void_p(pos_t.data_ptr()), c_void_p(vel_t.data_ptr()),
                                                   c_void_p(z_t.data_ptr()),
                                                   c_void_p(fixed.data_ptr()) if fixed is not None else None, _ptr(cell_h),
                                                   _ptr(pbc_h), ctypes.byref(params), int(n_steps), self._stream(),
                                                   c_void_p(F.data_ptr()), c_void_p(trace.data_ptr()),
                                                   c_void_p(beta.data_ptr()) if beta is not None else None,
                                                   c_void_p(fire.data_ptr()), c_void_p(state.data_ptr())))

    def check_status(self):
        """``sgpr_check`` without raising: (status, message) -- SGPR_ERR_RETRY (-7) is a step to repeat, not a failure."""
        st = self.lib.sgpr_check(self._h, None)
        return int(st), (self.lib.sgpr_last_error().decode(errors="replace") if st else "")

    def set_async(self, on=True):
        """Device-pointer entry points (predict_device, peer exchange) enqueue warm steps without synchronising; call
        ``check()`` after synchronising the stream (include/sgpr_b200.h, "Asynchronous steps")."""
        _check(self.lib, self.lib.sgpr_set_async(self._h, 1 if on else 0))

    def check(self):
        """Validate the asynchronous steps since the last check; returns the pair count of the last step.  Raises
        ``RuntimeError`` (SGPR_ERR_RETRY ...) if one of them was invalid: repeat it."""
        n = c_int64(0)
        _check(self.lib, self.lib.sgpr_check(self._h, ctypes.byref(n)))
        return int(n.value)

    def enable_timing(self, on=True):
        _check(self.lib, self.lib.sgpr_enable_timing(self._h, 1 if on else 0))

    def stats(self):
        s = sgpr_stats()
        _check(self.lib, self.lib.sgpr_get_stats(self._h, ctypes.byref(s)))
        return {k: getattr(s, k) for k, _ in sgpr_stats._fields_}
