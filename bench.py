#!/usr/bin/env python
"""bench.py -- atom-steps/sec of SGPR E+F+stress prediction (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl reference] [--dump-outputs DIR]

A step = one full evaluation (neighbour list -> descriptors -> kernel GEMMs -> energy,
forces, virial) of one synthetic structure.  Workload (default c3, the configuration the
metric's target is quoted on): 4-species Li/P/S/O-like 97,556-atom fcc-derived solid,
random-init frozen model with M = 2000 inducing LCEs, SeSoap lmax=3 nmax=3 rc=6.
Prints ONE JSON line (see DESIGN.md "Measurement").
"""
from __future__ import annotations

import os
import sys

if "--impl" in sys.argv and "reference" in sys.argv:
    # the CPU arm runs one single-threaded process per core: pin the BLAS/OpenMP pools BEFORE numpy / torch load
    for _k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[_k] = "1"

import argparse
import json
import statistics
import subprocess
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "atom-steps/sec (E+F+stress) SGPR MD prediction"
UNIT = "atom-steps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="c3")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="atoms in the CPU-baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--variants", type=int, default=4, help="pre-generated perturbed position sets cycled over the steps")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "p2p-nccl", "halo"],
                    help="multi-GPU force exchange: peer-memory adds over NVLink with the fused mailbox/flag exchange step "
                         "(default), the same with an NCCL all-reduce of E + virial as the barrier, or halo recompute")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's energy, forces and virial to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the GPU path (--impl b200)")
    return args


def dump_outputs(dirname, E, F, W):
    """What a caller of the timed path receives from its last step: energy [1], forces [N,3], virial [3,3], float64.
    The inputs are seeded, so two builds run with the same arguments can be compared output for output: energy and
    virial repeat bit for bit, forces to rounding (atomic adds in the force scatter; 2e-15 eV/A apart at c3 on a B200).
    The largest workload (c5, 1,000,188 atoms) writes 24 MB."""
    os.makedirs(dirname, exist_ok=True)
    for name, a in (("energy", [E]), ("forces", F), ("virial", W)):
        np.save(os.path.join(dirname, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def workload_inputs(name, variants):
    from autoforce_b200 import synth

    w = synth.WORKLOADS[name]
    pos, cell, numbers = synth.fcc(w["rep"], w["Zs"], 0.1, 0)
    rng = np.random.default_rng(123)
    # every step sees perturbed positions, N(0, 0.03 A) (SURVEY.md 8d); generated before timing
    pos_variants = [pos + rng.normal(0, 0.03, pos.shape) for _ in range(max(1, variants))]
    return w, pos_variants, cell, numbers


def config_of(name, w, N, M, world):
    """Identical for the b200 and the reference arm of one (workload, N GPUs) pair."""
    return {
        "workload": f"{name}: fcc-derived {N}-atom {'/'.join(str(z) for z in w['Zs'])} solid, frozen random-init SGPR model "
                    f"M={M}, SeSoap lmax={w['lmax']} nmax={w['nmax']} rc={w['rc']}, xi=4",
        "atoms": N, "inducing": M, "species": len(w["Zs"]),
        "parallelism": f"atoms sharded over {world} GPU(s); positions replicated; all-reduce of E + 3x3 virial only",
        "cache": "working set (pair list + descriptor/gradient matrices, >500 MB at c3) exceeds the 126 MB L2; positions change every step",
    }


DTYPE = "f64 results (neighbour list, descriptors, forces in float64; kernel GEMMs as exact int8 x 6-slice tcgen05 products of 46-bit fixed-point operands, float64 epilogues)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class NvmlSampler:
    """SM clock + throttle reasons through NVML from a polling thread (every ~2 ms): the timed region of a sharded run is
    a few milliseconds, shorter than the start-up of an `nvidia-smi -lms` process.  Same result keys as ClockSampler."""
    REASONS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, torch_index):
        import threading

        import pynvml
        import torch

        self.nv = pynvml
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(torch_index).uuid)
        if not uuid.startswith("GPU-"):
            uuid = "GPU-" + uuid
        self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
        self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        self.sm, self.bits, self.stop_flag = [], 0, False
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _once(self):
        self.sm.append(float(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
        try:
            self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            self.bits |= int(self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _run(self):
        while not self.stop_flag:
            self._once()
            time.sleep(0.002)

    def start(self):
        self.thread.start()

    def stop(self):
        self._once()          # at least one sample, taken while the last steps are still in flight or just retired
        self.stop_flag = True
        self.thread.join(timeout=2)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "samples": len(self.sm),
                "reasons": sorted(k for k, b in self.REASONS.items() if self.bits & b), "source": "nvml"}


def make_sampler(index):
    try:
        return NvmlSampler(index)
    except Exception:
        return ClockSampler(index)


def dgemm_peak_tflops():
    """FP64 GEMM peak of this GPU measured in-run (cuBLAS DGEMM 8192^3, best of 5):
    MEASURED_PEAKS.json only lists bf16, and the kernel GEMMs run on the FP64 pipe."""
    import torch

    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n**3 / (best * 1e-3) / 1e12


def int8_peak_tops():
    """Dense int8 tensor throughput of this GPU measured in-run: cuBLASLt IMMA 8192^3 through torch._int_mm
    (2 N^3 operations, best of 10).  MEASURED_PEAKS.json lists bf16 only."""
    import torch

    n = 8192
    a = torch.randint(-100, 100, (n, n), dtype=torch.int8, device="cuda")
    b = torch.randint(-100, 100, (n, n), dtype=torch.int8, device="cuda")
    torch._int_mm(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(10):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch._int_mm(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n**3 / (best * 1e-3) / 1e12


def reference_sample_plan(w, procs):
    """Atoms per process of the reference's bounded sample: ~3 s of reference work per step
    (3.8 ms N + 0.34 ms N M_sameZ per process, BASELINE.md section 2)."""
    m_same = w["M"] / len(w["Zs"])
    apc = max(2, min(16, int(round(3.0 / (0.0038 + 0.00034 * m_same)))))
    return apc


def run_reference(workload, steps, warmup, procs=None):
    """The reference's own ActiveCalculator.calculate on the host cores (oracle/ref_bench.py); falls back to the numpy
    port when the reference package is not available (neither /root/reference nor oracle/_ref)."""
    from autoforce_b200 import synth
    from oracle import ref_bench, ref_runner

    w = synth.WORKLOADS[workload]
    procs = procs or min(os.cpu_count() or 1, 64)
    if ref_runner.reference_available():
        apc = reference_sample_plan(w, procs)
        out = ref_bench.run(workload, steps, warmup, procs, rep=ref_bench.sample_rep(procs, apc), timeout=1500)
        nodes = out["node_seconds"]
        sample = (f"the UNMODIFIED reference (theforce ActiveCalculator.calculate, prediction mode, {out['reference']} copy) on a "
                  f"{out['atoms']}-atom periodic cell of the same family (fcc rep {out['rep']}, same species mix / rattle / per-step "
                  f"perturbation / kernel / all {out['M']} inducing LCEs), evaluated in full every step by {procs} processes x 1 thread "
                  f"(the reference's own atom decomposition + all-reduces over a gloo-backed mpi4py stand-in; OMP/MKL threads = 1); "
                  f"reference cost is linear in atoms at fixed M; per-step nodes [s]: nl+desc {nodes['nl_desc']:.3g}, kernel "
                  f"{nodes['kernel']:.3g}, autograd {nodes['results']:.3g}, covloss {nodes['covloss']:.3g}; neighbour list from the "
                  f"ase stand-in (ASE is not installed)")
        return dict(value=out["value"], ms_per_step=out["ms_per_step"], cores=procs, kind="reference", sample=sample, work=out["work"])
    return run_port(workload, steps, warmup, procs)


def run_port(workload, steps, warmup, procs=None, timeout=300):
    """The numpy restatement (oracle/sgpr_oracle.py) on the host cores: a sample of the full-size structure's
    environments per step.  Second CPU figure next to the reference's (it is vectorised where the reference loops in
    Python, so it is the faster of the two), and the fallback when the reference package is absent.
    Runs in a fresh interpreter (its worker pool forks; this process may hold a CUDA context) with a hard time limit."""
    procs = procs or min(os.cpu_count() or 1, 64)
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "OPENBLAS_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        env[k] = "1"
    env["CUDA_VISIBLE_DEVICES"] = ""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--port-worker", workload, str(steps), str(warmup), str(procs)]
    r = subprocess.run(cmd, env=env, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    if r.returncode != 0:
        raise RuntimeError("numpy port worker failed: " + r.stderr[-500:])
    return json.loads(r.stdout.strip().splitlines()[-1])


def port_worker(workload, steps, warmup, procs):
    from autoforce_b200 import synth
    from oracle.cpu_bench import CpuBench
    from oracle.sgpr_oracle import neighbor_list

    w = synth.WORKLOADS[workload]
    pos_variants, cell, numbers = workload_inputs(workload, 4)[1:]
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"], neighbors_fn=neighbor_list)
    cb = CpuBench(model, pos_variants, cell, numbers, 32 * procs, procs)
    value, sec = cb.run(steps, warmup)
    cb.close()
    print(json.dumps(dict(value=value, ms_per_step=sec * 1e3, cores=procs, kind="port",
                          sample=f"{cb.sample} of {len(numbers)} atoms per step (full neighbour environments, all {model.M} inducing "
                                 f"LCEs), {procs} worker processes x 1 thread; oracle/sgpr_oracle.py (vectorised numpy restatement)",
                          work=None)), flush=True)


def cpu_arm(args, world, rank):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores."""
    if rank != 0:
        return
    from autoforce_b200 import synth

    w = synth.WORKLOADS[args.workload]
    N = 4 * w["rep"] ** 3
    r = run_reference(args.workload, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": config_of(args.workload, w, N, w["M"], max(1, args.gpus)),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- parity (outside the timed regions)
def _periodic_nl(pos, cell, rc, centres):
    """(first, J, S) rows of ``centres`` in an orthorhombic periodic cell with L > 2 rc: k-d tree candidates, then the
    reference's own distance test (descriptor/atoms.py:366-368 op order via oracle.displacements)."""
    from scipy.spatial import cKDTree

    from oracle import sgpr_oracle as o

    L = np.diag(cell)
    wrapped = pos - np.floor(pos / L) * L
    wrapped = np.where(wrapped >= L, wrapped - L, wrapped)
    tree = cKDTree(wrapped, boxsize=L)
    cand = tree.query_ball_point(wrapped[centres], rc * (1 + 1e-9) + 1e-9)
    N = len(pos)
    first = np.zeros(N + 1, np.int64)
    rows = {}
    for i, js in zip(centres, cand):
        js = np.array(sorted(j for j in js if j != i), dtype=np.int64)
        S = -np.round((pos[js] - pos[i]) / L).astype(np.int64)
        d = o.displacements(pos, cell, int(i), js, S)
        keep = np.sqrt((d * d).sum(axis=1)) < rc
        rows[int(i)] = (js[keep], S[keep])
    J, S = [], []
    for i in range(N):
        if i in rows:
            J.append(rows[i][0])
            S.append(rows[i][1])
            first[i + 1] = len(rows[i][0])
    first = np.cumsum(first)
    return first, (np.concatenate(J) if J else np.zeros(0, np.int64)), (np.concatenate(S) if S else np.zeros((0, 3), np.int64))


def parity_full_size(eng, model, pos, cell, numbers, F_gpu, n_probe=3, want_nl=True):
    """Sampled atoms of the FULL-SIZE structure against the oracle port: neighbour rows as sets, and the complete force
    on each probe atom (its own environment + every environment it is a neighbour of)."""
    from oracle import sgpr_oracle as o
    from oracle.cpu_bench import to_oracle_model

    rc = model.rc
    rng = np.random.default_rng(99)
    probes = np.sort(rng.choice(len(pos), n_probe, replace=False))
    f0, J0, S0 = _periodic_nl(pos, cell, rc, probes)
    centres = np.unique(np.concatenate([probes] + [J0[f0[i]:f0[i + 1]] for i in probes]))
    nl = _periodic_nl(pos, cell, rc, centres)
    om = to_oracle_model(model)
    ref = o.predict(om, pos, cell, True, numbers.astype(np.int64), atoms=centres, nl=nl, chunk=64)
    out = {"probe_atoms": [int(i) for i in probes], "environments_checked": int(len(centres)),
           "max_abs_dF": float(np.abs(F_gpu[probes] - ref["forces"][probes]).max())}
    if want_nl:
        first, J, S = eng.neighbors(pos, numbers, cell, True)
        same = True
        for i in centres:
            a = sorted(zip(J[first[i]:first[i + 1]].tolist(), map(tuple, S[first[i]:first[i + 1]].astype(np.int64).tolist())))
            b = sorted(zip(nl[1][nl[0][i]:nl[0][i + 1]].tolist(), map(tuple, nl[2][nl[0][i]:nl[0][i + 1]].tolist())))
            same &= a == b
        out["neighbour_rows_identical"] = bool(same)
        out["pairs_total"] = int(len(J))
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        cpu_arm(args, world, rank)
        return
    import torch
    import torch.distributed as dist

    import autoforce_b200 as ab
    from autoforce_b200 import synth

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # all device work of the bench runs on ONE explicit (non-default) stream: the library captures its warm steps into
    # CUDA graphs, which the legacy default stream does not allow; the CUDA events below are recorded on the same stream
    torch.cuda.set_stream(torch.cuda.Stream(device=dev))

    w, pos_variants, cell, numbers = workload_inputs(args.workload, args.variants)
    N = len(numbers)
    model = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"])
    eng = ab.SgprEngine(model, species=w["Zs"], device=local_rank)
    pbc = True
    pos_d = [torch.as_tensor(p, device=dev) for p in pos_variants]
    z_d = torch.as_tensor(numbers.astype(np.int32), device=dev)
    out = (torch.empty(1, dtype=torch.float64, device=dev), torch.empty((N, 3), dtype=torch.float64, device=dev),
           torch.empty(9, dtype=torch.float64, device=dev))
    ew = torch.zeros(10, dtype=torch.float64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def pick_exchange(engine, n_atoms):
        """-> (mode, PeerForceExchange | None), agreed by all ranks."""
        if world == 1:
            return "none", None
        mode, px_ = args.exchange, None
        if mode in ("p2p", "p2p-nccl"):
            try:
                px_ = engine.peer_exchange(n_atoms, fused=(mode == "p2p"))
            except Exception as ex:  # symmetric memory unavailable -> halo recompute
                if rank == 0:
                    print(f"bench: peer-memory exchange unavailable ({ex}); falling back to halo recompute", file=sys.stderr)
                mode = "halo"
        ok = torch.tensor([1 if px_ is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            mode, px_ = "halo", None
        return mode, px_

    exchange, px = pick_exchange(eng, N)
    # host buffers of the end-to-end leg are page-locked (inputs and the force output)
    pin_variants = [torch.from_numpy(p).pin_memory() for p in pos_variants]
    pin_F = torch.empty((N, 3), dtype=torch.float64).pin_memory()
    pin_F_np = pin_F.numpy()
    pin_Z = torch.from_numpy(np.ascontiguousarray(numbers, dtype=np.int32)).pin_memory()
    dev_pos = torch.empty((N, 3), dtype=torch.float64, device=dev) if px is not None else None

    def step_device(it):
        if px is not None:
            return px.step(pos_d[it % len(pos_d)], z_d, cell, pbc)
        E, F, W = eng.predict_device(pos_d[it % len(pos_d)], z_d, cell, pbc, rank=rank, world=world, out=out)
        if world > 1:  # the only collective of the path: 10 doubles
            ew[0:1].copy_(E)
            ew[1:].copy_(W)
            dist.all_reduce(ew)
        return E, F, W, None

    def step_host(it):
        if px is not None:   # host buffers in and out around the peer-memory step
            dev_pos.copy_(pin_variants[it % len(pin_variants)], non_blocking=True)
            E, F, W, owned = px.step(dev_pos, z_d, cell, pbc)
            pin_F.copy_(F, non_blocking=True)
            Eh = float(E.item())   # D2H of the reduced energy: synchronises the step
            torch.cuda.current_stream().synchronize()
            return Eh
        E, F, W, owned = eng.predict(pin_variants[it % len(pin_variants)].numpy(), pin_Z.numpy(), cell, pbc, rank=rank,
                                     world=world, out_forces=pin_F_np)
        if world > 1:
            t = torch.tensor([E] + list(W.reshape(-1)), dtype=torch.float64, device=dev)
            dist.all_reduce(t)
            E = float(t[0].item())
        return E

    def timed(fn, steps, warmup):
        """-> (device ms, wall ms, what the last timed step returned)"""
        for it in range(warmup):
            fn(it)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for it in range(steps):
            last = fn(it)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = max(e0.elapsed_time(e1), 0.0)
        t = torch.tensor([ms, wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0].item()), float(t[1].item()), last

    def full_results(res):
        """(E, F [N,3] device tensor, W [3,3]) of one step_device() result, summed over the ranks where the step leaves
        partial results.  A collective when sharded: every rank calls it; read it before the next step overwrites it."""
        if px is not None:
            Fd = res[1] * res[3].to(torch.float64)[:, None]
            dist.all_reduce(Fd)
            return float(res[0].item()), Fd, res[2].cpu().numpy().reshape(3, 3)
        Fd = res[1].clone()
        if world > 1:
            dist.all_reduce(Fd)   # halo mode: forces only on owned atoms, zeros elsewhere
            return float(ew[0].item()), Fd, ew[1:].cpu().numpy().reshape(3, 3)
        return float(res[0].item()), Fd, res[2].cpu().numpy().reshape(3, 3)

    # ---- device-resident leg (value): no in-library events, no stats calls inside the timed region; after the first
    # (sizing) step the library enqueues every step without host synchronisation -- validated after the timed region
    eng.set_async(True)
    sampler = make_sampler(local_rank)
    sampler.start()
    ms_dev, wall_dev, last = timed(step_device, args.steps, args.warmup)
    clocks = sampler.stop()
    eng.check()          # raises if any asynchronous step was invalid (pair list outgrew its capacity ...)
    if args.dump_outputs:
        E_last, F_last, W_last = full_results(last)
        if rank == 0:
            dump_outputs(args.dump_outputs, E_last, F_last.cpu().numpy(), W_last)
    launches_per_step = eng.stats()["kernel_launches"] + (1 if px is not None else 0)
    # ---- stage split: a separate, untimed pass with CUDA events between the stages inside the library
    eng.enable_timing(True)
    stage = {"ms_nl": 0.0, "ms_desc": 0.0, "ms_gemm": 0.0, "ms_force": 0.0, "ms_beta": 0.0, "ms_total": 0.0, "gemm_flops": 0.0, "i8_ops": 0.0}
    n_stage = max(1, min(args.steps, 10))
    samples = {k: [] for k in stage}
    for it in range(n_stage):
        step_device(it)
        st_ = eng.stats()
        for k in samples:
            samples[k].append(st_[k])
        stage["n_active"], stage["n_pairs"] = st_["n_active"], st_["n_pairs"]
    for k in ("ms_nl", "ms_desc", "ms_gemm", "ms_force", "ms_beta", "ms_total", "gemm_flops", "i8_ops"):
        stage[k] = statistics.median(samples[k])   # (the pass synchronises every step: a median, not a mean)
    eng.enable_timing(False)
    if os.environ.get("SGPR_BENCH_ALLRANKS"):
        print(f"rank {rank}: " + " ".join(f"{k[3:]}={stage[k]:.4f}" for k in ("ms_nl", "ms_desc", "ms_gemm", "ms_force", "ms_beta", "ms_total")),
              file=sys.stderr, flush=True)
    # ---- end-to-end leg: host buffers through the public host API (H2D + D2H inside)
    ms_e2e, wall_e2e, _ = timed(step_host, args.steps, args.warmup)
    eng.check()

    # ---- parity, outside the timed regions, every N
    parity = {}
    try:
        # (1) full-size structure: sampled atoms against the oracle port
        res = step_device(0)
        torch.cuda.synchronize()
        E_sh, Fd, W_sh = full_results(res)
        F_gpu = Fd.cpu().numpy()
        if rank == 0:
            parity["full_size_vs_oracle_port"] = parity_full_size(eng, model, pos_variants[0], cell, numbers, F_gpu,
                                                                   n_probe=3 if N <= 200000 else 2)
            if world > 1:   # the sharded step (this run's exchange mode) against the unsharded one on rank 0's GPU
                E1, F1, W1 = eng.predict_device(pos_d[0], z_d, cell, pbc, rank=0, world=1)
                torch.cuda.synchronize()
                parity["sharded_vs_unsharded_full_size"] = {
                    "dE_per_atom": abs(E_sh - float(E1.item())) / N, "max_abs_dF": float((Fd - F1).abs().max().item()),
                    "max_abs_dW": float(np.abs(W_sh - W1.cpu().numpy().reshape(3, 3)).max())}
        # (2) a small cell of the same family against committed results of the UNMODIFIED reference
        fx_path = os.path.join(ROOT, "tests", "golden", f"bench_{args.workload}_sample.npz")
        if os.path.exists(fx_path):
            fx = np.load(fx_path)
            model_c = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"], with_choli=True)
            eng_c = ab.SgprEngine(model_c, species=w["Zs"], device=local_rank)
            Nc = len(fx["numbers"])
            # sharded runs take the owner-computes (halo) entry point here: the peer-memory exchange is checked at full
            # size above (sharded == unsharded); beta only at N = 1
            r_ = eng_c.predict(fx["pos"], fx["numbers"], fx["cell"], True, rank=rank, world=world, want_beta=(world == 1))
            Ec, Fc, Wc = r_[0], r_[1], r_[2]
            beta = r_[4] if world == 1 else None
            if world > 1:
                t = torch.tensor([Ec] + list(Wc.reshape(-1)), dtype=torch.float64, device=dev)
                dist.all_reduce(t)
                Ft = torch.as_tensor(Fc, device=dev)
                dist.all_reduce(Ft)
                Ec, Wc, Fc = float(t[0].item()), t[1:].cpu().numpy().reshape(3, 3), Ft.cpu().numpy()
            vol = abs(np.linalg.det(fx["cell"]))
            stress = (np.asarray(Wc).reshape(3, 3) / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]]
            parity["sample_cell_vs_reference"] = {
                "what": f"{Nc}-atom cell of the same family, results of the unmodified reference committed in tests/golden/"
                        f"bench_{args.workload}_sample.npz (tests/golden/make_bench_fixture.py)",
                "dE_per_atom": abs(Ec - float(fx["energy"])) / Nc, "max_abs_dF": float(np.abs(Fc - fx["forces"]).max()),
                "max_abs_dstress": float(np.abs(stress - fx["stress"]).max()),
                "max_abs_dcovloss": None if beta is None else float(np.abs(beta - fx["covloss"]).max()),
                "tolerances": {"dE_per_atom": 1e-6, "dF": 1e-5, "dstress": 1e-6},
            }
            eng_c.close()
            p_ = parity["sample_cell_vs_reference"]
            parity["ok"] = bool(p_["dE_per_atom"] < 1e-6 and p_["max_abs_dF"] < 1e-5 and p_["max_abs_dstress"] < 1e-6)
        if rank == 0 and "full_size_vs_oracle_port" in parity:
            f_ = parity["full_size_vs_oracle_port"]
            parity["ok"] = bool(parity.get("ok", True) and f_["max_abs_dF"] < 1e-5 and f_.get("neighbour_rows_identical", True))
            if "sharded_vs_unsharded_full_size" in parity:
                s_ = parity["sharded_vs_unsharded_full_size"]
                parity["ok"] = bool(parity["ok"] and s_["dE_per_atom"] < 1e-9 and s_["max_abs_dF"] < 1e-8)
    except Exception as ex:  # pragma: no cover
        parity["error"] = f"{type(ex).__name__}: {ex}"
        parity["ok"] = False

    if rank == 0:
        K = args.steps
        value = N * K / (ms_dev * 1e-3)
        e2e = N * K / (wall_e2e * 1e-3)
        gemm_s = stage["ms_gemm"] * 1e-3
        fp64_equiv = stage["gemm_flops"] / gemm_s / 1e12 if gemm_s > 0 else None
        try:
            dgemm_peak = dgemm_peak_tflops()
        except Exception:  # pragma: no cover
            dgemm_peak = None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6536.0))
        use_i8 = stage["i8_ops"] > 0
        if use_i8:
            # the GEMMs run on tcgen05 as int8 digit-slice products: roofline in int8 tensor operations
            achieved = stage["i8_ops"] / gemm_s / 1e12
            try:
                peak = int8_peak_tops()
                peak_src = "measured in-run: cuBLASLt int8 GEMM 8192^3 via torch._int_mm, best of 10 (MEASURED_PEAKS.json lists bf16 only: 2 x its burst figure = %.0f)" % (2.0 * float(peaks.get("bf16_tflops", 1645.4)))
            except Exception as ex:  # pragma: no cover
                peak = 2.0 * float(peaks.get("bf16_tflops", 1645.4))
                peak_src = f"2 x measured dense bf16 peak of MEASURED_PEAKS.json (int8 probe failed: {ex})"
            kernel_name = "i8gemm_kernel (tcgen05.mma kind::i8, TMA + TMEM): FP64-accurate kernel GEMM + back projection as int8 digit-slice products"
            unit = "TOP/s (int8)"
        else:
            achieved = fp64_equiv
            peak = dgemm_peak if dgemm_peak else 40.0
            peak_src = "measured in-run: cuBLAS DGEMM 8192^3 (MEASURED_PEAKS.json has no FP64 entry)"
            kernel_name = "gemm_tn_kernel (FP64 DMMA kernel-matrix GEMM + back projection)"
            unit = "TFLOP/s"
        prof = {}
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            try:
                prof = json.load(open(tpath)).get(args.workload, {})
            except Exception:
                prof = {}
        traffic = prof.get("i8gemm_dram_bytes_per_launch" if use_i8 else "gemm_dram_bytes_per_launch")
        # per-stage HBM rooflines (north_star: achieved HBM GB/s of the descriptor and force stages): algorithmic bytes
        # per atom from SURVEY.md 8(d) / DESIGN.md 4 x atoms evaluated by this rank / measured stage time; ncu's
        # dram bytes and pipe utilisation of the same kernels come from the committed capture (profiles/)
        nn = stage.get("n_pairs", 0) / max(1, stage.get("n_active", 1))
        S_, nb_, L_ = len(w["Zs"]), w["nmax"] + 1, w["lmax"] + 1
        A_ = S_ * nb_
        Dp = A_ * (A_ + 1) // 2 * L_
        n_act = stage.get("n_active", N)
        alg = {
            "nl": n_act * (28 + 8 * nn),
            "desc": n_act * (32 * (1 + nn) + 8 * nn + 6 * Dp + 8 * A_ * L_ * L_),
            "force": n_act * (8 * Dp + 32 * (1 + nn) + 8 * nn + 8 * A_ * L_ * L_ + 24),
        }
        stages = {}
        for key, ms_key in (("nl", "ms_nl"), ("desc", "ms_desc"), ("force", "ms_force")):
            ms = stage[ms_key]
            gbs = alg[key] / (ms * 1e-3) / 1e9 if ms > 0 else None
            stages[key] = {"ms": ms, "algorithmic_bytes": alg[key], "achieved_gbs": gbs, "frac_hbm": gbs / hbm_peak if gbs else None,
                           "ncu": prof.get(f"stage_{key}")}
        stages["gemm"] = {"ms": stage["ms_gemm"], "achieved": achieved, "unit": unit, "frac_tensor": (achieved / peak) if achieved else None,
                          "ncu": prof.get("stage_gemm")}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": ms_dev / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE,
            "data": "synthetic", "config": config_of(args.workload, w, N, model.M, world),
            "exchange": {"p2p": "peer-memory adds over NVLink into the owner's buffer (no halo recompute); E + virial through "
                                "peer-mapped mailboxes with stamped flags (sgpr_p2p_step: no NCCL call in the step, one CUDA graph)",
                         "p2p-nccl": "peer-memory adds over NVLink into the owner's buffer; NCCL all-reduce of 10 doubles as barrier",
                         "halo": "owner-computes with one-cutoff halo recompute", "none": "single GPU"}[exchange],
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": wall_e2e / K,
                    "h2d_bytes_per_step": int(N * 24 + N * 4), "d2h_bytes_per_step": int(N * 24 + 16 * 8 + N)},
            "gpu_launches": int(launches_per_step * K),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": kernel_name,
                         "achieved": achieved, "peak": peak, "unit": unit, "frac": (achieved / peak) if achieved else None,
                         "traffic": traffic, "peak_source": peak_src,
                         "fp64_equivalent_tflops": fp64_equiv, "cublas_dgemm_tflops_in_run": dgemm_peak,
                         "int8_ops_per_step": stage["i8_ops"], "useful_int8_ops_per_step": 21 * stage["gemm_flops"],
                         "flops_per_step": stage["gemm_flops"], "gemm_ms_per_step": stage["ms_gemm"]},
            "roofline_stages": stages,
            "stages_ms_per_step": dict({k[3:]: stage[k] for k in ("ms_nl", "ms_desc", "ms_gemm", "ms_force", "ms_total")},
                                       **({"exchange": stage["ms_beta"]} if world > 1 else {})),
            "pairs": int(stage.get("n_pairs", 0)), "active_envs_rank0": int(stage.get("n_active", 0)),
            "parity": parity,
        }
        if world == 1:
            # covloss (calculator/active.py:781-804) runs every prediction step in the reference but is not part
            # of the metric (SURVEY.md 8d): reported separately, same structure, model with a dense lower-triangular choli
            try:
                model_c = synth.synth_model(w["Zs"], w["M"], 1, lmax=w["lmax"], nmax=w["nmax"], rc=w["rc"], with_choli="tril")
                eng_c = ab.SgprEngine(model_c, species=w["Zs"], device=local_rank)
                eng_c.enable_timing(True)
                tb, fl = [], 0.0
                for it in range(4):
                    eng_c.predict(pos_variants[it % len(pos_variants)], numbers, cell, pbc, want_beta=True)
                    st_c = eng_c.stats()
                    if it > 0:
                        tb.append(st_c["ms_beta"])
                        fl = st_c["covloss_flops"]
                eng_c.close()
                mb = sum(tb) / len(tb)
                line["covloss"] = {"ms_per_step": mb, "tflops": fl / (mb * 1e-3) / 1e12, "flops_per_step": fl,
                                   "note": "extra device time per step when beta is requested; tcgen05 int8 digit-slice GEMM K.choli^T (26 slice products; dense lower-triangular synthetic choli like the reference's L^-1, whose zero K-chunks are skipped; flops counted for the dense product) + row sum of squares"}
            except Exception as ex:  # pragma: no cover
                line["covloss"] = {"error": str(ex)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                r = run_reference(args.workload, 2, 1)
                line["cpu_baseline"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                                        "sample": "2 timed steps after 1 warm-up: " + r["sample"]}
            except Exception as ex:  # pragma: no cover
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {ex}"}
            if line["cpu_baseline"].get("kind") == "reference":
                try:   # the vectorised numpy port as a second CPU figure (VERDICT r1 item 3)
                    r = run_port(args.workload, 2, 1)
                    line["cpu_baseline_port"] = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                                                 "sample": "2 timed steps after 1 warm-up: " + r["sample"]}
                except Exception as ex:  # pragma: no cover
                    line["cpu_baseline_port"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {ex}"}
        elif world > 1:
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference",
                                    "sample": "timed at N = 1 only (it does not depend on the number of GPUs): see the N = 1 line, "
                                              "or `bench.py --impl reference`"}
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    if len(sys.argv) >= 6 and sys.argv[1] == "--port-worker":
        port_worker(sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]))
    else:
        main()
