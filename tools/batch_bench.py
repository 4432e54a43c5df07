"""Batched prediction against a loop of single-structure calls, on seeded workloads of small structures.

    python tools/batch_bench.py [--repeats R] [--scale S] [--out FILE]

For each workload, in one process on one GPU:
  batch        one sgpr_predict_batch call over all frames (device inputs and outputs);
  loop_device  one warm device-pointer sgpr_predict per frame (sgpr_set_async, frames copied into one fixed input
               buffer per atom count so that a steady shape replays its CUDA graph -- the loop's best case);
  loop_host    SgprEngine.predict per frame (host arrays: the calculator's path).
Times are medians over R repeats after one warm-up of every path, host clock around work that ends in a device
synchronisation.  The batch's working set (descriptor rows, digit slices, neighbour lists) is far above the 126 MB of
L2; a single small frame fits in it by nature.  Also reported: the largest batch-vs-loop difference in E/N, F and
stress, the batch's stage split (sgpr_enable_timing, a separate call), the per-atom time of a warm single step of the
c2 / c3 cells with the same models, and the card's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # pragma: no cover
        return {"gpu": None, "error": str(e)}


def frames_uniform(B, rep, Zs, seed):
    from autoforce_b200.synth import fcc

    out = []
    for b in range(B):
        pos, cell, Z = fcc(rep, Zs, 0.1, seed + b)
        out.append((pos, Z.astype(np.int32), cell, (True, True, True)))
    return out


def frames_mixed(B, Zs, seed):
    """32 .. 512 atoms, pbc (T,T,T), (T,T,F) or none."""
    from autoforce_b200.synth import fcc

    rng = np.random.default_rng(seed)
    reps = [(2, 2, 2), (3, 3, 2), (3, 3, 3), (4, 4, 2), (4, 4, 3), (4, 4, 4), (5, 5, 4), (4, 4, 8)]
    pbcs = [(True, True, True), (True, True, False), (False, False, False)]
    out = []
    for b in range(B):
        rep = reps[rng.integers(len(reps))]
        pbc = pbcs[rng.integers(len(pbcs))]
        pos, cell, Z = fcc(rep, Zs, 0.1, seed + 1000 + b)
        out.append((pos, Z.astype(np.int32), cell if pbc[0] else np.zeros((3, 3)), pbc))
    return out


def sync():
    import torch

    torch.cuda.synchronize()


def median_time(fn, repeats):
    ts = []
    for _ in range(repeats):
        sync()
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), [float(t) for t in ts]


def stress(W, cell):
    vol = abs(np.linalg.det(np.asarray(cell, dtype=float).reshape(3, 3))) or -2.0
    return (W / vol).reshape(-1)[[0, 4, 8, 5, 2, 1]]


def run_workload(name, model, frames, repeats):
    import torch

    import autoforce_b200 as ab

    species = sorted(set(int(z) for f in frames for z in np.unique(f[1])))
    eng = ab.SgprEngine(model, species=species)
    dev = torch.device("cuda", 0)
    B = len(frames)
    counts = np.array([len(f[1]) for f in frames])
    first = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    N = int(first[-1])
    pos_all = torch.as_tensor(np.concatenate([f[0] for f in frames]), device=dev)
    z_all = torch.as_tensor(np.concatenate([f[1] for f in frames]), device=dev)
    cells = np.ascontiguousarray(np.stack([np.asarray(f[2], dtype=float).reshape(9) for f in frames]))
    pbcs = np.ascontiguousarray(np.array([f[3] for f in frames], dtype=np.int32))
    E_d = torch.zeros(B, dtype=torch.float64, device=dev)
    F_d = torch.zeros((N, 3), dtype=torch.float64, device=dev)
    W_d = torch.zeros((B, 9), dtype=torch.float64, device=dev)
    from ctypes import c_void_p

    from autoforce_b200.engine import _check, _ptr

    def batch():
        _check(eng.lib, eng.lib.sgpr_predict_batch(eng._h, B, _ptr(first), c_void_p(pos_all.data_ptr()),
                                                   c_void_p(z_all.data_ptr()), _ptr(cells), _ptr(pbcs), eng._stream(),
                                                   c_void_p(E_d.data_ptr()), c_void_p(F_d.data_ptr()),
                                                   c_void_p(W_d.data_ptr()), None))

    # device loop: one fixed input / output set per atom count (graph replay while the shape stays)
    bufs = {}
    for n in sorted(set(counts.tolist())):
        bufs[n] = (torch.zeros((n, 3), dtype=torch.float64, device=dev), torch.zeros(n, dtype=torch.int32, device=dev),
                   torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros((n, 3), dtype=torch.float64, device=dev),
                   torch.zeros(9, dtype=torch.float64, device=dev))
    loop_E = torch.zeros(B, dtype=torch.float64, device=dev)
    loop_F = torch.zeros((N, 3), dtype=torch.float64, device=dev)
    loop_W = torch.zeros((B, 9), dtype=torch.float64, device=dev)
    eng.set_async(True)

    def loop_device():
        for b in range(B):
            n = int(counts[b])
            p, z, E, F, W = bufs[n]
            p.copy_(pos_all[first[b]:first[b + 1]], non_blocking=True)
            z.copy_(z_all[first[b]:first[b + 1]], non_blocking=True)
            eng.predict_device(p, z, frames[b][2], frames[b][3], out=(E, F, W))
            loop_E[b:b + 1].copy_(E, non_blocking=True)
            loop_F[first[b]:first[b + 1]].copy_(F, non_blocking=True)
            loop_W[b].copy_(W, non_blocking=True)
        sync()
        eng.check()

    host_out = [None] * B

    def loop_host():
        for b, f in enumerate(frames):
            host_out[b] = eng.predict(f[0], f[1], f[2], f[3])[:3]

    res = {"workload": name, "frames": B, "atoms": N, "atoms_per_frame": [int(counts.min()), int(counts.max())],
           "M": int(model.M), "species": species}
    for label, fn in (("batch", batch), ("loop_device", loop_device), ("loop_host", loop_host)):
        fn()   # warm-up (module loads, sizing steps, graph captures)
        t, ts = median_time(fn, repeats)
        res[label] = {"s": t, "frames_per_s": B / t, "atom_steps_per_s": N / t, "ns_per_atom": 1e9 * t / N,
                      "repeats_s": ts}
    res["batch_vs_loop_device"] = res["loop_device"]["s"] / res["batch"]["s"]
    res["batch_vs_loop_host"] = res["loop_host"]["s"] / res["batch"]["s"]
    # agreement: batch against the host loop (and the device loop)
    batch()
    sync()
    E, F, W = E_d.cpu().numpy(), F_d.cpu().numpy(), W_d.cpu().numpy()
    dE = dF = dS = 0.0
    for b, f in enumerate(frames):
        e1, f1, w1 = host_out[b]
        n = int(counts[b])
        dE = max(dE, abs(E[b] - e1) / n)
        dF = max(dF, float(np.abs(F[first[b]:first[b + 1]] - f1).max()))
        dS = max(dS, float(np.abs(stress(W[b], f[2]) - stress(np.asarray(w1), f[2])).max()))
    res["max_diff_vs_loop_host"] = {"E_per_atom": dE, "F": dF, "stress": dS}
    res["max_diff_vs_loop_device"] = {"E_per_atom": float(np.max(np.abs(E - loop_E.cpu().numpy()) / counts)),
                                      "F": float(np.abs(F - loop_F.cpu().numpy()).max()),
                                      "W": float(np.abs(W - loop_W.cpu().numpy()).max())}
    eng.enable_timing(True)
    batch()
    st = eng.stats()
    eng.enable_timing(False)
    res["batch_stages_ms"] = {k: float(st[k]) for k in ("ms_nl", "ms_desc", "ms_gemm", "ms_force", "ms_beta", "ms_total")}
    res["batch_pairs"] = int(st["n_pairs"])
    eng.close()
    return res


def single_step_ns_per_atom(model, workload, repeats):
    """Warm device-pointer step (graph replay) of bench.py's cell of the same family, per atom."""
    import torch

    import autoforce_b200 as ab
    from autoforce_b200 import synth

    w = synth.WORKLOADS[workload]
    pos, cell, Z = synth.fcc(w["rep"], w["Zs"], 0.1, 2)
    eng = ab.SgprEngine(model, species=w["Zs"])
    eng.set_async(True)
    p = torch.as_tensor(pos, device="cuda")
    z = torch.as_tensor(Z.astype(np.int32), device="cuda")
    out = eng.predict_device(p, z, cell, True)
    steps = 50

    def run():
        for _ in range(steps):
            eng.predict_device(p, z, cell, True, out=out)

    run()
    sync()
    t, _ = median_time(run, repeats)
    eng.check()
    eng.close()
    return {"workload": workload, "atoms": len(Z), "ns_per_atom": 1e9 * t / steps / len(Z), "step_ms": 1e3 * t / steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the frame counts (rehearsals)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("batch_bench.py needs a CUDA device")
    from autoforce_b200 import synth

    out = {"tool": "tools/batch_bench.py", **gpu_info(), "repeats": args.repeats, "workloads": []}
    c2, c3 = synth.WORKLOADS["c2"], synth.WORKLOADS["c3"]
    m2 = synth.synth_model(c2["Zs"], c2["M"], 1, lmax=c2["lmax"], nmax=c2["nmax"], rc=c2["rc"])
    m3 = synth.synth_model(c3["Zs"], c3["M"], 1, lmax=c3["lmax"], nmax=c3["nmax"], rc=c3["rc"])
    n = lambda k: max(1, int(round(k * args.scale)))   # noqa: E731
    out["workloads"].append(run_workload("cu108_c2model", m2, frames_uniform(n(2048), 3, [29], 100), args.repeats))
    out["workloads"].append(run_workload("4sp128_c3model", m3, frames_uniform(n(512), (4, 4, 2), c3["Zs"], 200), args.repeats))
    out["workloads"].append(run_workload("mixed32to512_c2model", m2, frames_mixed(n(1024), [29], 300), args.repeats))
    out["single_step"] = [single_step_ns_per_atom(m2, "c2", args.repeats), single_step_ns_per_atom(m3, "c3", args.repeats)]
    txt = json.dumps(out, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
