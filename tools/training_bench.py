"""Training-time kernels of many structures: one sgpr_kernel_jacobian_batch call against loops of single-structure calls.

    python tools/training_bench.py [--parent ROOT] [--repeats R] [--scale S] [--out FILE]

For each workload, in one run on one GPU, alternating repeat by repeat (median of R, host clock around work that ends
in a device synchronisation, every path warmed up first):
  batch        SgprEngine.training_kernels over all frames (Ke, Kf, Kv of every frame against every inducing LCE);
  loop         SgprEngine.kernel_jacobian per frame on this build (one Jacobian launch per frame);
  loop_parent  the same loop on the library and package under --parent (another checkout, built), run in a worker
               process -- e.g. the per-LCE backward passes the Jacobian kernel replaced.
Also reported: the Jacobian stage's time from CUDA events (sgpr_enable_timing, a separate call) and its achieved FP64
rate from the operation count below, a cuBLAS DGEMM (torch.matmul) measured in the same run, the largest differences
batch vs loop and batch vs loop_parent on the first frames, and the card's name and power limit.
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
N_COMPARE = 8   # frames whose outputs are compared between the paths


def jacobian_flops(model, frames, n_pairs):
    """FP64 operations of the Jacobian kernel (multiply-add = 2), from the shapes:
    per environment and LCE of its species  U_m = sum_b (z_m ttab) c   : 2 A^2 L2
    per pair and LCE of the centre's species  B = D f, Tn = D Y        : 4 nb L2, + 6 L2 (gradient), + 2 nb (radial)
    n_pairs[b][i]: neighbour count of atom i of frame b."""
    S = len(model.species())
    nb, L2 = model.nmax + 1, (model.lmax + 1) ** 2
    A = S * nb
    Ms = {int(z): int(np.sum(np.asarray(model.ind_Z) == z)) for z in model.species()}
    env = pair = 0.0
    for (pos, Z, cell, pbc), npb in zip(frames, n_pairs):
        for z, npi in zip(Z, npb):
            m = Ms.get(int(z), 0)
            if npi == 0 or m == 0:
                continue
            env += m * 2.0 * A * A * L2
            pair += m * npi * (4.0 * nb * L2 + 6.0 * L2 + 2.0 * nb)
    return env + pair


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clk = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:   # pragma: no cover
        return {"gpu": None, "error": str(e)}


def workloads(scale):
    from autoforce_b200 import synth

    sys.path.insert(0, os.path.join(ROOT, "tools"))
    from batch_bench import frames_mixed, frames_uniform

    c2, c3 = synth.WORKLOADS["c2"], synth.WORKLOADS["c3"]
    n = lambda k: max(1, int(round(k * scale)))   # noqa: E731
    m2 = lambda: synth.synth_model(c2["Zs"], c2["M"], 1, lmax=c2["lmax"], nmax=c2["nmax"], rc=c2["rc"])   # noqa: E731
    m3 = lambda: synth.synth_model(c3["Zs"], c3["M"], 1, lmax=c3["lmax"], nmax=c3["nmax"], rc=c3["rc"])   # noqa: E731
    return [("cu108_c2model", m2, lambda: frames_uniform(n(256), 3, [29], 100)),
            ("4sp128_c3model", m3, lambda: frames_uniform(n(128), (4, 4, 2), c3["Zs"], 200)),
            ("mixed32to256_c2model", m2, lambda: [f for f in frames_mixed(n(512), [29], 300) if len(f[1]) <= 256][:n(256)])]


def sync():
    import torch

    torch.cuda.synchronize()


def loop_outputs(eng, frames, keep):
    """kernel_jacobian per frame; Kf / Kv of the first `keep` frames as host arrays."""
    out = []
    for b, f in enumerate(frames):
        _, Kf, Kv = eng.kernel_jacobian(f[0], f[1], f[2], f[3])
        if b < keep:
            out.append((Kf.cpu().numpy(), Kv.cpu().numpy()))
    sync()
    return out


def worker(args):
    """Loop on the package under --root (the parent build), driven over stdin: "run" times one loop, "dump" writes the
    outputs of the first frames, "quit" ends."""
    sys.path.insert(0, args.root)
    import autoforce_b200 as ab

    name, mk_model, mk_frames = [w for w in workloads(args.scale) if w[0] == args.workload][0]
    model, frames = mk_model(), mk_frames()
    eng = ab.SgprEngine(model, species=sorted(set(int(z) for f in frames for z in np.unique(f[1]))))
    loop_outputs(eng, frames[:2], 0)
    print("ready", flush=True)
    for line in sys.stdin:
        cmd = line.split()
        if cmd[0] == "run":
            sync()
            t0 = time.perf_counter()
            loop_outputs(eng, frames, 0)
            print(time.perf_counter() - t0, flush=True)
        elif cmd[0] == "dump":
            out = loop_outputs(eng, frames, N_COMPARE)
            np.savez(cmd[1], *[a for kv in out for a in kv])
            print("ok", flush=True)
        else:
            break
    eng.close()


def run_workload(name, mk_model, mk_frames, args, tmp):
    import torch

    import autoforce_b200 as ab

    model, frames = mk_model(), mk_frames()
    species = sorted(set(int(z) for f in frames for z in np.unique(f[1])))
    eng = ab.SgprEngine(model, species=species)
    B, counts = len(frames), np.array([len(f[1]) for f in frames])
    first = np.concatenate([[0], np.cumsum(counts)])
    dev = torch.device("cuda", 0)
    pos = torch.as_tensor(np.concatenate([f[0] for f in frames]), device=dev)
    Z = torch.as_tensor(np.concatenate([f[1] for f in frames]).astype(np.int32), device=dev)
    cells = np.stack([np.asarray(f[2], dtype=float).reshape(3, 3) for f in frames])
    pbcs = np.array([f[3] for f in frames])
    batch = lambda: eng.training_kernels(pos, Z, first, cells, pbcs)   # noqa: E731
    parent = None
    if args.parent:
        parent = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", "--root", os.path.abspath(args.parent),
                                   "--workload", name, "--scale", str(args.scale)], stdin=subprocess.PIPE,
                                  stdout=subprocess.PIPE, text=True, cwd=os.path.abspath(args.parent))
        assert parent.stdout.readline().strip() == "ready"
    res = {"workload": name, "frames": B, "atoms": int(first[-1]), "atoms_per_frame": [int(counts.min()), int(counts.max())],
           "M": int(model.M), "species": species}
    batch()
    loop_outputs(eng, frames[:2], 0)
    sync()
    times = {"batch": [], "loop": [], "loop_parent": []}
    for _ in range(args.repeats):
        sync()
        t0 = time.perf_counter()
        batch()
        sync()
        times["batch"].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        loop_outputs(eng, frames, 0)
        times["loop"].append(time.perf_counter() - t0)
        if parent:
            parent.stdin.write("run\n")
            parent.stdin.flush()
            times["loop_parent"].append(float(parent.stdout.readline()))
    for k, ts in times.items():
        if ts:
            t = float(np.median(ts))
            res[k] = {"s": t, "frames_per_s": B / t, "repeats_s": ts}
    res["speedup_vs_loop"] = res["loop"]["s"] / res["batch"]["s"]
    if parent:
        res["speedup_vs_loop_parent"] = res["loop_parent"]["s"] / res["batch"]["s"]
    # the Jacobian stage from CUDA events, and its operation count
    eng.enable_timing(True)
    batch()
    st = eng.stats()
    eng.enable_timing(False)
    res["batch_stages_ms"] = {"nl": float(st["ms_nl"]), "desc": float(st["ms_desc"]), "kernel_matrix_and_Ke": float(st["ms_gemm"]),
                              "jacobian": float(st["ms_force"]), "total": float(st["ms_total"])}
    n_pairs = []
    for f in frames:
        fst, _, _ = eng.neighbors(f[0], f[1], f[2], f[3])
        n_pairs.append(np.diff(fst))
    flops = jacobian_flops(model, frames, n_pairs)
    res["jacobian_flop"] = flops
    res["jacobian_fp64_tflops"] = flops / (1e-3 * st["ms_force"]) / 1e12
    # agreement on the first frames
    Ke, Kf, Kv = (x.cpu().numpy() for x in batch())
    single = loop_outputs(eng, frames, N_COMPARE)
    diffs = {}

    def compare(label, outs):
        dF = dV = 0.0
        for b, (kf, kv) in enumerate(outs):
            kf_b = Kf[3 * first[b]:3 * first[b + 1]]
            dF = max(dF, float(np.abs(kf_b - kf).max(initial=0.0) / max(1e-300, np.abs(kf).max(initial=0.0))))
            dV = max(dV, float(np.abs(Kv[6 * b:6 * b + 6] - kv).max() / max(1e-300, np.abs(kv).max())))
        diffs[label] = {"Kf_rel": dF, "Kv_rel": dV, "frames": len(outs)}

    compare("batch_vs_loop", single)
    if parent:
        path = os.path.join(tmp, name + ".npz")
        parent.stdin.write(f"dump {path}\n")
        parent.stdin.flush()
        assert parent.stdout.readline().strip() == "ok"
        z = np.load(path)
        arrs = [z[f"arr_{i}"] for i in range(len(z.files))]
        compare("batch_vs_loop_parent", list(zip(arrs[0::2], arrs[1::2])))
        parent.stdin.write("quit\n")
        parent.stdin.flush()
        parent.wait(timeout=120)
    res["max_diff"] = diffs
    eng.close()
    return res


def dgemm_tflops():
    """cuBLAS DGEMM through torch, 8192^3, CUDA events."""
    import torch

    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(2):
        a @ b
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        a @ b
    e1.record()
    e1.synchronize()
    s = e0.elapsed_time(e1) * 1e-3 / reps
    return {"n": n, "s": s, "tflops": 2.0 * n ** 3 / s / 1e12}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", default=None, help="root of another built checkout: its kernel_jacobian loop is timed too")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the frame counts (rehearsals)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--root", default=ROOT, help=argparse.SUPPRESS)
    ap.add_argument("--workload", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    sys.path.insert(0, ROOT)
    import tempfile

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("training_bench.py needs a CUDA device")
    out = {"tool": "tools/training_bench.py", **gpu_info(), "repeats": args.repeats, "workloads": []}
    with tempfile.TemporaryDirectory() as tmp:
        for name, mk_model, mk_frames in workloads(args.scale):
            out["workloads"].append(run_workload(name, mk_model, mk_frames, args, tmp))
    out["cublas_dgemm"] = dgemm_tflops()
    for w in out["workloads"]:
        w["jacobian_share_of_dgemm"] = w["jacobian_fp64_tflops"] / out["cublas_dgemm"]["tflops"]
    txt = json.dumps(out, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
