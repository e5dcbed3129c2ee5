"""Jacobi-PCG with and without the compact values (spmv_compact = 0 / 1) on the benchmark's matrix, in one process.

    python tools/pcg_compact_probe.py OUT_DIR [--size 5792] [--rounds 7] [--cg-iters 25]

The workload is bench.py's: the P2 strip of `dist.strip_partition_device(n, n, 0, 1, jitter_amp=0.2, seed=1234)`,
assembled with its Dirichlet rows and columns.  Each round times, with CUDA events after a warm-up, one Jacobi-PCG of
exactly `--cg-iters` iterations per mode, alternating which mode goes first; the iterates must be equal bit for bit.
Bytes per apply are counted from the plan's shapes (values, one id byte per node row, x read and y written):

    full:    32 B per node block
    compact: 32 B per kept node block: every block but the 6 per cell of the vertex / opposite-edge pairs

Also reports the device memory left with the compact copy allocated (torch.cuda.mem_get_info) and writes
OUT_DIR/pcg_compact_probe.json with the card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "fem-libraries_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

MODES = {"compact": 0, "full": 1}   # spmv_compact value of each mode


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception as e:   # report what could be read
        name, power = torch.cuda.get_device_name(0), f"unavailable ({e})"
    return {"name": name, "power_limit": power}


def run(args) -> dict:
    import torch
    from femb200 import dist, fem
    torch.cuda.set_device(0)
    out = {"size": args.size, "card": card(), "rounds": args.rounds, "cg_iters": args.cg_iters}
    part = dist.strip_partition_device(args.size, args.size, 0, 1, jitter_amp=0.2, seed=1234)
    form = fem.ElasticityForm(part.mesh, part.E, 0.3)
    A = fem.create_matrix(form)
    A.set_bcs([fem.DirichletBC(part.bc, part.g)])
    fem.assemble_matrix(A, form)
    out["nnz_blocks"], out["nnodes"] = A.nnz_blocks, A.nnodes
    out["spmv_compact_keys"] = A.get_option("spmv_compact_keys")
    if out["spmv_compact_keys"] == 0:
        raise SystemExit("pcg_compact_probe: the plan has no compact keys")
    b = torch.where(part.bc != 0, part.g, torch.ones_like(part.g))
    cg = fem.CGSolver(rel_tol=0.0, max_iter=args.cg_iters)
    cg.SetOperator(A)
    cg.SetPreconditioner("jacobi")
    xs = {}
    for mode, v in MODES.items():          # warm-up; the first compact solve allocates the copy
        A.set_option("spmv_compact", v)
        xs[mode] = cg.Mult(b, fixed_iters=args.cg_iters).clone()
    torch.cuda.synchronize()
    kept = A.nnz_blocks - 6 * part.mesh.ncells
    out["kept_blocks"] = int(kept)
    out["compact_copy_gb"] = 32 * kept / 1e9
    out["mem_free_gb_with_copy"] = torch.cuda.mem_get_info()[0] / 1e9
    out["mem_total_gb"] = torch.cuda.mem_get_info()[1] / 1e9
    out["bitwise_equal_pcg_x"] = bool(torch.equal(xs["compact"], xs["full"]))
    ev = lambda: torch.cuda.Event(enable_timing=True)
    times = {m: [] for m in MODES}
    for r in range(args.rounds):
        for mode in (MODES if r % 2 == 0 else list(MODES)[::-1]):
            A.set_option("spmv_compact", MODES[mode])
            a, e = ev(), ev()
            a.record()
            cg.Mult(b, fixed_iters=args.cg_iters)
            e.record()
            torch.cuda.synchronize()
            times[mode].append(a.elapsed_time(e))
    # per-launch device time of the apply kernels (torch.profiler, one solve per mode after the timed rounds)
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for mode, v in MODES.items():
        A.set_option("spmv_compact", v)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            cg.Mult(b, fixed_iters=args.cg_iters)
            torch.cuda.synchronize()
        for ev_ in prof.events():
            if "spmv_tma_kernel" in ev_.name and ev_.device_time_total > 0:
                k = kern.setdefault(mode + ": " + ev_.name.split("(")[0].split("femb::")[-1], [])
                k.append(ev_.device_time_total / 1e3)
    out["apply_kernels_ms"] = {k: {"launches": len(v), "median_ms": float(np.median(v))} for k, v in kern.items()}
    A.set_option("spmv_compact", 0)
    bytes_apply = {"full": 32 * A.nnz_blocks + 33 * A.nnodes, "compact": 32 * int(kept) + 33 * A.nnodes}
    out["bytes_per_apply"] = bytes_apply
    out["modes"] = {}
    for mode, t in times.items():
        t = np.array(t)
        out["modes"][mode] = {"spmv_compact": MODES[mode], "pcg_ms_median": float(np.median(t)),
                              "pcg_ms_spread": float(t.max() - t.min()), "pcg_ms": t.tolist()}
    out["pcg_speedup"] = out["modes"]["full"]["pcg_ms_median"] / out["modes"]["compact"]["pcg_ms_median"]
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("out_dir")
    ap.add_argument("--size", type=int, default=5792, help="cells per side of the P2 mesh (bench.py's --size)")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--cg-iters", type=int, default=25)
    args = ap.parse_args(argv)
    if args.size < 1 or args.rounds < 1 or args.cg_iters < 1:
        ap.error("--size, --rounds and --cg-iters must be positive")
    res = run(args)
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "pcg_compact_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "modes"}), flush=True)
    for mode, r in res["modes"].items():
        print(mode, {k: v for k, v in r.items() if k != "pcg_ms"}, flush=True)
    if not res["bitwise_equal_pcg_x"]:
        raise SystemExit("pcg_compact_probe: the two modes disagree")
    return res


if __name__ == "__main__":
    main()
