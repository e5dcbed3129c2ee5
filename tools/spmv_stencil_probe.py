"""SpMV column modes side by side: stencil ids (spmv_cols = 0, the default where the plan has a dictionary) against
16-bit column offsets (spmv_cols = 2), on one matrix in one process.

    python tools/spmv_stencil_probe.py OUT_DIR [--size 5792] [--rounds 7] [--spmv-reps 10] [--cg-iters 25] [--dry-run]

The workload is bench.py's: the P2 strip of `dist.strip_partition_device(n, n, 0, 1, jitter_amp=0.2, seed=1234)`,
assembled with its Dirichlet rows and columns.  Each round times, for each mode in turn and with CUDA events after a
warm-up, `--spmv-reps` SpMVs and one Jacobi-PCG of exactly `--cg-iters` iterations; the y of the SpMV and the PCG
iterate must be equal bit for bit between the modes.  Bytes per SpMV are counted from the plan's shapes:

    stencil: 32 B of values per node block + 1 id byte per node row + x read and y written (32 B per node row)
    16-bit:  32 B of values + 2 B of bcol16 per node block + 8 B of brp per node row + x and y

Writes OUT_DIR/spmv_stencil_probe.json with the card name and power limit read in the same run.  `--dry-run` stops
before the device: it builds the mesh of `--size` on the CPU and writes the byte counts only.
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

MODES = {"stencil": 0, "bcol16": 2}   # spmv_cols value of each mode


def spmv_bytes(mode: str, nnz_blocks: int, nnodes: int) -> int:
    """Bytes one SpMV streams from / to HBM in `mode`, by design (values, indices, row data, x and y)."""
    vec = 32 * nnodes
    if mode == "stencil":
        return 32 * nnz_blocks + nnodes + vec
    if mode == "bcol16":
        return 34 * nnz_blocks + 8 * nnodes + vec
    raise ValueError(f"unknown mode {mode!r}")


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"])
    return None


def card():
    import torch
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception as e:   # report what could be read
        name, power = torch.cuda.get_device_name(0), f"unavailable ({e})"
    return {"name": name, "power_limit": power}


def shapes(nnz_blocks: int, nnodes: int) -> dict:
    return {"nnz_blocks": nnz_blocks, "nnodes": nnodes,
            "bytes_per_spmv": {m: spmv_bytes(m, nnz_blocks, nnodes) for m in MODES}}


def dry_run(args) -> dict:
    from femb200 import dist
    from oracle import oracle
    m = dist.strip_partition(args.size, args.size, 2, 0, 1).mesh
    rowptr, _ = oracle.build_pattern(m.nnodes, m.dofmap)
    return {"dry_run": True, "size": args.size, **shapes(int(rowptr[-1]) // 4, m.nnodes)}


def run(args) -> dict:
    import torch
    from femb200 import dist, fem
    torch.cuda.set_device(0)
    out = {"dry_run": False, "size": args.size, "card": card(), "rounds": args.rounds, "spmv_reps": args.spmv_reps,
           "cg_iters": args.cg_iters}
    part = dist.strip_partition_device(args.size, args.size, 0, 1, jitter_amp=0.2, seed=1234)
    form = fem.ElasticityForm(part.mesh, part.E, 0.3)
    A = fem.create_matrix(form)
    A.set_bcs([fem.DirichletBC(part.bc, part.g)])
    fem.assemble_matrix(A, form)
    out.update(shapes(A.nnz_blocks, A.nnodes))
    out["spmv_stencils"] = A.get_option("spmv_stencils")
    if out["spmv_stencils"] == 0:
        raise SystemExit("spmv_stencil_probe: the plan has no stencil dictionary")
    b = torch.where(part.bc != 0, part.g, torch.ones_like(part.g))
    y = torch.empty_like(b)
    cg = fem.CGSolver(rel_tol=0.0, max_iter=args.cg_iters)
    cg.SetOperator(A)
    cg.SetPreconditioner("jacobi")
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(fn, reps):
        a, e = ev(), ev()
        a.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        return a.elapsed_time(e) / reps

    times = {m: {"spmv_ms": [], "pcg_ms": []} for m in MODES}
    results = {}
    for mode, v in MODES.items():          # warm-up of both kernels
        A.set_option("spmv_cols", v)
        A.mult(b, y)
        cg.Mult(b, fixed_iters=args.cg_iters)
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for mode in (MODES if r % 2 == 0 else list(MODES)[::-1]):
            A.set_option("spmv_cols", MODES[mode])
            times[mode]["spmv_ms"].append(timed(lambda: A.mult(b, y), args.spmv_reps))
            times[mode]["pcg_ms"].append(timed(lambda: cg.Mult(b, fixed_iters=args.cg_iters), 1))
            if r == 0:
                results[mode] = (y.clone(), cg.Mult(b, fixed_iters=args.cg_iters).clone())
    A.set_option("spmv_cols", 0)
    ys, xs = results["stencil"], results["bcol16"]
    out["bitwise_equal"] = {"spmv_y": bool(torch.equal(ys[0], xs[0])), "pcg_x": bool(torch.equal(ys[1], xs[1]))}
    peak = hbm_peak()
    out["hbm_peak_gbs"] = peak
    out["hbm_peak_source"] = "MEASURED_PEAKS.json" if peak else None
    out["modes"] = {}
    for mode, t in times.items():
        s, c = np.array(t["spmv_ms"]), np.array(t["pcg_ms"])
        nb = out["bytes_per_spmv"][mode]
        gbs = nb / (np.median(s) * 1e-3) / 1e9
        out["modes"][mode] = {"spmv_cols": MODES[mode], "spmv_ms_median": float(np.median(s)),
                              "spmv_ms_spread": float(s.max() - s.min()), "pcg_ms_median": float(np.median(c)),
                              "pcg_ms_spread": float(c.max() - c.min()), "spmv_gbs": gbs,
                              "spmv_frac_of_peak": gbs / peak if peak else None, "spmv_ms": t["spmv_ms"],
                              "pcg_ms": t["pcg_ms"]}
    st, c16 = out["modes"]["stencil"], out["modes"]["bcol16"]
    out["spmv_speedup"] = c16["spmv_ms_median"] / st["spmv_ms_median"]
    out["pcg_speedup"] = c16["pcg_ms_median"] / st["pcg_ms_median"]
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("out_dir")
    ap.add_argument("--size", type=int, default=5792, help="cells per side of the P2 mesh (bench.py's --size)")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--spmv-reps", type=int, default=10)
    ap.add_argument("--cg-iters", type=int, default=25)
    ap.add_argument("--dry-run", action="store_true", help="CPU only: mesh and byte counts, no device")
    args = ap.parse_args(argv)
    if args.size < 1 or args.rounds < 1 or args.spmv_reps < 1 or args.cg_iters < 1:
        ap.error("--size, --rounds, --spmv-reps and --cg-iters must be positive")
    res = dry_run(args) if args.dry_run else run(args)
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "spmv_stencil_probe.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "modes"}), flush=True)
    for mode, r in res.get("modes", {}).items():
        print(mode, {k: v for k, v in r.items() if k not in ("spmv_ms", "pcg_ms")}, flush=True)
    if not res["dry_run"] and not all(res["bitwise_equal"].values()):
        raise SystemExit("spmv_stencil_probe: the two column modes disagree")
    return res


if __name__ == "__main__":
    main()
