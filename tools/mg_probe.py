"""Multigrid preconditioner probe: memory, set-up split, V-cycle cost per level, Galerkin-kernel bandwidth and
time-to-solution of multigrid-PCG against Jacobi-PCG, on large P2 lattices and refined square.msh meshes.

    python tools/mg_probe.py OUT_DIR [--lattice 1024 2048 4096] [--square 8 9] [--jacobi-cap 20]

Writes OUT_DIR/mg_probe.json with the card name and power limit read in the same run.  Times are CUDA-event
times after a warm-up; the working sets are larger than L2 except on the coarse levels.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "fem-libraries_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

from femb200 import _capi as capi  # noqa: E402
from femb200 import fem, mesh as fm  # noqa: E402

HBM_BPS = 6451.2e9


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
    except Exception as e:   # report what could be read
        name, power = torch.cuda.get_device_name(0), f"unavailable ({e})"
    return {"name": name, "power_limit": power}


def ev_time(fn, reps=3, warm=1):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps * 1e-3


def host_time(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t, out


def square_mesh():
    with open(os.path.join(ROOT, "tests", "golden", "square_mesh.json")) as f:
        m = json.load(f)
    x = np.array([[float(a), float(b)] for a, b in m["x"]], dtype=np.float64)
    tri = np.array(m["triangles"], dtype=np.int32)
    meta = {"kind": "gmsh22", "cell_tags": np.array(m["triangle_tag"], dtype=np.int32),
            "facets": np.array(m["edges"], dtype=np.int32), "facet_tags": np.array(m["edge_tag"], dtype=np.int32)}
    return fm.Mesh(fm.P1, x, tri, tri.copy(), 0, 0, meta)


def run_case(label, hier, jacobi_cap):
    m = hier[-1]
    out = {"case": label, "ndofs": m.ndofs, "ncells": m.ncells}
    E = fm.young_from_tags(m.meta["cell_tags"]) if "cell_tags" in m.meta else fm.young_per_cell(m.ncells)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, E, 0.3)
    A = fem.create_matrix(form)
    fem.assemble_matrix_nobc(A, form)
    gd = torch.from_numpy(g).cuda()
    b = -A.mult(gd)
    bcd = torch.from_numpy(bc).cuda() != 0
    b[bcd] = gd[bcd]
    fem.assemble_matrix(A, form, bcs=[fem.DirichletBC(bc, g)])
    torch.cuda.synchronize()

    t_create, mg = host_time(lambda: fem.MultigridPreconditioner(A, hier))
    L = mg.nlevels
    # set-up split: Galerkin cascade, smoother (D^-1 + power iteration), coarse inverse
    t_setup, _ = host_time(lambda: capi.call("femb200_mg_setup", mg.handle, fem._p(A.values), fem._stream()))
    t_inv, _ = host_time(mg.set_coarse_inverse)
    rap = [ev_time(lambda l=l: mg.galerkin(l)) for l in range(L)]
    mg.setup()
    nd, nz, lam, mg_bytes = mg.sizes()
    plan_bytes = []
    for l in range(1, L + 1):
        v = [C.c_int64() for _ in range(4)]
        deg, by = C.c_int32(), C.c_int64()
        capi.call("femb200_plan_sizes", mg._plans[l - 1], *[C.byref(x) for x in v], C.byref(deg), C.byref(by))
        plan_bytes.append(by.value)
    # Galerkin kernel: algorithmic bytes (fine values, fine block pattern, map, slot list, coarse values once)
    rap_rows = []
    for l in range(L):
        nnzb_f, nnzb_c = nz[l] // 4, nz[l + 1] // 4
        byts = 8 * nz[l] + 4 * nnzb_f + 8 * (nd[l] // 2) + 8 * (nd[l] // 2 + 1) + 4 * nnzb_c + 8 * nz[l + 1]
        rap_rows.append({"level": l, "seconds": rap[l], "bytes": byts, "GBps": byts / rap[l] / 1e9,
                         "hbm_fraction": byts / rap[l] / HBM_BPS})
    # V-cycle: total (events around 10 cycles), and per level the kernels inside the cycle (an event after every
    # launch, femb200_mg_vcycle_timed; event-to-event, so launch gaps are charged to the launch that follows them),
    # averaged over 5 timed cycles
    r = torch.randn(A.ndofs, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    z = torch.empty_like(r)
    t_v = ev_time(lambda: mg.apply(r, z), reps=10, warm=2)
    ms = sum(mg.apply_timed(r, z) for _ in range(5)) / 5
    x = torch.randn(A.ndofs, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)
    fine_spmv = ev_time(lambda: A.mult(x, y), reps=10)
    kinds = ("spmv", "chebyshev_pass", "restrict", "prolong", "coarse_gemv")
    levels = []
    for l in range(L + 1):
        row = {"level": l, "ndofs": nd[l], "nnz": nz[l], "values_bytes": 8 * nz[l],
               "plan_bytes": None if l == 0 else plan_bytes[l - 1],
               "in_vcycle_s": {k: float(ms[l, i]) * 1e-3 for i, k in enumerate(kinds)}}
        if l < L:
            row.update({"lambda": lam[l], "spmv_per_vcycle": 2 * mg.degree, "chebyshev_passes_per_vcycle": 2 * mg.degree})
        else:
            row["coarse_inverse_bytes"] = 8 * nd[L] ** 2
        levels.append(row)
    # time to solution
    x = torch.empty_like(b)
    mg.solve(b, x, 1e-12, 0.0, 5)   # warm
    t_sol, res = host_time(lambda: mg.solve(b, x, 1e-12, 0.0, 500))
    its, fnorm, conv = res
    # Jacobi-PCG to the same tolerance under a wall-clock cap
    cg = fem.CGSolver(rel_tol=1e-12, max_iter=50)
    cg.SetOperator(A)
    cg.SetPreconditioner("jacobi")
    cg.Mult(b, fixed_iters=50)
    t50, _ = host_time(lambda: cg.Mult(b, fixed_iters=50))
    cap_its = max(50, int(jacobi_cap / (t50 / 50)))
    cg.SetMaxIter(cap_its)
    cg.check_every = 200
    t_jac, _ = host_time(lambda: cg.Mult(b))
    out.update({"levels": levels, "nlevels": L, "mg_device_bytes": mg_bytes, "fine_matrix_bytes": 8 * A.nnz,
                "setup": {"create_s (coarse plans + maps + nesting check)": t_create,
                          "galerkin_s (sum over levels)": sum(rap),
                          "smoother_s (setup minus Galerkin: D^-1 + power iteration)": t_setup - sum(rap),
                          "coarse_inverse_s": t_inv},
                "galerkin_kernel": rap_rows,
                "vcycle": {"seconds": t_v, "fine_spmv_s (alone)": fine_spmv, "fine_spmv_equivalents": t_v / fine_spmv,
                           "timed_cycle_s (sum of the per-level kernel times)": float(ms.sum()) * 1e-3,
                           "coarse_levels_share (levels >= 1 of the timed cycle)": float(ms[1:].sum() / ms.sum())},
                "mg_pcg": {"iterations": its, "converged": conv, "seconds": t_sol, "final_norm": fnorm},
                "jacobi_pcg": {"wall_cap_s": jacobi_cap, "max_iter_in_cap": cap_its, "iterations": cg.GetNumIterations(),
                               "converged": cg.GetConverged(), "seconds": t_jac, "final_norm": cg.GetFinalNorm(),
                               "seconds_per_iteration": t50 / 50}})
    mg.close()
    del A, form
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--lattice", type=int, nargs="*", default=[1024, 2048, 4096])
    ap.add_argument("--square", type=int, nargs="*", default=[8, 9])
    ap.add_argument("--jacobi-cap", type=float, default=20.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mg_probe needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    res = {"card": card(), "hbm_roofline_Bps": HBM_BPS, "cases": []}
    cases = [(f"P2 lattice n={n}", lambda n=n: fm.lattice_hierarchy(fm.structured_triangles(n, order=2))) for n in a.lattice]
    cases += [(f"square.msh r={r}", lambda r=r: fm.refine_uniform_hierarchy(square_mesh(), r)) for r in a.square]
    for label, make in cases:
        t = time.perf_counter()
        try:
            res["cases"].append(run_case(label, make(), a.jacobi_cap))
        except Exception as e:   # keep the other cases (e.g. out of memory on the largest)
            res["cases"].append({"case": label, "error": f"{type(e).__name__}: {e}"})
        res["cases"][-1]["host_wall_s"] = time.perf_counter() - t
        print(json.dumps(res["cases"][-1])[:600], flush=True)
        torch.cuda.empty_cache()
        with open(os.path.join(a.out, "mg_probe.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
