"""Multigrid preconditioner probe: memory, set-up split, V-cycle cost per level, Galerkin-kernel bandwidth and
time-to-solution of multigrid-PCG against Jacobi-PCG, on large P2 lattices and refined square.msh meshes (assembled),
on jittered Q2 meshes (matrix-free, as bench.py config 3) and, with --pa, on the P2 lattices matrix-free as well.

    python tools/mg_probe.py OUT_DIR [--lattice 1024 2048 4096] [--square 8 9] [--quad 1024 2048 4096] [--pa]
                                     [--jacobi-cap 20]

A matrix-free case never assembles the fine matrix: its first coarse operator comes from the element Galerkin step
(per-cell P_e^T K_e P_e from the PA data, gathered into the coarse pattern), reported with its algorithmic bytes.

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


def run_case(label, hier, jacobi_cap, matrix_free=False):
    m = hier[-1]
    out = {"case": label, "operator": "matrix-free (PA)" if matrix_free else "assembled", "ndofs": m.ndofs,
           "ncells": m.ncells}
    E = fm.young_from_tags(m.meta["cell_tags"]) if "cell_tags" in m.meta else fm.young_per_cell(m.ncells)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, E, 0.3)
    gd = torch.from_numpy(g).cuda()
    bcd = torch.from_numpy(bc).cuda() != 0
    if matrix_free:
        A = fem.PAOperator(form)
        b = -A.mult(gd)
        A = fem.PAOperator(form, bcs=[fem.DirichletBC(bc, g)])
        fine_values = None
    else:
        A = fem.create_matrix(form)
        fem.assemble_matrix_nobc(A, form)
        b = -A.mult(gd)
        fem.assemble_matrix(A, form, bcs=[fem.DirichletBC(bc, g)])
        fine_values = fem._p(A.values)
    b[bcd] = gd[bcd]
    torch.cuda.synchronize()
    mem0 = torch.cuda.memory_allocated()

    t_create, mg = host_time(lambda: fem.MultigridPreconditioner(A, hier))
    L = mg.nlevels
    # set-up split: Galerkin cascade, smoother (D^-1 + power iteration), coarse inverse
    t_setup, _ = host_time(lambda: capi.call("femb200_mg_setup", mg.handle, fine_values, fem._stream()))
    t_inv, _ = host_time(mg.set_coarse_inverse)
    rap = [ev_time(lambda l=l: mg.galerkin(l)) for l in range(L)]
    mg.setup()
    nd, nz, lam, mg_bytes = mg.sizes()
    plan_bytes, nnzb = [], [nz[0] // 4]
    for l in range(1, L + 1):
        v = [C.c_int64() for _ in range(4)]
        deg, by = C.c_int32(), C.c_int64()
        capi.call("femb200_plan_sizes", mg._plans[l - 1], *[C.byref(x) for x in v], C.byref(deg), C.byref(by))
        plan_bytes.append(by.value)
        nnzb.append(v[2].value)
    # Galerkin kernel: algorithmic bytes (fine values, fine block pattern, map, slot list, coarse values once); the
    # element step of a matrix-free level 0: per cell its PA geometry + Lame pair, mask and cell number, the per-cell
    # coarse matrix written and read once, the coarse visit records, and the coarse values written once
    rap_rows = []
    W = mg.width
    for l in range(L):
        if matrix_free and l == 0:
            c = hier[-2]
            nv, n2 = c.nv, 2 * c.nv
            byts = m.ncells * ((2 * form.nv + 2) * 8 + 8 + 2 * 8 * n2 * n2 + 16 * nv) + 8 * nz[1] + 16 * (c.nnodes + 1)
            kind = "element Galerkin (P_e^T K_e P_e from the PA data + gather)"
        else:
            nnzb_f, nnzb_c = nz[l] // 4, nz[l + 1] // 4
            byts = 8 * nz[l] + 4 * nnzb_f + 4 * W * (nd[l] // 2) + 8 * (nd[l] // 2 + 1) + 4 * nnzb_c + 8 * nz[l + 1]
            kind = "CSR Galerkin (P^T A P gather)"
        rap_rows.append({"level": l, "kind": kind, "seconds": rap[l], "bytes": byts, "GBps": byts / rap[l] / 1e9,
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
    kinds = ("spmv" if not matrix_free else "operator_apply (level 0: PA, else SpMV)", "chebyshev_pass", "restrict",
             "prolong", "coarse_gemv")
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
    mem_peak = torch.cuda.max_memory_allocated()
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
    out.update({"levels": levels, "nlevels": L, "map_width": W, "mg_device_bytes": mg_bytes,
                "fine_matrix_bytes": None if matrix_free else 8 * A.nnz,
                "device_memory": {"torch_allocated_before_mg_bytes": mem0, "torch_peak_bytes": mem_peak,
                                  "mg_handle_bytes": mg_bytes, "coarse_plan_bytes": sum(plan_bytes)},
                "setup": {"create_s (coarse plans + maps + nesting check)": t_create,
                          "element_galerkin_s (level 0 -> 1, matrix-free)": rap[0] if matrix_free else None,
                          "galerkin_cascade_s (CSR Galerkin steps)": sum(rap[1:] if matrix_free else rap),
                          "smoother_s (setup minus Galerkin: D^-1 + power iteration)": t_setup - sum(rap),
                          "coarse_inverse_s": t_inv},
                "galerkin_kernel": rap_rows,
                "vcycle": {"seconds": t_v, "fine_apply_s (alone)": fine_spmv, "fine_apply_equivalents": t_v / fine_spmv,
                           "timed_cycle_s (sum of the per-level kernel times)": float(ms.sum()) * 1e-3,
                           "coarse_levels_share (levels >= 1 of the timed cycle)": float(ms[1:].sum() / ms.sum())},
                "mg_pcg": {"iterations": its, "converged": conv, "seconds": t_sol, "final_norm": fnorm,
                           "setup_plus_solve_s": t_setup + t_inv + t_sol},
                "jacobi_pcg": {"wall_cap_s": jacobi_cap, "max_iter_in_cap": cap_its, "iterations": cg.GetNumIterations(),
                               "converged": cg.GetConverged(), "seconds": t_jac, "final_norm": cg.GetFinalNorm(),
                               "seconds_per_iteration": t50 / 50}})
    mg.close()
    del A, form, mg, cg
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out")
    ap.add_argument("--lattice", type=int, nargs="*", default=[1024, 2048, 4096])
    ap.add_argument("--square", type=int, nargs="*", default=[8, 9])
    ap.add_argument("--quad", type=int, nargs="*", default=[], help="jittered Q2 n x n, matrix-free (bench.py config 3)")
    ap.add_argument("--pa", action="store_true", help="also solve the P2 lattices matrix-free")
    ap.add_argument("--jacobi-cap", type=float, default=20.0)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mg_probe needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    res = {"card": card(), "hbm_roofline_Bps": HBM_BPS, "cases": []}
    cases = []
    for n in a.lattice:
        make = lambda n=n: fm.lattice_hierarchy(fm.structured_triangles(n, order=2))
        cases.append((f"P2 lattice n={n}", make, False))
        if a.pa:
            cases.append((f"P2 lattice n={n} matrix-free", make, True))
    cases += [(f"square.msh r={r}", lambda r=r: fm.refine_uniform_hierarchy(square_mesh(), r), False) for r in a.square]
    cases += [(f"Q2 jittered n={n} matrix-free",
               lambda n=n: fm.quad_lattice_hierarchy(fm.jitter(fm.structured_quads_q2(n), 0.2, seed=1234)), True)
              for n in a.quad]
    for label, make, matrix_free in cases:
        t = time.perf_counter()
        try:
            res["cases"].append(run_case(label, make(), a.jacobi_cap, matrix_free))
        except Exception as e:   # keep the other cases (e.g. out of memory on the largest)
            res["cases"].append({"case": label, "error": f"{type(e).__name__}: {e}"})
        res["cases"][-1]["host_wall_s"] = time.perf_counter() - t
        print(json.dumps(res["cases"][-1])[:600], flush=True)
        torch.cuda.empty_cache()
        with open(os.path.join(a.out, "mg_probe.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
