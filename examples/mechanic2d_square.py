"""The reference's driver sequence on its shipped mesh, through femb200 (one GPU).

Mirrors FEniCSx/mechanic2d/asym_elasto_damage_model_symb_sym.py (F.py) and the MFEM driver (M.cc) stage by
stage, with the stage numbers of their timers:

  1    mesh            Gmsh 2.2 file (M.cc:1017-1020; gmsh_to_xdmf + read_mesh, F.cc:153-193)
  4.1  materials       E = E_range[cell tag % 200], nu = 0.3 (M.cc:1074-1098, F.py:213-222)
  4.2  damage field    MAX_DAM on the nodes of the facets tagged 4 (DEBUG_SQUARE, M.cc:1164-1167), then
                       8 (max_refine + 1) smoothing double sweeps over the vertex graph (M.cc:1258-1315)
  5    boundary conds  x = 0 clamped, x = 1 pulled by 0.01 (F.cc:627-664); body force M.cc:1431-1440
  7    non-linear      Newton (rel 1e-7, abs 5e-8, M.cc:1531-1543) around residual / tangent assembly and
                       (Jacobi-)PCG at 1e-12 (M.cc:1502-1528; BoomerAMG is third party, out of scope)
  8.1  strain/stress   DG0 fields at the cell centroids (M.cc:1551-1563, F.cc:909-942)

    python examples/mechanic2d_square.py [--mg] [path/to/square.msh [path/to/mfem_disp_0]]

With a second argument the displacement is compared with an OUT_COMP dump of the reference (M.cc:1660-1725) and the
reference's own two error norms are printed (femb200.compare).

Without an argument the mesh is rebuilt from tests/golden/square_mesh.json (the fixture derived from
common/data/square.msh of the reference).
"""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "fem-libraries_b200")]
from femb200 import compare, fem, mesh as fm  # noqa: E402


def fixture_msh(path: str) -> None:
    with open(os.path.join(ROOT, "tests", "golden", "square_mesh.json")) as f:
        m = json.load(f)
    with open(path, "w") as f:
        f.write("$MeshFormat\n2.2 0 8\n$EndMeshFormat\n$Nodes\n%d\n" % len(m["x"]))
        for i, p in enumerate(m["x"]):
            f.write("%d %.17g %.17g 0\n" % (i + 1, float(p[0]), float(p[1])))
        f.write("$EndNodes\n$Elements\n%d\n" % (len(m["edges"]) + len(m["triangles"])))
        k = 1
        for e, t in zip(m["edges"], m["edge_tag"]):
            f.write("%d 1 2 %d %d %d %d\n" % (k, t, t, e[0] + 1, e[1] + 1))
            k += 1
        for c, t in zip(m["triangles"], m["triangle_tag"]):
            f.write("%d 2 2 %d %d %d %d %d\n" % (k, t, t, c[0] + 1, c[1] + 1, c[2] + 1))
            k += 1
        f.write("$EndElements\n")


def run(msh_path: str, max_refine: int = 0, damaged_facet_tags=(4,), verbose: bool = True, multigrid: bool = False):
    """`multigrid`: solve the Newton steps with multigrid-PCG on the refinement hierarchy instead of Jacobi-PCG."""
    # 1: the MFEM driver reads the Gmsh file (M.cc:1017-1020), the FEniCSx driver its XDMF conversion (F.cc:155-163)
    mesh = fm.read_xdmf(msh_path) if msh_path.endswith(".xdmf") else fm.read_gmsh22(msh_path)
    if multigrid:
        if max_refine < 1:
            raise ValueError("multigrid needs at least one refinement (MAX_REFINE >= 1): the coarse levels are the "
                             "meshes of the -r loop")
        hierarchy = fm.refine_uniform_hierarchy(mesh, max_refine)           # its finest mesh is refine_uniform's
        mesh = hierarchy[-1]
    else:
        hierarchy = None
        mesh = fm.refine_uniform(mesh, max_refine)                           # 1: the -r loop (M.cc:1037-1038, F.cc:166-185)
    E = fm.young_from_tags(mesh.meta["cell_tags"])                           # 4.1
    d0 = fm.damage_seed(mesh, list(damaged_facet_tags), max_dam=1.0)         # 4.2
    d = fem.DamageSmoother(mesh).smooth(d0, niter=8 * (max_refine + 1))
    bc, g = fm.dirichlet_markers(mesh)                                       # 5
    load = fm.body_force(mesh)
    form = fem.ElasticityForm(mesh, E, 0.3, d=d)                             # 7
    newton = fem.NewtonSolver(form, [fem.DirichletBC(bc, g)], f=load, rel_tol=1e-7, abs_tol=5e-8, max_iter=10,
                               **({"preconditioner": "mg", "hierarchy": hierarchy} if multigrid else {}))
    u = newton.solve()
    form.set_u(u)
    strain, stress = fem.cell_strain_stress(form)                            # 8.1
    if verbose:
        print(f"mesh: {mesh.nnodes} nodes, {mesh.ncells} triangles; damaged nodes {int((d0 > 0).sum())} -> "
              f"{int((d.cpu().numpy() > 0).sum())} after smoothing")
        print(f"Newton: {newton.iterations} iterations, |r| = " + ", ".join(f"{r:.3e}" for r in newton.residual_norms))
        print(f"PCG iterations per Newton step: {newton.linear_iterations}")
        print(f"max |u| = {float(u.abs().max()):.6e}, max |stress| = {float(stress.abs().max()):.6e}")
    return {"mesh": mesh, "E": E, "d0": d0, "d": d, "bc": bc, "g": g, "load": load, "u": u, "strain": strain,
            "stress": stress, "newton": newton}


if __name__ == "__main__":
    mg = "--mg" in sys.argv                                                  # multigrid-PCG instead of Jacobi-PCG
    sys.argv = [a for a in sys.argv if a != "--mg"]
    if len(sys.argv) > 1:
        refine = int(os.environ.get("MAX_REFINE", "0"))                      # the reference's -r / MAX_REFINE
        out = run(sys.argv[1], max_refine=refine, multigrid=mg)
        if len(sys.argv) > 2:                                                # IN_COMP (M.cc:1689-1725)
            l2x, l2y = compare.compare_disp_file(sys.argv[2], out["mesh"].x, out["u"].cpu().numpy())
            print(f"Error L2 x:{l2x}\nError L2 y:{l2y}")
    else:
        with tempfile.TemporaryDirectory() as tmp:
            p = os.path.join(tmp, "square.msh")
            fixture_msh(p)
            run(p)
