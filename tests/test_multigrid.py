"""Geometric multigrid preconditioner: mesh hierarchies and transfer maps (CPU), and the device Galerkin operators,
transfers, V-cycle and multigrid-PCG against a scipy restatement kept here (GPU)."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from femb200 import mesh as fm
from oracle import oracle

LO_FRAC = 0.25


def square_mesh(square):
    meta = {"kind": "gmsh22", "cell_tags": square["tag"], "facets": square["edges"], "facet_tags": square["edge_tag"]}
    return fm.Mesh(fm.P1, square["x"].copy(), square["tri"].copy(), square["tri"].copy(), 0, 0, meta)


# ---- scipy restatement ------------------------------------------------------------------------------------------
def node_P(tmap, ncoarse):
    """Scalar (node) prolongation of a transfer map."""
    nf = len(tmap)
    a, b = tmap[:, 0].astype(np.int64), tmap[:, 1].astype(np.int64)
    rows = np.concatenate([np.arange(nf), np.arange(nf)])
    P = sp.csr_matrix((np.full(2 * nf, 0.5), (rows, np.concatenate([a, b]))), shape=(nf, ncoarse))
    P.sum_duplicates()
    return P


def vec_P(tmap, ncoarse, bcf=None, bcc=None):
    P = sp.kron(node_P(tmap, ncoarse), sp.identity(2), format="csr")
    if bcf is not None:
        P = sp.diags((bcf == 0).astype(float)) @ P @ sp.diags((bcc == 0).astype(float))
    return P.tocsr()


def galerkin_levels(A, hier, fine_marker, nlevels):
    """[A_0 .. A_L] and [P_0 .. P_{L-1}] for the last nlevels + 1 meshes of the hierarchy."""
    marks = hier.markers(fine_marker)
    levels, Ps = [A], []
    for k in range(len(hier) - 2, len(hier) - 2 - nlevels, -1):
        P = vec_P(hier.maps[k], hier[k].nnodes, marks[k + 1], marks[k])
        Ac = (P.T @ levels[-1] @ P).tocsr() + sp.diags((marks[k] != 0).astype(float))
        levels.append(Ac.tocsr())
        Ps.append(P)
    return levels, Ps


def cheb(A, dinv, lmax, b, x, deg):
    a, bb = LO_FRAC * lmax, lmax
    theta, delta = 0.5 * (bb + a), 0.5 * (bb - a)
    sigma = theta / delta
    rho = 1 / sigma
    r = dinv * (b - A @ x)
    d = r / theta
    for k in range(deg):
        x = x + d
        if k == deg - 1:
            break
        r = r - dinv * (A @ d)
        rho_n = 1 / (2 * sigma - rho)
        d = rho_n * rho * d + 2 * rho_n / delta * r
        rho = rho_n
    return x


def vcycle(levels, Ps, lams, Cinv, b, l=0, deg=2):
    if l == len(levels) - 1:
        return Cinv @ b
    A = levels[l]
    dinv = 1 / A.diagonal()
    x = cheb(A, dinv, lams[l], b, np.zeros_like(b), deg)
    x = x + Ps[l] @ vcycle(levels, Ps, lams, Cinv, Ps[l].T @ (b - A @ x), l + 1, deg)
    return cheb(A, dinv, lams[l], b, x, deg)


# ---- CPU: hierarchies ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_refine_hierarchy_finest_is_refine_uniform(square, k):
    m = square_mesh(square)
    h = fm.refine_uniform_hierarchy(m, k)
    ref = fm.refine_uniform(m, k)
    assert len(h) == k + 1 and len(h.maps) == k
    assert np.array_equal(h[-1].x, ref.x) and np.array_equal(h[-1].dofmap, ref.dofmap)
    assert np.array_equal(h[-1].xdofmap, ref.xdofmap)
    for key in ("cell_tags", "facets", "facet_tags"):
        assert np.array_equal(h[-1].meta[key], ref.meta[key])
    for j in range(k):
        assert np.array_equal(h[j + 1].x[:h[j].nnodes], h[j].x)


def hierarchies(square):
    out = {"p2_lattice": fm.lattice_hierarchy(fm.structured_triangles(16, order=2)),
           "p1_lattice_rect": fm.lattice_hierarchy(fm.structured_triangles(24, 8, order=1)),
           "p2_jitter": fm.lattice_hierarchy(fm.jitter(fm.structured_triangles(16, order=2), 0.2, seed=7)),
           "square_r3": fm.refine_uniform_hierarchy(square_mesh(square), 3)}
    return out


def test_lattice_hierarchy_levels():
    h = fm.lattice_hierarchy(fm.structured_triangles(16, order=2))
    assert [m.etype for m in h] == [fm.P1] * 5 + [fm.P2]
    assert [m.nx for m in h] == [1, 2, 4, 8, 16, 16]
    h = fm.lattice_hierarchy(fm.structured_triangles(24, 8, order=1))
    assert [(m.nx, m.ny) for m in h] == [(3, 1), (6, 2), (12, 4), (24, 8)]


def test_transfer_maps_reproduce_linear_functions(square):
    """P I_c(f) = I_f(f) for f linear, on every step (P2 -> P1, lattice halving, red refinement)."""
    for name, h in hierarchies(square).items():
        for k in range(len(h) - 1):
            c, f = h[k], h[k + 1]
            if name == "p2_jitter" and k < len(h) - 2:
                continue   # the coarse lattices of a jittered mesh are nested in topology only
            P = node_P(h.maps[k], c.nnodes)
            for coef in ((1.0, 0.0, 0.0), (0.3, 2.0, -1.5)):
                lin = lambda x: coef[0] + coef[1] * x[:, 0] + coef[2] * x[:, 1]
                np.testing.assert_allclose(P @ lin(c.x), lin(f.x), rtol=0, atol=1e-13, err_msg=f"{name} level {k}")


def test_coarse_markers(square):
    for name, h in hierarchies(square).items():
        fine = h[-1]
        bc, _ = fm.dirichlet_markers(fine)
        marks = h.markers(bc)
        assert len(marks) == len(h) and np.array_equal(marks[-1], bc)
        for k, m in enumerate(h.meshes):
            want, _ = fm.dirichlet_markers(m)   # coarse nodes carry the coordinates of their coincident fine nodes
            assert marks[k].dtype == np.uint8 and np.array_equal(marks[k], want), f"{name} level {k}"
        for k in range(len(h) - 1):
            tm = h.maps[k]
            co = fm.coincident_nodes(tm, h[k].nnodes)
            assert np.array_equal(marks[k].reshape(-1, 2), marks[k + 1].reshape(-1, 2)[co])


def test_galerkin_pattern_is_coarse_mesh_pattern(square):
    """The structural pattern of P^T A P is the coarse mesh's own P1 pattern, bit for bit."""
    for name, h in hierarchies(square).items():
        for k in range(len(h) - 1):
            c, f = h[k], h[k + 1]
            rp, ci = oracle.build_pattern(f.nnodes, f.dofmap)
            S = sp.csr_matrix((np.ones(len(ci)), ci, rp), shape=(f.ndofs, f.ndofs))
            P = vec_P(h.maps[k], c.nnodes)
            G = (P.T @ S @ P).tocsr()
            G.sort_indices()
            rpc, cic = oracle.build_pattern(c.nnodes, c.dofmap)
            assert np.array_equal(G.indptr.astype(np.int64), rpc) and np.array_equal(G.indices.astype(np.int32), cic), \
                f"{name} level {k}"


def test_hierarchy_errors():
    with pytest.raises(ValueError):
        fm.lattice_hierarchy(fm.structured_quads_q2(4))
    h = fm.lattice_hierarchy(fm.structured_triangles(8, order=1))
    with pytest.raises(ValueError):
        h.markers(np.zeros(3, np.uint8))


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _problem(m, E=None, damaged=False, variant=0):
    """Assembled constrained operator on the device and a lifted right-hand side with a body force."""
    import torch
    from femb200 import fem
    E = fm.young_per_cell(m.ncells) if E is None else E
    bc, g = fm.dirichlet_markers(m)
    d = u = None
    if damaged:
        d = fm.damage_band(m)
        u = 1e-3 * np.random.default_rng(1).standard_normal(m.ndofs)
    form = fem.ElasticityForm(m, E, 0.3, d=d, u=u, variant=variant)
    A = fem.create_matrix(form)
    fem.assemble_matrix_nobc(A, form)
    gd = torch.from_numpy(g).cuda()
    Kg = A.mult(gd).cpu().numpy()
    f = np.zeros(m.ndofs)
    f[0::2] = fm.body_force(m)[:, 0] * 1e-6
    b = f - Kg
    b[bc != 0] = g[bc != 0]
    fem.assemble_matrix(A, form, bcs=[fem.DirichletBC(bc, g)])
    return A, torch.from_numpy(b).cuda(), bc


def _cases(square):
    return {"p2_lattice": (fm.structured_triangles(32, order=2), False, 0),
            "p1_lattice": (fm.structured_triangles(64, order=1), False, 0),
            "p2_jitter": (fm.jitter(fm.structured_triangles(32, order=2), 0.2, seed=3), False, 0),
            "square_r4": (fm.refine_uniform(square_mesh(square), 4), False, 0),
            "square_r4_damaged_closed": (fm.refine_uniform(square_mesh(square), 4), True, 0),
            "square_r4_damaged_ad": (fm.refine_uniform(square_mesh(square), 4), True, 1)}


def _hier(m, square):
    if m.meta.get("kind") == "structured-tri-right":
        return fm.lattice_hierarchy(m)
    return fm.refine_uniform_hierarchy(square_mesh(square), int(m.meta["refined"]))


def _E(m):
    return fm.young_from_tags(m.meta["cell_tags"]) if "cell_tags" in m.meta else fm.young_per_cell(m.ncells)


@pytest.mark.gpu
def test_galerkin_levels_match_scipy(square):
    from femb200 import fem
    for name, (m, damaged, variant) in _cases(square).items():
        A, _, bc = _problem(m, _E(m), damaged, variant)
        h = _hier(m, square)
        mg = fem.MultigridPreconditioner(A, h, coarse_max=600)
        mg.setup()
        levels, _ = galerkin_levels(A.to_scipy(), h, bc, mg.nlevels)
        for l in range(1, mg.nlevels + 1):
            rp, ci = (t.cpu().numpy() for t in mg.level_csr(l))
            got = sp.csr_matrix((mg.level_values(l).cpu().numpy(), ci, rp), shape=levels[l].shape)
            err = spla.norm(got - levels[l]) / spla.norm(levels[l])
            assert err <= 1e-12, f"{name} level {l}: {err:.3e}"
        first = [mg.level_values(l).cpu().numpy() for l in range(1, mg.nlevels + 1)]
        mg.setup()
        for l in range(1, mg.nlevels + 1):
            assert np.array_equal(first[l - 1], mg.level_values(l).cpu().numpy()), f"{name}: setup is not deterministic"
        mg.close()


@pytest.mark.gpu
def test_transfers_match_scipy(square):
    import torch
    from femb200 import fem
    rng = np.random.default_rng(5)
    for name in ("p2_lattice", "square_r4"):
        m = _cases(square)[name][0]
        A, _, bc = _problem(m, _E(m))
        h = _hier(m, square)
        mg = fem.MultigridPreconditioner(A, h, coarse_max=600)
        marks = h.markers(bc)
        for l in range(mg.nlevels):
            k = len(h) - 2 - l
            P = vec_P(h.maps[k], h[k].nnodes, marks[k + 1], marks[k])
            xc, x = rng.standard_normal(P.shape[1]), rng.standard_normal(P.shape[0])
            got = mg.prolong(l, torch.from_numpy(xc).cuda(), torch.from_numpy(x).cuda()).cpu().numpy()
            assert np.array_equal(got, x + P @ xc), f"{name} prolongation level {l}"
            b, t = rng.standard_normal(P.shape[0]), rng.standard_normal(P.shape[0])
            for tt in (None, t):
                want = P.T @ (b - (0 if tt is None else tt))
                got = mg.restrict(l, torch.from_numpy(b).cuda(), None if tt is None else torch.from_numpy(tt).cuda())
                err = np.linalg.norm(got.cpu().numpy() - want) / np.linalg.norm(want)
                assert err <= 1e-15, f"{name} restriction level {l}: {err:.3e}"
        mg.close()


@pytest.mark.gpu
def test_vcycle_matches_restatement_and_is_spd(square):
    import torch
    from femb200 import fem
    rng = np.random.default_rng(11)
    for name in ("p2_lattice", "p2_jitter", "square_r4_damaged_ad"):
        m, damaged, variant = _cases(square)[name]
        A, _, bc = _problem(m, _E(m), damaged, variant)
        h = _hier(m, square)
        mg = fem.MultigridPreconditioner(A, h, coarse_max=600)
        mg.setup()
        lams = mg.lambdas
        assert all(l > 0 for l in lams[:-1])
        levels, Ps = galerkin_levels(A.to_scipy(), h, bc, mg.nlevels)
        Cinv = np.linalg.inv(levels[-1].toarray())
        for _ in range(2):
            r = rng.standard_normal(A.ndofs)
            want = vcycle(levels, Ps, lams, Cinv, r)
            got = mg.apply(torch.from_numpy(r).cuda()).cpu().numpy()
            err = np.linalg.norm(got - want) / np.linalg.norm(want)
            assert err <= 1e-11, f"{name}: V-cycle {err:.3e}"
        x, y = (torch.from_numpy(rng.standard_normal(A.ndofs)).cuda() for _ in range(2))
        Bx, By = mg.apply(x), mg.apply(y)
        asym = abs(torch.dot(Bx, y).item() - torch.dot(x, By).item())
        assert asym <= 1e-12 * Bx.norm().item() * y.norm().item(), f"{name}: V-cycle not symmetric ({asym:.3e})"
        assert torch.dot(Bx, x).item() > 0 and torch.dot(By, y).item() > 0
        mg.close()


@pytest.mark.gpu
def test_mg_pcg_solution_matches_spsolve(square):
    from femb200 import fem
    for name in ("p2_lattice", "p1_lattice", "square_r4_damaged_closed"):
        m, damaged, variant = _cases(square)[name]
        A, b, bc = _problem(m, _E(m), damaged, variant)
        cg = fem.CGSolver(rel_tol=1e-12, max_iter=200)
        cg.SetOperator(A)
        cg.SetPreconditioner("mg", hierarchy=_hier(m, square))
        x = cg.Mult(b).cpu().numpy()
        xs = spla.spsolve(A.to_scipy().tocsc(), b.cpu().numpy())
        err = np.linalg.norm(x - xs) / np.linalg.norm(xs)
        assert cg.GetConverged() and err <= 1e-10, f"{name}: {cg.GetNumIterations()} its, error {err:.3e}"
        cg.mg.close()


def _iterations(m, square, jacobi_cap):
    from femb200 import fem
    A, b, _ = _problem(m, _E(m))
    mg = fem.MultigridPreconditioner(A, _hier(m, square))
    mg.setup()
    x = b.clone()
    its, _, conv = mg.solve(b, x, 1e-12, 0.0, 200)
    assert conv
    mg.close()
    cg = fem.CGSolver(rel_tol=1e-12, max_iter=jacobi_cap * its)
    cg.SetOperator(A)
    cg.SetPreconditioner("jacobi")
    cg.Mult(b)
    return its, cg.GetConverged()


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["p2_lattice", "square"])
def test_mg_iterations_do_not_grow_with_resolution(square, family):
    sizes = (64, 128, 256, 512) if family == "p2_lattice" else (3, 4, 5, 6)
    its = []
    for s in sizes:
        m = fm.structured_triangles(s, order=2) if family == "p2_lattice" else fm.refine_uniform(square_mesh(square), s)
        it, jac_conv = _iterations(m, square, 10)
        assert it <= 30, f"{family} {s}: {it} iterations"
        assert not jac_conv, f"{family} {s}: Jacobi-PCG converged within 10 x {it} iterations"
        its.append(it)
    assert its[-1] <= its[0] + 5, its


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["p2_lattice", "square"])
def test_newton_with_mg_matches_jacobi(square, family):
    import torch
    from femb200 import fem
    m = fm.structured_triangles(64, order=2) if family == "p2_lattice" else fm.refine_uniform(square_mesh(square), 4)
    E = _E(m)
    bc, g = fm.dirichlet_markers(m)
    f = fm.body_force(m)
    runs = {}
    for prec in ("jacobi", "mg"):
        form = fem.ElasticityForm(m, E, 0.3, d=fm.damage_band(m))
        ns = fem.NewtonSolver(form, [fem.DirichletBC(bc, g)], f=f, cg_max_iter=20000, preconditioner=prec,
                              hierarchy=_hier(m, square) if prec == "mg" else None)
        u = ns.solve()
        runs[prec] = (ns.iterations, list(ns.residual_norms), list(ns.linear_iterations), list(ns.linear_converged),
                      u.cpu().numpy())
        ns.close()
        torch.cuda.synchronize()
    (itj, rj, _, cj, uj), (itm, rm, lm, cm, um) = runs["jacobi"], runs["mg"]
    assert itj == itm and all(cj) and all(cm)
    assert max(lm) <= 30, lm
    # Both linear solves stop at rtol 1e-12, but in different norms (<D^-1 r, r> and <B r, r>), and the damaged tangent
    # is not smooth in u, so the Newton steps carry those ~1e-12 differences forward.  Measured on a B200 (relative to
    # each step's own |r_k|): at most 2.5e-9 (P2 n = 64) and 2.5e-8 (square.msh r = 4), both at step 5; so every step
    # is held to 1e-9 |r_0| and to 1e-7 |r_k|.
    rel = [abs(a - b) / abs(a) for a, b in zip(rj, rm)]
    print(f"{family}: |r_k| {rj}, relative differences {rel}")
    for k, (a, b) in enumerate(zip(rj, rm)):
        assert abs(a - b) <= 1e-9 * rj[0], f"step {k}: {a!r} vs {b!r} (|r_0| = {rj[0]!r}, all {rj})"
        assert rel[k] <= 1e-7, f"step {k}: {a!r} vs {b!r}, relative {rel[k]:.3e}"
    assert np.linalg.norm(um - uj) <= 1e-8 * np.linalg.norm(uj)


@pytest.mark.gpu
def test_mg_pcg_with_direct_spmv_kernel_on_a_fresh_stream():
    """MG-PCG on a plan whose SpMV takes the direct kernel (plan option spmv_path = 1), first solve on a new stream:
    that SpMV grows the stream's fused-reduction scratch (more than 131 k nodes), and the <B r, r> reductions of the
    solve must use the grown scratch.  Same iterations and solution as with the default SpMV kernel."""
    import torch
    from femb200 import fem
    m = fm.structured_triangles(256, order=2)          # 263 169 nodes
    out = {}
    for path in (0, 1):
        with torch.cuda.stream(torch.cuda.Stream()):
            A, b, _ = _problem(m)
            A.set_option("spmv_path", path)
            mg = fem.MultigridPreconditioner(A, fm.lattice_hierarchy(m))
            mg.setup()
            x = torch.empty_like(b)
            its, _, conv = mg.solve(b, x, 1e-12, 0.0, 100)
            torch.cuda.current_stream().synchronize()
            out[path] = (its, conv, x.cpu().numpy())
            mg.close()
    (i0, c0, x0), (i1, c1, x1) = out[0], out[1]
    assert c0 and c1 and abs(i0 - i1) <= 1, (i0, i1)
    assert np.linalg.norm(x1 - x0) <= 1e-10 * np.linalg.norm(x0)


@pytest.mark.gpu
def test_vcycle_refuses_aliased_vectors():
    from femb200 import fem
    m = fm.structured_triangles(16, order=2)
    A, b, _ = _problem(m)
    mg = fem.MultigridPreconditioner(A, fm.lattice_hierarchy(m))
    mg.setup()
    with pytest.raises(ValueError):
        mg.apply(b, b)
    mg.close()


@pytest.mark.gpu
def test_mg_errors(square):
    from femb200 import fem
    m = fm.structured_triangles(33, order=1)       # odd: no coarser lattice
    A, _, _ = _problem(m)
    with pytest.raises(ValueError, match="no mesh coarser"):
        fem.MultigridPreconditioner(A, fm.lattice_hierarchy(m))
    m = fm.structured_triangles(66, order=1)
    A, _, _ = _problem(m)
    with pytest.raises(ValueError, match="coarse_max"):
        fem.MultigridPreconditioner(A, fm.lattice_hierarchy(m), coarse_max=1000)
    m = fm.structured_triangles(16, order=2)
    A, _, _ = _problem(m)
    with pytest.raises(ValueError):
        fem.NewtonSolver(fem.ElasticityForm(m, fm.young_per_cell(m.ncells)), [fem.DirichletBC(*fm.dirichlet_markers(m))],
                         preconditioner="mg", hierarchy=fm.lattice_hierarchy(m), part=object())
