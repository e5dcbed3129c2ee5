"""Multigrid for quadrilateral meshes and for the matrix-free operator: width-4 transfer maps and the Q2 -> Q1 -> Q1/2
hierarchy (CPU), the pattern-only Q1 plan, assembled Q2 multigrid, and multigrid-PCG with a matrix-free (PA) P2 / Q2 fine
level whose first coarse operator is built from the per-cell data without assembling the fine matrix (GPU), against a
scipy restatement kept here."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla

from femb200 import mesh as fm

LO_FRAC = 0.25


# ---- scipy restatement ------------------------------------------------------------------------------------------
def node_P(tmap, ncoarse):
    """Scalar (node) prolongation of a transfer map of width 2 or 4: each distinct entry of a row weighs
    1 / (number of distinct entries); columns sorted."""
    tmap = np.asarray(tmap, dtype=np.int64)
    nf, w = tmap.shape
    first = [np.ones(nf, bool)]
    for k in range(1, w):
        first.append(np.all(tmap[:, [k]] != tmap[:, :k], axis=1))
    ndist = np.sum(first, axis=0)
    rows = np.concatenate([np.nonzero(f)[0] for f in first])
    cols = np.concatenate([tmap[f, k] for k, f in enumerate(first)])
    vals = 1.0 / ndist[rows]
    P = sp.csr_matrix((vals, (rows, cols)), shape=(nf, ncoarse))
    P.sort_indices()
    return P


def vec_P(tmap, ncoarse, bcf=None, bcc=None):
    P = sp.kron(node_P(tmap, ncoarse), sp.identity(2), format="csr")
    if bcf is not None:
        P = sp.diags((bcf == 0).astype(float)) @ P @ sp.diags((bcc == 0).astype(float))
    P = P.tocsr()
    P.sort_indices()
    return P


def cell_pattern(mesh):
    """Scalar pattern of a mesh: every pair of dofs of every cell (both components)."""
    dm = np.asarray(mesh.dofmap, dtype=np.int64)
    nd = dm.shape[1]
    r = np.repeat(dm, nd, axis=1).ravel()
    c = np.tile(dm, (1, nd)).ravel()
    S = sp.csr_matrix((np.ones(len(r)), (r, c)), shape=(mesh.nnodes, mesh.nnodes))
    S = sp.kron(S, np.ones((2, 2)), format="csr")
    S.data[:] = 1.0
    S.sort_indices()
    return S


def galerkin_levels(A, hier, fine_marker, nlevels):
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


def quad_hierarchies():
    return {"q2_lattice": fm.quad_lattice_hierarchy(fm.structured_quads_q2(16)),
            "q2_rect": fm.quad_lattice_hierarchy(fm.structured_quads_q2(24, 8)),
            "q2_jitter": fm.quad_lattice_hierarchy(fm.jitter(fm.structured_quads_q2(16), 0.2, seed=7)),
            "q2_odd": fm.quad_lattice_hierarchy(fm.structured_quads_q2(5, 3))}


# ---- CPU: hierarchies and maps --------------------------------------------------------------------------------------
def test_quad_lattice_hierarchy_levels():
    h = fm.quad_lattice_hierarchy(fm.structured_quads_q2(16))
    assert [m.etype for m in h] == [fm.Q1] * 5 + [fm.Q2]
    assert [m.nx for m in h] == [1, 2, 4, 8, 16, 16]
    h = fm.quad_lattice_hierarchy(fm.structured_quads_q2(24, 8))
    assert [(m.nx, m.ny) for m in h] == [(3, 1), (6, 2), (12, 4), (24, 8), (24, 8)]
    h = fm.quad_lattice_hierarchy(fm.structured_quads_q2(5, 3))
    assert [(m.etype, m.nx, m.ny) for m in h] == [(fm.Q1, 5, 3), (fm.Q2, 5, 3)]
    for h in quad_hierarchies().values():
        assert all(np.asarray(t).shape == (h[k + 1].nnodes, 4) and np.asarray(t).dtype == np.int32
                   for k, t in enumerate(h.maps))
        assert all(m.nd == 4 and m.nv == 4 for m in h.meshes[:-1])
        # the first Q1 level keeps the Q2 cell order: its vertices are those of the Q2 cell with the same number
        co = fm.coincident_nodes(h.maps[-1], h[-2].nnodes)
        assert np.array_equal(co[h[-2].dofmap], h[-1].dofmap[:, [0, 2, 6, 8]])
    with pytest.raises(ValueError):
        fm.quad_lattice_hierarchy(fm.structured_triangles(8, order=2))
    with pytest.raises(ValueError):
        fm.quad_lattice_hierarchy(fm.structured_triangles(8, order=1))


def test_width4_maps_follow_the_convention():
    for name, h in quad_hierarchies().items():
        for k, t in enumerate(h.maps):
            t = np.asarray(t)
            co = (t == t[:, [0]]).all(axis=1)
            edge = (t[:, 0] == t[:, 2]) & (t[:, 1] == t[:, 3]) & (t[:, 0] != t[:, 1])
            quad = np.array([len(set(r)) == 4 for r in t.tolist()])
            assert np.all(co | edge | quad), f"{name} level {k}"
            assert np.array_equal(co, t[:, 0] == t[:, 1]), f"{name} level {k}: column 0 == 1 only when coincident"
            assert co.sum() == h[k].nnodes
            # every (coarse node, partner) slot of the coarse pattern is named by exactly one fine node
            owners = {}
            for i, r in enumerate(t.tolist()):
                for j in range(4):
                    owners.setdefault((r[j], r[3 - j]), set()).add(i)
            assert all(len(v) == 1 for v in owners.values()), f"{name} level {k}"
            Sn = cell_pattern(h[k])[0::2, 0::2].tocoo()
            assert set(zip(Sn.row.tolist(), Sn.col.tolist())) == set(owners), f"{name} level {k}"


def test_width4_maps_reproduce_linear_and_bilinear_functions():
    """P I_c f = I_f f: linear f on every step of the unjittered meshes and on the Q2 -> Q1 step of the jittered one
    (the coarse lattices of a jittered mesh are nested in topology only); lattice-bilinear f on unjittered meshes."""
    for name, h in quad_hierarchies().items():
        for k in range(len(h) - 1):
            c, f = h[k], h[k + 1]
            if name == "q2_jitter" and k < len(h) - 2:
                continue
            P = node_P(h.maps[k], c.nnodes)
            fs = [lambda x: 0.3 + 2.0 * x[:, 0] - 1.5 * x[:, 1], lambda x: np.ones(len(x))]
            if name != "q2_jitter":
                fs.append(lambda x: 0.7 - x[:, 0] + 0.4 * x[:, 1] + 3.0 * x[:, 0] * x[:, 1])
            for fn in fs:
                np.testing.assert_allclose(P @ fn(c.x), fn(f.x), rtol=0, atol=1e-13, err_msg=f"{name} level {k}")


def test_quad_coarse_markers():
    for name, h in quad_hierarchies().items():
        bc, _ = fm.dirichlet_markers(h[-1])
        marks = h.markers(bc)
        for k, m in enumerate(h.meshes):
            want, _ = fm.dirichlet_markers(m)
            assert marks[k].dtype == np.uint8 and np.array_equal(marks[k], want), f"{name} level {k}"


def test_galerkin_pattern_is_q1_pattern():
    """The structural pattern of P^T S P is the Q1 mesh's all-pairs-per-cell pattern."""
    for name, h in quad_hierarchies().items():
        for k in range(len(h) - 1):
            c, f = h[k], h[k + 1]
            P = vec_P(h.maps[k], c.nnodes)
            G = (P.T @ cell_pattern(f) @ P).tocsr()
            G.sort_indices()
            Sc = cell_pattern(c)
            assert np.array_equal(G.indptr, Sc.indptr) and np.array_equal(G.indices, Sc.indices), f"{name} level {k}"


def test_q1_mesh_has_no_form():
    pytest.importorskip("torch")
    from femb200 import fem
    c = fm.quad_lattice_hierarchy(fm.structured_quads_q2(4))[-2]
    with pytest.raises(ValueError, match="Q1"):
        fem.ElasticityForm(c, np.ones(c.ncells))


# ---- GPU ------------------------------------------------------------------------------------------------------------
def _problem(m, matrix_free=False):
    """Assembled constrained operator (and the PA operator of the same form), lifted right-hand side with a body force."""
    import torch
    from femb200 import fem
    E = fm.young_per_cell(m.ncells)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, E, 0.3)
    A = fem.create_matrix(form)
    fem.assemble_matrix_nobc(A, form)
    gd = torch.from_numpy(g).cuda()
    Kg = A.mult(gd).cpu().numpy()
    f = np.zeros(m.ndofs)
    f[0::2] = fm.body_force(m)[:, 0] * 1e-6
    b = f - Kg
    b[bc != 0] = g[bc != 0]
    fem.assemble_matrix(A, form, bcs=[fem.DirichletBC(bc, g)])
    pa = fem.PAOperator(form, bcs=[fem.DirichletBC(bc, g)]) if matrix_free else None
    return A, pa, torch.from_numpy(b).cuda(), bc


def _pa_problem(m):
    """PA operator and right-hand side without an assembled matrix (large meshes)."""
    import torch
    from femb200 import fem
    E = fm.young_per_cell(m.ncells)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, E, 0.3)
    pa0 = fem.PAOperator(form)
    Kg = pa0.mult(torch.from_numpy(g).cuda()).cpu().numpy()
    del pa0
    f = np.zeros(m.ndofs)
    f[0::2] = fm.body_force(m)[:, 0] * 1e-6
    b = f - Kg
    b[bc != 0] = g[bc != 0]
    return fem.PAOperator(form, bcs=[fem.DirichletBC(bc, g)]), torch.from_numpy(b).cuda()


def _hier(m):
    return fm.quad_lattice_hierarchy(m) if m.etype == fm.Q2 else fm.lattice_hierarchy(m)


def _level_matrix(mg, l, shape):
    rp, ci = (t.cpu().numpy() for t in mg.level_csr(l))
    return sp.csr_matrix((mg.level_values(l).cpu().numpy(), ci, rp), shape=shape)


@pytest.mark.gpu
def test_q1_plan_pattern_spmv_and_refusals():
    import ctypes as C
    import torch
    from femb200 import capi, fem
    h = fm.quad_lattice_hierarchy(fm.jitter(fm.structured_quads_q2(12, 6), 0.2, seed=2))
    c = h[-2]
    st = fem._stream()
    dm = fem.to_device(c.dofmap, np.int32)
    plan = C.c_void_p()
    capi.call("femb200_plan_create", capi.Q1, c.nnodes, c.ncells, fem._p(dm), fem._p(dm), st, C.byref(plan))
    try:
        nn, nc, nzb, nz, md, by = (C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int32(), C.c_int64())
        capi.call("femb200_plan_sizes", plan, C.byref(nn), C.byref(nc), C.byref(nzb), C.byref(nz), C.byref(md), C.byref(by))
        assert md.value == 9
        rp = torch.empty(c.ndofs + 1, dtype=torch.int64, device="cuda")
        ci = torch.empty(nz.value, dtype=torch.int32, device="cuda")
        capi.call("femb200_plan_scalar_csr", plan, fem._p(rp), fem._p(ci), st)
        S = cell_pattern(c)
        assert np.array_equal(rp.cpu().numpy(), S.indptr) and np.array_equal(ci.cpu().numpy(), S.indices)
        rng = np.random.default_rng(3)
        vals = rng.standard_normal(nz.value)
        x = rng.standard_normal(c.ndofs)
        y = torch.empty(c.ndofs, dtype=torch.float64, device="cuda")
        vd, xd = torch.from_numpy(vals).cuda(), torch.from_numpy(x).cuda()
        capi.call("femb200_spmv", plan, fem._p(vd), fem._p(xd), fem._p(y), st)
        M = sp.csr_matrix((vals, S.indices, S.indptr), shape=S.shape)
        want = M @ x
        assert np.linalg.norm(y.cpu().numpy() - want) <= 1e-14 * np.linalg.norm(want)
        dg = torch.empty(c.ndofs, dtype=torch.float64, device="cuda")
        capi.call("femb200_extract_diagonal", plan, fem._p(vd), fem._p(dg), st)
        assert np.array_equal(dg.cpu().numpy(), M.diagonal())
        bc, g = fm.dirichlet_markers(c)
        bcd = fem.to_device(bc, np.uint8)
        capi.call("femb200_plan_set_dirichlet", plan, fem._p(bcd), st)
        capi.call("femb200_apply_dirichlet", plan, fem._p(vd), 1.0, st)
        keep = sp.diags((bc == 0).astype(float))
        Md = (keep @ M @ keep + sp.diags((bc != 0).astype(float))).tocsr()
        got = sp.csr_matrix((vd.cpu().numpy(), S.indices, S.indptr), shape=S.shape)
        assert abs(got - Md).max() == 0.0
        # element-level entry points refuse the pattern-only family, naming it
        xg = fem.to_device(c.x, np.float64)
        E = fem.to_device(np.ones(c.ncells), np.float64)
        u = torch.zeros(c.ndofs, dtype=torch.float64, device="cuda")
        out = torch.empty(c.ncells * 64 + nz.value, dtype=torch.float64, device="cuda")
        calls = {
            "femb200_tabulate_tensor_batched": (capi.Q1, c.ncells, fem._p(out), fem._p(xg), 2, fem._p(dm), fem._p(dm),
                                                fem._p(E), 0.3, None, None, 0, 0, st),
            "femb200_element_grad_batched": (capi.Q1, c.ncells, fem._p(out), fem._p(xg), 2, fem._p(dm), fem._p(dm),
                                             fem._p(E), 0.3, None, None, 0, st),
            "femb200_assemble_matrix": (plan, fem._p(xg), 2, fem._p(E), 0.3, None, None, 0, fem._p(out), st),
            "femb200_assemble_matrix_nobc": (plan, fem._p(xg), 2, fem._p(E), 0.3, None, None, 0, fem._p(out), st),
            "femb200_assemble_vector": (plan, fem._p(xg), 2, fem._p(E), 0.3, None, fem._p(u), None, fem._p(out), st),
            "femb200_apply_lifting": (plan, fem._p(vd), fem._p(u), fem._p(u), -1.0, fem._p(out), None, st),
            "femb200_cell_strain_stress": (capi.Q1, c.ncells, fem._p(dm), fem._p(dm), fem._p(xg), 2, fem._p(E), 0.3, None,
                                           fem._p(u), fem._p(out), None, st),
            "femb200_smooth_damage": (plan, fem._p(out), fem._p(out), 1, 0.01, st),
        }
        for name, args in calls.items():
            with pytest.raises(capi.Femb200Error, match="Q1"):
                capi.call(name, *args)
        pa = C.c_void_p()
        for name in ("femb200_pa_create", "femb200_assemble_pa"):
            with pytest.raises(capi.Femb200Error, match="Q1"):
                capi.call(name, capi.Q1, c.nnodes, c.ncells, fem._p(dm), fem._p(dm), fem._p(xg), 2, fem._p(E), 0.3, st,
                          C.byref(pa))
    finally:
        capi.lib().femb200_plan_destroy(plan)


def _assembled_quad_cases():
    return {"q2_jitter": fm.jitter(fm.structured_quads_q2(32), 0.2, seed=3),
            "q2_rect": fm.structured_quads_q2(48, 16)}


@pytest.mark.gpu
def test_assembled_q2_galerkin_and_transfers_match_scipy():
    import torch
    from femb200 import fem
    rng = np.random.default_rng(5)
    for name, m in _assembled_quad_cases().items():
        A, _, _, bc = _problem(m)
        h = fm.quad_lattice_hierarchy(m)
        mg = fem.MultigridPreconditioner(A, h, coarse_max=600)
        mg.setup()
        levels, _ = galerkin_levels(A.to_scipy(), h, bc, mg.nlevels)
        first = []
        for l in range(1, mg.nlevels + 1):
            got = _level_matrix(mg, l, levels[l].shape)
            err = spla.norm(got - levels[l]) / spla.norm(levels[l])
            assert err <= 1e-12, f"{name} level {l}: {err:.3e}"
            first.append(got.data.copy())
        mg.setup()
        for l in range(1, mg.nlevels + 1):
            assert np.array_equal(first[l - 1], mg.level_values(l).cpu().numpy()), f"{name}: setup is not deterministic"
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


def _pa_cases():
    return {"p2_lattice": fm.structured_triangles(32, order=2),
            "p2_jitter": fm.jitter(fm.structured_triangles(32, order=2), 0.2, seed=3),
            "q2_lattice": fm.structured_quads_q2(32),
            "q2_jitter": fm.jitter(fm.structured_quads_q2(32), 0.2, seed=3)}


@pytest.mark.gpu
def test_matrix_free_galerkin_levels_match_assembled_cascade():
    """Every level >= 1 built from the PA handle (element Galerkin step, then the cascade) matches scipy's cascade from
    the assembled constrained matrix; a second setup() reproduces them bit for bit."""
    from femb200 import fem
    for name, m in _pa_cases().items():
        A, pa, _, bc = _problem(m, matrix_free=True)
        d = pa.diagonal().cpu().numpy()
        assert np.all(d[bc != 0] == 1.0), f"{name}: the PA diagonal must carry the unit Dirichlet diagonal"
        h = _hier(m)
        mg = fem.MultigridPreconditioner(pa, h, coarse_max=600)
        mg.setup()
        nd, nz, _, _ = mg.sizes()
        assert nz[0] == 0 and nd[0] == m.ndofs
        levels, _ = galerkin_levels(A.to_scipy(), h, bc, mg.nlevels)
        first = []
        for l in range(1, mg.nlevels + 1):
            got = _level_matrix(mg, l, levels[l].shape)
            err = spla.norm(got - levels[l]) / spla.norm(levels[l])
            assert err <= 1e-12, f"{name} level {l}: {err:.3e}"
            first.append(got.data.copy())
        mg.galerkin(0)
        assert np.array_equal(first[0], mg.level_values(1).cpu().numpy()), f"{name}: galerkin(0) differs from setup()"
        mg.setup()
        for l in range(1, mg.nlevels + 1):
            assert np.array_equal(first[l - 1], mg.level_values(l).cpu().numpy()), f"{name}: setup is not deterministic"
        mg.close()


@pytest.mark.gpu
def test_matrix_free_vcycle_matches_restatement_and_is_spd():
    import torch
    from femb200 import fem
    rng = np.random.default_rng(11)
    for name in ("p2_jitter", "q2_jitter"):
        m = _pa_cases()[name]
        A, pa, _, bc = _problem(m, matrix_free=True)
        h = _hier(m)
        mg = fem.MultigridPreconditioner(pa, h, coarse_max=600)
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
            assert err <= 1e-10, f"{name}: V-cycle {err:.3e}"
        x, y = (torch.from_numpy(rng.standard_normal(A.ndofs)).cuda() for _ in range(2))
        Bx, By = mg.apply(x), mg.apply(y)
        asym = abs(torch.dot(Bx, y).item() - torch.dot(x, By).item())
        assert asym <= 1e-12 * Bx.norm().item() * y.norm().item(), f"{name}: V-cycle not symmetric ({asym:.3e})"
        assert torch.dot(Bx, x).item() > 0 and torch.dot(By, y).item() > 0
        with pytest.raises(ValueError):
            mg.apply(x, x)
        mg.close()


@pytest.mark.gpu
def test_matrix_free_mg_pcg_matches_spsolve_and_assembled():
    from femb200 import fem
    for name in ("p2_lattice", "q2_jitter"):
        m = _pa_cases()[name]
        A, pa, b, _ = _problem(m, matrix_free=True)
        h = _hier(m)
        xs = spla.spsolve(A.to_scipy().tocsc(), b.cpu().numpy())
        mg = fem.MultigridPreconditioner(pa, h)
        mg.setup()
        x = b.clone()
        its, _, conv = mg.solve(b, x, 1e-12, 0.0, 200)
        err = np.linalg.norm(x.cpu().numpy() - xs) / np.linalg.norm(xs)
        assert conv and err <= 1e-10, f"{name}: {its} its, error {err:.3e}"
        cg = fem.CGSolver(rel_tol=1e-12, max_iter=200)
        cg.SetOperator(pa)
        cg.SetPreconditioner("mg", hierarchy=h)
        xc = cg.Mult(b)
        assert cg.GetConverged() and cg.GetNumIterations() == its
        assert np.linalg.norm(xc.cpu().numpy() - x.cpu().numpy()) <= 1e-12 * np.linalg.norm(xs)
        cg2 = fem.CGSolver(rel_tol=1e-12, max_iter=200)
        cg2.SetOperator(pa)
        cg2.SetPreconditioner(mg)
        cg2.Mult(b)
        assert cg2.GetConverged() and cg2.GetNumIterations() == its
        if m.etype == fm.P2:
            ma = fem.MultigridPreconditioner(A, h)
            ma.setup()
            its_a, _, conv_a = ma.solve(b, b.clone(), 1e-12, 0.0, 200)
            assert conv_a and abs(its_a - its) <= 1, (its_a, its)
            ma.close()
        cg.mg.close()
        mg.close()


@pytest.mark.gpu
def test_matrix_free_q2_iterations_do_not_grow_with_resolution():
    from femb200 import fem
    its = []
    for s in (32, 64, 128, 256):
        m = fm.jitter(fm.structured_quads_q2(s), 0.2, seed=1234)
        pa, b = _pa_problem(m)
        mg = fem.MultigridPreconditioner(pa, fm.quad_lattice_hierarchy(m))
        mg.setup()
        x = b.clone()
        it, _, conv = mg.solve(b, x, 1e-12, 0.0, 200)
        assert conv, f"{s}: multigrid-PCG did not converge in 200 iterations"
        mg.close()
        cg = fem.CGSolver(rel_tol=1e-12, max_iter=10 * it)
        cg.SetOperator(pa)
        cg.SetPreconditioner("jacobi")
        cg.Mult(b)
        print(f"Q2 jittered {s} x {s}: multigrid {it}, Jacobi converged within {10 * it}: {cg.GetConverged()}")
        assert not cg.GetConverged(), f"{s}: Jacobi-PA-PCG converged within 10 x {it} iterations"
        its.append(it)
    # Measured on a B200: 18, 20, 19, 20 iterations at 32, 64, 128, 256 cells per side; Jacobi-PA-PCG does not
    # converge within ten times those counts.
    assert all(it <= 25 for it in its), its
    assert its[-1] <= its[0] + 5, its


@pytest.mark.gpu
def test_matrix_free_mg_pcg_on_a_fresh_stream():
    """First matrix-free multigrid solve on a new stream, more than 131 k nodes: the PA apply grows the stream's
    fused-reduction scratch and the <B r, r> reductions must use the grown scratch.  Same result as on the default
    stream."""
    import torch
    from femb200 import fem
    m = fm.structured_quads_q2(256)                    # 263 169 nodes
    out = {}
    for fresh in (False, True):
        ctx = torch.cuda.stream(torch.cuda.Stream()) if fresh else torch.cuda.stream(torch.cuda.current_stream())
        with ctx:
            pa, b = _pa_problem(m)
            mg = fem.MultigridPreconditioner(pa, fm.quad_lattice_hierarchy(m))
            mg.setup()
            x = torch.empty_like(b)
            its, _, conv = mg.solve(b, x, 1e-12, 0.0, 100)
            torch.cuda.current_stream().synchronize()
            out[fresh] = (its, conv, x.cpu().numpy())
            mg.close()
    (i0, c0, x0), (i1, c1, x1) = out[False], out[True]
    assert c0 and c1 and abs(i0 - i1) <= 1, (i0, i1)
    assert np.linalg.norm(x1 - x0) <= 1e-10 * np.linalg.norm(x0)


@pytest.mark.gpu
def test_matrix_free_mg_errors():
    import torch
    from femb200 import capi, fem
    # h-coarsening first step (a P1 operator on a refined triangulation)
    h = fm.refine_uniform_hierarchy(fm.structured_triangles(4, order=1), 2)
    _, pa, _, _ = _problem(h[-1], matrix_free=True)
    with pytest.raises(ValueError, match="p-coarsening"):
        fem.MultigridPreconditioner(pa, h)
    # a hierarchy of another mesh
    m = fm.structured_quads_q2(16)
    _, pa, b, _ = _problem(m, matrix_free=True)
    with pytest.raises(ValueError, match="not the mesh of the operator"):
        fem.MultigridPreconditioner(pa, fm.quad_lattice_hierarchy(fm.structured_quads_q2(32, 8)))
    with pytest.raises(ValueError, match="not the mesh of the operator"):
        fem.MultigridPreconditioner(pa, fm.quad_lattice_hierarchy(fm.jitter(m, 0.2, seed=1)))
    # a first coarse mesh whose cells are numbered differently from the fine mesh's
    h = fm.quad_lattice_hierarchy(m)
    perm = np.random.default_rng(0).permutation(h[-2].ncells)
    c = h[-2]
    h.meshes[-2] = fm.Mesh(fm.Q1, c.x, c.xdofmap[perm].copy(), c.dofmap[perm].copy(), c.nx, c.ny, dict(c.meta))
    with pytest.raises(capi.Femb200Error, match="p-coarsening"):
        fem.MultigridPreconditioner(pa, h)
    # a map that is nested (every coarse slot named once) but not the element interpolation: two edge midpoints swapped
    h = fm.quad_lattice_hierarchy(m)
    t = h.maps[-1].copy()
    mid = np.nonzero((t[:, 0] == t[:, 2]) & (t[:, 0] != t[:, 1]))[0]
    t[[mid[0], mid[-1]]] = t[[mid[-1], mid[0]]]
    h.maps[-1] = t
    with pytest.raises(capi.Femb200Error, match="p-coarsening"):
        fem.MultigridPreconditioner(pa, h)
    # fine values handed to a matrix-free handle
    mg = fem.MultigridPreconditioner(pa, fm.quad_lattice_hierarchy(m))
    junk = torch.zeros(16, dtype=torch.float64, device="cuda")
    for name, args in (("femb200_mg_setup", (fem._p(junk), fem._stream())),
                       ("femb200_mg_galerkin", (fem._p(junk), 0, fem._stream()))):
        with pytest.raises(capi.Femb200Error, match="matrix-free"):
            capi.call(name, mg.handle, *args)
    mg.close()


@pytest.mark.gpu
def test_matrix_free_mg_follows_reassembly_of_the_operator():
    """PAOperator.AssemblePA replaces the device operator the multigrid handle borrows: the V-cycle and the solve refuse
    to run on the old one, setup() rebuilds the handle on the new one and gives the same solve."""
    import torch
    from femb200 import fem
    m = fm.jitter(fm.structured_quads_q2(32), 0.2, seed=3)
    _, pa, b, _ = _problem(m, matrix_free=True)
    h = fm.quad_lattice_hierarchy(m)
    mg = fem.MultigridPreconditioner(pa, h)
    mg.setup()
    x0 = torch.empty_like(b)
    its0, _, conv0 = mg.solve(b, x0, 1e-12, 0.0, 200)
    levels0 = [mg.level_values(l).cpu().numpy() for l in range(1, mg.nlevels + 1)]
    cg = fem.CGSolver(rel_tol=1e-12, max_iter=200)
    cg.SetOperator(pa)
    cg.SetPreconditioner(mg)
    for _ in range(2):
        pa.AssemblePA()
        with pytest.raises(RuntimeError, match="AssemblePA"):
            mg.apply(b)
        with pytest.raises(RuntimeError, match="AssemblePA"):
            mg.solve(b, torch.empty_like(b))
        with pytest.raises(RuntimeError, match="AssemblePA"):
            cg.Mult(b)
        mg.setup()
        for l in range(1, mg.nlevels + 1):
            assert np.array_equal(levels0[l - 1], mg.level_values(l).cpu().numpy()), f"level {l} after reassembly"
        x = cg.Mult(b)
        assert conv0 and cg.GetConverged() and abs(cg.GetNumIterations() - its0) <= 1
        assert np.linalg.norm((x - x0).cpu().numpy()) <= 1e-10 * np.linalg.norm(x0.cpu().numpy())
    mg.close()


@pytest.mark.gpu
def test_transfers_follow_a_reset_of_the_fine_dirichlet_marker():
    """Clearing the fine Matrix's Dirichlet conditions frees the plan's marker and setting them again allocates a new
    one: restriction and prolongation read the current marker."""
    import torch
    from femb200 import fem
    rng = np.random.default_rng(9)
    m = fm.structured_quads_q2(24, 8)
    A, _, _, bc = _problem(m)
    h = fm.quad_lattice_hierarchy(m)
    mg = fem.MultigridPreconditioner(A, h, coarse_max=600)
    A.set_bcs(None)
    A.set_bcs([fem.DirichletBC(*fm.dirichlet_markers(m))])
    marks = h.markers(bc)
    k = len(h) - 2
    P = vec_P(h.maps[k], h[k].nnodes, marks[k + 1], marks[k])
    xc, x, b = rng.standard_normal(P.shape[1]), rng.standard_normal(P.shape[0]), rng.standard_normal(P.shape[0])
    got = mg.prolong(0, torch.from_numpy(xc).cuda(), torch.from_numpy(x).cuda()).cpu().numpy()
    assert np.array_equal(got, x + P @ xc)
    want = P.T @ b
    got = mg.restrict(0, torch.from_numpy(b).cuda()).cpu().numpy()
    assert np.linalg.norm(got - want) <= 1e-15 * np.linalg.norm(want)
    mg.close()
