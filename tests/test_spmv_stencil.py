"""SpMV with stencil ids: each node row's column offsets J - I come from a per-plan dictionary of the distinct offset
lists, so the staged SpMV streams the values and one id byte per row.  The stencil mode (spmv_cols = 0, the default
where the plan has a dictionary) must give the same y, the same fused <x, y> and the same PCG iterates, bit for bit,
as the 16-bit offsets (spmv_cols = 2) and the 32-bit indices (spmv_cols = 1)."""
import ctypes as C
import json
import os

import numpy as np
import pytest

from femb200 import mesh as fm

K_MAX, D_MAX = 64, 32   # dictionary caps of the plan


def stencil_count(brp, bcol):
    """Number of stencil ids the plan should have: the distinct offset lists of the block pattern, or 0 when there
    are more than K_MAX, a row is longer than D_MAX or an offset does not fit in 16 bits."""
    brp, bcol = np.asarray(brp, dtype=np.int64), np.asarray(bcol, dtype=np.int64)
    nn = brp.size - 1
    off = bcol - np.repeat(np.arange(nn), np.diff(brp))
    if np.diff(brp).max() > D_MAX or np.abs(off).max() > 32767:
        return 0
    lists = {tuple(off[brp[i]:brp[i + 1]]) for i in range(nn)}
    return len(lists) if len(lists) <= K_MAX else 0


def _blocks_of(m):
    """Block CSR (brp, bcol) of a mesh from the oracle's scalar pattern: rowptr[2I] = 4 brp[I], colidx of row 2I =
    2 bcol, 2 bcol + 1."""
    from oracle import oracle
    rp, ci = oracle.build_pattern(m.nnodes, m.dofmap)
    return (np.append(rp[0:-1:2] // 4, rp[-1] // 4),
            np.concatenate([ci[rp[2 * i]:rp[2 * i + 1]:2] // 2 for i in range(m.nnodes)]))


def test_stencil_count_restatement():
    m = fm.structured_triangles(12, 7, order=2)
    brp, bcol = _blocks_of(m)
    n = stencil_count(brp, bcol)
    assert 0 < n <= K_MAX
    assert n == stencil_count(*_blocks_of(fm.structured_triangles(20, 9, order=2)))   # independent of the size
    perm = np.random.default_rng(1).permutation(m.nnodes)
    assert stencil_count(brp, perm[bcol]) == 0   # no locality: more than K_MAX lists


def test_probe_rehearsal(tmp_path):
    """tools/spmv_stencil_probe.py without a device: arguments, mesh and the byte counts of both column modes."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("spmv_stencil_probe", os.path.join(root, "tools", "spmv_stencil_probe.py"))
    probe = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(probe)
    res = probe.main([str(tmp_path), "--size", "6", "--dry-run"])
    with open(tmp_path / "spmv_stencil_probe.json") as f:
        assert json.load(f) == res
    m = fm.structured_triangles(6, order=2)
    brp, _ = _blocks_of(m)
    nb, nn = int(brp[-1]), m.nnodes
    assert res["nnz_blocks"] == nb and res["nnodes"] == nn
    assert res["bytes_per_spmv"] == {"stencil": 32 * nb + nn + 32 * nn, "bcol16": 34 * nb + 8 * nn + 32 * nn}
    with pytest.raises(SystemExit):
        probe.main([str(tmp_path), "--rounds", "0"])


# ---- GPU ------------------------------------------------------------------------------------------------------------
class _Plan:
    """A plan handle with values: an assembled Matrix, or a pattern-only plan (Q1) with random values."""

    def __init__(self, plan, values, nnodes, keep=None):
        self.plan, self.values, self.nnodes, self.keep = plan, values, nnodes, keep

    def option(self, key, value=None):
        from femb200 import capi
        if value is not None:
            capi.call("femb200_plan_set_option", self.plan, key.encode(), int(value))
            return value
        v = C.c_int()
        capi.call("femb200_plan_get_option", self.plan, key.encode(), C.byref(v))
        return v.value

    def blocks(self, nnzb):
        import torch
        from femb200 import capi, fem
        brp = torch.empty(self.nnodes + 1, dtype=torch.int64, device="cuda")
        bcol = torch.empty(nnzb, dtype=torch.int32, device="cuda")
        capi.call("femb200_plan_copy_block_csr", self.plan, fem._p(brp), fem._p(bcol), fem._stream())
        return brp.cpu().numpy(), bcol.cpu().numpy()


def _assembled(m):
    from femb200 import fem
    form = fem.ElasticityForm(m, fm.young_per_cell(m.ncells))
    A = fem.assemble_matrix(fem.create_matrix(form), form)
    return _Plan(A.plan, A.values, A.nnodes, keep=A), A.nnz_blocks


def _pattern_only(m, etype):
    import torch
    from femb200 import capi, fem
    dm = fem.to_device(m.dofmap, np.int32)
    plan = C.c_void_p()
    capi.call("femb200_plan_create", etype, m.nnodes, m.ncells, fem._p(dm), fem._p(dm), fem._stream(), C.byref(plan))
    nn, nc, nzb, nz, md, by = (C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int32(), C.c_int64())
    capi.call("femb200_plan_sizes", plan, C.byref(nn), C.byref(nc), C.byref(nzb), C.byref(nz), C.byref(md), C.byref(by))
    vals = torch.from_numpy(np.random.default_rng(4).standard_normal(nz.value)).cuda()

    class Owner:
        def __del__(self):
            capi.lib().femb200_plan_destroy(plan)
    return _Plan(plan, vals, m.nnodes, keep=(dm, Owner())), nzb.value


def _cases():
    lattice_p1 = fm.structured_triangles(6, order=1)
    return {
        "p2_lattice": lambda: _assembled(fm.jitter(fm.structured_triangles(40, 23, order=2), 0.2, seed=3)),
        "p1": lambda: _assembled(fm.jitter(fm.structured_triangles(30, 17, order=1), 0.2, seed=3)),
        "q2": lambda: _assembled(fm.jitter(fm.structured_quads_q2(12, 9), 0.2, seed=3)),
        "q1_hierarchy": lambda: _pattern_only(fm.quad_lattice_hierarchy(fm.structured_quads_q2(24, 12))[-2], fm.Q1),
        "refined_p1": lambda: _assembled(fm.refine_uniform_hierarchy(lattice_p1, 2)[-1]),
    }


def _apply_all(P, x):
    """Full apply, fused-dot apply and ragged row ranges (with their dots) under the plan's current options."""
    import torch
    from femb200 import capi, fem
    n = P.nnodes
    out = []
    y = torch.empty_like(x)
    capi.call("femb200_spmv", P.plan, fem._p(P.values), fem._p(x), fem._p(y), fem._stream())
    out.append(y.clone())
    dot = torch.zeros(1, dtype=torch.float64, device="cuda")
    capi.call("femb200_spmv_dot", P.plan, fem._p(P.values), fem._p(x), fem._p(y), fem._p(dot), fem._stream())
    out += [y.clone(), dot.clone()]
    for lo, hi in ((1, n - 1), (163, min(n, 1000)), (n - 5, n), (17, 17 + 64), (0, n)):
        lo = min(lo, n)
        y = torch.full_like(x, -3.0)
        dot = torch.full((1,), 2.0, dtype=torch.float64, device="cuda")
        capi.call("femb200_spmv_rows", P.plan, fem._p(P.values), fem._p(x), fem._p(y), lo, hi, fem._p(dot), 1, None,
                  fem._stream())
        out += [y, dot]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(_cases()))
def test_stencil_spmv_bitwise(case):
    import torch
    P, nnzb = _cases()[case]()
    brp, bcol = P.blocks(nnzb)
    want = stencil_count(brp, bcol)
    assert P.option("spmv_stencils") == want
    if case != "refined_p1":
        assert want > 0, "lattice numberings have a dictionary"
    assert P.option("spmv_col_bits") == (0 if want else 16)
    x = torch.from_numpy(np.random.default_rng(11).standard_normal(2 * P.nnodes)).cuda()
    got = {}
    for cols in (0, 2, 1):
        P.option("spmv_cols", cols)
        got[cols] = _apply_all(P, x)
    assert P.option("spmv_col_bits") == 32
    P.option("spmv_cols", 2)
    assert P.option("spmv_col_bits") == 16 and P.option("spmv_stencils") == want
    P.option("spmv_cols", 0)
    for cols in (2, 1):
        for k, (a, b) in enumerate(zip(got[0], got[cols])):
            assert torch.equal(a, b), f"{case}: output {k} differs between spmv_cols 0 and {cols}"
    # against the scalar CSR on the host
    from femb200 import capi, fem
    import scipy.sparse as sp
    rp = torch.empty(2 * P.nnodes + 1, dtype=torch.int64, device="cuda")
    ci = torch.empty(4 * nnzb, dtype=torch.int32, device="cuda")
    capi.call("femb200_plan_scalar_csr", P.plan, fem._p(rp), fem._p(ci), fem._stream())
    M = sp.csr_matrix((P.values.cpu().numpy(), ci.cpu().numpy(), rp.cpu().numpy()))
    ref = M @ x.cpu().numpy()
    assert np.linalg.norm(got[0][0].cpu().numpy() - ref) <= 1e-13 * np.linalg.norm(ref)


@pytest.mark.gpu
def test_stencil_refusals():
    """Numberings without a small dictionary keep the index paths: the random permutation of a 40 401-node P1 mesh
    (offsets beyond 2^15: 32-bit indices) and of a 441-node one (offsets fit 16 bits, but hundreds of lists)."""
    import torch
    from femb200 import fem
    for n, bits in ((200, 32), (20, 16)):
        m1 = fm.structured_triangles(n, order=1)
        perm = np.random.default_rng(7).permutation(m1.nnodes).astype(np.int32)
        inv = np.empty_like(perm)
        inv[perm] = np.arange(m1.nnodes, dtype=np.int32)
        mp = fm.Mesh(m1.etype, np.ascontiguousarray(m1.x[inv]), perm[m1.xdofmap], perm[m1.dofmap], 0, 0, {})
        form = fem.ElasticityForm(mp, fm.young_per_cell(mp.ncells))
        A = fem.assemble_matrix(fem.create_matrix(form), form)
        assert A.get_option("spmv_col_bits") == bits and A.get_option("spmv_stencils") == 0
        x = torch.from_numpy(np.random.default_rng(2).standard_normal(mp.ndofs)).cuda()
        y0 = A.mult(x).clone()
        A.set_option("spmv_cols", 1)
        assert torch.equal(A.mult(x), y0)
    with pytest.raises(fem.capi.Femb200Error, match="spmv_cols"):
        A.set_option("spmv_cols", 3)


@pytest.mark.gpu
def test_stencil_pcg_bitwise():
    """Jacobi-PCG with 25 fixed iterations, and multigrid-PCG on a lattice hierarchy (every level's plan switched):
    the same iterate under stencil ids and under 16-bit offsets."""
    import torch
    from femb200 import capi, fem
    m = fm.jitter(fm.structured_triangles(48, 40, order=2), 0.2, seed=5)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, fm.young_per_cell(m.ncells))
    A = fem.assemble_matrix(fem.create_matrix(form), form, bcs=[fem.DirichletBC(bc, g)])
    assert A.get_option("spmv_col_bits") == 0
    b = torch.from_numpy(np.where(bc != 0, g, 1.0)).cuda()
    xs = {}
    for cols in (0, 2):
        A.set_option("spmv_cols", cols)
        cg = fem.CGSolver(rel_tol=0.0, max_iter=25)
        cg.SetOperator(A)
        cg.SetPreconditioner("jacobi")
        xs[cols] = cg.Mult(b, fixed_iters=25).clone()
    assert torch.equal(xs[0], xs[2])
    mg = fem.MultigridPreconditioner(A, fm.lattice_hierarchy(m), coarse_max=600)
    try:
        for cols in (0, 2):
            A.set_option("spmv_cols", cols)
            for p in mg._plans:
                capi.call("femb200_plan_set_option", p, b"spmv_cols", cols)
            mg.setup()
            x = torch.zeros_like(b)
            mg.solve(b, x, 0.0, 0.0, 8)
            xs[("mg", cols)] = x
        assert torch.equal(xs[("mg", 0)], xs[("mg", 2)])
    finally:
        mg.close()
