"""Compact values of the PCG: on a P2 mesh the block of a vertex and of the midpoint of its opposite edge is zero on
every straight-sided cell, and only that cell holds the pair, so the PCG applies stream a copy of the values without
those blocks (spmv_compact = 0, the default where the plan has compact keys).  The first apply of a solve writes the
copy and checks that every dropped block is +-0; when one is not, the solve streams the CSR values.  Either way the
iterates, scalars and iteration counts must equal those of spmv_compact = 1 bit for bit."""

import numpy as np
import pytest

from femb200 import mesh as fm

K_MAX = 64   # compact keys of a plan


def dropped_pairs(dofmap):
    """(I, J) node pairs every cell holding both has as a vertex / opposite-edge pair (P2, basix order: edge 3 + i is
    opposite vertex i), both directions."""
    dm = np.asarray(dofmap, dtype=np.int64).reshape(-1, 6)
    opp, other = set(), set()
    for a in range(6):
        for b in range(6):
            pairs = set(zip(dm[:, a].tolist(), dm[:, b].tolist()))
            (opp if b == a + 3 or a == b + 3 else other).update(pairs)
    return opp - other


def compact_keys(brp, bcol, dropped):
    """Number of compact keys the plan should have: distinct (column offsets, kept slots) of the node rows, in the
    plan's column order; 0 when there are more than K_MAX or nothing is dropped."""
    keys = set()
    for i in range(brp.size - 1):
        cols = bcol[brp[i]:brp[i + 1]].tolist()
        keys.add((tuple(c - i for c in cols), tuple((i, c) not in dropped for c in cols)))
    return len(keys) if (len(keys) <= K_MAX and dropped) else 0


@pytest.mark.parametrize("nx,ny", [(6, 4), (13, 9), (32, 20)])
def test_dropped_pairs_restatement(nx, ny):
    m = fm.jitter(fm.structured_triangles(nx, ny, order=2), 0.2, seed=1)
    assert len(dropped_pairs(m.dofmap)) == 6 * m.ncells


def _problem(nx=48, ny=40):
    import torch
    from femb200 import fem
    m = fm.jitter(fm.structured_triangles(nx, ny, order=2), 0.2, seed=5)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, fm.young_per_cell(m.ncells))
    A = fem.assemble_matrix(fem.create_matrix(form), form, bcs=[fem.DirichletBC(bc, g)])
    b = torch.from_numpy(np.where(bc != 0, g, 1.0)).cuda()
    return m, form, A, b


def _blocks(A):
    import torch
    from femb200 import capi, fem
    brp = torch.empty(A.nnodes + 1, dtype=torch.int64, device="cuda")
    bcol = torch.empty(A.nnz_blocks, dtype=torch.int32, device="cuda")
    capi.call("femb200_plan_copy_block_csr", A.plan, fem._p(brp), fem._p(bcol), fem._stream())
    return brp.cpu().numpy(), bcol.cpu().numpy()


def _solves(A, b):
    """Jacobi and unpreconditioned PCG, 25 fixed iterations and to convergence: (x, iterations, final norm) each."""
    from femb200 import fem
    out = []
    for pre in ("jacobi", "none"):
        for rtol, fixed in ((0.0, 25), (1e-9, 0)):
            cg = fem.CGSolver(rel_tol=rtol, max_iter=4000)
            cg.SetOperator(A)
            cg.SetPreconditioner(pre)
            x = cg.Mult(b, fixed_iters=fixed).clone()
            out.append((x, cg.GetNumIterations(), cg.GetFinalNorm()))
    return out


def _assert_same(a, b, what):
    import torch
    for k, ((x0, i0, f0), (x1, i1, f1)) in enumerate(zip(a, b)):
        assert torch.equal(x0, x1) and i0 == i1 and f0 == f1, f"{what}: solve {k} differs"


@pytest.mark.gpu
def test_compact_keys_and_pcg_bitwise():
    m, _, A, b = _problem()
    brp, bcol = _blocks(A)
    want = compact_keys(brp, bcol, dropped_pairs(m.dofmap))
    assert 0 < want <= K_MAX
    assert A.get_option("spmv_compact_keys") == want
    assert A.get_option("spmv_compact") == 0
    on = _solves(A, b)
    A.set_option("spmv_compact", 1)
    off = _solves(A, b)
    A.set_option("spmv_compact", 0)
    _assert_same(on, off, "spmv_compact 0 / 1")
    assert on[1][1] < 4000 and on[3][1] < 4000, "the converged solves stop before max_iter"
    _assert_same(_solves(A, b), on, "second solve on the same plan")


@pytest.mark.gpu
def test_compact_fallback_on_nonzero_dropped_blocks():
    """A dropped block edited to non-zero through torch, and a damaged tangent: the solve streams the CSR values and
    gives the spmv_compact = 1 result; an undamaged reassembly brings the compact path back with the same result."""
    import torch
    from femb200 import fem
    m, form, A, b = _problem(24, 18)
    brp, bcol = _blocks(A)
    drop = dropped_pairs(m.dofmap)
    I = next(i for i in range(A.nnodes) if any((i, int(c)) in drop for c in bcol[brp[i]:brp[i + 1]]))
    s = next(s for s, c in enumerate(bcol[brp[I]:brp[I + 1]]) if (I, int(c)) in drop)
    deg = int(brp[I + 1] - brp[I])
    base = 4 * int(brp[I])
    assert A.values[base + 2 * s].item() == 0 and A.values[base + 2 * deg + 2 * s + 1].item() == 0
    ref = _solves(A, b)

    def both(what):
        on = _solves(A, b)
        A.set_option("spmv_compact", 1)
        off = _solves(A, b)
        A.set_option("spmv_compact", 0)
        _assert_same(on, off, what)
        return on

    A.values[base + 2 * deg + 2 * s + 1] = 1.0
    edited = both("edited dropped block")
    assert not torch.equal(edited[0][0], ref[0][0]), "the edited block reaches the iterate"
    rng = np.random.default_rng(0)
    fd = fem.ElasticityForm(m, fm.young_per_cell(m.ncells), 0.3, d=fm.damage_band(m),
                            u=1e-3 * rng.standard_normal(m.ndofs), variant=1)
    fem.assemble_matrix_nobc(A, fd)
    both("damaged tangent")
    bc, g = fm.dirichlet_markers(m)
    fem.assemble_matrix(A, form, bcs=[fem.DirichletBC(bc, g)])
    A2 = fem.assemble_matrix(fem.create_matrix(form), form, bcs=[fem.DirichletBC(bc, g)])
    _assert_same(both("reassembled"), _solves(A2, b), "reassembled against a fresh matrix")


@pytest.mark.gpu
def test_compact_refusals():
    """P1 and Q2 have no dropped blocks; a P2 numbering without a stencil dictionary has no compact keys; the option
    takes 0 or 1 only."""
    import torch
    from femb200 import fem
    for m in (fm.structured_triangles(12, order=1), fm.structured_quads_q2(8)):
        A = fem.create_matrix(fem.ElasticityForm(m, fm.young_per_cell(m.ncells)))
        assert A.get_option("spmv_compact_keys") == 0
    m2 = fm.structured_triangles(20, order=2)
    perm = np.random.default_rng(7).permutation(m2.nnodes).astype(np.int32)
    inv = np.empty_like(perm)
    inv[perm] = np.arange(m2.nnodes, dtype=np.int32)
    mp = fm.Mesh(m2.etype, np.ascontiguousarray(m2.x[inv]), perm[m2.xdofmap], perm[m2.dofmap], 0, 0, {})
    form = fem.ElasticityForm(mp, fm.young_per_cell(mp.ncells))
    A = fem.assemble_matrix(fem.create_matrix(form), form)
    assert A.get_option("spmv_stencils") == 0 and A.get_option("spmv_compact_keys") == 0
    b = torch.ones(mp.ndofs, dtype=torch.float64, device="cuda")
    cg = fem.CGSolver(rel_tol=0.0, max_iter=10)
    cg.SetOperator(A)
    cg.SetPreconditioner("jacobi")
    assert torch.isfinite(cg.Mult(b, fixed_iters=10)).all()
    with pytest.raises(fem.capi.Femb200Error, match="spmv_compact"):
        A.set_option("spmv_compact", 2)
