"""Synthetic meshes, dof maps and problem data for the mechanic2d hot path.

Input generation only (host side, numpy): nothing here is on the timed path.
Conventions are the ones fixed in SURVEY.md 8c:

* unit square [0,1]^2 (or [0,1] x [0,ny/nx]), structured nx x ny cells; triangles
  are each cell split by the "right" diagonal into {v0,v1,v3}, {v0,v2,v3};
* P2/Q2 nodes live on the (2nx+1) x (2ny+1) lattice, numbered lexicographically
  (x fastest); P1 nodes on the (nx+1) x (ny+1) lattice;
* P2 local dof order is basix': three vertices, then the midpoint of the edge
  opposite to vertex i; Q2 local order is tensor / lexicographic (ix + 3 iy);
* global dof = 2 * node + component (blocked, bs = 2: `M.cc:1107`, `F.cc:691`);
* materials: the reference's 200 Young moduli (`M.cc:1076-1085`) indexed by
  `cell_id % 200`, nu = 0.3 (`M.cc:1074`);
* Dirichlet: all dofs on x = 0 clamped, on x = 1: ux = +0.01, uy = 0
  (`F.cc:627-664`); body force `M.cc:1431-1440`.

All `file:line` citations are relative to /root/reference (M.cc =
MFEM/mechanic2d/asym_elasto_damage_model.cc, F.cc = FEniCSx/mechanic2d/...).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass, field

import numpy as np

P1, P2, Q2 = 0, 1, 2
Q1 = 3          # pattern only (coarse levels of a quadrilateral multigrid hierarchy): no element kernel accepts it
ELEM_ND = {P1: 3, P2: 6, Q2: 9, Q1: 4}
ELEM_NV = {P1: 3, P2: 3, Q2: 4, Q1: 4}
ELEM_NAME = {P1: "P1", P2: "P2", Q2: "Q2", Q1: "Q1"}


@dataclass
class Mesh:
    """A 2-D mesh with one vector-valued Lagrange space on it.

    x        (nnodes, 2) float64   coordinates of every node of the space
    xdofmap  (ncells, nv) int32    geometry vertices of each cell (node ids)
    dofmap   (ncells, nd) int32    scalar dofs (node ids) of each cell
    """

    etype: int
    x: np.ndarray
    xdofmap: np.ndarray
    dofmap: np.ndarray
    nx: int = 0
    ny: int = 0
    meta: dict = field(default_factory=dict)

    @property
    def nnodes(self) -> int:
        return int(self.x.shape[0])

    @property
    def ncells(self) -> int:
        return int(self.dofmap.shape[0])

    @property
    def ndofs(self) -> int:
        return 2 * self.nnodes

    @property
    def nd(self) -> int:
        return ELEM_ND[self.etype]

    @property
    def nv(self) -> int:
        return ELEM_NV[self.etype]


def young_table() -> np.ndarray:
    """The reference's 200 Young moduli: glibc `srand(6575)`, `rand() % 200`
    (`M.cc:1076-1085`, `F.cc:533-541`, `F.py:213-222`)."""
    libc = ctypes.CDLL("libc.so.6")
    libc.srand(6575)
    a = (1.0e8 - 5.0e6) / 199.0
    tab = np.array([a * (libc.rand() % 200) + 5.0e6 for _ in range(200)], dtype=np.float64)
    # SURVEY.md 8c: E_range[1], E_range[2] with glibc 2.39
    assert abs(tab[1] - 70402010.05025125) < 1e-6 and abs(tab[2] - 26005025.12562814) < 1e-6, \
        "libc rand() does not reproduce the reference's Young-modulus table"
    return tab


def young_per_cell(ncells: int, first_cell: int = 0) -> np.ndarray:
    """E per cell = table[cell_id % 200] (SURVEY.md 8d, config 2)."""
    tab = young_table()
    return tab[(np.arange(first_cell, first_cell + ncells, dtype=np.int64) % 200)].copy()


def _lattice(nx: int, ny: int, sub: int, ly: float, y0: float = 0.0):
    mx, my = sub * nx + 1, sub * ny + 1
    xs = np.linspace(0.0, 1.0, mx)
    ys = y0 + np.linspace(0.0, ly, my)
    X, Y = np.meshgrid(xs, ys, indexing="xy")
    x = np.stack([X.ravel(), Y.ravel()], axis=1).astype(np.float64)
    return x, mx, my


def structured_triangles(nx: int, ny: int | None = None, order: int = 2, ly: float | None = None,
                         y0: float = 0.0) -> Mesh:
    """nx x ny cells, right-diagonal split, P1 (order 1) or P2 (order 2)."""
    ny = nx if ny is None else ny
    ly = (ny / nx) if ly is None else ly
    sub = 1 if order == 1 else 2
    x, mx, _ = _lattice(nx, ny, sub, ly, y0)
    cx, cy = np.meshgrid(np.arange(nx, dtype=np.int64), np.arange(ny, dtype=np.int64), indexing="xy")
    cx, cy = cx.ravel(), cy.ravel()
    node = lambda i, j: i + mx * j
    v0 = node(sub * cx, sub * cy)
    v1 = node(sub * cx + sub, sub * cy)
    v2 = node(sub * cx, sub * cy + sub)
    v3 = node(sub * cx + sub, sub * cy + sub)
    ncell = 2 * nx * ny
    tri = np.empty((ncell, 3), dtype=np.int64)
    tri[0::2] = np.stack([v0, v1, v3], axis=1)
    tri[1::2] = np.stack([v0, v2, v3], axis=1)
    if order == 1:
        dm = tri
        et = P1
    else:
        # midpoint lattice node of two vertex lattice nodes = their average index
        mid = lambda a, b: (a + b) // 2
        dm = np.empty((ncell, 6), dtype=np.int64)
        dm[:, :3] = tri
        dm[:, 3] = mid(tri[:, 1], tri[:, 2])
        dm[:, 4] = mid(tri[:, 0], tri[:, 2])
        dm[:, 5] = mid(tri[:, 0], tri[:, 1])
        et = P2
    return Mesh(et, x, tri.astype(np.int32), dm.astype(np.int32), nx, ny,
                {"kind": "structured-tri-right", "order": order})


def structured_quads_q2(nx: int, ny: int | None = None, ly: float | None = None, y0: float = 0.0) -> Mesh:
    """nx x ny Q2 quads on the (2nx+1) x (2ny+1) lattice; local order ix + 3 iy."""
    ny = nx if ny is None else ny
    ly = (ny / nx) if ly is None else ly
    x, mx, _ = _lattice(nx, ny, 2, ly, y0)
    cx, cy = np.meshgrid(np.arange(nx, dtype=np.int64), np.arange(ny, dtype=np.int64), indexing="xy")
    cx, cy = cx.ravel(), cy.ravel()
    dm = np.empty((nx * ny, 9), dtype=np.int64)
    for iy in range(3):
        for ix in range(3):
            dm[:, ix + 3 * iy] = (2 * cx + ix) + mx * (2 * cy + iy)
    xd = dm[:, [0, 2, 6, 8]]
    return Mesh(Q2, x, xd.astype(np.int32), dm.astype(np.int32), nx, ny, {"kind": "structured-quad"})


def jitter(mesh: Mesh, amp: float = 0.2, seed: int = 1234) -> Mesh:
    """Move interior *vertex* nodes by U(-amp*h, amp*h) (SURVEY.md 8d); edge
    (and Q2 face) nodes are re-placed at the average of their vertices so that
    triangles stay straight-sided and quads bilinear."""
    nx, ny = mesh.nx, mesh.ny
    h = 1.0 / nx
    rng = np.random.default_rng(seed)
    x = mesh.x.copy()
    if mesh.etype == P1:
        mx, my = nx + 1, ny + 1
        I, J = np.meshgrid(np.arange(mx), np.arange(my), indexing="xy")
        interior = ((I > 0) & (I < mx - 1) & (J > 0) & (J < my - 1)).ravel()
        x[interior] += rng.uniform(-amp * h, amp * h, size=(int(interior.sum()), 2))
        return Mesh(mesh.etype, x, mesh.xdofmap, mesh.dofmap, nx, ny, dict(mesh.meta, jitter=amp))
    mx, my = 2 * nx + 1, 2 * ny + 1
    I, J = np.meshgrid(np.arange(mx), np.arange(my), indexing="xy")
    isv = ((I % 2 == 0) & (J % 2 == 0))
    interior = (isv & (I > 0) & (I < mx - 1) & (J > 0) & (J < my - 1)).ravel()
    x[interior] += rng.uniform(-amp * h, amp * h, size=(int(interior.sum()), 2))
    dm = mesh.dofmap.astype(np.int64)
    if mesh.etype == P2:
        for loc, (p, q) in zip((3, 4, 5), ((1, 2), (0, 2), (0, 1))):
            x[dm[:, loc]] = 0.5 * (x[dm[:, p]] + x[dm[:, q]])
    else:
        for loc, vs in ((1, (0, 2)), (3, (0, 6)), (5, (2, 8)), (7, (6, 8)), (4, (0, 2, 6, 8))):
            x[dm[:, loc]] = np.mean([x[dm[:, v]] for v in vs], axis=0)
    return Mesh(mesh.etype, x, mesh.xdofmap, mesh.dofmap, nx, ny, dict(mesh.meta, jitter=amp))


def dirichlet_markers(mesh: Mesh, eps: float = 1e-10, traction: bool = True):
    """Per-dof marker (uint8) and imposed values: x = 0 clamped, x = 1:
    ux = +0.01 (traction) / -0.01, uy = 0 (`F.cc:627-664`, `M.cc:1403-1415`)."""
    bc = np.zeros(mesh.ndofs, dtype=np.uint8)
    g = np.zeros(mesh.ndofs, dtype=np.float64)
    left = np.nonzero(np.abs(mesh.x[:, 0]) < eps)[0]
    right = np.nonzero(np.abs(mesh.x[:, 0] - 1.0) < eps)[0]
    for nodes in (left, right):
        bc[2 * nodes] = 1
        bc[2 * nodes + 1] = 1
    g[2 * right] = 0.01 if traction else -0.01
    return bc, g


def body_force(mesh: Mesh) -> np.ndarray:
    """Nodal load f = (-1e5 (x-.5)^3 (1600 (y-.5)^2 - 500), 0), interpolated at
    the nodes (`M.cc:1431-1447`, `F.cc:564-585`).  Returns (nnodes, 2)."""
    r = mesh.x[:, 0] - 0.5
    y = mesh.x[:, 1] - 0.5
    xf = 100000.0 * (-r * r * r)
    f = np.zeros((mesh.nnodes, 2))
    f[:, 0] = (1600.0 * y * y - 500.0) * xf
    return f


def damage_band(mesh: Mesh) -> np.ndarray:
    """Synthetic nodal damage field in [0,1) for the reassembly workload
    (SURVEY.md 8d, config 5): max(0, 1 - |y - 0.5 - 0.1 sin 6x| / 0.05),
    capped below 1."""
    x, y = mesh.x[:, 0], mesh.x[:, 1]
    d = np.maximum(0.0, 1.0 - np.abs(y - 0.5 - 0.1 * np.sin(6.0 * x)) / 0.05)
    return np.minimum(d, 0.95)


def _remap_checked(remap: np.ndarray, ids: np.ndarray, path: str) -> np.ndarray:
    if ids.size and (ids.min() < 0 or ids.max() >= len(remap) or (remap[ids] < 0).any()):
        raise ValueError(f"{path}: an element refers to a node id that $Nodes does not define")
    return remap[ids]


def read_gmsh22(path: str) -> Mesh:
    """Gmsh 2.2 ASCII reader for triangulations (role of `Mesh(mesh_file, 1, 0, true)`, M.cc:1017-1020,
    and of the gmsh -> XDMF conversion + `read_mesh` / `read_meshtags`, gmsh_to_xdmf_neper_dam.py:1-16,
    F.cc:153-193): 2-node lines (type 1) and 3-node triangles (type 2) with their first (physical)
    tag.  Returns a P1 Mesh; meta holds `cell_tags` (ncells), `facets` (nfacets, 2) and `facet_tags`.
    Orientation is left as in the file: the element kernels use |det J| (SURVEY.md B6)."""
    with open(path) as f:
        tok = f.read().split("\n")
    sec = {}
    i = 0
    while i < len(tok):
        ln = tok[i].strip()
        if ln.startswith("$") and not ln.startswith("$End"):
            j = i + 1
            while j < len(tok) and tok[j].strip() != "$End" + ln[1:]:
                j += 1
            sec[ln[1:]] = tok[i + 1:j]
            i = j
        i += 1
    if "MeshFormat" in sec and not sec["MeshFormat"][0].split()[0].startswith("2"):
        raise ValueError(f"{path}: only the Gmsh 2.x ASCII format is supported")
    nn = int(sec["Nodes"][0])
    rows = np.array([r.split() for r in sec["Nodes"][1:1 + nn]], dtype=np.float64)
    ids = rows[:, 0].astype(np.int64)
    remap = np.full(int(ids.max()) + 1, -1, dtype=np.int64)
    remap[ids] = np.arange(nn)
    x = np.ascontiguousarray(rows[:, 1:3])
    tris, ttag, lines, ltag = [], [], [], []
    ne = int(sec["Elements"][0])
    for r in sec["Elements"][1:1 + ne]:
        p = [int(t) for t in r.split()]
        et, ntags = p[1], p[2]
        tag = p[3] if ntags > 0 else 0
        nodes = p[3 + ntags:]
        if et == 2:
            tris.append(nodes), ttag.append(tag)
        elif et == 1:
            lines.append(nodes), ltag.append(tag)
    if not tris:
        raise ValueError(f"{path}: no triangles")
    tri_ids = np.array(tris, dtype=np.int64)
    if tri_ids.min() < 0 or tri_ids.max() >= len(remap) or (remap[tri_ids] < 0).any():
        raise ValueError(f"{path}: an element refers to a node id that $Nodes does not define")
    tri = remap[tri_ids].astype(np.int32)
    meta = {"kind": "gmsh22", "cell_tags": np.array(ttag, dtype=np.int32),
            "facets": _remap_checked(remap, np.array(lines, dtype=np.int64).reshape(-1, 2), path).astype(np.int32),
            "facet_tags": np.array(ltag, dtype=np.int32)}
    return Mesh(P1, x, tri, tri.copy(), 0, 0, meta)


def refine_uniform(mesh: Mesh, levels: int = 1) -> Mesh:
    """Uniform refinement of a P1 triangulation, `levels` times: the role of `pmesh->UniformRefinement(0)` in the
    `-r` loop (M.cc:1037-1038) and of `plaza::refine` + `transfer_cell_meshtag` / `transfer_facet_meshtag`
    (F.cc:166-185).  Every triangle (v0, v1, v2) becomes (v0, m01, m20), (m01, v1, m12), (m20, m12, v2) and
    (m12, m20, m01) with m_ab the midpoint of edge (a, b): children keep the orientation of the parent, child c of
    cell k is cell 4 k + c, the new vertices follow the old ones in the order of the sorted unique (min, max) edges.
    Cell tags are inherited, every tagged facet becomes its two halves with the same tag (what the tag transfer of
    both libraries does).  The vertex / cell NUMBERING the two libraries produce is theirs (un-vendored: unpinned);
    the refined geometry, tags and everything computed from them do not depend on it."""
    if mesh.etype != P1:
        raise ValueError("refine_uniform: P1 triangulations only (refine before building the P2 space)")
    for _ in range(int(levels)):
        tri = mesh.xdofmap.astype(np.int64)
        nv = mesh.nnodes
        ea = np.stack([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]], axis=1).reshape(-1, 2)   # (3 ncells, 2)
        key = np.minimum(ea[:, 0], ea[:, 1]) * nv + np.maximum(ea[:, 0], ea[:, 1])
        ukey, inv = np.unique(key, return_inverse=True)
        mid = (nv + inv).reshape(-1, 3)                                     # m01, m12, m20 of every cell
        x = np.vstack([mesh.x, 0.5 * (mesh.x[ukey // nv] + mesh.x[ukey % nv])])
        v0, v1, v2 = tri[:, 0], tri[:, 1], tri[:, 2]
        m01, m12, m20 = mid[:, 0], mid[:, 1], mid[:, 2]
        child = np.stack([np.stack([v0, m01, m20], 1), np.stack([m01, v1, m12], 1), np.stack([m20, m12, v2], 1),
                          np.stack([m12, m20, m01], 1)], axis=1).reshape(-1, 3).astype(np.int32)
        meta = dict(mesh.meta)
        if "cell_tags" in meta:
            meta["cell_tags"] = np.repeat(np.asarray(meta["cell_tags"]), 4)
        if "facets" in meta and len(meta["facets"]):
            f = np.asarray(meta["facets"], dtype=np.int64)
            fk = np.minimum(f[:, 0], f[:, 1]) * nv + np.maximum(f[:, 0], f[:, 1])
            pos = np.searchsorted(ukey, fk)
            if np.any(pos >= len(ukey)) or np.any(ukey[np.minimum(pos, len(ukey) - 1)] != fk):
                raise ValueError("refine_uniform: a tagged facet is not an edge of the triangulation")
            fm_ = nv + pos
            meta["facets"] = np.stack([np.stack([f[:, 0], fm_], 1), np.stack([fm_, f[:, 1]], 1)], axis=1).reshape(-1, 2).astype(np.int32)
            meta["facet_tags"] = np.repeat(np.asarray(meta["facet_tags"]), 2)
        meta["refined"] = int(meta.get("refined", 0)) + 1
        mesh = Mesh(P1, np.ascontiguousarray(x), child, child.copy(), 0, 0, meta)
    return mesh


@dataclass
class MeshHierarchy:
    """Nested meshes for geometric multigrid, coarsest first: meshes[-1] is the finest (the mesh being solved on),
    every other mesh is P1 (triangles) or Q1 (quadrilaterals).  maps[k] is the transfer from meshes[k + 1] to
    meshes[k], one row of coarse node ids per fine node, both components alike:

    * (nf, 2) int32 pairs (a, b): a == b for a node that coincides with coarse node a (weight 1), otherwise the
      midpoint of the coarse edge (a, b) (weight 1/2 on each);
    * (nf, 4) int32 rows: (a, a, a, a) a coincident node, (a, b, a, b) the midpoint of the coarse edge (a, b),
      (v00, v10, v01, v11) the centre of a coarse quad; each distinct entry weighs 1 / (number of distinct entries).

    Entry k and its partner (width - 1 - k) name the coarse pairs a fine node stands for (its node, its edge, the two
    diagonals of its quad).  In both widths column 0 equals column 1 for a coincident node only.  Indexing and len()
    go over the meshes."""
    meshes: list
    maps: list

    def __len__(self) -> int:
        return len(self.meshes)

    def __getitem__(self, k):
        return self.meshes[k]

    def markers(self, fine_marker) -> list:
        """Per-dof Dirichlet markers (uint8) of every mesh, coarsest first, from the finest mesh's marker: a coarse
        dof is constrained when the fine dof of its coincident node is."""
        out = [np.asarray(fine_marker, dtype=np.uint8).reshape(-1)]
        if out[0].size != self.meshes[-1].ndofs:
            raise ValueError(f"the marker has {out[0].size} entries, the finest mesh {self.meshes[-1].ndofs} dofs")
        for k in range(len(self.meshes) - 2, -1, -1):
            co = coincident_nodes(self.maps[k], self.meshes[k].nnodes)
            m = out[0].reshape(-1, 2)[co].reshape(-1)
            out.insert(0, np.ascontiguousarray(m))
        return out


def coincident_nodes(tmap: np.ndarray, ncoarse: int) -> np.ndarray:
    """Fine node that coincides with each coarse node of a transfer map (raises when one has none)."""
    tmap = np.asarray(tmap)
    sel = np.nonzero(tmap[:, 0] == tmap[:, 1])[0]
    co = np.full(ncoarse, -1, dtype=np.int64)
    co[tmap[sel, 0]] = sel
    if (co < 0).any():
        raise ValueError(f"transfer map: {int((co < 0).sum())} coarse nodes have no coincident fine node")
    return co


def _lattice_map(mxf: int, myf: int) -> np.ndarray:
    """(a, b) of the (mxf x myf)-node lattice halved: node (i, j) -> coarse (i // 2, j // 2) and ((i + 1) // 2,
    (j + 1) // 2); equal for even (i, j), the two ends of the horizontal, vertical or right-diagonal coarse edge
    through the node otherwise."""
    mxc = (mxf - 1) // 2 + 1
    i, j = np.meshgrid(np.arange(mxf, dtype=np.int64), np.arange(myf, dtype=np.int64), indexing="xy")
    i, j = i.ravel(), j.ravel()
    a = (i // 2) + mxc * (j // 2)
    b = ((i + 1) // 2) + mxc * ((j + 1) // 2)
    return np.ascontiguousarray(np.stack([a, b], axis=1).astype(np.int32))


def lattice_hierarchy(fine: Mesh) -> MeshHierarchy:
    """Hierarchy of a `structured_triangles` mesh (P1 or P2, any nx x ny, jittered or not): a P2 mesh is coarsened
    to P1 on the same vertices (its nodes are those of the P1 lattice of 2nx x 2ny cells), then the P1 lattice is
    halved while both cell counts are even.  Coarse nodes take the coordinates of their coincident fine nodes."""
    if fine.meta.get("kind") != "structured-tri-right" or fine.etype not in (P1, P2):
        raise ValueError("lattice_hierarchy: needs a P1 / P2 mesh of structured_triangles")
    nx, ny = fine.nx, fine.ny
    meshes, maps = [fine], []
    sub = 2 if fine.etype == P2 else 1
    mfx, mfy = sub * nx + 1, sub * ny + 1      # fine node lattice
    cur = fine
    while True:
        if fine.etype == P2 and cur is fine:
            cx, cy = nx, ny
        elif cur.nx % 2 == 0 and cur.ny % 2 == 0:
            cx, cy = cur.nx // 2, cur.ny // 2
        else:
            break
        tmap = _lattice_map(mfx, mfy)
        c = structured_triangles(cx, cy, order=1)
        co = coincident_nodes(tmap, c.nnodes)
        c = Mesh(P1, np.ascontiguousarray(cur.x[co]), c.xdofmap, c.dofmap, cx, cy, dict(c.meta))
        meshes.insert(0, c)
        maps.insert(0, tmap)
        cur, mfx, mfy = c, cx + 1, cy + 1
    return MeshHierarchy(meshes, maps)


def _quad_lattice_map(mxf: int, myf: int) -> np.ndarray:
    """Width-4 map of the (mxf x myf)-node lattice halved: node (i, j) -> the coarse lattice nodes (i // 2 or
    (i + 1) // 2, j // 2 or (j + 1) // 2): (a, a, a, a) for even (i, j), (a, b, a, b) for the midpoint of a horizontal
    or vertical coarse edge, (v00, v10, v01, v11) for odd (i, j), the centre of a coarse quad."""
    mxc = (mxf - 1) // 2 + 1
    i, j = np.meshgrid(np.arange(mxf, dtype=np.int64), np.arange(myf, dtype=np.int64), indexing="xy")
    i, j = i.ravel(), j.ravel()
    c = lambda ii, jj: ii + mxc * jj
    i0, i1, j0, j1 = i // 2, (i + 1) // 2, j // 2, (j + 1) // 2
    m = np.stack([c(i0, j0), c(i1, j0), c(i0, j1), c(i1, j1)], axis=1)
    vert = (i % 2 == 0) & (j % 2 == 1)          # (a, a, b, b) -> (a, b, a, b)
    m[vert] = m[vert][:, [0, 2, 0, 2]]
    return np.ascontiguousarray(m.astype(np.int32))


def _quads_q1(nx: int, ny: int, x: np.ndarray) -> Mesh:
    """Q1 mesh of nx x ny cells on the (nx + 1) x (ny + 1) vertex lattice, cells in the order of structured_quads_q2
    (x fastest), local order (v00, v10, v01, v11)."""
    mx = nx + 1
    cx, cy = np.meshgrid(np.arange(nx, dtype=np.int64), np.arange(ny, dtype=np.int64), indexing="xy")
    v00 = (cx + mx * cy).ravel()
    dm = np.stack([v00, v00 + 1, v00 + mx, v00 + mx + 1], axis=1).astype(np.int32)
    return Mesh(Q1, np.ascontiguousarray(x), dm, dm.copy(), nx, ny, {"kind": "structured-quad", "order": 1})


def quad_lattice_hierarchy(fine: Mesh) -> MeshHierarchy:
    """Hierarchy of a `structured_quads_q2` mesh (any nx x ny, jittered or not): Q2 -> Q1 on the same vertices and the
    same cells (cell k of the Q1 mesh is cell k of the Q2 mesh; the Q2 node lattice maps like a halved lattice), then
    the Q1 lattice halved while both cell counts are even.  Width-4 maps; coarse nodes take the coordinates of their
    coincident fine nodes."""
    if fine.meta.get("kind") != "structured-quad" or fine.etype != Q2:
        raise ValueError("quad_lattice_hierarchy: needs a Q2 mesh of structured_quads_q2")
    meshes, maps = [fine], []
    cur, mfx, mfy = fine, 2 * fine.nx + 1, 2 * fine.ny + 1
    while True:
        if cur is fine:
            cx, cy = fine.nx, fine.ny
        elif cur.nx % 2 == 0 and cur.ny % 2 == 0:
            cx, cy = cur.nx // 2, cur.ny // 2
        else:
            break
        tmap = _quad_lattice_map(mfx, mfy)
        co = coincident_nodes(tmap, (cx + 1) * (cy + 1))
        c = _quads_q1(cx, cy, cur.x[co])
        meshes.insert(0, c)
        maps.insert(0, tmap)
        cur, mfx, mfy = c, cx + 1, cy + 1
    return MeshHierarchy(meshes, maps)


def refine_uniform_hierarchy(coarse: Mesh, levels: int) -> MeshHierarchy:
    """refine_uniform(coarse, 1) `levels` times, keeping every mesh and the transfer maps: the first nv nodes of a
    refined mesh are the coarse ones, the midpoints follow in sorted-edge order (refine_uniform's numbering), so
    the finest mesh is refine_uniform(coarse, levels) bit for bit."""
    meshes, maps = [coarse], []
    for _ in range(int(levels)):
        m = meshes[-1]
        tri = m.xdofmap.astype(np.int64)
        nv = m.nnodes
        ea = np.stack([tri[:, [0, 1]], tri[:, [1, 2]], tri[:, [2, 0]]], axis=1).reshape(-1, 2)
        ukey = np.unique(np.minimum(ea[:, 0], ea[:, 1]) * nv + np.maximum(ea[:, 0], ea[:, 1]))
        a = np.concatenate([np.arange(nv, dtype=np.int64), ukey // nv])
        b = np.concatenate([np.arange(nv, dtype=np.int64), ukey % nv])
        meshes.append(refine_uniform(m, 1))
        maps.append(np.ascontiguousarray(np.stack([a, b], axis=1).astype(np.int32)))
    return MeshHierarchy(meshes, maps)


def young_from_tags(cell_tags: np.ndarray) -> np.ndarray:
    """E per cell from the physical tag: E_range[tag % 200] (M.cc:1580-1583, F.py:221)."""
    return young_table()[np.asarray(cell_tags, dtype=np.int64) % 200].copy()


def damage_seed(mesh: Mesh, facet_tags, max_dam: float = 1.0) -> np.ndarray:
    """Initial nodal damage: MAX_DAM on the nodes of the facets carrying one of `facet_tags`
    (M.cc:1160-1205,1251-1255; F.py:113-127; the square mesh uses tag 4, M.cc:1164-1167)."""
    d = np.zeros(mesh.nnodes)
    sel = np.isin(mesh.meta["facet_tags"], np.asarray(facet_tags))
    d[np.unique(mesh.meta["facets"][sel])] = max_dam
    return d


# ---- XDMF (the FEniCSx driver's mesh file) ---------------------------------------------------------------------------
def _xdmf_item(node, base: str, dtype):
    """One <DataItem>: Format="XML" (numbers inline) and Format="Binary" (raw side file) are read here; Format="HDF"
    (what dolfinx writes by default, "file.h5:/path") needs h5py, which this image does not ship: it is used when
    importable, else the error says so."""
    import os
    item = node if node.tag == "DataItem" else node.find("DataItem")
    if item is None:
        raise ValueError("read_xdmf: element without a DataItem")
    dims = [int(t) for t in item.get("Dimensions", "").split()]
    fmt = item.get("Format", "XML").upper()
    if fmt == "XML":
        a = np.array((item.text or "").split(), dtype=dtype)
    elif fmt == "HDF":
        try:
            import h5py
        except ImportError as e:
            raise ValueError("read_xdmf: this file keeps its arrays in HDF5 and h5py is not installed; convert it with "
                             "write_xdmf (inline XML data) or read the Gmsh 2.2 source with read_gmsh22") from e
        fname, path = (item.text or "").strip().split(":", 1)
        with h5py.File(os.path.join(base, fname), "r") as h:
            a = np.asarray(h[path], dtype=dtype)
    elif fmt == "BINARY":
        # raw side file (XDMF "Binary" format): NumberType / Precision / Endian / Seek attributes
        kind = {"FLOAT": "f", "INT": "i", "UINT": "u", "CHAR": "i", "UCHAR": "u"}.get(item.get("NumberType", "Float").upper())
        if kind is None:
            raise ValueError(f"read_xdmf: NumberType={item.get('NumberType')!r} is not supported")
        prec = int(item.get("Precision", "4"))
        order = {"BIG": ">", "LITTLE": "<"}.get(item.get("Endian", "Native").upper(), "=")
        count = int(np.prod(dims)) if dims else -1
        a = np.fromfile(os.path.join(base, (item.text or "").strip()), dtype=np.dtype(f"{order}{kind}{prec}"), count=count,
                        offset=int(item.get("Seek", "0"))).astype(dtype)
    else:
        raise ValueError(f"read_xdmf: DataItem Format={fmt!r} is not supported")
    return a.reshape(dims) if dims else a


def read_xdmf(path: str, name: str | None = None) -> Mesh:
    """XDMF reader for the layout the FEniCSx driver reads (F.cc:155-163: `read_mesh(tria, ..., name)` +
    `read_meshtags(mesh, name + "_cells")` + `read_meshtags(mesh, name + "_facets")`, written by
    gmsh_to_xdmf_neper_dam.py:1-16): grid `name` with a Triangle topology and an XY / XYZ geometry, grid
    `name_cells` = cell topology + one cell-centred attribute, grid `name_facets` = 2-node PolyLine topology + one
    attribute.  `name` defaults to the first grid of the file.  Returns the same Mesh (P1, meta cell_tags / facets /
    facet_tags) as read_gmsh22.  Mesh-tag grids list their entities by vertex numbers: cell tags are matched to the
    mesh cells by their sorted vertex triple, as `read_meshtags` does."""
    import os
    import xml.etree.ElementTree as ET
    root = ET.parse(path).getroot()
    base = os.path.dirname(os.path.abspath(path))
    grids = {g.get("Name"): g for g in root.iter("Grid")}
    if not grids:
        raise ValueError(f"{path}: no Grid")
    if name is None:
        name = next(iter(grids))
    if name not in grids:
        raise ValueError(f"{path}: no grid named {name!r} (has {sorted(grids)})")
    g = grids[name]
    topo, geom = g.find("Topology"), g.find("Geometry")
    if topo is None or geom is None:
        raise ValueError(f"{path}: grid {name!r} needs a Topology and a Geometry")
    if topo.get("TopologyType", "").lower() != "triangle":
        raise ValueError(f"{path}: only Triangle topologies are supported, got {topo.get('TopologyType')!r}")
    tri = _xdmf_item(topo, base, np.int64).reshape(-1, 3)
    x = _xdmf_item(geom, base, np.float64)
    x = np.ascontiguousarray(x.reshape(-1, 3 if geom.get("GeometryType", "XY").upper() == "XYZ" else 2)[:, :2])
    if tri.size and (tri.min() < 0 or tri.max() >= len(x)):
        raise ValueError(f"{path}: a cell refers to a vertex outside the geometry")
    meta = {"kind": "xdmf", "cell_tags": np.zeros(len(tri), dtype=np.int32), "facets": np.zeros((0, 2), dtype=np.int32),
            "facet_tags": np.zeros(0, dtype=np.int32)}

    def tags(gname, npe):
        tg = grids.get(gname)
        if tg is None:
            return None
        ent = _xdmf_item(tg.find("Topology"), base, np.int64).reshape(-1, npe)
        att = tg.find("Attribute")
        val = _xdmf_item(att, base, np.float64).reshape(-1).astype(np.int32)
        if len(val) != len(ent):
            raise ValueError(f"{path}: grid {gname!r} has {len(ent)} entities and {len(val)} values")
        return ent, val

    ct = tags(name + "_cells", 3)
    if ct is not None:
        nv = len(x)
        key = lambda t: (np.sort(t, axis=1) * np.array([nv * nv, nv, 1], dtype=np.int64)).sum(axis=1)
        kc = key(tri)
        order = np.argsort(kc)
        pos = np.searchsorted(kc[order], key(ct[0]))
        if np.any(pos >= len(kc)) or np.any(kc[order][np.minimum(pos, len(kc) - 1)] != key(ct[0])):
            raise ValueError(f"{path}: a tagged cell is not a cell of the mesh")
        meta["cell_tags"][order[pos]] = ct[1]
    ft = tags(name + "_facets", 2)
    if ft is not None:
        meta["facets"], meta["facet_tags"] = ft[0].astype(np.int32), ft[1]
    tri = tri.astype(np.int32)
    return Mesh(P1, x, tri, tri.copy(), 0, 0, meta)


def write_xdmf(path: str, mesh: Mesh, name: str = "mesh") -> None:
    """Writes a P1 triangulation with its cell and facet tags in the layout read_xdmf / the FEniCSx driver reads, arrays
    inline (Format="XML", repr-exact floats): the role of gmsh_to_xdmf_neper_dam.py without the HDF5 side file."""
    tri, x = np.asarray(mesh.xdofmap), np.asarray(mesh.x)

    def item(a, fmtf):
        a = np.asarray(a)
        dims = " ".join(str(d) for d in a.shape)
        num = "Float" if a.dtype.kind == "f" else "Int"
        body = "\n".join(" ".join(fmtf(v) for v in row) for row in a.reshape(len(a), -1))
        return f'<DataItem Dimensions="{dims}" NumberType="{num}" Precision="8" Format="XML">\n{body}\n</DataItem>'

    fi, ff = (lambda v: str(int(v))), (lambda v: repr(float(v)))
    geo = f'<Geometry GeometryType="XY">{item(x, ff)}</Geometry>'
    out = ['<?xml version="1.0"?>', '<Xdmf Version="3.0"><Domain>',
           f'<Grid Name="{name}" GridType="Uniform"><Topology TopologyType="Triangle" NumberOfElements="{len(tri)}" '
           f'NodesPerElement="3">{item(tri, fi)}</Topology>{geo}</Grid>']
    ctag = mesh.meta.get("cell_tags")
    if ctag is not None:
        out.append(f'<Grid Name="{name}_cells" GridType="Uniform"><Topology TopologyType="Triangle" '
                   f'NumberOfElements="{len(tri)}" NodesPerElement="3">{item(tri, fi)}</Topology>{geo}'
                   f'<Attribute Name="{name}_cells" AttributeType="Scalar" Center="Cell">'
                   f'{item(np.asarray(ctag).reshape(-1, 1), fi)}</Attribute></Grid>')
    fac = mesh.meta.get("facets")
    if fac is not None and len(fac):
        out.append(f'<Grid Name="{name}_facets" GridType="Uniform"><Topology TopologyType="PolyLine" '
                   f'NumberOfElements="{len(fac)}" NodesPerElement="2">{item(fac, fi)}</Topology>{geo}'
                   f'<Attribute Name="{name}_facets" AttributeType="Scalar" Center="Cell">'
                   f'{item(np.asarray(mesh.meta["facet_tags"]).reshape(-1, 1), fi)}</Attribute></Grid>')
    out.append("</Domain></Xdmf>")
    with open(path, "w") as f:
        f.write("\n".join(out) + "\n")
