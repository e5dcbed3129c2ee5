"""bench.py --dump-outputs: the arrays the timed step computed, sampled reproducibly, and equal to the oracle's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sample_output_is_reproducible_and_capped():
    import torch
    v = torch.arange(1000, dtype=torch.float32)
    whole = bench.sample_output(v, 1000)
    assert whole.dtype == np.float64 and np.array_equal(whole, np.arange(1000.0))
    a, b = bench.sample_output(v, 100), bench.sample_output(v, 100)
    assert a.dtype == np.float64 and 0 < a.size <= 100 and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and np.isin(a, whole).all()     # sorted distinct entries of v
    assert sum(bench.DUMP_ENTRIES.values()) * 8 <= 64 << 20


@pytest.mark.gpu
def test_dump_outputs_match_oracle(tmp_path):
    """A small run of the flagship step writes the constrained matrix and the 25-iteration PCG iterate of its last
    timed step; both equal the oracle's on the same mesh, and --steps sets the number of timed steps."""
    from oracle import oracle
    from femb200 import dist
    n, steps = 48, 2
    out = tmp_path / "dump"
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--size", str(n), "--steps", str(steps),
                          "--warmup", "1", "--skip-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-4000:]
    line = json.loads([s for s in res.stdout.splitlines() if s.startswith("{")][-1])
    assert line["steps"] == steps and line["e2e"]["steps"] == steps and line["parity"]["ok"]
    assert sorted(os.listdir(out)) == ["cg_x.npy", "e2e_du.npy", "matrix_values.npy"]
    p = dist.strip_partition(n, n, 2, 0, 1)                  # the mesh bench.py generates on the device
    m = p.mesh
    rowptr, colidx = oracle.build_pattern(m.nnodes, m.dofmap)
    K = oracle.assemble_matrix(m.etype, m.x, m.xdofmap, m.dofmap, p.E, 0.3, rowptr, colidx, bc=p.bc)
    x, _, _, _ = oracle.pcg(rowptr, colidx, K, np.where(p.bc != 0, p.g, 1.0), rtol=0.0, atol=0.0, maxit=25, jacobi=True)
    vals, xs, du = (np.load(out / f) for f in ("matrix_values.npy", "cg_x.npy", "e2e_du.npy"))
    assert vals.dtype == xs.dtype == du.dtype == np.float64
    assert vals.shape == K.shape and np.linalg.norm(vals - K) <= 1e-12 * np.linalg.norm(K)
    assert xs.shape == x.shape and np.linalg.norm(xs - x) <= 1e-10 * np.linalg.norm(x)
    assert du.shape == (m.ndofs,) and np.isfinite(du).all() and np.abs(du).max() > 0
