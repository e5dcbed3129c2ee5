#!/usr/bin/env python
"""bench.py -- the hot path of the mechanic2d elasticity examples on N B200s.

Workload (BASELINE.json configs[3], the configuration the north-star target is quoted on): P2 triangles on
the structured n x n mesh split by the right diagonal, n = 5792 -> 67 094 528 elements, 268 424 450 dofs,
6 173 067 268 CSR non-zeros; jittered vertices, the reference's 200-value Young-modulus table, nu = 0.3,
Dirichlet x = 0 / x = 1.  The SAME global mesh at every N: `--gpus N` cuts it into N strips of cell rows
(strong scaling); N = 1 holds all of it on one GPU (49 GB of values).

One timed STEP = one pass of the hot path = one Newton linearisation:
    full tangent assembly (element integration + write-once gather into the CSR + Dirichlet rows/columns,
    the setJ lambda F.cc:847-862)  +  `--cg-iters` (25) Jacobi-PCG iterations on it (operator apply with
    the ghost update of the search direction and the all-reduce of the dot products: CGSolver::Mult
    M.cc:1502-1528 / KSP cg F.cc:718-722).
`value` = dofs / step time (GDOF/s), whole job.  The same run times the assembly alone, the SpMV alone and
the PCG iterations alone (sub-keys "assembly", "cg", each with its own roofline), checks parity in-run at
every N (golden norms of the oracle, rigid-body modes through the distributed operator, recurrence vs true
residual of the PCG), and at N = 1 also reports BASELINE configs[2] (Q2 matrix-free), configs[4] (damaged
reassembly at 10 / 50 / 100 % damage), the FP64 roofline of the element kernels and the CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--size n] [--dump-outputs DIR]

`--dump-outputs DIR` writes, after the timed steps, what the last of them computed as float64 .npy files: matrix_values
(the constrained CSR values), cg_x (the PCG iterate, owned dofs) and e2e_du (the Newton increment of the end-to-end leg,
owned dofs); an output longer than DUMP_ENTRIES allows is a fixed, seeded sample of it.  The inputs are generated from
fixed seeds, so two builds of the project can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "fem-libraries_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "assembly GDOF/s & CG SpMV GB/s (% HBM roofline): P2 elasticity Newton linearisation (CSR assembly + PCG)"
UNIT = "GDOF/s"
GOLDEN = os.path.join(ROOT, "tests", "golden", "config_norms.json")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------
# algorithmic bytes (DESIGN.md section 4, SURVEY.md 8d)
# ---------------------------------------------------------------------------
def assembly_bytes(nnz: int, ncells: int, nnodes: int) -> int:
    """write nnz values once + read connectivity (6 x int32), E (8 B) per cell and
    coordinates (16 B) per node: ~808 B per P2 element."""
    return 8 * nnz + ncells * (6 * 4 + 8) + nnodes * 16


def spmv_bytes(nnz_blocks: int, nnodes: int) -> int:
    """block pattern: 32 B of values + 4 B column index per 2x2 block; per node 8 B of
    row pointer, 16 B of x read, 16 B of y written."""
    return 36 * nnz_blocks + nnodes * (8 + 16 + 16)


def cg_iter_bytes(nnz_blocks: int, nnodes: int) -> int:
    """SpMV + update_r (read Ad, r, dinv; write r) + update_xdir (read r, dinv, d, x; write d, x: the x update rides
    with the direction update), 16 B per node per vector pass."""
    return spmv_bytes(nnz_blocks, nnodes) + 10 * 16 * nnodes


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])), mx.append(float(r[1])), pw.append(float(r[2]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if r[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def host_threads() -> int:
    """Cores this process may use: the affinity mask, NOT OMP_NUM_THREADS (torchrun exports OMP_NUM_THREADS=1
    to its workers, which made the round-1 reference arm single-threaded at N > 1)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


# ---------------------------------------------------------------------------
# reference arm: the CPU restatement of the reference (oracle) on the host cores
# ---------------------------------------------------------------------------
def cpu_reference(n_sample: int, steps: int, warmup: int, cg_iters: int):
    """The same step on the host: oracle assembly (domain-decomposed over the threads, as the reference's MPI
    ranks) + `cg_iters` Jacobi-PCG iterations (OpenMP SpMV, dots, axpys), all-core and one-thread figures, median
    and best of `steps` repetitions (BASELINE.md section 3)."""
    from oracle import oracle
    from femb200 import dist
    nt_all = host_threads()
    part = dist.strip_partition(n_sample, n_sample, 2, 0, 1)
    m, E, bc, g = part.mesh, part.E, part.bc, part.g
    rowptr, colidx = oracle.build_pattern(m.nnodes, m.dofmap)
    vals = np.empty(int(rowptr[-1]))
    b = np.where(bc != 0, g, 1.0)
    out = {}
    for nt in sorted({1, nt_all}, reverse=True):
        k = steps if nt == nt_all else max(1, min(steps, 2))     # the one-thread figure is context: keep it short
        w = warmup if nt == nt_all else 0
        ta, tc = [], []
        for i in range(w + k):
            t0 = time.perf_counter()
            oracle.assemble_matrix(m.etype, m.x, m.xdofmap, m.dofmap, E, 0.3, rowptr, colidx, bc=bc, nthreads=nt, values=vals)
            t1 = time.perf_counter()
            oracle.pcg(rowptr, colidx, vals, b, rtol=0.0, atol=0.0, maxit=cg_iters, jacobi=True, nthreads=nt)
            t2 = time.perf_counter()
            if i >= w:
                ta.append(t1 - t0), tc.append(t2 - t1)
        ts = np.array(ta) + np.array(tc)
        v = np.random.default_rng(0).standard_normal(m.ndofs)
        y = np.empty(m.ndofs)
        oracle.spmv(rowptr, colidx, vals, v, nthreads=nt, y=y)
        t0 = time.perf_counter()
        reps = 5 if nt == nt_all else 2
        for _ in range(reps):
            oracle.spmv(rowptr, colidx, vals, v, nthreads=nt, y=y)
        t_spmv = (time.perf_counter() - t0) / reps
        out[nt] = {"threads": nt, "step_s_median": float(np.median(ts)), "step_s_best": float(ts.min()),
                   "step_gdofs": m.ndofs / float(np.median(ts)) / 1e9, "assembly_s": float(np.median(ta)),
                   "assembly_gdofs": m.ndofs / float(np.median(ta)) / 1e9, "cg_iter_s": float(np.median(tc)) / (cg_iters + 1),
                   "spmv_s": t_spmv, "spmv_gbs": (12 * int(rowptr[-1]) + 24 * m.ndofs + 8) / t_spmv / 1e9,
                   "spmv_gdofs": m.ndofs / t_spmv / 1e9, "repetitions": k}
    best = out[nt_all]
    best["one_thread"] = out.get(1) if nt_all != 1 else None
    best["sample"] = (f"P2 n={n_sample} ({m.ncells} elements, {m.ndofs} dofs), same mesh family / materials / BCs as the "
                      f"GPU arm; step = assembly + {cg_iters} Jacobi-PCG iterations; oracle/fem_oracle.c -O3 OpenMP, "
                      f"{nt_all} threads (os.sched_getaffinity), median of {best['repetitions']}")
    return best


def reference_element_kernel_rate(n_elems: int = 400000):
    """The reference's OWN element code (damIntegrator::AssembleElementGrad, M.cc:639-916, compiled in place
    into oracle/_ref by oracle/ref_shim/build_ref.sh), one host thread, P1 triangles, d = 0: elements per
    second, next to the 5.5 M elements/s/core the reference publishes (curve_time.txt col 84).  None when
    oracle/_ref does not exist on this box."""
    import ctypes as C
    so = os.path.join(ROOT, "oracle", "_ref", "libref_B.so")
    if not os.path.exists(so):
        return None
    L = C.CDLL(so)
    if not hasattr(L, "ref_element_grad_batch"):
        return None
    dp = C.POINTER(C.c_double)
    L.ref_element_grad_batch.argtypes = [C.c_long, dp, dp, dp, dp, dp]
    rng = np.random.default_rng(0)
    xv = np.tile(np.array([0.0, 0.0, 1.0, 0.1, 0.2, 0.9]), (n_elems, 1)) + 0.05 * rng.random((n_elems, 6))
    lam, mu, d = np.full(n_elems, 4.0e7), np.full(n_elems, 2.7e7), np.zeros(n_elems)
    out = np.empty((n_elems, 36))
    P = lambda a: a.ctypes.data_as(dp)
    L.ref_element_grad_batch(1000, P(xv), P(lam), P(mu), P(d), P(out))
    t = time.perf_counter()
    L.ref_element_grad_batch(n_elems, P(xv), P(lam), P(mu), P(d), P(out))
    dt = time.perf_counter() - t
    return {"melems_per_s_per_core": n_elems / dt / 1e6, "elements": n_elems,
            "what": "the reference's own damIntegrator::AssembleElementGrad (M.cc:639-916, P1, d = 0) compiled in place "
                    "against the MFEM stand-in of oracle/ref_shim, 1 thread, -O3 -DNDEBUG",
            "published_melems_per_s_per_core": 5.5}


def workload_text(n: int, rows: int) -> str:
    return (f"P2 triangles, structured {n} x {rows} cells ({2 * n * rows} elements, {2 * (2 * n + 1) * (2 * rows + 1)} dofs), "
            "jittered, E = reference 200-value table, nu = 0.3, Dirichlet x = 0 / x = 1 (BASELINE configs[3] at n = 5792)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference(args.cpu_n, args.steps, args.warmup, args.cg_iters)
    line = {"impl": "reference", "metric": METRIC, "value": r["step_gdofs"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["step_s_median"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(args.n, args.n), "timed_on": r["sample"], "cg_iters": args.cg_iters},
            "cpu_baseline": {"value": r["step_gdofs"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                             "sample": r["sample"], "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
            "assembly": {"gdofs": r["assembly_gdofs"], "ms": 1e3 * r["assembly_s"]},
            "cg": {"spmv_gbs": r["spmv_gbs"], "spmv_gdofs": r["spmv_gdofs"], "cg_iter_ms": 1e3 * r["cg_iter_s"]},
            "one_thread": r["one_thread"],
            "e2e": {"value": r["step_gdofs"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------
def bind_to_gpu_numa(index: int):
    """Pin this process to the CPU cores next to its GPU (NVML's ideal affinity) so that the pinned host buffers of the
    end-to-end leg are first-touched on that GPU's NUMA node: eight ranks sharing one node's memory controller was
    the round-1 e2e bottleneck (torchrun does not bind its workers).  Returns the number of cores, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class Env:
    """rank / world, barrier, max-over-ranks timing."""

    def __init__(self):
        import torch
        import torch.distributed as td
        self.torch, self.td = torch, td
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the B200 arm has no CPU fallback)")
        torch.cuda.set_device(self.local)
        self.orig_affinity = os.sched_getaffinity(0)
        self.cpu_binding = bind_to_gpu_numa(self.local)
        if self.world > 1:
            td.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        if self.world > 1:
            self.td.barrier()
        self.torch.cuda.synchronize()

    def maxf(self, v: float) -> float:
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.float64, device="cuda")
        self.td.all_reduce(t, op=self.td.ReduceOp.MAX)
        return float(t.item())

    def sumi(self, v: int) -> int:
        if self.world == 1:
            return v
        t = self.torch.tensor([v], dtype=self.torch.int64, device="cuda")
        self.td.all_reduce(t)
        return int(t.item())

    def timed(self, fn, k):
        """k calls bracketed by barrier + synchronize; device time by CUDA events on the launching stream;
        returns (total ms, max over ranks; per-call ms of this rank)."""
        torch = self.torch
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        self.barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for a, b in evs:
            a.record()
            fn()
            b.record()
        e.record()
        self.barrier()
        return self.maxf(s.elapsed_time(e)), [a.elapsed_time(b) for a, b in evs]

    def close(self):
        if self.world > 1:
            self.td.destroy_process_group()


def parity_checks(env, fem, dist, A, form, part, op, n, rows, bvec):
    """In-run parity (every N): (1) all-reduced |K|_F^2 and trace K of the constrained matrix against the oracle's
    golden sums for this workload (tests/golden/config_norms.json, when n is listed there); (2) rigid-body modes
    through the DISTRIBUTED operator: K_unconstrained t = 0 for the two translations and the rotation (exact
    property of any elasticity tangent; exercises assembly + ghost update + owned-row SpMV); returns a dict."""
    torch = env.torch
    lo, hi = 2 * part.own_lo, 2 * part.own_hi
    out = {"ok": True}
    # (2) first: needs the unconstrained matrix
    fem.assemble_matrix_nobc(A, form)
    x = form.x
    modes = {"tx": lambda: torch.stack([torch.ones_like(x[:, 0]), torch.zeros_like(x[:, 0])], dim=1),
             "ty": lambda: torch.stack([torch.zeros_like(x[:, 0]), torch.ones_like(x[:, 0])], dim=1),
             "rot": lambda: torch.stack([-x[:, 1], x[:, 0]], dim=1)}
    nrm = torch.zeros(2, dtype=torch.float64, device="cuda")
    fem.capi.call("femb200_matrix_norms", A.plan, fem._p(A.values), fem._p(nrm), fem._stream())
    y = torch.empty(2 * x.shape[0], dtype=torch.float64, device="cuda")
    worst = 0.0
    for name, make in modes.items():
        v = make().reshape(-1).contiguous()
        v[:lo] = float("nan")
        v[hi:] = float("nan")          # the ghosts must come through the transport
        op.mult(v, y)
        r = torch.stack([y[lo:hi].abs().max(), torch.zeros((), dtype=torch.float64, device="cuda")])
        if env.world > 1:
            env.td.all_reduce(r, op=env.td.ReduceOp.MAX)
        worst = max(worst, float(r[0].item()))
    # local Frobenius norm is enough for the scale (same order on every rank)
    scale = float(np.sqrt(nrm[0].item()))
    out["rigid_body_max_abs_over_fro"] = worst / scale
    out["ok"] &= bool(np.isfinite(worst) and worst / scale < 1e-12)
    # (1) the constrained matrix (left in A.values for the timed steps)
    sums = torch.zeros(2, dtype=torch.float64, device="cuda")
    fem.assemble_matrix(A, form, norms_out=sums)
    if part.world > 1 or part.own_lo != 0 or part.own_hi != A.nnodes:
        # owned rows only: recompute on the owned value range
        sums = owned_norms(torch, fem, A, part)
    op.allreduce_sum(sums)
    f2, tr = (float(v) for v in sums.tolist())
    out["fro2"], out["trace"] = f2, tr
    gold = None
    if os.path.exists(GOLDEN) and rows == n:
        with open(GOLDEN) as f:
            gold = json.load(f).get(str(n))
    if gold is not None:
        out["fro2_rel_err"] = abs(f2 - gold["fro2"]) / gold["fro2"]
        out["trace_rel_err"] = abs(tr - gold["trace"]) / abs(gold["trace"])
        out["golden"] = "tests/golden/config_norms.json (oracle, strip by strip)"
        out["ok"] &= out["fro2_rel_err"] < 1e-12 and out["trace_rel_err"] < 1e-12
    else:
        out["golden"] = None
    return out


# entries kept per output by --dump-outputs, all ranks together: (4 + 1 + 1) M float64 = 48 MB
DUMP_ENTRIES = {"matrix_values": 4 << 20, "cg_x": 1 << 20, "e2e_du": 1 << 20}


def sample_output(v, k: int, seed: int = 0) -> np.ndarray:
    """A 1-D tensor as float64 on the host: whole when it has at most `k` entries, else the entries at (up to) `k`
    sorted indices drawn from `seed`, the same indices on every run with an output of the same length."""
    import torch
    n = v.numel()
    if n > k:
        idx = np.unique(np.random.default_rng(seed).integers(0, n, size=k))
        v = v[torch.from_numpy(idx).to(v.device)]
    return v.detach().to("cpu", torch.float64).numpy()


def dump_outputs(path: str, outputs: dict, rank: int, world: int) -> None:
    """`<path>/<name>.npy` for every output (`<name>_rank<r>.npy` at N > 1)."""
    os.makedirs(path, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(path, name + (f"_rank{rank}" if world > 1 else "") + ".npy"), a)


def owned_norms(torch, fem, A, part):
    """(|K|_F^2, trace K) over the owned rows of this rank (device; torch reductions on slices: checker code)."""
    brp, _ = A.block_csr()
    v0, v1 = 4 * int(brp[part.own_lo].item()), 4 * int(brp[part.own_hi].item())
    f2 = torch.zeros((), dtype=torch.float64, device="cuda")
    chunk = 1 << 28
    for s in range(v0, v1, chunk):
        seg = A.values[s:min(s + chunk, v1)]
        f2 += torch.dot(seg, seg)
    d = A.diagonal()[2 * part.own_lo:2 * part.own_hi]
    return torch.stack([f2, d.sum()])


def run_b200(args):
    env = Env()
    torch, td, world, rank = env.torch, env.td, env.world, env.rank
    from femb200 import fem, dist
    K, W, n = args.steps, max(args.warmup, 3), args.n
    rows = args.rows if args.rows else n
    if rows % world:
        raise SystemExit(f"bench.py: {rows} cell rows do not split into {world} strips")
    t0 = time.perf_counter()
    part = dist.strip_partition_device(n, rows, rank, world, jitter_amp=0.2, seed=1234)
    m = part.mesh
    torch.cuda.synchronize()
    mesh_s = time.perf_counter() - t0
    form = fem.ElasticityForm(m, part.E, 0.3)
    # load the library's CUDA module (lazy, one-off) outside the pattern-build timing
    from femb200 import mesh as _fm
    _tiny = _fm.structured_triangles(4, order=2)
    fem.create_matrix(fem.ElasticityForm(_tiny, _fm.young_per_cell(_tiny.ncells), 0.3))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    A = fem.create_matrix(form)
    A.set_bcs([fem.DirichletBC(part.bc, part.g)])
    torch.cuda.synchronize()
    pattern_ms = 1e3 * (time.perf_counter() - t0)
    owned_nodes, owned_dofs = part.n_owned, 2 * part.n_owned
    total_dofs, total_cells = env.sumi(owned_dofs), env.sumi(part.n_owned_cells)
    lo, hi = 2 * part.own_lo, 2 * part.own_hi

    op = dist.DistOperator(A, part, transport=args.transport)
    bvec = torch.where(part.bc != 0, part.g, torch.ones_like(part.g))
    parity = parity_checks(env, fem, dist, A, form, part, op, n, rows, bvec)
    dcg = dist.DistCG(A, part, rel_tol=0.0, abs_tol=0.0, max_iter=args.cg_iters, op=op, use_graph=not args.no_graph)
    xsol = torch.zeros_like(bvec)
    ytmp = torch.empty_like(bvec)
    vtmp = bvec.clone()

    def asm():
        fem.assemble_matrix(A, form)

    def cg_run():
        dcg.solve(bvec, xsol, fixed_iters=args.cg_iters)

    def spmv_run():
        op.mult(vtmp, ytmp)            # ghost update, then the owned rows

    def step():
        asm()
        cg_run()

    for _ in range(W):
        step()
    spmv_run()
    sampler = ClockSampler(env.local)
    if rank == 0:
        sampler.start()
    step_total, _ = env.timed(step, K)
    step_ms = step_total / K
    value = total_dofs / (step_ms * 1e-3) / 1e9
    outputs = {}
    if args.dump_outputs:
        outputs["matrix_values"] = sample_output(A.values, DUMP_ENTRIES["matrix_values"] // world)
        outputs["cg_x"] = sample_output(xsol[lo:hi], DUMP_ENTRIES["cg_x"] // world)
    asm_total, asm_calls = env.timed(asm, K)
    asm_ms = asm_total / K
    kc = max(1, min(K, 5))
    cg_total, _ = env.timed(cg_run, kc)
    cg_iter_ms = cg_total / kc / (args.cg_iters + 1)      # one PCG call = setup (init + first apply) + cg_iters iterations
    ks = max(K, 10)
    spmv_total, spmv_calls = env.timed(spmv_run, ks)
    spmv_ms = spmv_total / ks
    clocks = sampler.stop() if rank == 0 else None

    # PCG consistency (parity check 3): the recurrence residual of the last solve equals b - A x through the
    # distributed operator, and (where the oracle's PCG state is committed) the 25-iteration iterate matches it
    r_rec = op.vectors()[0][lo:hi].clone()
    op.mult(xsol, ytmp)
    chk = torch.stack([((bvec - ytmp)[lo:hi] - r_rec).pow(2).sum(), bvec[lo:hi].pow(2).sum(), xsol[lo:hi].pow(2).sum()])
    op.allreduce_sum(chk)
    parity["pcg_residual_consistency"] = float((chk[0] / chk[1]).sqrt().item())
    parity["pcg_x_norm"] = float(chk[2].sqrt().item())
    parity["pcg_final_norm"] = dcg.final_norm
    parity["ok"] &= parity["pcg_residual_consistency"] < 1e-10
    if os.path.exists(GOLDEN) and rows == n and args.cg_iters == 25:
        with open(GOLDEN) as f:
            gold = json.load(f).get(str(n), {}).get("pcg25")
        if gold:
            parity["pcg_x_norm_rel_err"] = abs(parity["pcg_x_norm"] - gold["x_norm"]) / gold["x_norm"]
            parity["pcg_final_norm_rel_err"] = abs(dcg.final_norm - gold["final_norm"]) / gold["final_norm"]
            parity["ok"] &= parity["pcg_x_norm_rel_err"] < 1e-10 and parity["pcg_final_norm_rel_err"] < 1e-8

    # transports side by side at N > 1: the NCCL baseline of the same iteration
    comm = {"transport": op.transport, "graph": not args.no_graph}
    if world > 1 and op.transport == "p2p" and not args.no_nccl_compare:
        op.use("nccl")
        for _ in range(2):
            cg_run()
        t_nccl, _ = env.timed(cg_run, kc)
        comm["nccl_cg_iter_ms"] = t_nccl / kc / (args.cg_iters + 1)
        comm["p2p_cg_iter_ms"] = cg_iter_ms
        op.use("p2p")

    # ---- end to end: one Newton linearisation through the public API, host buffers ------------------
    e2e_du, e2e = e2e_newton(env, fem, dist, form, part, op, A, args, total_dofs)
    if args.dump_outputs:
        outputs["e2e_du"] = sample_output(e2e_du, DUMP_ENTRIES["e2e_du"] // world)
        dump_outputs(args.dump_outputs, outputs, rank, world)

    # BASELINE configs[4] over the ranks (N > 1; at N = 1 it is part of `extras`)
    c5 = config5_ranks(env, fem, dist, assembly_bytes) if (world > 1 and not args.skip_extras) else None

    nnzb_owned = part.owned_nnz_blocks(A)
    plan_bytes = A.plan_bytes
    a_bytes = assembly_bytes(A.nnz, m.ncells, m.nnodes)            # this rank's launch (ghost cell row included)
    s_bytes = spmv_bytes(nnzb_owned, owned_nodes)
    col_bits = A.get_option("spmv_col_bits")                       # 16: column offsets from the row's node, 2 B per block
    s_moved = s_bytes - (4 - col_bits // 8) * nnzb_owned           # bytes the kernel is designed to move
    c_bytes = cg_iter_bytes(nnzb_owned, owned_nodes) - (s_bytes - s_moved)   # bytes the iteration's kernels move
    c_bytes_survey = s_bytes + 56 * 2 * owned_nodes                # SURVEY 8(d): SpMV + 7 vector passes (56 B per dof)
    if rank != 0:
        if world == 1:
            pass
        op.close()
        env.close()
        return

    peak, peak_src = measured_peaks()
    a_ms = float(np.mean(asm_calls))
    s_ms = float(np.mean(spmv_calls))
    a_gbs, s_gbs, c_gbs = a_bytes / (a_ms * 1e-3) / 1e9, s_bytes / (s_ms * 1e-3) / 1e9, c_bytes / (cg_iter_ms * 1e-3) / 1e9
    # PCG call: init, scalar, apply, scalar; cg_iters - 1 full iterations of 5 kernels (update_r, scalar, update_xdir,
    # apply, scalar); the last one 3 (update_r, scalar, x update); one ghost-update kernel per apply on the P2P transport
    launches_pcg = 4 + 5 * (args.cg_iters - 1) + 3 + (args.cg_iters if (world > 1 and op.transport == "p2p") else 0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_text(n, rows), "step": f"full CSR assembly + Dirichlet, then {args.cg_iters} Jacobi-PCG "
                   "iterations (ghost update + all-reduces inside at N > 1)", "elements": total_cells, "dofs": total_dofs,
                   "nnz_rank0": A.nnz, "plan_bytes_rank0": plan_bytes,
                   "l2": "values + vectors per step (>= 6 GB per GPU at N = 8) exceed the 126 MB L2; no explicit flush",
                   "parallelism": f"{world} strips of cell rows, one ghost cell row, owner = lowest rank" if world > 1 else "single GPU",
                   "cg_iters": args.cg_iters, "pattern_build_ms": pattern_ms, "mesh_generation_s": mesh_s},
        "parity": parity,
        "roofline": {"kernel": "spmv_tma_kernel<DOT,64,2,4> (dominant: cg_iters + 1 launches per step)", "bound": "hbm",
                     "achieved": s_gbs, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": s_gbs / peak,
                     "algorithmic_bytes_per_launch": s_bytes, "kernel_ms": s_ms,
                     "bytes_moved_by_design": s_moved, "frac_of_bytes_moved": s_moved / (s_ms * 1e-3) / 1e9 / peak,
                     "column_index_bits": col_bits,
                     "traffic": traffic_from_profile("spmv", n, world), "note": "rank 0's owned rows; timed alone over "
                     f"{ks} launches (with the ghost update at N > 1); achieved = SURVEY 8(d)'s algorithmic bytes "
                     "(36 B per node block + 40 B per node) / time; the kernel reads 16-bit column offsets where the "
                     "pattern allows (34 B per block): bytes_moved_by_design / frac_of_bytes_moved"},
        "assembly": {"ms": asm_ms, "gdofs": total_dofs / (asm_ms * 1e-3) / 1e9,
                     "roofline": {"kernel": "assemble_fast_kernel<P2> (+ cell_setup_kernel, dirichlet_kernel)", "bound": "hbm",
                                  "achieved": a_gbs, "peak": peak, "unit": "GB/s", "frac": a_gbs / peak,
                                  "algorithmic_bytes_per_launch": a_bytes, "kernel_ms": a_ms,
                                  "traffic": traffic_from_profile("assemble", n, world)}},
        "cg": {"spmv_ms": spmv_ms, "spmv_gbs": s_gbs, "spmv_frac": s_gbs / peak, "spmv_gdofs": total_dofs / (spmv_ms * 1e-3) / 1e9,
               "cg_iter_ms": cg_iter_ms, "cg_iter_gbs": c_gbs, "cg_iter_frac": c_gbs / peak,
               "cg_iter_bytes": c_bytes, "cg_iter_frac_at_survey_bytes": c_bytes_survey / (cg_iter_ms * 1e-3) / 1e9 / peak,
               "cg_iter_what": "bytes moved by design: SpMV (34 or 36 B per block + 40 B per node) + 10 vector passes "
                               "(update_r: 3 reads 1 write; update_xdir: 4 reads 2 writes, Jacobi included); "
                               "SURVEY 8(d) counts SpMV at 36 B per block + 7 passes",
               "cg_iter_gdofs": total_dofs / (cg_iter_ms * 1e-3) / 1e9, "precond": "jacobi", "iters": args.cg_iters,
               "comm": comm},
        "e2e": e2e,
        "gpu_launches": K * (3 + launches_pcg),
        "clocks": clocks,
    }
    if c5 is not None:
        line["config5_over_ranks"] = c5
    del dcg, xsol, ytmp, vtmp, bvec
    op.close()
    if world == 1 and not args.skip_extras:
        del A, form, part, m, op
        torch.cuda.empty_cache()
        line["extras"] = extras(env, fem, peak, args)
    if world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, env.orig_affinity)      # the CPU arm gets every core of the box back
        r = cpu_reference(args.cpu_baseline_n, 3, 1, args.cg_iters)
        line["cpu_baseline"] = {"value": r["step_gdofs"], "unit": UNIT, "cores": r["threads"], "kind": "port",
                                "sample": r["sample"], "assembly_gdofs": r["assembly_gdofs"], "spmv_gbs": r["spmv_gbs"],
                                "spmv_gdofs": r["spmv_gdofs"], "one_thread": r["one_thread"],
                                "reference_element_kernel": reference_element_kernel_rate()}
    print(json.dumps(line), flush=True)
    env.close()
    if not parity["ok"]:
        raise SystemExit("bench.py: in-run parity check FAILED: " + json.dumps(parity))


def e2e_newton(env, fem, dist, form, part, op, A, args, total_dofs):
    """The same step end to end through the public API with HOST buffers: per step the current iterate u goes up
    from pinned host memory, NewtonSolver.residual (F(u) + lifting) and NewtonSolver.increment (tangent assembly +
    Dirichlet + `cg_iters` PCG iterations) run, and the increment du comes back to pinned host memory.  Geometry,
    materials and the pattern are resident (uploaded once: they do not change between Newton iterations).  Returns the
    host buffer holding the last step's du and the result line's "e2e" entry."""
    torch = env.torch
    K = args.e2e_steps or args.steps
    ns = fem.NewtonSolver.__new__(fem.NewtonSolver)          # reuse the bench's matrix / operator (no second 49 GB)
    ns.form, ns.f, ns.A, ns.part = form, None, A, part
    ns.rel_tol, ns.abs_tol, ns.max_iter, ns.convention = 1e-7, 5e-8, 10, "mfem"
    ns.g = part.g
    ns.cg = dist.DistCG(A, part, rel_tol=0.0, abs_tol=0.0, max_iter=args.cg_iters, op=op, jacobi=False,
                        use_graph=not args.no_graph)
    ns._lo, ns._hi = 2 * part.own_lo, 2 * part.own_hi
    ns._b = torch.empty(A.ndofs, dtype=torch.float64, device="cuda")
    ns._du = torch.zeros(A.ndofs, dtype=torch.float64, device="cuda")
    ns._nrm = torch.zeros(1, dtype=torch.float64, device="cuda")
    ns._lifted, ns._tangent_ready = False, False
    ns.residual_norms, ns.linear_iterations = [], []
    nloc = A.ndofs
    hu = torch.zeros(nloc, dtype=torch.float64).pin_memory()
    hu.copy_(torch.from_numpy(1e-4 * np.cos(np.arange(nloc, dtype=np.float64) * 1e-3)))
    hdu = torch.empty(ns._hi - ns._lo, dtype=torch.float64).pin_memory()
    du_dev = torch.empty(nloc, dtype=torch.float64, device="cuda")

    copy_stream, up = torch.cuda.Stream(), torch.cuda.Event()

    def e2e_step():
        main = torch.cuda.current_stream()
        copy_stream.wait_stream(main)                             # the previous step is done with the buffer
        with torch.cuda.stream(copy_stream):
            du_dev.copy_(hu, non_blocking=True)                   # H2D: the iterate (owned + ghost window)
            up.record(copy_stream)
        ns._lifted = False
        ns.prepare_tangent()                                      # the tangent of this (undamaged) form does not read u:
        main.wait_event(up)                                       # it is assembled while u is on its way
        b = ns.residual(du_dev)                                   # F(u), lifting (unconstrained tangent already there)
        du = ns.increment(b, fixed_iters=args.cg_iters)           # Dirichlet rows/cols, Jacobi, PCG
        hdu.copy_(du[ns._lo:ns._hi], non_blocking=True)           # D2H: the increment (owned dofs)
        torch.cuda.current_stream().synchronize()                 # the host consumes du

    for _ in range(2):
        e2e_step()
    tot, _ = env.timed(lambda: [e2e_step() for _ in range(K)], 1)
    ms = tot / K
    return hdu, {"value": total_dofs / (ms * 1e-3) / 1e9, "unit": UNIT, "ms_per_step": ms, "steps": K,
                 "h2d_bytes_per_step": int(hu.numel() * 8), "d2h_bytes_per_step": int(hdu.numel() * 8),
                 "cpu_cores_bound_to_gpu_numa_node": env.cpu_binding,
                 "du_checksum": float(hdu.abs().sum().item()),
                 "what": "per step and per rank: pinned host u -> device on a copy stream while NewtonSolver.prepare_tangent "
                         "assembles the tangent (it does not read u: the form is undamaged), NewtonSolver.residual (F(u) + "
                         "apply_lifting: work the device-timed `value` does not contain), NewtonSolver.increment (Dirichlet "
                         "rows / columns + Jacobi + PCG), owned du -> pinned host, host waits for it; geometry / materials / "
                         "pattern resident (constant across Newton iterations)"}


def extras(env, fem, peak, args):
    """The other BASELINE configurations on one GPU, in the default run: configs[2] (Q2 quads, matrix-free CG,
    16.8 M elements), configs[4] (damaged-tangent reassembly of 16.8 M P2 elements at 10 / 50 / 100 % damaged cells,
    closed form and AD), and the FP64 roofline of the element kernels."""
    torch = env.torch
    from femb200 import mesh as fm, dist
    capi = fem.capi
    out = {}
    # ---- FP64 peak (measured) + element kernels -------------------------------------------------------
    nb, fl = ctypes.c_int64(), ctypes.c_double()
    capi.call("femb200_fp64_probe", 8, 4096, None, ctypes.byref(nb), ctypes.byref(fl), None)
    buf = torch.empty(nb.value * 256, dtype=torch.float64, device="cuda")
    probe = lambda: capi.call("femb200_fp64_probe", 8, 4096, fem._p(buf), ctypes.byref(nb), ctypes.byref(fl), fem._stream())
    for _ in range(3):
        probe()
    tot, calls = env.timed(probe, 10)
    fp64_peak = fl.value / (min(calls) * 1e-3) / 1e12
    out["fp64"] = {"peak_tflops": fp64_peak, "how": "femb200_fp64_probe: 8 x 148 blocks x 256 threads x 8 independent DFMA "
                   "chains x 4096 rounds, best of 10, CUDA events", "flops_per_launch": fl.value}
    n = 1448
    p = dist.strip_partition_device(n, n, 0, 1)
    m = p.mesh
    form = fem.ElasticityForm(m, p.E, 0.3)
    Ae = torch.empty((m.ncells, 12, 12), dtype=torch.float64, device="cuda")
    for _ in range(2):
        fem.tabulate_tensor_batched(form, out=Ae)
    tot, calls = env.timed(lambda: fem.tabulate_tensor_batched(form, out=Ae), 10)
    ms = float(np.mean(calls))
    # undamaged straight-sided triangles: closed form from the nine P1 blocks: 9 x bdb_block (38 flops) + the 36 blocks
    # (9 x 4 + 12 x 4 + 9 x 4 x 8 flops) + geometry (~30)
    FL_CLOSED = 9 * 38 + 36 + 48 + 288 + 30
    out["fp64"]["tabulate_kernel_p2"] = {
        "ms": ms, "cells": m.ncells, "flops_per_element": FL_CLOSED, "tflops": FL_CLOSED * m.ncells / (ms * 1e-3) / 1e12,
        "frac_fp64": FL_CLOSED * m.ncells / (ms * 1e-3) / 1e12 / fp64_peak, "bytes_written_per_element": 1152,
        "frac_hbm": (1152 + 40) * m.ncells / (ms * 1e-3) / 1e9 / peak,
        "what": "femb200_tabulate_tensor_batched (ufcx / AssembleElementGrad surface), undamaged cells: all 12 x 12 element "
                "tangents to HBM from the closed form (exact for the 3-point rule on straight-sided triangles): HBM-bound"}
    # the same kernel on damaged cells (d > 0 at every point): per-point integration, B_q D_q B_q^t with the reference's
    # closed-form tangent (M.cc:736-872): the FP64-heavy form of the element kernel
    xy = m.x
    dfull = torch.full((m.nnodes,), 0.5, dtype=torch.float64, device="cuda")
    ufull = 1e-3 * torch.randn(2 * m.nnodes, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    formd = fem.ElasticityForm(m, p.E, 0.3, d=dfull, u=ufull)
    for _ in range(2):
        fem.tabulate_tensor_batched(formd, out=Ae)
    tot, calls = env.timed(lambda: fem.tabulate_tensor_batched(formd, out=Ae), 10)
    msd = float(np.mean(calls))
    FL_TAB = 36 * 3 * 38 + 3 * 70 + 3 * 150   # 36 block pairs x 3 points x bdb_block (38) + 3 x point geometry (~70) + 3 x tangent (~150)
    out["fp64"]["tabulate_kernel_p2_damaged"] = {
        "ms": msd, "cells": m.ncells, "flops_per_element": FL_TAB, "tflops": FL_TAB * m.ncells / (msd * 1e-3) / 1e12,
        "frac_fp64": FL_TAB * m.ncells / (msd * 1e-3) / 1e12 / fp64_peak,
        "frac_hbm": (1152 + 40 + 6 * 16 + 24) * m.ncells / (msd * 1e-3) / 1e9 / peak,
        "what": "the same kernel with every cell damaged: per-point triple products + the closed-form damaged tangent"}
    del formd, dfull, ufull
    # the reference's own element: P1, one point (damIntegrator::AssembleElementGrad, M.cc:639-916; the CPU figure of the
    # same kernel compiled from the reference's source is in cpu_baseline.reference_element_kernel)
    from femb200 import mesh as _fm
    m1 = _fm.jitter(_fm.structured_triangles(2896, order=1), 0.2, seed=1234)
    f1 = fem.ElasticityForm(m1, _fm.young_per_cell(m1.ncells), 0.3)
    A1 = torch.empty((m1.ncells, 6, 6), dtype=torch.float64, device="cuda")
    for _ in range(2):
        fem.tabulate_tensor_batched(f1, layout=fem.capi.COLMAJOR_BYNODES, out=A1)
    tot, calls = env.timed(lambda: fem.tabulate_tensor_batched(f1, layout=fem.capi.COLMAJOR_BYNODES, out=A1), 10)
    ms1 = float(np.mean(calls))
    out["fp64"]["element_grad_p1"] = {
        "ms": ms1, "cells": m1.ncells, "gelems_per_s": m1.ncells / (ms1 * 1e-3) / 1e9, "bytes_written_per_element": 288,
        "frac_hbm": (288 + 12 + 8 + 8) * m1.ncells / (ms1 * 1e-3) / 1e9 / peak,
        "what": "femb200_element_grad_batched on 16.8 M P1 triangles, MFEM layout (column-major, byNODES): the batched "
                "form of the reference's AssembleElementGrad, d = 0"}
    del A1, f1, m1
    del Ae
    A = fem.create_matrix(form)
    for _ in range(3):
        fem.assemble_matrix(A, form)
    tot, calls = env.timed(lambda: fem.assemble_matrix(A, form), 10)
    ms = float(np.mean(calls))
    FL_FAST = 900
    out["fp64"]["assemble_fast_kernel_p2"] = {
        "ms": ms, "cells": m.ncells, "flops_per_element": FL_FAST, "tflops": FL_FAST * m.ncells / (ms * 1e-3) / 1e12,
        "frac_fp64": FL_FAST * m.ncells / (ms * 1e-3) / 1e12 / fp64_peak,
        "frac_hbm": assembly_bytes(A.nnz, m.ncells, m.nnodes) / (ms * 1e-3) / 1e9 / peak,
        "what": "the fused element + gather kernel of the timed path at n = 1448 (closed-form P2 blocks: ~0.9 kflop per "
                "element); HBM-bound, the FP64 pipe idles"}
    out["config2_p2_n1448"] = {"assembly_ms": ms, "assembly_gdofs": m.ndofs / (ms * 1e-3) / 1e9,
                               "assembly_frac_hbm": out["fp64"]["assemble_fast_kernel_p2"]["frac_hbm"]}
    del A, form, p, m
    torch.cuda.empty_cache()

    # ---- config 3: Q2 matrix-free ----------------------------------------------------------------------
    n = 4096
    m = fm.jitter(fm.structured_quads_q2(n), 0.2, seed=1234)
    E = fm.young_per_cell(m.ncells)
    bc, g = fm.dirichlet_markers(m)
    form = fem.ElasticityForm(m, E, 0.3)
    pa = fem.PAOperator(form, bcs=[fem.DirichletBC(bc, g)])
    v = torch.randn(m.ndofs, dtype=torch.float64, device="cuda")
    y = torch.empty_like(v)
    for _ in range(3):
        pa.mult(v, y)
    tot, calls = env.timed(lambda: pa.mult(v, y), 10)
    ms = float(np.mean(calls))
    nbytes = m.nnodes * 32 + m.ncells * (8 * (2 * m.nv + 2) + 4 * m.nd + 4)
    r = {"workload": f"Q2 quads n={n}: {m.ncells} elements, {m.ndofs} dofs, 3x3 Gauss, sum-factorised (BASELINE configs[2])",
         "pa_apply_ms": ms, "gdofs": m.ndofs / (ms * 1e-3) / 1e9, "gbs": nbytes / (ms * 1e-3) / 1e9,
         "frac": nbytes / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes": nbytes,
         "bytes_per_element": nbytes / m.ncells, "survey_bytes_per_element": 596,
         "frac_at_survey_bytes": 596 * m.ncells / (ms * 1e-3) / 1e9 / peak}
    cg = fem.CGSolver(rel_tol=0.0, max_iter=10)
    cg.SetOperator(pa)
    cg.SetPreconditioner("jacobi")
    b = torch.ones(m.ndofs, dtype=torch.float64, device="cuda")
    x = torch.empty_like(b)
    cg.Mult(b, x, fixed_iters=10)
    tot, _ = env.timed(lambda: cg.Mult(b, x, fixed_iters=10), 3)
    r.update({"pa_cg_iter_ms": tot / 3 / 11, "pa_cg_iter_gdofs": m.ndofs / (tot / 3 / 11 * 1e-3) / 1e9})
    out["config3_q2_matrix_free"] = r
    del pa, cg, form, b, x, v, y
    torch.cuda.empty_cache()

    # ---- config 5: damaged reassembly ---------------------------------------------------------------------
    n = 2896
    p = dist.strip_partition_device(n, n, 0, 1)
    m = p.mesh
    xy = m.x
    u = 1e-3 * torch.randn(2 * m.nnodes, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    res = {"workload": f"P2 n={n} ({m.ncells} elements, BASELINE configs[4] on one GPU), values-only reassembly on a frozen "
                       "pattern, damage band of the stated width"}
    form0 = fem.ElasticityForm(m, p.E, 0.3)
    A = fem.create_matrix(form0)
    for _ in range(2):
        fem.assemble_matrix(A, form0)
    tot, calls = env.timed(lambda: fem.assemble_matrix(A, form0), 5)
    res["undamaged_ms"] = float(np.mean(calls))
    a_bytes = assembly_bytes(A.nnz, m.ncells, m.nnodes)
    for label, half_width in (("10pct", 0.05), ("50pct", 0.25), ("100pct", 10.0)):
        d = torch.clamp(1.0 - (xy[:, 1] - 0.5 - 0.1 * torch.sin(6.0 * xy[:, 0])).abs() / half_width, min=0.0, max=0.95)
        share = float((d[m.xdofmap.long()].max(dim=1).values > 0).double().mean().item())
        rec = {"damaged_cell_share": share}
        for variant, name in ((0, "closed_form"), (1, "ad")):
            form = fem.ElasticityForm(m, p.E, 0.3, d=d, u=u, variant=variant)
            for _ in range(3):  # a Newton loop has a solve between two assemblies: let the plan's damage-share word
                fem.assemble_matrix(A, form)  # (written by the previous assembly) settle, and with it the one-off slot map
                torch.cuda.synchronize()
            tot, calls = env.timed(lambda: fem.assemble_matrix(A, form), 5)
            ms = float(np.mean(calls))
            rec[name + "_ms"] = ms
            rec[name + "_gdofs"] = m.ndofs / (ms * 1e-3) / 1e9
            rec[name + "_frac_hbm"] = (a_bytes + 8 * m.nnodes + 16 * m.nnodes) / (ms * 1e-3) / 1e9 / peak
            del form
        rec["ad_over_closed"] = rec["ad_ms"] / rec["closed_form_ms"]
        res[label] = rec
    out["config5_damaged_reassembly"] = res
    return out


def config5_ranks(env, fem, dist, abytes):
    """BASELINE configs[4] ("repeated tangent reassembly on 16 M P2 elements, 8 B200") inside the default multi-GPU run:
    the nx = 2896 mesh in `world` strips, a vertical damage band of 10 % / 100 % of the cells through every strip,
    values-only reassembly on the frozen pattern (no communication: ghost cell row), closed form and AD."""
    torch = env.torch
    nx = 2896
    rows = nx - nx % env.world
    part = dist.strip_partition_device(nx, rows, env.rank, env.world, jitter_amp=0.2, seed=1234)
    m = part.mesh
    x, y = m.x[:, 0], m.x[:, 1]
    u = 1e-3 * torch.randn(2 * m.nnodes, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(env.rank))
    form0 = fem.ElasticityForm(m, part.E, 0.3)
    A = fem.create_matrix(form0)
    dofs = env.sumi(2 * part.n_owned)
    peak, _ = measured_peaks()
    out = {"workload": f"P2 nx = {nx}, {rows} cell rows in {env.world} strips ({2 * nx * rows} elements), vertical damage band, "
                       "values-only reassembly on a frozen pattern, no communication", "dofs": dofs}
    for label, hw in (("10pct", 0.05), ("100pct", 10.0)):
        d = torch.clamp(1.0 - (x - 0.5 - 0.1 * torch.sin(6.0 * y)).abs() / hw, min=0.0, max=0.95)
        rec = {}
        for variant, name in ((0, "closed_form"), (1, "ad")):
            form = fem.ElasticityForm(m, part.E, 0.3, d=d, u=u, variant=variant)
            for _ in range(3):
                fem.assemble_matrix(A, form)
                torch.cuda.synchronize()  # see extras(): the schedule follows the previous assembly's damage share
            tot, calls = env.timed(lambda: fem.assemble_matrix(A, form), 10)
            ms = tot / 10
            rec[name + "_ms"] = ms
            rec[name + "_gdofs"] = dofs / (ms * 1e-3) / 1e9
            rec[name + "_frac_hbm_rank0"] = abytes(A.nnz, m.ncells, m.nnodes) / (float(np.mean(calls)) * 1e-3) / 1e9 / peak
        rec["ad_over_closed"] = rec["ad_ms"] / rec["closed_form_ms"]
        out[label] = rec
    return out


def config5(args, rank, world, local):
    """BASELINE config 5 over the ranks: repeated tangent reassembly (closed-form and AD tangents, M.cc:736-872 /
    752-765) of 16 773 632 P2 elements on `world` GPUs: strips of the nx = 2896 mesh, a vertical damage band through
    every strip, 10 reassemblies on the frozen pattern.  Assembly needs no communication (ghost cell row)."""
    import torch
    import torch.distributed as td
    from femb200 import fem, dist
    torch.cuda.set_device(local)
    if world > 1:
        td.init_process_group("nccl", device_id=torch.device("cuda", local))
    nx = 2896
    part = dist.strip_partition_device(nx, nx - nx % world, rank, world, jitter_amp=0.2, seed=1234)
    m, E, owned_dofs = part.mesh, part.E, 2 * part.n_owned
    x, y = m.x[:, 0], m.x[:, 1]
    d = torch.clamp(1.0 - (x - 0.5 - 0.1 * torch.sin(6.0 * y)).abs() / args.damage_half_width, min=0.0, max=0.95)
    u = 1e-3 * torch.randn(2 * m.nnodes, dtype=torch.float64, device="cuda", generator=torch.Generator("cuda").manual_seed(rank))
    share = float((d[m.xdofmap.long()].max(dim=1).values > 0).double().mean().item())
    reps = 10

    def sync():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    out = {}
    for variant, name in ((0, "closed_form"), (1, "ad")):
        form = fem.ElasticityForm(m, E, 0.3, d=d, u=u, variant=variant)
        A = fem.create_matrix(form)
        for _ in range(3):
            fem.assemble_matrix(A, form)
        sync()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(reps):
            fem.assemble_matrix(A, form)
        e.record()
        sync()
        t = torch.tensor([s.elapsed_time(e), float(owned_dofs)], dtype=torch.float64, device="cuda")
        if world > 1:
            tmax = t.clone()
            td.all_reduce(tmax, op=td.ReduceOp.MAX)
            td.all_reduce(t, op=td.ReduceOp.SUM)
            ms, dofs = tmax[0].item() / reps, t[1].item()
        else:
            ms, dofs = t[0].item() / reps, t[1].item()
        out[name] = {"ms_per_reassembly": ms, "gdofs": dofs / (ms * 1e-3) / 1e9}
        del A, form
        torch.cuda.empty_cache()
    if rank == 0:
        print(json.dumps({"metric": "damaged-tangent reassembly GDOF/s (BASELINE config 5)", "unit": UNIT,
                          "value": out["closed_form"]["gdofs"], "n_gpus": world, "reassemblies": reps,
                          "higher_is_better": True, "dtype": "f64", "data": "synthetic",
                          "config": {"workload": f"P2 triangles nx = {nx}, strips over {world} GPU(s), vertical damage band "
                                                 f"on {100 * share:.1f} % of rank 0's cells, values-only reassembly on a frozen "
                                                 "pattern", "elements_total": 2 * nx * (nx - nx % world)},
                          "closed_form": out["closed_form"], "ad": out["ad"],
                          "ad_over_closed": out["ad"]["ms_per_reassembly"] / out["closed_form"]["ms_per_reassembly"]}),
              flush=True)
    if world > 1:
        td.destroy_process_group()


def traffic_from_profile(which: str, n: int, world: int):
    """dram__bytes (read + write) per launch of the kernel from the committed `ncu --set full` capture of THIS workload
    size on one GPU (profiles/traffic.json: {"<n>": {"assemble": ..., "spmv": ...}}); null when no capture of this size
    is committed.  ncu cannot run inside the timed process: a number printed under a profiler is never a bench value."""
    if world != 1:
        return None
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        with open(path) as f:
            return json.load(f).get(str(n), {}).get(which)
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--size", dest="n", type=int, default=5792, help="cells per side of the global mesh (5792 -> 67 M P2 triangles)")
    ap.add_argument("--rows", type=int, default=0, help="cell rows of the global mesh (default: --size)")
    ap.add_argument("--cg-iters", type=int, default=25)
    ap.add_argument("--cpu-n", type=int, default=1448, help="cells per side of the CPU sample of --impl reference")
    ap.add_argument("--cpu-baseline-n", type=int, default=1024, help="cells per side of the cpu_baseline leg of the default run")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed steps of the end-to-end leg (default: --steps)")
    ap.add_argument("--transport", default="auto", choices=["auto", "p2p", "nccl"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-nccl-compare", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="N = 1 only: skip configs 3 / 5 and the FP64 roofline")
    ap.add_argument("--config5", action="store_true",
                    help="BASELINE config 5 over the ranks instead of the headline step: repeated damaged-tangent reassembly "
                         "(closed form and AD) of 16.8 M P2 elements (nx = 2896)")
    ap.add_argument("--damage-half-width", type=float, default=0.05)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.e2e_steps < 0:
        ap.error("--steps must be at least 1 and --e2e-steps not negative")
    if args.dump_outputs and (args.impl == "reference" or args.config5):
        ap.error("--dump-outputs applies to the B200 step (not --impl reference, not --config5)")
    sys.dont_write_bytecode = True      # the tree may be read-only: no __pycache__ next to the imported modules
    if args.impl == "reference":
        run_reference(args)
    elif args.config5:
        config5(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")),
                int(os.environ.get("LOCAL_RANK", "0")))
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
