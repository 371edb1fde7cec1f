#!/usr/bin/env python
"""bench.py -- pair-solves/sec of the focal-pair Laplacian solve loop on B200.

Contract (one JSON line on stdout from rank 0):
  python bench.py --gpus N --steps K --warmup W            (N>1 under torchrun)
  python bench.py --impl reference ...                     (CPU CG+AMG arm)
  python bench.py ... --dump-outputs DIR                   (also write the last timed step's results
                                                            as DIR/<name>.npy, see dump_outputs)

Default workload = the configuration BASELINE.json's metric is quoted on, "10^7-node raster":
3163 x 3163 synthetic resistance raster (R ~ U[1,10], seed 42; n = 10 004 569, nnz = 90 003 169),
8-neighbour average-conductance stencil, fp64, 128 focal pairs (17 focal nodes, rng 7) -- a fixed
job that is sharded over the N GPUs (STRONG scaling, the split of BASELINE config C4: pairs
round-robin over ranks, 16 pairs = two full 8-column panels per GPU at N = 8).
`--config c2` is BASELINE configs[1] (1000 x 1000, 10 pairs per GPU, weak), the round-1 line.

A *step* = one pass of the hot path over the rank's pairs: RHS build, batched AMG-PCG to
rtol 1e-6, true-residual gate, resistance extraction, node currents accumulated into the
cumulative / max vectors -- all on the device through `cs_b200_solve_pairs`; for N > 1 the step
ends with the gather of the resistances and the SUM / MAX reduction of the current maps.
The operator + preconditioner are resident before the timed region (the reference's "construct
cholesky factor" / "construct preconditioner" is likewise once per component, src/core.jl:164-167,
379); its cost is in `setup` together with the setup-INCLUSIVE rate of the whole job.
  value        pair-solves/s, whole job, device-timed (CUDA events on the solve stream)
  e2e          the same pairs through the plug-in hook `solve_linear_system(factor, matrix, rhs)` in
               batches of `--bs` columns (cholmod_batch_size, src/core.jl:448-452) with pinned HOST
               n x bs RHS / solution buffers (H2D + D2H inside), all `--steps` steps
  roofline     dominant kernel (finest-level k_spmm_win, k = 8) timed per launch with CUDA events in
               an instrumented repeat of one step; `spmv_1e7` = the SpMV / SpMM micro-benchmark
  cpu_baseline the oracle's CG+AMG port on the host cores, one pair per core, bounded sample
  parity       max relative deviation of R from the oracle's CG+AMG run to rtol 1e-10
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: rows, cols, pairs (total when strong / per GPU when weak), scaling
    "headline": dict(rows=3163, cols=3163, pairs=128, scaling="strong"),
    "c2": dict(rows=1000, cols=1000, pairs=10, scaling="weak"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS))
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--pairs", type=int, default=0, help="total pairs (strong) / pairs per GPU (weak)")
    ap.add_argument("--scaling", default="", choices=["", "strong", "weak"])
    ap.add_argument("--bs", type=int, default=32, help="columns per solve_linear_system call in the e2e leg")
    ap.add_argument("--precision", default="double")
    ap.add_argument("--precond", default="amg", choices=["amg", "jacobi"])
    ap.add_argument("--rtol", type=float, default=1e-6)
    ap.add_argument("--loop", default="device", choices=["device", "chunk", "plain"],
                    help="PCG loop control: device-side WHILE graph | host-polled graph chunks | plain launches")
    ap.add_argument("--setup", default="auto", choices=["auto", "device", "host"],
                    help="where the AMG hierarchy / window records are built")
    ap.add_argument("--skip-spmv1e7", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-direct", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=16, help="pairs per CPU step (one per core)")
    ap.add_argument("--ref-budget-s", type=float, default=330.0,
                    help="--impl reference: wall budget that bounds the warm-up steps after the first")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    c = CONFIGS[a.config]
    a.rows = a.rows or c["rows"]
    a.cols = a.cols or c["cols"]
    a.pairs = a.pairs or c["pairs"]
    a.scaling = a.scaling or c["scaling"]
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        return json.load(open(p))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_SAMPLE = 1 << 20        # entries kept of a longer output: a 10^7-node map becomes 8 MB in fp64


def dump_outputs(path, arrays):
    """Write each array as path/<name>.npy.  An array longer than DUMP_SAMPLE is cut to the same
    seeded sample of its entries on every run, so runs with the same arguments compare entry for entry."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.size > DUMP_SAMPLE:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(path, f"{name}.npy"), a)


def b_spmm(n, nnz, k, sv):
    """SURVEY.md §8d / BASELINE.md: algorithmic bytes of one SpMM launch."""
    return nnz * (sv + 4) + (n + 1) * 4 + 2 * n * k * sv


def total_pairs(args, world):
    return args.pairs if args.scaling == "strong" else args.pairs * world


def workload(args, npairs):
    from circuitscape_b200 import graph
    L, _ = graph.synthetic_raster_laplacian(args.rows, args.cols, seed=42,
                                            dtype=np.float64 if args.precision == "double" else np.float32)
    npts = 2
    while npts * (npts - 1) // 2 < npairs:
        npts += 1
    nodes = graph.focal_nodes(L.shape[0], npts, seed=7)
    src, dst = graph.all_pairs(nodes, limit=npairs)
    return L, src, dst


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.proc = None
        self.lines = []
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------
# CPU arm: the oracle's CG+AMG port, one pair per core (mirrors src/core.jl:262-272)
# ---------------------------------------------------------------------------
_CPU = {}


def _cpu_init():
    try:                                   # one BLAS thread per worker: no oversubscription
        from threadpoolctl import threadpool_limits
        _CPU["_tp"] = threadpool_limits(1)
    except Exception:
        pass


def _cpu_one(job):
    from oracle import amg
    i, rtol = job
    A, ml, src, dst = _CPU["A"], _CPU["ml"], _CPU["src"], _CPU["dst"]
    if rtol < 0:                 # parity reference: the UNregularised Laplacian, converged far below rtol
        A, rtol = _CPU["A0"], -rtol
    n = A.shape[0]
    b = np.zeros(n); b[src[i]] = -1.0; b[dst[i]] = 1.0
    if rtol >= 1e-6:
        v, it = amg.pcg(A, b, ml, rtol=rtol, itmax=100_000)          # src/core.jl:639 (atol = sqrt(eps))
    else:
        v, it = amg.pcg(A, b, ml, rtol=rtol, atol=0.0, itmax=100_000)  # tight run
    res = np.linalg.norm(A @ v - b) / np.sqrt(2.0)
    assert res < 1e-4                                                # src/core.jl:640-641
    return float(v[dst[i]] - v[src[i]]), it


class CpuArm:
    """The oracle's SA-AMG(sym. GS, pinv coarse)-preconditioned CG on the host cores: hierarchy once
    (src/core.jl:164-167), then one pair per process (src/core.jl:262-272)."""

    def __init__(self, L, src, dst, sample):
        import multiprocessing as mp
        from oracle import amg
        self.host_cores = len(os.sched_getaffinity(0))
        A0 = L.astype(np.float64).tocsr()
        A = A0.copy()
        A.data = A.data + np.finfo(np.float64).eps * np.linalg.norm(A.data)     # src/core.jl:161
        _CPU["A0"] = A0
        t0 = time.time()
        ml = amg.smoothed_aggregation(A)
        self.setup_s = time.time() - t0
        self.levels = [l.n for l in ml.levels]
        self.sample = min(sample, len(src), self.host_cores)
        _CPU.update(A=A, ml=ml, src=src, dst=dst)
        self.pool = mp.get_context("fork").Pool(self.sample, initializer=_cpu_init)

    def step(self, rtol=1e-6, count=None):
        count = self.sample if count is None else count
        t0 = time.time()
        out = self.pool.map(_cpu_one, [(i, rtol) for i in range(count)], chunksize=1)
        return time.time() - t0, [o[0] for o in out], [o[1] for o in out]

    def close(self):
        self.pool.close()
        self.pool.join()


def config_dict(args, L, npairs, world):
    n = int(L.shape[0])
    if args.config == "c2":
        name = "C2"
    elif n >= 9_000_000 and n <= 11_000_000:
        name = "10^7-node raster"
    elif (args.rows, args.cols) == (4000, 4000):
        name = "C4 raster"
    else:
        name = f"{n}-node raster (size override)"
    per = (f"{npairs} focal pairs sharded over {world} GPU(s)" if args.scaling == "strong"
           else f"{args.pairs} focal pairs per GPU")
    ws_gb = (L.nnz * 12 + L.nnz * 6 + 10 * n * 8 * 8) / 1e9      # CSR + fp32 operator copy + ~10 fp64 k = 8 panels
    l2 = (f"working set per iteration (operator {L.nnz * 12 / 1e9:.2f} GB + its fp32 copy + panels, ~{ws_gb:.1f} GB) "
          + ("exceeds the 126 MB L2" if ws_gb > 0.126 else "FITS the 126 MB L2: not an HBM measurement"))
    return {"workload": f"{name}: {args.rows}x{args.cols} synthetic raster (R~U[1,10] seed 42), 8-neighbour "
                        f"avg-conductance, {per}, {args.precision}",
            "n": int(L.shape[0]), "nnz": int(L.nnz), "pairs_total": int(npairs), "rtol": args.rtol,
            "preconditioner": args.precond, "parallelism": f"pair-shard x{world}",
            "l2_policy": l2}


def run_reference(args):
    """--impl reference: the reference's CPU CG+AMG path (oracle port; Julia is not in the image)
    on the same matrix, every step a bounded sample of the job's pairs, one pair per core."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    npairs = total_pairs(args, max(world, args.gpus))
    L, src, dst = workload(args, npairs)
    arm = CpuArm(L, src, dst, args.cpu_sample)
    t1, _, _ = arm.step()                                   # warm-up 1 (page-in, worker start)
    # a 10^7-node solve takes ~10 s per core: more warm-up only while the run stays inside the budget
    warm = 1
    while warm < args.warmup and (args.warmup - warm + args.steps) * t1 < args.ref_budget_s:
        arm.step(); warm += 1
    times, iters = [], None
    for _ in range(args.steps):
        t, R, iters = arm.step()
        times.append(t)
    arm.close()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"resistances": R})
    wall = float(np.mean(times))
    value = arm.sample / wall
    line = {
        "impl": "reference", "metric": "pair_solves_per_sec", "value": value, "unit": "pair-solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warm, "ms_per_step": wall * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args, L, npairs, max(world, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "pair-solves/s", "cores": arm.sample, "kind": "port",
                         "sample": f"{arm.sample} of {len(src)} pairs per step, one pair per process on "
                                   f"{arm.host_cores} host cores (SA-AMG + symmetric-GS PCG rtol 1e-6, oracle/amg.py; "
                                   f"AMG setup {arm.setup_s:.1f}s excluded, levels {arm.levels}; iterations {iters}); "
                                   f"warm-up requested {args.warmup}, bounded by --ref-budget-s"},
        "setup": {"amg_setup_s": arm.setup_s,
                  "setup_inclusive_pair_solves_per_s": arm.sample / (arm.setup_s + wall)},
        "e2e": {"value": value, "unit": "pair-solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_direct_leg(rows=1000, cols=1000, npairs=10):
    """CHOLMOD-like path (factor once + batched solves, src/core.jl:379,448-463,519-523) with SciPy
    SuperLU standing in for CHOLMOD, on the C2-size raster (the 10^7-node factorisation does not fit
    the time / memory of a bench run and is reported as skipped)."""
    import scipy.sparse as _sp
    import scipy.sparse.linalg as _spla
    from circuitscape_b200 import graph
    L, _ = graph.synthetic_raster_laplacian(rows, cols, seed=42)
    n = L.shape[0]
    nodes = graph.focal_nodes(n, 5, seed=7)
    src, dst = graph.all_pairs(nodes, limit=npairs)
    t0 = time.time()
    Md = (L.astype(np.float64) + 10 * np.finfo(np.float64).eps * _sp.identity(n)).tocsc()   # core.jl:521
    lu = _spla.splu(Md, permc_spec="MMD_AT_PLUS_A", diag_pivot_thresh=0.0, options=dict(SymmetricMode=True))
    tf = time.time() - t0
    rhs_d = np.zeros((n, len(src)))
    rhs_d[src, np.arange(len(src))] = -1.0
    rhs_d[dst, np.arange(len(src))] = 1.0
    t0 = time.time()
    Xd = lu.solve(rhs_d)
    tsv = time.time() - t0
    Rd = Xd[dst, np.arange(len(src))] - Xd[src, np.arange(len(src))]
    return {"kind": "port (SciPy SuperLU standing in for CHOLMOD)", "cores": 1, "raster": f"{rows}x{cols}",
            "factor_s": tf, "solve_s": tsv, "pairs": len(src),
            "pair_solves_per_s_incl_factor": len(src) / (tf + tsv),
            "pair_solves_per_s_excl_factor": len(src) / tsv, "R": [float(x) for x in Rd]}, (L, src, dst)


# ---------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import circuitscape_b200 as cb
    from circuitscape_b200 import dist as cdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback on the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if distributed:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist = None

    npairs = total_pairs(args, world)
    solver = cb.CUDASolver(precision=args.precision, device=local, rtol=args.rtol, precond=args.precond,
                           use_graph={"device": True, "chunk": "chunk", "plain": False}[args.loop],
                           setup=args.setup)
    t_asm = time.time()
    L = src = dst = None
    if rank == 0:
        L, src, dst = workload(args, npairs)
    t_asm = time.time() - t_asm
    # ---- replicate the operator: one NCCL broadcast of the CSR (SURVEY §8e), behind the C ABI:
    # torch.distributed only carries the 128-byte NCCL id and three integers between the ranks
    t0 = time.time()
    comm = None
    if distributed:
        def exchange(raw):
            t = torch.zeros(128, dtype=torch.uint8, device=dev)
            if raw is not None:
                t = torch.tensor(list(raw), dtype=torch.uint8, device=dev)
            dist.broadcast(t, src=0)
            return bytes(t.cpu().tolist())
        comm = cdist.Comm(local, rank, world, exchange)
        meta = torch.zeros(3, dtype=torch.int64, device=dev)
        if rank == 0:
            meta = torch.tensor([L.shape[0], L.nnz, npairs], dtype=torch.int64, device=dev)
        dist.broadcast(meta, src=0)
        n, nnz = int(meta[0]), int(meta[1])
        pairs = torch.zeros((2, npairs), dtype=torch.int64, device=dev)
        if rank == 0:
            pairs = torch.as_tensor(np.stack([src, dst]), device=dev)
        dist.broadcast(pairs, src=0)
        src, dst = pairs[0].cpu().numpy(), pairs[1].cpu().numpy()
        t0 = time.time()
        factor = comm.create_factor(L if rank == 0 else None, solver, shape=(n, nnz))
    else:
        n, nnz = L.shape[0], L.nnz
        factor = cb.construct_cholesky_factor(L, solver)
    torch.cuda.synchronize()
    setup_cold_s = time.time() - t0
    # the first create of a process also pays the one-time CUDA module load of the library; a job pays
    # that once however many connected components it factors (src/core.jl:148-168 loops over them),
    # so the per-component figure is the SECOND create of the same matrix
    warm = []
    for _ in range(2):          # two more creates of the same matrix: the steady per-component cost
        factor.close()
        if distributed:
            comm.barrier()
        t0 = time.time()
        factor = (comm.create_factor(L if rank == 0 else None, solver, shape=(n, nnz)) if distributed
                  else cb.construct_cholesky_factor(L, solver))
        torch.cuda.synchronize()
        warm.append(time.time() - t0)
    setup_s = min(warm)
    mine = cdist.shard_pairs(npairs, rank, world)
    msrc, mdst = src[mine], dst[mine]
    ext = torch.cuda.ExternalStream(factor.stream_ptr(), device=dev)

    def step():
        factor.reset_currents()
        out = factor.solve_pairs(msrc, mdst, accumulate=True)
        if distributed:                                   # end of the job: one gather, one reduction
            R = comm.gather_pairs(mine, out["R"], npairs)
            comm.reduce_currents(factor)
        else:
            R = out["R"]
        return R, out, factor.stats()

    def timed(fn, steps):
        if distributed:
            comm.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        t0 = time.time()
        res = [fn() for _ in range(steps)]
        e1.record(ext)
        torch.cuda.synchronize()
        wall = time.time() - t0
        ms = e0.elapsed_time(e1)
        if distributed:                                   # device time: max over ranks
            ms, wallms = comm.max([ms, wall * 1e3])
            wall = wallms / 1e3
        return ms, wall, res

    # clocks are sampled from the first warm-up step to the end of the timed region (the
    # timed region alone can be shorter than nvidia-smi's start-up + sampling period)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        step()
    t_w = time.time()
    while rank == 0 and sampler and len(sampler.lines) < 2 and time.time() - t_w < 3.0:
        factor.solve_pairs(msrc[:8], mdst[:8])    # local work only (no collective): load until samples arrive
    ms, wall, res = timed(step, args.steps)
    clocks = sampler.stop() if sampler else None
    R, out, st = res[-1]
    if args.dump_outputs and rank == 0:
        # what a caller of the step receives: every pair's resistance and the job's current maps
        # (cumulative and max over pairs, summed / maxed over ranks); iterations and residuals are in the JSON line
        cum, mx = factor.read_currents()
        dump_outputs(args.dump_outputs, {"resistances": R, "cum_current": cum, "max_current": mx})
    launches = sum(r[2]["kernel_launches"] for r in res)
    iters = out["iters"]
    value = npairs * args.steps / (ms / 1e3)
    it_all = None
    if distributed:
        t = torch.tensor([float(iters.sum()), float(iters.max()), float(len(iters))], dtype=torch.float64, device=dev)
        g = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(g, t)
        it_all = [[int(x) for x in gi.tolist()] for gi in g]

    # ---- e2e: plug-in hook #2 with host RHS / solution buffers, bs columns per call ----
    e2e = None
    if not args.skip_e2e:
        k = len(msrc)
        bs = max(1, min(args.bs, k))
        tdt = torch.float64 if factor.dtype == np.float64 else torch.float32
        # pinned host buffers, column-major n x bs (a Julia Matrix): torch (bs, n) row-major == (n, bs) F-order
        rhs = torch.zeros((bs, n), dtype=tdt).pin_memory().numpy().T
        lhs_buf = torch.zeros((bs, n), dtype=tdt).pin_memory().numpy().T
        h2d = d2h = 0

        def step_e2e():
            nonlocal h2d, d2h
            r = np.zeros(k)
            h2d = d2h = 0
            for c0 in range(0, k, bs):                          # src/core.jl:448-452 (batches of bs columns)
                c1 = min(k, c0 + bs)
                kk = c1 - c0
                cols = np.arange(kk)
                rhs[msrc[c0:c1], cols] = -1.0                    # src/core.jl:459-460
                rhs[mdst[c0:c1], cols] = 1.0
                lhs, _, _ = factor.solve_rhs(rhs[:, :kk], out=lhs_buf[:, :kk])          # hook #2
                r[c0:c1] = lhs[mdst[c0:c1], cols] - lhs[msrc[c0:c1], cols]             # core.jl:466-472, 486-492
                rhs[msrc[c0:c1], cols] = 0.0
                rhs[mdst[c0:c1], cols] = 0.0
                s_ = factor.stats()
                h2d += int(s_["h2d_bytes"]); d2h += int(s_["d2h_bytes"])
            if distributed:
                r = comm.gather_pairs(mine, r, npairs)
            return r

        rhs[:] = 0.0
        step_e2e()
        ms_e, wall_e, res_e = timed(step_e2e, args.steps)
        e2e_value = npairs * args.steps / max(wall_e, ms_e / 1e3)
        e2e = {"value": e2e_value, "unit": "pair-solves/s",
               "h2d_bytes_per_step": int(h2d) * world, "d2h_bytes_per_step": int(d2h) * world,
               "ms_per_step": wall_e * 1e3 / args.steps, "steps": args.steps,
               "through": f"solve_linear_system(factor, matrix, rhs::Matrix) in batches of {bs} columns with "
                          f"pinned host n x {bs} buffers"}
        assert np.abs(np.asarray(res_e[-1]) - np.asarray(R)).max() <= 1e-6 * np.abs(R).max()
        del rhs, lhs_buf

    # ---- roofline of the dominant kernel: instrumented repeat of one timed step ---
    peak, peak_src = peaks()
    roof = None
    extra = {}
    sv = 8 if args.precision == "double" else 4
    if rank == 0:
        kk = min(len(msrc), 16) // 8 * 8 or len(msrc)          # full k = 8 panels only: like-for-like bytes
        factor.profile_spmm(True)
        factor.reset_currents()
        factor.solve_pairs(msrc[:kk], mdst[:kk], accumulate=True)
        pbytes = factor.profile_bytes()
        pclasses = factor.profile_classes()
        pms, pl = factor.profile_spmm(False)
        avg_bytes = pbytes / max(pl, 1)
        achieved = pbytes / (pms * 1e-3) / 1e9
        traffic = None
        tnote = "no ncu --set full capture for this size"
        tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath)).get(f"finest_level_{args.rows}x{args.cols}")
            if tj:
                traffic = tj.get("traffic_bytes_per_launch")
                tnote = tj.get("note", "")
        t_full = time.time()
        factor.reset_currents()
        o2 = factor.solve_pairs(msrc[:kk], mdst[:kk], accumulate=True)
        t_full = (time.time() - t_full) * 1e3
        form = factor.operator_form()
        roof = {"bound": "hbm",
                "kernel": ("k_stencil (9-diagonal form)" if form == "stencil" else "k_spmm_win (windowed CSR records)")
                          + " on the finest-level operator, k = 8 panels, every epilogue of the AMG-PCG "
                          "iteration (fp64 CG SpMM / residual gate, fp32 residual + Jacobi sweep of the V-cycle)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_note": tnote, "peak_source": peak_src, "launches": int(pl),
                "avg_launch_ms": pms / max(pl, 1), "algorithmic_bytes_per_launch": avg_bytes,
                "spmm_share_of_step": pms / max(t_full, 1e-9),
                "by_kernel": {k: {"launches": c, "avg_ms": m / c, "GB/s": b / (m * 1e-3) / 1e9, "frac": b / (m * 1e-3) / 1e9 / peak}
                              for k, (m, b, c) in pclasses.items()},
                "note": "per-launch CUDA events on the solve stream in an instrumented repeat of the first "
                        f"{kk} pairs of the step (plain launches, same kernels as the graph); bytes = "
                        "nnz(s_v+4)+(n+1)4+panel passes summed per launch by the library (DESIGN.md section 4); "
                        "share = event time of those launches / wall time of the same pairs un-instrumented"}
        for kq in (1, 8):
            t_it = factor.bench_cg_iter(kq, reps=20)
            extra[f"pcg_iter_k{kq}_ms"] = t_it

    # ---- headline SpMV at 10^7 nodes ---------------------------------------------
    spmv = None
    if rank == 0 and not args.skip_spmv1e7:
        f7, own = factor, False
        n7, nnz7 = n, nnz
        if n < 9_000_000 or args.precision != "double":
            from circuitscape_b200 import graph
            factor.close()
            L7, _ = graph.synthetic_raster_laplacian(3163, 3163, seed=42)
            f7 = cb.construct_cholesky_factor(L7, cb.CUDASolver(device=local, precond="jacobi"))
            n7, nnz7, own = L7.shape[0], L7.nnz, True
            del L7
        form = f7.operator_form()
        spmv = {"n": n7, "nnz": nnz7, "peak": peak, "peak_source": peak_src, "dtype": "f64",
                "l2": "flushed (256 MB write) between repetitions", "operator_form": form,
                "note": "frac = CSR-algorithmic bytes (SURVEY.md 8d: nnz(s_v+4)+(n+1)4+2nk s_v) / time / peak; "
                        "actual = bytes the kernel's format really streams (stencil form: 9 n s_v values, no "
                        "column stream; windowed records: 10 B per entry) / time / peak"}
        for kq in (1, 8):
            t = f7.bench_spmm(kq, reps=20, flush_l2=True)
            b = b_spmm(n7, nnz7, kq, 8)
            actual = (9 * n7 * 8 if form == "stencil" else nnz7 * 10 + n7 * 10) + 2 * n7 * kq * 8
            spmv[f"k{kq}"] = {"ms": t, "algorithmic_bytes": b, "GB/s": b / (t * 1e-3) / 1e9,
                              "frac": b / (t * 1e-3) / 1e9 / peak, "actual_bytes": actual,
                              "actual_frac": actual / (t * 1e-3) / 1e9 / peak}
        if own:
            f7.close()

    # ---- CPU baseline + R parity (rank 0, N = 1 only) ------------------------------
    cpu = parity = None
    setup = {"assemble_s": t_asm, "create_s": setup_s, "create_first_in_process_s": setup_cold_s,
             "create_repeats_s": warm,
             "create_ms_device": st["setup_ms"],
             "setup_inclusive_pair_solves_per_s": npairs / (setup_s + ms / 1e3 / args.steps),
             "setup_inclusive_pair_solves_per_s_first_create": npairs / (setup_cold_s + ms / 1e3 / args.steps),
             "note": "create_s = wall time of construct_cholesky_factor (upload"
                     + (" on the root + NCCL broadcast of the CSR and of the aggregation seeds" if distributed else "")
                     + " + hierarchy + operator records), best of the second and third create of the process; create_first_in_process_s "
                     "adds the one-time CUDA module load of libcsb200.so; the rates are pairs_total / (create + one step)"}
    if rank == 0 and world == 1 and not args.skip_cpu:
        arm = CpuArm(L, src, dst, args.cpu_sample)
        arm.step(count=min(2, arm.sample))                      # page-in
        wall_c, Rc, itc = arm.step()
        ntight = min(3, arm.sample)
        _, Rt, itt = arm.step(rtol=-1e-10, count=ntight)        # exact: no regularisation, rtol 1e-10
        _, Rreg, _ = arm.step(rtol=1e-10, count=ntight)         # the regularised system, converged
        arm.close()
        cpu = {"value": arm.sample / wall_c, "unit": "pair-solves/s", "cores": arm.sample, "kind": "port",
               "sample": f"{arm.sample} of {len(src)} pairs, one pair per process on {arm.host_cores} host cores, "
                         f"SA-AMG(sym. GS, pinv coarse)-PCG rtol 1e-6 (oracle/amg.py; Julia absent); "
                         f"AMG setup {arm.setup_s:.1f}s excluded; {wall_c:.1f}s wall; iterations {itc}",
               "amg_setup_s": arm.setup_s,
               "setup_inclusive_pair_solves_per_s": arm.sample / (arm.setup_s + wall_c),
               "max_rel_dev_from_gpu_R": float(np.max(np.abs(np.array(Rc) - np.asarray(R)[:arm.sample])
                                                      / np.asarray(R)[:arm.sample]))}
        Rg = np.asarray(R)[:ntight]
        parity = {"max_rel_dev_of_R": float(np.max(np.abs(np.array(Rt) - Rg) / np.array(Rt))),
                  "pairs": ntight, "tolerance": 1e-6,
                  "oracle": f"CPU PCG (oracle/amg.py) on the Laplacian as assembled, rtol 1e-10, atol 0 ({itt} iterations) "
                            "= what the direct solvers (CHOLMOD + 10 eps I, src/core.jl:521) return",
                  "R_gpu": [float(x) for x in Rg], "R_oracle": [float(x) for x in Rt],
                  "vs_regularised_cg_amg": {
                      "max_rel_dev_of_R": float(np.max(np.abs(np.array(Rreg) - Rg) / np.array(Rreg))),
                      "R": [float(x) for x in Rreg],
                      "note": "the reference's cg+amg path first adds eps*norm(nzval) to EVERY stored entry "
                              "(src/core.jl:161): a leak of 9 eps ||nzval||_2 per node that grows like n^1.5 and "
                              "moves R by ~2e-6 at 10^7 nodes -- a property of that regularisation, not of either solver"}}
    if rank == 0 and world == 1 and not args.skip_direct:
        try:
            d, (Ld, sd, dd) = cpu_direct_leg()
            with cb.construct_cholesky_factor(Ld, cb.CUDASolver(device=local)) as fd:
                Rg = fd.solve_pairs(sd, dd)["R"]
            d["max_rel_dev_from_gpu_R"] = float(np.max(np.abs(np.array(d.pop("R")) - Rg) / Rg))
            if L.shape[0] > 2_000_000:
                d["at_bench_size"] = ("skipped: a supernodal factor of the 10^7-node stencil needs ~30 n log2 n "
                                      "= 7e9 entries (56 GB) and minutes of single-threaded SuperLU; the reference "
                                      "itself switches large jobs to cg+amg")
            extra["cpu_direct"] = d
        except Exception as exc:                                 # never let a side leg break the line
            extra["cpu_direct"] = {"error": repr(exc)}
    if rank == 0:
        line = {
            "metric": "pair_solves_per_sec", "value": value, "unit": "pair-solves/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f64" if args.precision == "double" else "f32", "data": "synthetic",
            "config": config_dict(args, L, npairs, world), "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu, "parity": parity,
            "setup": setup, "spmv_1e7": spmv,
            "detail": {"iterations_rank0": [int(x) for x in iters], "iterations_per_rank_sum_max_count": it_all,
                       "wall_s_timed_region": wall, "relres_max": float(out["relres"].max()),
                       "R_first": [float(x) for x in np.asarray(R)[:3]], **extra},
        }
        print(json.dumps(line), flush=True)
    if distributed:
        factor.close()
        comm.barrier()
        comm.close()
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
