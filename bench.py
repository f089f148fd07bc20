#!/usr/bin/env python
"""Headline benchmark: randsvd (K=200, p=10, q=2) of a matrix-free covariance operator.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c5|c5s|small|dense]
                    [--impl reference] [--generation table|arithmetic] [--dump-outputs DIR]

One "step" = one complete randsvd(A, K, p, q) of the workload (sketch GEMM, 2q power
products with pivot-faithful LU normalisation, final Householder QR, projection, TSQR +
Jacobi SVD, Z = V sqrt(S)).  Default workload c3 = BASELINE.json configs[2]: 3-D
64x56x56 = 200 704-point Gaussian covariance, single B200; with N > 1 the rows of the
operator and of every iterate are sharded over the ranks (strong scaling, same problem).
`--workload dense` is the same algorithm on a dense `A::Matrix` (32 768^2 exponential
covariance materialised in HBM, 8.6 GB) -- the TMA-fed dense DMMA GEMM of north_star
subsystem 1; its CPU arm runs the SAME matrix (same_config).

metric  = randsvd throughput in FP64 TFLOP/s, F = (2q+2)*2*n^2*(K+p) algorithmic flops
          (SURVEY.md §8d) / time of the step (factorisations are in the time, not in the
          numerator);  ms_per_step = randsvd time.
value   : Omega already resident in HBM, Z left in HBM.
e2e     : through the public API with HOST buffers -- Omega uploaded from pinned host
          memory and Z downloaded to pinned host memory inside the timed region.
dump    : `--dump-outputs DIR` writes what the last timed step returned: DIR/S.npy (the l singular
          values) and DIR/Z.npy (rows of Z, float64; all n rows when they fit in 64 MB, otherwise the
          rows `dump_rows(n, l)` picks, a fixed seeded sample in ascending order).  Omega and the
          operator are seeded, so two builds run with the same arguments can be compared file by file.
parity  : BEFORE the timed region, at every N, the reduced workload (17 472-point Gaussian,
          same K, p, q; dense: n = 4096) is factored row-sharded over the N ranks; rank 0 compares
          it with the CPU oracle (singular values, subspace sine, exact-zero tail) after the ranks
          have left the process group, so that no rank spins on a host core meanwhile;
          `sigma_head` are the first singular values of the TIMED workload, so that agreement
          across N is visible in the scaling run.
"""
import os
import sys

# The CPU arms (oracle on SciPy/OpenBLAS) must see the same BLAS thread count whatever launched
# this process: torch.distributed.run exports OMP_NUM_THREADS=1, which made the round-1 reference
# arm 5.6x slower at N >= 2 than at N = 1.  Pin before NumPy loads OpenBLAS.
def _usable_cpus():
    """Cores this process may really use: the affinity mask, capped by a cgroup CPU quota if one is set
    (a container can see more cores than it is allowed to run on; oversubscribing them with BLAS
    threads makes the CPU arm several times slower)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


_NCPU = _usable_cpus()
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ[_v] = str(_NCPU)

import argparse          # noqa: E402
import json              # noqa: E402
import subprocess        # noqa: E402
import threading         # noqa: E402
import time              # noqa: E402

import numpy as np       # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (kind, grid, ell, K, p, q, description)
    "c3": ("gaussian", (64, 56, 56), (9.0, 7.0, 5.0), 200, 10, 2,
           "BASELINE configs[2]: randsvd of matrix-free 200704-point (64x56x56) 3-D Gaussian covariance, K=200 p=10 q=2"),
    "c5": ("exponential", (1000, 1000), (120.0, 80.0), 200, 10, 2,
           "BASELINE configs[4]: row-sharded randsvd of matrix-free 10^6-point (1000x1000) exponential covariance, K=200 p=10 q=2"),
    "c5s": ("exponential", (512, 500), (60.0, 40.0), 200, 10, 2,
            "reduced configs[4]: 256000-point (512x500) exponential covariance, K=200 p=10 q=2"),
    "small": ("gaussian", (28, 26, 24), (9.0, 7.0, 5.0), 200, 10, 2,
              "reduced configs[2]: 17472-point (28x26x24) 3-D Gaussian covariance, K=200 p=10 q=2"),
    "dense": ("exponential", (256, 128), (30.0, 20.0), 200, 10, 2,
              "dense A::Matrix: 32768x32768 exponential covariance (256x128 grid) materialised in HBM (8.6 GB), K=200 p=10 q=2"),
}
# dense sample the CPU baseline / reference arm runs (a 200704^2 dense matrix is 322 GB)
CPU_SAMPLE = {"c3": (28, 26, 24), "small": (20, 18, 16), "c5": (132, 132), "c5s": (132, 132), "dense": (256, 128)}
# reduced workload of the pre-run parity check
PARITY_GRID = {"c3": (28, 26, 24), "small": (20, 18, 16), "c5": (132, 132), "c5s": (132, 132), "dense": (64, 64)}
KIND_ID = {"exponential": 0, "gaussian": 1, "powerlaw": 2}
DUMP_BYTES = 64_000_000        # what --dump-outputs may write in all, .npy headers included


def dump_rows(n, l):
    """Row indices of Z that --dump-outputs writes: every row if Z and S fit in DUMP_BYTES, else a
    sample drawn from a fixed seed, so that every run with the same n and l writes the same rows."""
    k = min(n, (DUMP_BYTES - 8 * l - 4096) // (8 * l))
    if k == n:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))


def grid_coords(shape):
    axes = [np.arange(s, dtype=np.float64) for s in shape]
    grids = np.meshgrid(*axes, indexing="ij")
    return np.stack([g.ravel(order="F") for g in grids], axis=0)


def randsvd_flops(n, l, q):
    return (2 * q + 2) * 2.0 * n * n * l


def blas_threads():
    """Threads the host BLAS will actually use (threadpoolctl), after raising the limit to all cores."""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=_NCPU, user_api="blas")
        info = [i for i in threadpool_info() if i.get("user_api") == "blas"]
        return max((i.get("num_threads", 1) for i in info), default=1)
    except Exception:
        return int(os.environ.get("OPENBLAS_NUM_THREADS", "1"))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_fp64_peak():
    """cuBLAS DGEMM 8192^3 best-of-5 (MEASURED_PEAKS.json carries no FP64 entry)."""
    import torch
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device="cuda")
    b = torch.randn(n, n, dtype=torch.float64, device="cuda")
    for _ in range(2):
        c = a @ b
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); c = a @ b; e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b, c
    torch.cuda.empty_cache()
    return 2 * n ** 3 / best * 1e-9


def dense_matrix(kind, grid, ell):
    """The dense workload's A: exponential covariance of a 2-D grid, built block-wise on the host."""
    import oracle          # checker-side helper used as the INPUT GENERATOR of the dense workload only
    coords = grid_coords(grid)
    return np.asfortranarray(oracle.kernel_cov_dense(KIND_ID[kind], coords, ell[:len(grid)]))


def cpu_oracle_run(workload, steps, warmup):
    """Times the oracle (reference algorithm restated on SciPy/OpenBLAS, all host cores) on a
    bounded dense sample of the workload (the dense workload: the full matrix, same config).
    Returns a dict for the JSON line."""
    import oracle
    kind, grid, ell, K, p, q, _ = WORKLOADS[workload]
    sgrid = CPU_SAMPLE[workload]
    threads = blas_threads()
    coords = grid_coords(sgrid)
    n = coords.shape[1]
    C = oracle.kernel_cov_dense(KIND_ID[kind], coords, ell[:len(sgrid)])
    Omega = np.random.default_rng(0).standard_normal((n, K + p))
    for _ in range(warmup):
        oracle.randsvd(C, Omega, K, p, q)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.randsvd(C, Omega, K, p, q)
    dt = (time.perf_counter() - t0) / steps
    same = tuple(sgrid) == tuple(grid)
    sample = (f"dense n={n} ({'x'.join(map(str, sgrid))} grid, {kind}) oracle randsvd K={K} p={p} q={q}; "
              + ("the full workload (same config)" if same else
                 "flops-normalised (the full-size dense matrix cannot be materialised)"))
    return {"value": randsvd_flops(n, K + p, q) / dt * 1e-12, "unit": "TFLOP/s", "cores": _NCPU, "threads": threads,
            "kind": "port", "sample": sample, "ms_per_step_sample": dt * 1e3, "same_config": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="gsi", choices=["gsi", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip extra.arith_tflops and (N = 8) extra.c5")
    ap.add_argument("--generation", default="table", choices=["table", "arithmetic"],
                    help="kernel values: lattice-table look-up (structured grid) or exp/sqrt arithmetic from coordinates")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write Z (rows, see dump_rows) and S of the last timed step as DIR/Z.npy, DIR/S.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    kind, grid, ell, K, p, q, desc = WORKLOADS[args.workload]
    l = K + p
    dense = args.workload == "dense"

    if args.impl == "reference":
        # The reference (pure Julia) cannot run here: its CPU algorithm restated on
        # SciPy/OpenBLAS is timed on the host cores; rank 0 only, same thread count at every N.
        if args.dump_outputs:
            ap.error("--dump-outputs needs the CUDA path (--impl gsi)")
        if rank != 0:
            return
        steps = args.steps
        cb = cpu_oracle_run(args.workload, steps, 1)
        print(json.dumps({
            "impl": "reference", "metric": "randsvd_fp64_tflops", "value": cb["value"], "unit": "TFLOP/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": cb["ms_per_step_sample"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": desc, "sample": cb["sample"]},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "TFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }))
        return

    import torch
    import gsi_b200 as gsi
    torch.cuda.set_device(local_rank)
    dist = None
    uid = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        t = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            t = torch.tensor(list(gsi.Context.unique_id()), dtype=torch.uint8, device="cuda")
        dist.broadcast(t, 0)
        uid = bytes(t.cpu().tolist())
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"

    peak = measured_fp64_peak() if rank == 0 else None

    ctx = gsi.Context(local_rank, rank, world, uid)
    gsi.set_default_context(ctx)

    def make_operator(kind_, grid_, ell_, dense_=False, generation="table"):
        n_ = int(np.prod(grid_))
        r0_, ml_ = gsi.partition_rows(n_, world, rank)
        if dense_:
            A = dense_matrix(kind_, grid_, ell_)
            return gsi.DenseMatrix(A[r0_:r0_ + ml_], ctx=ctx, row0=r0_, m_global=n_), n_, r0_, ml_
        if generation == "table":
            return gsi.GridKernelCovMatrix(kind_, grid_, ell_, ctx=ctx, row0=r0_, mloc=ml_), n_, r0_, ml_
        return gsi.KernelCovMatrix(kind_, grid_coords(grid_), ell_, ctx=ctx, row0=r0_, mloc=ml_), n_, r0_, ml_

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ------------------------------------------------------------------ parity evidence, before timing
    parity, parity_job = None, None
    if not args.no_parity:
        pgrid = PARITY_GRID[args.workload]
        pell = ell[:len(pgrid)]
        opp, pn, _, _ = make_operator(kind, pgrid, pell, dense, args.generation)
        pl = min(l, pn // 2)
        pK = pl - p
        Om = np.random.default_rng(0).standard_normal((pn, pl))
        Zp = gsi.randsvd(opp, pK, p, q, Omega=Om, full=True)          # gathered on every rank
        opp.free()
        parity_job = (Zp, Om, pgrid, pell, pn, pK) if rank == 0 else None     # compared with the oracle at the end
        del Zp
        barrier()

    # ------------------------------------------------------------------ the timed workload
    op, n, row0, mloc = make_operator(kind, grid, ell, dense, args.generation)

    # host-seeded Omega in pinned memory (the reference draws randn(n, l) on the host)
    omega_pinned = torch.empty((l, n), dtype=torch.float64, pin_memory=True)      # (l, n) C-order == (n, l) F-order
    Omega_h = omega_pinned.numpy().T
    Omega_h[...] = np.random.default_rng(0).standard_normal((n, l))
    zrows = n if dense else mloc            # a dense operator returns the replicated Z (its A'Q is all-reduced)
    z_pinned = torch.empty((l, zrows), dtype=torch.float64, pin_memory=True)
    Z_h = z_pinned.numpy().T
    Omega_d = gsi.DeviceMatrix.from_host(ctx, Omega_h)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local_rank))
    sigma_head = []
    last = {}                   # Z (on the device) and S of the latest step_resident, for --dump-outputs

    def step_resident():
        if last:
            last.pop("Z").free()        # back to the library's pool before this step allocates its Z
        Z, S = gsi.randsvd(op, K, p, q, Omega=Omega_d, device_out=True, return_singular_values=True)
        sigma_head[:] = [float(s) for s in S[:5]]
        last.update(Z=Z, S=S)

    def step_e2e():
        Z = gsi.randsvd(op, K, p, q, Omega=Omega_h, device_out=True)     # uploads Omega from pinned host memory
        Z.numpy(out=Z_h)                                                 # downloads this rank's rows of Z
        Z.free()

    def timed(fn, steps, with_timing):
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        ctx.launch_count(reset=True)
        if with_timing:
            ctx.gemm_timing(enable=True)
            ctx.phase_timing(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ctx.launch_count()
        gemm = ctx.gemm_timing(enable=False) if with_timing else None
        phases = ctx.phase_timing() if with_timing else None
        clocks = sampler.stop() if rank == 0 else None
        if dist is not None:
            tt = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
            lt = torch.tensor([launches], dtype=torch.float64, device="cuda")
            dist.all_reduce(lt, op=dist.ReduceOp.SUM)
            launches = int(lt.item())
        return ms, launches, gemm, clocks, phases

    for _ in range(args.warmup):
        step_resident()
    ms, launches, gemm, clocks, phases = timed(step_resident, args.steps, True)
    if args.dump_outputs:
        # each rank holds the rows of its own block of Z (a dense operator's Z is replicated): gather the sample on rank 0
        rows = dump_rows(n, l)
        z0 = 0 if dense else row0
        mine = rows[(rows >= z0) & (rows < z0 + zrows)]
        Zs = last["Z"].numpy()[mine - z0]
        if dist is not None and not dense:
            parts = [None] * world if rank == 0 else None
            dist.gather_object(Zs, parts, dst=0)
            Zs = np.concatenate(parts) if rank == 0 else None
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "Z.npy"), Zs)
            np.save(os.path.join(args.dump_outputs, "S.npy"), last["S"])
    last.pop("Z").free()
    ms_per_step = ms / args.steps
    F = randsvd_flops(n, l, q)
    value = F / (ms_per_step * 1e-3) * 1e-12

    e2e = None
    if not args.no_e2e:
        step_e2e()
        ms2, _, _, _, _ = timed(step_e2e, args.steps, False)
        e2e_ms = ms2 / args.steps
        e2e = {"value": F / (e2e_ms * 1e-3) * 1e-12, "unit": "TFLOP/s", "ms_per_step": e2e_ms,
               "h2d_bytes_per_step": int(world * n * l * 8), "d2h_bytes_per_step": int(world * zrows * l * 8)}

    # ------------------------------------------------------------------ extras (outside the timed regions)
    extra = {}

    def product_tflops(opx, nx, trans, reps=3):
        """CUDA-event time of `reps` single operator products on the library stream."""
        X = gsi.DeviceMatrix.from_host(ctx, np.random.default_rng(1).standard_normal((nx, l)))
        opx.apply(X, trans=trans).free()
        barrier()
        ctx.gemm_timing(enable=True)
        for _ in range(reps):
            opx.apply(X, trans=trans).free()
        barrier()
        g_ms, g_n, g_fl = ctx.gemm_timing(enable=False)
        X.free()
        return (g_fl / (g_ms * 1e-3) * 1e-12, g_ms / max(g_n, 1)) if g_ms > 0 else (None, None)

    if not args.no_extras:
        if dense:
            # the two variants of the dense DMMA GEMM separately: A*X (UTMALDG tiles of A) and A'*X
            for nm, tr in (("dense_n", False), ("dense_t", True)):
                tf, lms = product_tflops(op, n, tr)
                if rank == 0:
                    extra[nm] = {"tflops_per_gpu": tf, "ms_per_launch": lms,
                                 "algorithmic_bytes": 8.0 * mloc * n + 16.0 * n * l,
                                 "hbm_gbs_algorithmic": (8.0 * mloc * n + 16.0 * n * l) / (lms * 1e-3) * 1e-9 if lms else None}
        elif args.generation == "table":
            # the coordinate-based (arithmetic exp/sqrt) generation path of the same operator
            opa, _, _, _ = make_operator(kind, grid, ell, False, "arithmetic")
            tf, lms = product_tflops(opa, n, False, reps=2)
            opa.free()
            if rank == 0:
                extra["arith_tflops"] = {"tflops_per_gpu": tf, "ms_per_launch": lms,
                                         "what": "one product launch of KernelCovMatrix (kernel values by exp/sqrt "
                                                 "arithmetic from coordinates) on the same workload"}
        if world == 8 and args.workload == "c3":
            # the north-star configuration on the driver's box: 1 warm + 2 timed steps of the 10^6-point case
            kind5, grid5, ell5, K5, p5, q5, desc5 = WORKLOADS["c5"]
            op5, n5, _, _ = make_operator(kind5, grid5, ell5)
            Om5 = gsi.DeviceMatrix.from_host(ctx, np.random.default_rng(0).standard_normal((n5, K5 + p5)))

            def step5():
                gsi.randsvd(op5, K5, p5, q5, Omega=Om5, device_out=True).free()
            step5()
            ms5, _, gemm5, _, ph5 = timed(step5, 2, True)
            op5.free(); Om5.free()
            if rank == 0:
                F5 = randsvd_flops(n5, K5 + p5, q5)
                v5 = F5 / (ms5 / 2 * 1e-3) * 1e-12
                extra["c5"] = {"workload": desc5, "steps": 2, "warmup": 1, "ms_per_step": ms5 / 2, "tflops": v5,
                               "frac_of_peak_per_gpu": v5 / world / peak,
                               "product_tflops_per_gpu": gemm5[2] / (gemm5[0] * 1e-3) * 1e-12 if gemm5[0] > 0 else None,
                               "phase_ms_per_step": {k: v / 2 for k, v in ph5.items()}}

    # k-sweep schedule of the product kernel (gsi_ctx_set_option / GSI_SWEEP): groups,div,hint,window,epoch_shift
    schedule = ",".join(str(ctx.get_option(k)) for k in ("kcov.sweep_groups", "kcov.sweep_div", "kcov.l2_hint",
                                                         "kcov.window", "kcov.epoch_shift"))
    if rank == 0:
        gemm_ms, gemm_launches, gemm_flops = gemm
        traffic, traffic_source = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
                tj = json.load(f)
            key = args.workload
            if (world == 1 and args.generation == "table" and key in tj
                    and (dense or tj[key].get("schedule") == schedule)):
                traffic = tj[key]["bytes_per_launch"]
                traffic_source = ("NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one launch "
                                  "from the committed ncu capture " + tj[key].get("source", "profiles/traffic.json"))
        except Exception:
            traffic = None
        ach = gemm_flops / (gemm_ms * 1e-3) * 1e-12 if gemm_ms > 0 else None
        kname = ("dense_gemm_kernel (dense A x tall-skinny, A tiles by tiled TMA, DMMA.8x8x4)" if dense else
                 "kcov_gemm_kernel (matrix-free covariance x tall-skinny, DMMA.8x8x4)")
        roof = {"bound": "tensor", "kernel": kname,
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": (ach / peak) if ach else None,
                "traffic": traffic, "traffic_source": traffic_source,
                "peak_source": "builder-measured: cuBLAS DGEMM 8192^3 (torch.matmul fp64) best of 5 in this run; "
                               "MEASURED_PEAKS.json has no FP64 entry",
                "avg_launch_ms": gemm_ms / max(gemm_launches, 1), "launches_timed": gemm_launches,
                "algorithmic_flops_per_launch": gemm_flops / max(gemm_launches, 1),
                "gemm_share_of_step": gemm_ms / ms}
        cfg = {"workload": desc, "n": n, "K": K, "p": p, "q": q, "kernel": kind, "ell": list(ell),
               "normaliser": "LU_REF", "parallelism": f"row-shard x{world}",
               "l2": "operand streams (X 366 MB/pass) exceed L2; no flush needed" if not dense else
                     "A (8.6 GB) exceeds L2; no flush needed",
               "lu_panel": ctx.get_option("lu.panel"), "qr_panel": ctx.get_option("qr.panel"),
               "svd_fused": ctx.get_option("svd.fused")}
        if not dense:
            cfg["kernel_values"] = ("lattice table look-up (structured grid, n distinct values)"
                                    if args.generation == "table" else "exp/sqrt arithmetic from coordinates")
            cfg["kcov_schedule"] = schedule
        out = {"metric": "randsvd_fp64_tflops", "value": value, "unit": "TFLOP/s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
               "config": cfg, "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roof,
               "phase_ms_per_step": {k: v / args.steps for k, v in phases.items()},
               "parity": parity, "sigma_head": sigma_head, "extra": extra}
    # All collective work is done: the ranks leave the process group NOW, so that nothing spins on a host
    # core while rank 0 times the CPU baseline (ranks waiting in an NCCL barrier busy-wait, and OpenBLAS's
    # spinning worker threads then fight them for cores: measured 0.11 / 0.07 TF/s at N = 2 / 8 against
    # 0.40 at N = 1 on the same kind of box before this ordering).
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        if world > 1:
            time.sleep(2.0)               # let the other ranks exit
        if parity_job is not None:
            # the reduced workload was factored on the GPUs BEFORE the timed region; its CPU check runs here
            import oracle                                                # checker
            Zp, Om, pgrid, pell, pn, pK = parity_job
            Cd = oracle.kernel_cov_dense(KIND_ID[kind], grid_coords(pgrid), pell)
            c = oracle.compare_Z(Zp, oracle.randsvd(Cd, Om, pK, p, q), pK)
            out["parity"] = {"sv_rel": c["sv_rel"], "sine": c["sine"], "tail_zero": c["tail_zero"], "n_ranks": world,
                             "workload": f"{'x'.join(map(str, pgrid))} {kind}, n={pn}, K={pK} p={p} q={q}, factored row-sharded "
                                         f"over {world} rank(s) before the timed region, vs oracle.randsvd on the dense "
                                         f"matrix (same Omega)",
                             "ok": bool(c["tail_zero"] and c["sv_rel"] < 1e-10 and c["sine"] < 1e-8)}
            del Cd
        if not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_oracle_run(args.workload, 1, 1)
        print(json.dumps(out))


if __name__ == "__main__":
    main()
