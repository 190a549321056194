#!/usr/bin/env python
"""bench.py -- ALS user+item row-updates/sec at f=64 (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C2] [--scale S]
                    [--dump-outputs DIR]

A "step" is one ALS iteration of the hot path (user half + item half, each = Gramian + fused
per-row Cholesky solve [+ factor all-gather at N > 1]) over the synthetic last.fm-shaped matrix C2
(360k x 300k, 17M nnz power law, factors=64, Cholesky, lambda=0.01; SURVEY.md section 8(d) generator).
`value` = (users + items) * K / device time of K iterations with everything resident in HBM;
`e2e` = the same metric through the public API with HOST inputs: AlternatingLeastSquares.fit(csr) for
3 iterations from pinned host CSR arrays (H2D), device transpose, and the factors read back (D2H).

One process per GPU (torchrun-compatible env: RANK / LOCAL_RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT);
rank 0 prints exactly one JSON line.  --impl reference times the reference's own Cython/OpenMP CPU
path (oracle/_ref when it was built where /root/reference exists, else the C restatement) on a
bounded row sample of the same workload, on rank 0 only.
--dump-outputs DIR writes what the timed path computed in its last step as DIR/<name>.npy (see dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "ALS user+item row-updates/sec at f=64"
UNIT = "row-updates/s"
E2E_ITERS = 3
DUMP_BYTES = 60_000_000  # what --dump-outputs may write in all: under 64 MB with the .npy headers


def metric_name(cfg):
    return f"ALS user+item row-updates/sec at f={cfg['factors']}" + (" (CG, 3 steps)" if cfg["use_cg"] else "")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--config", default="C2")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink rows/cols/nnz together (debugging only)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU-baseline sample duration")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--trace-e2e", action="store_true", help="cProfile of the last end-to-end fit, to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")
    return args


# --------------------------------------------------------------------------------------- helpers
def algorithmic_bytes_half(nnz, rows, n_other, f):
    """SURVEY.md 8(d): compulsory bytes of one Cholesky half: index + value + gathered row per nonzero,
    indptr + written row per solved row; the Gramian read of the other side is its own kernel."""
    solve = nnz * (4 + 4 + 4 * f) + rows * 4 + rows * 4 * f
    gram = n_other * 4 * f + 4 * f * f
    return solve, gram


def ncu_traffic(kernel, scale, world):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, averaged over the
    two halves, from the committed ncu capture of this same workload (profiles/ncu_traffic.json, written by
    tools/ncu_traffic.py).  None when no capture matches the run (other scale / sharded run)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if scale != 1.0 or world != 1 or not os.path.exists(path):
        return None
    with open(path) as fh:
        return json.load(fh).get(kernel, {}).get("bytes_per_launch")


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe): `nvidia-smi -lms 100`, plus -- the
    timed region of a multi-GPU step is shorter than nvidia-smi's start-up and sampling period -- an in-process NVML
    poll every 10 ms (nvidia-ml-py; best effort: any failure leaves the nvidia-smi samples as the only source)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NVML_REASONS = (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                    ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                    ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                    ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap", 0x4))

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.nvml, self.nvml_samples, self.nvml_stop, self.nvml_thread = None, [], threading.Event(), None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nvml = (pynvml, pynvml.nvmlDeviceGetHandleByIndex(int(self.index)))
            self.nvml_thread = threading.Thread(target=self._poll, daemon=True)
            self.nvml_thread.start()
        except Exception:  # noqa: BLE001  (no NVML binding / no permission: nvidia-smi below is the recipe's source anyway)
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml
        while not self.nvml_stop.is_set():
            try:
                self.nvml_samples.append((int(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                          int(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)),
                                          int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
            except Exception:  # noqa: BLE001
                return
            time.sleep(0.010)

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        self.nvml_stop.set()
        if self.proc is None and not self.nvml_samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        n_smi = len(sm)
        try:
            nv = self.nvml[0] if self.nvml else None
            for c, m, bits in list(self.nvml_samples):
                sm.append(float(c))
                mx.append(float(m))
                for name, attr, default in self.NVML_REASONS:
                    if bits & int(getattr(nv, attr, default)):
                        reasons.add(name)
        except Exception:  # noqa: BLE001
            pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_nvidia_smi": n_smi, "reasons": sorted(reasons)}


def dump_outputs(path, arrays):
    """Writes each 2-D float32 / float64 array as <path>/<name>.npy.  An array above its share of DUMP_BYTES keeps a
    sample of its rows drawn with a fixed seed, in row order: runs with the same arguments write the same rows."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def pinned_csr(Cui):
    """Copy of a scipy CSR whose three arrays live in page-locked host memory."""
    import scipy.sparse as sp

    from implicit_b200 import _lib

    data = _lib.pinned_empty(Cui.data.shape, np.float32)
    indices = _lib.pinned_empty(Cui.indices.shape, np.int32)
    indptr = _lib.pinned_empty(Cui.indptr.shape, np.int32)
    data[:], indices[:], indptr[:] = Cui.data, Cui.indices, Cui.indptr
    return sp.csr_matrix((data, indices, indptr), shape=Cui.shape, copy=False)


# --------------------------------------------------------------------------------------- CPU reference
def cpu_reference_rate(Cui, X0, Y0, cfg, seconds, kind="auto"):
    """Times the reference's CPU Cholesky/CG half on a bounded ROW SAMPLE of the workload (all host
    threads, OPENBLAS_NUM_THREADS=1 as implicit/utils.py:18-62 asks).  Per-row cost depends only on the
    row's nonzeros, so a uniform row sample scales linearly to the whole iteration."""
    import oracle

    impl = oracle.get(kind)
    users, items = Cui.shape
    Ciu = Cui.T.tocsr()
    rng = np.random.default_rng(0)
    def solver(C, X, Y, nt):
        if cfg["use_cg"]:
            impl.least_squares_cg(C, X, Y, 0.01, num_threads=nt, cg_steps=3)
        else:
            impl.least_squares(C, X, Y, 0.01, num_threads=nt)

    def run(frac, nt):
        nu, ni = max(64, int(users * frac)), max(64, int(items * frac))
        su = np.sort(rng.choice(users, min(users, nu), replace=False))
        si = np.sort(rng.choice(items, min(items, ni), replace=False))
        Cu, Ci = Cui[su], Ciu[si]
        Xs, Ys = X0[su].copy(), Y0[si].copy()
        t = time.perf_counter()
        solver(Cu, Xs, Y0, nt)
        solver(Ci, Ys, X0, nt)
        return len(su) + len(si), time.perf_counter() - t, Cu.nnz + Ci.nnz

    # give the reference its best thread count: on many-core hosts its dynamic-chunk-8 OpenMP loop over
    # tiny BLAS calls can run slower with every hardware thread than with fewer
    ncpu = os.cpu_count() or 1
    cands = sorted({n for n in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8) if 1 <= n <= ncpu}, reverse=True)
    run(0.001, ncpu)  # warm the OpenMP pool
    best_nt, best_rate, t_best = ncpu, 0.0, 1.0
    for nt in cands:
        rows, t, _ = run(0.01, nt)
        if rows / t > best_rate:
            best_nt, best_rate, t_best = nt, rows / t, t
    frac = min(1.0, max(0.01, 0.01 * seconds / max(t_best, 1e-3)))
    rows, t, nnz = run(frac, best_nt)
    return {"value": rows / t, "unit": UNIT, "cores": best_nt, "host_cpus": ncpu,
            "kind": "reference" if impl.name == "ref" else "port",
            "sample": f"uniform {frac:.3%} row sample of both halves ({rows} rows, {nnz} nnz, {t:.1f} s), "
                      f"{'CG(3)' if cfg['use_cg'] else 'Cholesky'} f={cfg['factors']}, best of num_threads in {cands}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from implicit_b200 import synthetic

    ref_scale = args.scale * (0.02 if args.config == "C4" else 1.0)  # C4: a 1/50 instance of the same recipe on the host
    Cui, X0, Y0, cfg = synthetic.config(args.config, scale=ref_scale)
    rates = []
    for _ in range(args.warmup):
        cpu_reference_rate(Cui, X0, Y0, cfg, seconds=1.0)
    per_step = max(1.0, min(args.cpu_seconds, 150.0 / max(args.steps, 1)))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r = cpu_reference_rate(Cui, X0, Y0, cfg, seconds=per_step)
        rates.append(r)
    wall = time.perf_counter() - t0
    value = float(np.mean([r["value"] for r in rates]))
    base = dict(rates[-1], value=value)
    out = {
        "impl": "reference", "metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * (cfg["users"] + cfg["items"]) / value, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args, 1), "cpu_baseline": base,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": wall,
    }
    print(json.dumps(out))


def workload_config(cfg, args, world):
    return {"workload": f"{args.config}: synthetic power-law CSR {cfg['users']}x{cfg['items']}, {cfg['nnz']} nnz, "
                        f"factors={cfg['factors']}, {'CG(3)' if cfg['use_cg'] else 'Cholesky'}, lambda=0.01, seed={cfg['seed']}",
            "scale": args.scale, "l2": "inputs_exceed_l2 (CSR + factors > 126 MB)" if cfg["nnz"] * 8 > 126e6 else "l2_flush",
            "parallelism": (f"row-sharded dp{world}, solved rows mirrored to peer replicas over NVLink by the solve kernel"
                            if world > 1 else "single GPU"),
            "e2e_step": f"fit(host CSR) x {E2E_ITERS} iterations + factors read back"}


# --------------------------------------------------------------------------------------- our arm
def run_ours(args):
    from implicit_b200 import AlternatingLeastSquares, _lib, synthetic
    from implicit_b200.distributed import init_process_group
    from implicit_b200.utils import nnz_balanced_splits

    pg = init_process_group()
    rank, world, ctx = pg.rank, pg.world, pg.ctx
    on_device = args.config == "C4"  # 10M x 1M, 500M nnz: generated on the device (csrc/gen.cu), identically on every rank
    if on_device:
        cfg = dict(synthetic.CONFIGS["C4"])
        cfg.update(users=max(8, int(cfg["users"] * args.scale)), items=max(8, int(cfg["items"] * args.scale)),
                   nnz=max(8, int(cfg["nnz"] * args.scale)))
        Cui_host = X0 = Y0 = None
    else:
        Cui_host, X0, Y0, cfg = synthetic.config(args.config, scale=args.scale)
    users, items, f = cfg["users"], cfg["items"], cfg["factors"]
    use_cg = cfg["use_cg"]
    reg = 0.01

    def initial_factors_on_device():
        if on_device:
            A, B = _lib.DeviceFactors(ctx, users, f), _lib.DeviceFactors(ctx, items, f)
            A.fill_uniform(42, 0.01)   # the distribution of implicit/cpu/als.py:144-147, hashed instead of PCG64
            B.fill_uniform(43, 0.01)
            return A, B
        return _lib.DeviceFactors.from_host(ctx, X0), _lib.DeviceFactors.from_host(ctx, Y0)

    # ---- device-resident arm
    if on_device:
        Cui = _lib.DeviceCSR.generate(ctx, users, items, cfg["nnz"], cfg["seed"])
        cfg["nnz"] = int(Cui.shape3[2])
    else:
        Cui = _lib.DeviceCSR.upload(ctx, Cui_host)
    Ciu = Cui.transpose()
    X, Y = initial_factors_on_device()
    Cui_s, Ciu_s, usplit, isplit = Cui, Ciu, None, None
    p2p = world > 1 and os.environ.get("ALS_B200_NO_P2P") != "1"
    if world > 1:
        row_cost = 20 if use_cg else 60
        usplit = nnz_balanced_splits(Cui.indptr_host() if on_device else Cui_host.indptr, world, row_cost)
        isplit = nnz_balanced_splits(Ciu.indptr_host(), world, row_cost)
        Cui_s = Cui.slice_rows(usplit[rank], usplit[rank + 1])
        Ciu_s = Ciu.slice_rows(isplit[rank], isplit[rank + 1])
        if p2p:  # fused exchange: solved rows are stored into the peers' replicas by the solve kernel itself
            ctx.attach_peers(X)
            ctx.attach_peers(Y)
            _lib.gramian_shard(ctx, Y, isplit[rank], isplit[rank + 1] - isplit[rank])

    def half(C, A, B, split):
        if split is not None and p2p:
            # device-resident all-reduced Gramian; rows mirrored into the peers by the kernel; the all-reduce
            # of the next Gramian (over the rows just solved) orders the next half after every peer's stores
            _lib.half_pregram_async(ctx, C, A, B, reg, use_cg, 3)  # no host round trip: the halves queue back to back
            _lib.gramian_shard(ctx, A, split[rank], split[rank + 1] - split[rank])
            return
        if use_cg:
            _lib.least_squares_cg(ctx, C, A, B, reg, 3)
        else:
            _lib.least_squares(ctx, C, A, B, reg)
        if split is not None:
            ctx.allgather_rows(A, split)

    def iteration():
        half(Cui_s, X, Y, usplit)
        half(Ciu_s, Y, X, isplit)

    flush = cfg["nnz"] * 8 <= 126e6  # small debug scales fit in L2: flush it between iterations
    scaling = "weak" if on_device else "strong"  # C4 is the configuration sized for 8 GPUs; C2 / C3 are fixed problems
    for _ in range(max(args.warmup, 3)):
        iteration()
    ctx.sync()
    if world > 1:
        pg.barrier()
    sampler = ClockSampler(ctx.device)
    sampler.start()
    ctx.profile(True)
    ctx.profile_read()
    launches0 = ctx.launch_count()
    ctx.sync()
    if world > 1:
        pg.barrier()
    ctx.timer_start()
    for _ in range(args.steps):
        if flush:
            ctx.flush_l2()
        iteration()
    ms = ctx.timer_stop()
    ctx.sync()
    if world > 1:
        if p2p and not use_cg:
            _lib.solver_status(ctx)  # any non-PD row in the timed halves raises here
        pg.barrier()
    clocks = sampler.stop()
    prof = ctx.profile_read()
    ctx.profile(False)
    launches = ctx.launch_count() - launches0
    if args.dump_outputs and rank == 0:  # every rank holds both factor matrices whole
        dump_outputs(args.dump_outputs, {"user_factors": X.download(), "item_factors": Y.download()})
    ms_max = pg.allreduce_max(ms) if world > 1 else ms
    value = (users + items) * args.steps / (ms_max * 1e-3)

    # ---- N > 1: the sharded result against a single-GPU run of the same iterations (rank 0 holds full replicas
    #      and the whole CSR): every row of both factor matrices, so the scaling line is a checked result
    parity_vs_n1 = None
    if world > 1:
        total_iters = max(args.warmup, 3) + args.steps
        xs, ys = X.download(), Y.download()
        if rank == 0:
            X1, Y1 = initial_factors_on_device()
            for _ in range(total_iters):
                if use_cg:
                    _lib.least_squares_cg(ctx, Cui, X1, Y1, reg, 3)
                    _lib.least_squares_cg(ctx, Ciu, Y1, X1, reg, 3)
                else:
                    _lib.least_squares(ctx, Cui, X1, Y1, reg)
                    _lib.least_squares(ctx, Ciu, Y1, X1, reg)
            x1, y1 = X1.download(), Y1.download()
            X1.close()
            Y1.close()

            def rerr(a, b):
                a, b = a.astype(np.float64), b.astype(np.float64)
                den = np.linalg.norm(b, axis=1)
                return np.linalg.norm(a - b, axis=1) / np.maximum(den, 0.01 * np.median(den))

            e = np.concatenate([rerr(xs, x1), rerr(ys, y1)])
            parity_vs_n1 = {"iterations": total_iters, "rows": int(len(e)), "row_err_max": float(e.max()),
                            "row_err_median": float(np.median(e)), "row_err_p999": float(np.quantile(e, 0.999)),
                            "what": "||sharded - single GPU||_2 / ||single GPU||_2 per factor row, all rows of X and Y"}
        pg.barrier()

    # roofline of the dominant kernel (this rank's shard): algorithmic bytes / measured kernel time
    ru, _, nu = Cui_s.shape3
    ri, _, ni = Ciu_s.shape3
    su, gu = algorithmic_bytes_half(nu, ru, items, f)
    si, gi = algorithmic_bytes_half(ni, ri, users, f)
    main_kernel = "cg" if use_cg else "cholesky"
    aux = "cg_giant" if use_cg else "cholesky_finish"
    k_ms = prof[main_kernel][0] + prof[aux][0]
    k_n = prof[main_kernel][1]
    extra = (ru + ri) * 4 * f if use_cg else 0  # CG also reads the warm start
    bytes_per_launch = (su + si + extra) / 2.0
    peak, peak_src = measured_peak_gbs()
    achieved = (bytes_per_launch * k_n) / (k_ms * 1e-3) / 1e9 if k_ms > 0 else None
    roofline = {"bound": "hbm", "kernel": ("cholesky half: cholesky_half_kernel (rows > 48 nnz) + short_batch_kernel<4,{48..8}> + tcgen05 whitening + giant-row pass"
                           if not use_cg else "cg_rows_kernel (+ giant-row passes)"), "achieved": achieved,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak if achieved else None,
                "traffic": ncu_traffic(main_kernel, args.scale, world), "algorithmic_bytes_per_launch": bytes_per_launch,
                "avg_launch_ms": k_ms / k_n if k_n else None,
                "kernel_share_of_step": k_ms / ms if ms else None,
                "gramian_ms_per_launch": prof["gramian"][0] / max(prof["gramian"][1], 1)}
    whole_iter_bytes = su + si + gu + gi + extra
    roofline["whole_step_frac"] = whole_iter_bytes * args.steps / (ms * 1e-3) / 1e9 / peak

    # ---- end-to-end arm through the public API with host inputs.  Primary: the caller holds ORDINARY numpy / scipy
    #      arrays (pageable memory), which is what a user of the reference passes to fit(); secondary: the same
    #      arrays already page-locked (what a serving loop that re-fits from a staging buffer would hold).
    e2e = None
    if on_device and not args.no_e2e:
        # host copies of the device-generated inputs, for the public-API arm (fit() takes host arrays)
        Cui_host = Cui.download()
        X0, Y0 = initial_factors_on_device()
        X0, Y0 = (lambda a, b: (a.download(), b.download()))(X0, Y0)
    if not args.no_e2e:
        def timed_fits(Cin, X0in, Y0in, reps):
            times = []
            for rep in range(reps + 1):
                m = AlternatingLeastSquares(factors=f, regularization=reg, use_cg=use_cg, iterations=E2E_ITERS,
                                            process_group=pg)
                m.user_factors, m.item_factors = X0in, Y0in
                if world > 1:
                    pg.barrier()
                prof_e2e = None
                if args.trace_e2e and rep == reps:
                    import cProfile

                    prof_e2e = cProfile.Profile()
                    prof_e2e.enable()
                t = time.perf_counter()
                m.fit(Cin, show_progress=False)
                uf, vf = m.user_factors, m.item_factors  # D2H into (pooled) page-locked arrays
                dt = time.perf_counter() - t
                nbytes = uf.nbytes + vf.nbytes
                del uf, vf  # hand the page-locked result buffers back: a live reference would force the next fit to
                #             page-lock fresh ones (~30 ms per 90 MB), which is not what a user's second fit pays
                if prof_e2e is not None:
                    import pstats

                    prof_e2e.disable()
                    print(f"e2e fit: {dt * 1e3:.2f} ms; all reps so far {[round(x * 1e3, 2) for x in times]}", file=sys.stderr)
                    pstats.Stats(prof_e2e, stream=sys.stderr).sort_stats("cumulative").print_stats(25)
                assert nbytes == X0.nbytes + Y0.nbytes
                if rep > 0:  # first repetition is warm-up
                    times.append(pg.allreduce_max(dt) if world > 1 else dt)
                del m
            return times

        h2d = Cui_host.data.nbytes + Cui_host.indices.nbytes + Cui_host.indptr.nbytes + X0.nbytes + Y0.nbytes
        d2h = X0.nbytes + Y0.nbytes
        reps = 2 if on_device else max(3, min(7, args.steps))
        times = timed_fits(Cui_host, X0, Y0, reps)
        times_pinned = None
        if not on_device:  # (C4 would page-lock 7 GB per rank for this secondary figure)
            Cpin = pinned_csr(Cui_host)
            X0p, Y0p = _lib.pinned_empty(X0.shape, np.float32), _lib.pinned_empty(Y0.shape, np.float32)
            X0p[:], Y0p[:] = X0, Y0
            times_pinned = timed_fits(Cpin, X0p, Y0p, reps)
        # every fit is listed; the median is the reported figure, with the mean and the max / median ratio alongside
        e2e = {"value": (users + items) * E2E_ITERS / float(np.median(times)), "unit": UNIT,
               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "step": f"fit(ordinary scipy CSR + numpy factors in pageable memory) of {E2E_ITERS} iterations + both factor "
                       f"matrices read back, median of {len(times)} fits",
               "s_per_fit": float(np.median(times)), "s_per_fit_mean": float(np.mean(times)),
               "fits_ms": [round(1e3 * x, 2) for x in times], "max_over_median": float(np.max(times) / np.median(times)),
               "pinned_inputs": None if times_pinned is None else {
                   "value": (users + items) * E2E_ITERS / float(np.median(times_pinned)),
                   "s_per_fit": float(np.median(times_pinned)), "fits_ms": [round(1e3 * x, 2) for x in times_pinned]}}

    # ---- C4: the reference on a row sample (SURVEY.md 8(d): full-size C4 has no CPU run; 2000 user rows of one half)
    oracle_sample = None
    if on_device and rank == 0 and Cui_host is not None:
        import oracle

        impl = oracle.get("auto")
        sample = np.sort(np.random.default_rng(4).choice(users, 2000, replace=False))
        sub = Cui_host[sample]
        Yh = Y.download()
        exp = np.zeros((len(sample), f), dtype=np.float32)
        impl.least_squares(sub, exp, Yh, reg)
        Xt = _lib.DeviceFactors(ctx, users, f)
        _lib.least_squares(ctx, Cui, Xt, Y, reg)
        got = Xt.download()[sample]
        Xt.close()
        den = np.linalg.norm(exp.astype(np.float64), axis=1)
        err = np.linalg.norm(got.astype(np.float64) - exp, axis=1) / np.maximum(den, 0.01 * np.median(den))
        oracle_sample = {"rows": int(len(sample)), "row_err_max": float(err.max()), "row_err_median": float(np.median(err)),
                         "what": "one Cholesky user half on the final item factors: GPU vs the reference's least_squares on the sampled rows"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not on_device:
        cpu = cpu_reference_rate(Cui_host, X0, Y0, cfg, seconds=args.cpu_seconds)

    if rank == 0:
        out = {
            "metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "note_c4": ("inputs generated on the device (csrc/gen.cu), statistically equivalent to the host generator"
                        if on_device else None),
            "dtype": "f32 (tensor-core accumulation with 3-term hi/lo splits, fp32-faithful)", "data": "synthetic",
            "config": workload_config(cfg, args, world), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": cpu, "parity_vs_n1": parity_vs_n1, "oracle_sample": oracle_sample,
            "kernel_ms": {k: {"total_ms": v[0], "launches": v[1]} for k, v in prof.items() if v[1]},
        }
        print(json.dumps(out))
    if world > 1:
        pg.barrier()


# --------------------------------------------------------------------------------------- C5: recommend
# batch: two full waves of the top-k kernel's 256-query CTAs on 148 SMs (the 1M-user sweep is 13.2 such batches)
C5 = dict(users=1_000_000, items=1_000_000, factors=64, k=10, liked_per_user=20, batch=2 * 148 * 256, seed=5)


def c5_inputs(scale):
    """SURVEY.md 8(d): factors from default_rng(5).standard_normal * 0.1, liked-items CSR at 20 nnz / user."""
    from implicit_b200 import synthetic

    Q, I = max(1024, int(C5["users"] * scale)), max(1024, int(C5["items"] * scale))
    rng = np.random.default_rng(C5["seed"])
    users = rng.standard_normal((Q, C5["factors"]), dtype=np.float32) * np.float32(0.1)
    items = rng.standard_normal((I, C5["factors"]), dtype=np.float32) * np.float32(0.1)
    liked = synthetic.power_law_csr(Q, I, C5["liked_per_user"] * Q, C5["seed"])
    return users, items, liked


def c5_config(Q, I, batch, args):
    return {"workload": f"C5: recommend() top-k={C5['k']} for {Q} users against {I} items, factors={C5['factors']}, liked items "
                        f"filtered ({C5['liked_per_user']} per user), fused GEMM + top-k; one step = one batch of {batch} users",
            "scale": args.scale, "l2": "inputs_exceed_l2 (item factors, 256 MB, are streamed once per 128-query tile)",
            "parallelism": "single GPU", "e2e_step": "model.recommend(userids, user_items[userids]) with host ids / scores"}


def run_topk_reference(args):
    """The reference's topk (implicit/cpu/topk.pyx:15-67: sgemm + heap select) on a bounded sample of query rows."""
    import oracle

    if int(os.environ.get("RANK", "0")) != 0:
        return
    users, items, liked = c5_inputs(args.scale)
    Q, I = users.shape[0], items.shape[0]
    impl = oracle.get("auto")
    ncpu = os.cpu_count() or 1
    rows = 100
    rates = []
    t_all = time.perf_counter()
    for step in range(args.warmup + args.steps):
        sel = np.sort(np.random.default_rng(step).choice(Q, rows, replace=False))
        t = time.perf_counter()
        impl.topk(items, users[sel], C5["k"], filter_query_items=liked[sel], num_threads=0)
        dt = time.perf_counter() - t
        if step >= args.warmup:
            rates.append(rows / dt)
        rows = int(max(100, min(2000, rows * min(args.cpu_seconds, 150.0 / max(args.steps, 1)) / max(dt, 1e-3))))
    value = float(np.mean(rates))
    batch = min(C5["batch"], Q)
    base = {"value": value, "unit": "queries/s", "cores": ncpu, "kind": "reference" if impl.name == "ref" else "port",
            "sample": f"{rows} uniformly drawn query rows x all {I} items per step (topk.pyx batches of 100 rows), num_threads=0"}
    print(json.dumps({
        "impl": "reference", "metric": "recommend() user-queries/sec at f=64, k=10", "value": value, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * batch / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": c5_config(Q, I, batch, args), "cpu_baseline": base,
        "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_all}))


def run_topk(args):
    """C5: fused scores + filter + top-k.  value = queries/s with everything resident (the liked CSR of the whole
    user base, both factor matrices); e2e = model.recommend() per batch with host ids in, host (ids, scores) out."""
    from implicit_b200 import AlternatingLeastSquares, _lib

    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps({"metric": "recommend() user-queries/sec at f=64, k=10", "unavailable": "C5 is a single-GPU configuration"}))
        return
    users, items, liked = c5_inputs(args.scale)
    Q, I, f, k = users.shape[0], items.shape[0], C5["factors"], C5["k"]
    batch = min(C5["batch"], Q)
    ctx = _lib.Context(0)
    di, dq = _lib.DeviceFactors.from_host(ctx, items), _lib.DeviceFactors.from_host(ctx, users)
    liked_dev = {}

    def batch_rows(step):
        lo = (step * batch) % max(Q - batch + 1, 1)
        return lo, np.arange(lo, lo + batch, dtype=np.int32)

    warm = max(args.warmup, 3)
    for step in range(warm + args.steps):  # the liked lists of the batches this run touches, resident before timing
        lo, _ = batch_rows(step)
        if lo not in liked_dev:
            liked_dev[lo] = _lib.DeviceCSR.upload(ctx, liked[lo:lo + batch])
    for step in range(warm):
        lo, rows = batch_rows(step)
        _lib.topk(ctx, di, dq, k, query_rows=rows, liked=liked_dev[lo])
    ctx.sync()
    sampler = ClockSampler(ctx.device)
    sampler.start()
    ctx.profile(True)
    ctx.profile_read()
    launches0 = ctx.launch_count()
    t0 = time.perf_counter()
    for step in range(warm, warm + args.steps):
        lo, rows = batch_rows(step)
        ids, scores = _lib.topk(ctx, di, dq, k, query_rows=rows, liked=liked_dev[lo])
    ctx.sync()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    prof = ctx.profile_read()
    ctx.profile(False)
    launches = ctx.launch_count() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"ids": ids.astype(np.float64), "scores": scores})
    k_ms, k_n = prof["topk"]
    ms = k_ms  # device time of the fused kernel(s): CUDA events around each launch on the library's stream
    value = batch * args.steps / (ms * 1e-3)
    flops = 2.0 * batch * I * f
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            bf16 = float(json.load(fh)["bf16_tflops"])
        peak_src = "measured 16-bit tensor burst (MEASURED_PEAKS.json bf16_tflops) / 3: fp16 hi/lo operands, three MMAs per product"
    except Exception:
        bf16, peak_src = 1590.0, "fallback 16-bit tensor 1.59 PFLOP/s / 3 (fp16 hi/lo operands, three MMAs per product)"
    peak = bf16 / 3.0
    achieved = flops * k_n / (k_ms * 1e-3) / 1e12
    roofline = {"bound": "tensor", "kernel": "topk kernel (scores + filters + ordered select)", "achieved": achieved, "peak": peak,
                "peak_source": peak_src, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None,
                "algorithmic_flops_per_launch": flops, "avg_launch_ms": k_ms / max(k_n, 1),
                "candidates_per_s": batch * I * k_n / (k_ms * 1e-3),
                "full_c5_seconds_at_this_rate": Q / value}

    # ---- end to end through the public API
    e2e = None
    if not args.no_e2e:
        m = AlternatingLeastSquares(factors=f)
        m.user_factors, m.item_factors = users, items
        times = []
        h2d = d2h = 0
        for step in range(1 + max(3, min(args.steps, 7))):
            lo, rows = batch_rows(step)
            ui = liked[lo:lo + batch]
            t = time.perf_counter()
            ids, sc = m.recommend(rows, ui, N=k, filter_already_liked_items=True)
            dt = time.perf_counter() - t
            if step > 0:  # the first call uploads both factor matrices (model load), not a per-request cost
                times.append(dt)
            h2d = rows.nbytes + ui.data.nbytes + ui.indices.nbytes + ui.indptr.nbytes
            d2h = ids.nbytes + sc.nbytes
        e2e = {"value": batch / float(np.median(times)), "unit": "queries/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "step": f"recommend({batch} userids, their liked CSR) -> host (ids, scores)",
               "s_per_call": float(np.median(times)), "calls_ms": [round(1e3 * x, 2) for x in times]}

    cpu = None
    if not args.no_cpu_baseline:
        import oracle

        impl = oracle.get("auto")
        rows = 200
        sel = np.sort(np.random.default_rng(0).choice(Q, rows, replace=False))
        t = time.perf_counter()
        impl.topk(items, users[sel], k, filter_query_items=liked[sel], num_threads=0)
        dt = time.perf_counter() - t
        rows2 = int(max(200, min(4000, rows * args.cpu_seconds / max(dt, 1e-3))))
        sel = np.sort(np.random.default_rng(1).choice(Q, rows2, replace=False))
        t = time.perf_counter()
        impl.topk(items, users[sel], k, filter_query_items=liked[sel], num_threads=0)
        dt = time.perf_counter() - t
        cpu = {"value": rows2 / dt, "unit": "queries/s", "cores": os.cpu_count() or 1, "kind": "reference" if impl.name == "ref" else "port",
               "sample": f"{rows2} uniformly drawn query rows x all {I} items ({dt:.1f} s), reference topk with num_threads=0"}

    print(json.dumps({
        "metric": "recommend() user-queries/sec at f=64, k=10", "value": value, "unit": "queries/s", "n_gpus": 1,
        "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32 (fp16 hi/lo split tensor-core scores: three tcgen05 MMAs per product, fp32-faithful)", "data": "synthetic",
        "config": c5_config(Q, I, batch, args), "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
        "roofline": roofline, "cpu_baseline": cpu, "wall_s_timed_region": wall}))


# --------------------------------------------------------------------------------------- the reference's own CUDA kernel
def run_reference_gpu(args):
    """The reference's CUDA ALS solver (implicit/gpu/als.cu: cuBLAS Gramian + least_squares_cg_kernel), compiled
    unchanged into oracle/_ref/libref_gpu_als.so (oracle/build_ref_gpu.py), driven like implicit/gpu/als.py:159-165 on the
    same workload and initial factors, on GPU 0.  CG only (the reference has no GPU Cholesky); for the Cholesky
    configuration C2 this is its answer to the same problem.  Reports the SAME metric, plus parity with our CG path."""
    import ctypes

    if int(os.environ.get("RANK", "0")) != 0:
        return
    from implicit_b200 import _lib, synthetic

    path = os.path.join(ROOT, "oracle", "_ref", "libref_gpu_als.so")
    if not os.path.exists(path):
        print(json.dumps({"impl": "reference-gpu", "unavailable": "oracle/_ref/libref_gpu_als.so was not built (oracle/build_ref_gpu.py needs /root/reference)"}))
        return
    lib = ctypes.CDLL(path)
    Cui, X0, Y0, cfg = synthetic.config(args.config, scale=args.scale)
    users, items, f = cfg["users"], cfg["items"], cfg["factors"]
    Ciu = Cui.T.tocsr()
    iters = args.warmup + args.steps
    X, Y = X0.copy(), Y0.copy()
    ms = np.zeros(iters, dtype=np.float32)
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    ui = [np.ascontiguousarray(Cui.indptr, np.int32), np.ascontiguousarray(Cui.indices, np.int32), np.ascontiguousarray(Cui.data, np.float32)]
    iu = [np.ascontiguousarray(Ciu.indptr, np.int32), np.ascontiguousarray(Ciu.indices, np.int32), np.ascontiguousarray(Ciu.data, np.float32)]
    rc = lib.ref_gpu_als_cg_fit(users, items, f, p(ui[0]), p(ui[1]), p(ui[2]), int(Cui.nnz), p(iu[0]), p(iu[1]), p(iu[2]), p(X), p(Y),
                                ctypes.c_float(0.01), 3, iters, p(ms))
    if rc != 0:
        print(json.dumps({"impl": "reference-gpu", "unavailable": f"harness returned {rc}"}))
        return
    timed = ms[args.warmup:]
    value = (users + items) * len(timed) / (float(timed.sum()) * 1e-3)
    # parity of OUR CG path with the reference's CUDA kernel after the same number of iterations (both fp32, CG(3))
    ctx = _lib.Context(0)
    C = _lib.DeviceCSR.upload(ctx, Cui)
    T = C.transpose()
    dX, dY = _lib.DeviceFactors.from_host(ctx, X0), _lib.DeviceFactors.from_host(ctx, Y0)
    ctx.timer_start()
    for _ in range(iters):
        _lib.least_squares_cg(ctx, C, dX, dY, 0.01, 3)
        _lib.least_squares_cg(ctx, T, dY, dX, 0.01, 3)
    ours_ms = ctx.timer_stop() / iters
    gx = dX.download()
    den = np.linalg.norm(X.astype(np.float64), axis=1)
    err = np.linalg.norm(gx.astype(np.float64) - X, axis=1) / np.maximum(den, 0.01 * np.median(den))
    print(json.dumps({
        "impl": "reference-gpu", "metric": metric_name(dict(cfg, use_cg=True)), "value": value, "unit": UNIT, "n_gpus": 1,
        "steps": int(len(timed)), "warmup": args.warmup, "ms_per_step": float(timed.mean()), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(dict(cfg, use_cg=True), args, 1),
                       note="the reference's GPU path is CG-only: implicit/gpu/als.cu least_squares_cg_kernel + cublasSgemm Gramian, compiled for sm_100a"),
        "ms_per_iteration": [round(float(x), 3) for x in ms],
        "ours_cg_same_workload": {"ms_per_step": ours_ms, "value": (users + items) / (ours_ms * 1e-3),
                                  "speedup_over_reference_gpu": float(timed.mean()) / ours_ms,
                                  "row_err_vs_reference_gpu": {"median": float(np.median(err)), "p99": float(np.quantile(err, 0.99)),
                                                               "max": float(err.max()),
                                                               "note": f"user factors after {iters} CG(3) iterations from the same start"}},
        "gpu_launches": 4 * iters}))


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus != world and world == 1 and args.gpus > 1:
        # convenience: `python bench.py --gpus N` re-launches itself with one process per GPU
        port = 29500 + os.getpid() % 1000
        procs = []
        for r in range(args.gpus):
            env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(args.gpus), MASTER_ADDR="127.0.0.1",
                       MASTER_PORT=str(port))
            procs.append(subprocess.Popen([sys.executable] + sys.argv, env=env))
        sys.exit(max(p.wait() for p in procs))
    if args.impl == "reference-gpu":
        run_reference_gpu(args)
    elif args.config == "C5":
        (run_topk_reference if args.impl == "reference" else run_topk)(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
