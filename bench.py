#!/usr/bin/env python
"""bench.py — superblock H·psi throughput of the B200 path (BASELINE.json metric) with the reference-algorithm CPU
baseline beside it.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm on the host cores
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's y = H*psi as DIR/hpsi.npy

A step is one H·psi apply (MatMult_KronSumShell, src/DMRGKron.cpp:1827-1869) on the synthetic sweep-midpoint
superblock of BASELINE.json configs[2] (J1-J2 12x6 cylinder, J2/J1 = 0.5, m = 2048 kept states; the largest
single-GPU configuration the metric is quoted on).  `value` = algorithmic GB/s (SURVEY.md §8d: 16·D bytes of psi in/out
+ every distinct operator panel once) with psi resident in HBM; `e2e` = the same through the C-ABI call with HOST
buffers (dmrgx_hshell_apply_host: H2D + kernels + D2H inside the timed region).  The workload is bound by the FP64
tensor pipe, not by HBM (420 flop per algorithmic byte), so `tflops` / `roofline_frac` stand beside `value` at the top
level.  Every run compares the GPU result with the oracle on a sample of superblock rows (`parity`), at every N.
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="j1j2_12x6")
    ap.add_argument("--m", "--mstates", dest="m", type=int, default=2048, help="kept states of the synthetic blocks (use --mstates under torchrun: its parser "
                    "takes a bare --m for one of its own options)")
    ap.add_argument("--cpu-baseline-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle comparison on a row sample")
    ap.add_argument("--from-disk", default=None, help="BASELINE configs[4]: a Sweep_*/ directory of saved blocks (InitializeFromDisk layout) "
                    "to take the superblock from instead of the synthetic one")
    ap.add_argument("--no-sweep", action="store_true", help="skip the seconds-per-sweep measurement (DMRG-SquareLattice.x on the metric's config)")
    ap.add_argument("--sweep-msweeps", default="512,1024,2048", help="-msweeps of the seconds-per-sweep run (the last entry is the one reported)")
    ap.add_argument("--no-extras", action="store_true", help="only the H*psi line (no lanczos / sparse-sector / sweep sections)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write y = H*psi of the last timed step as DIR/hpsi.npy (float64; a fixed "
                    "seeded sample of rows when the whole vector exceeds %d MB), so that two builds can be compared output for output" % (DUMP_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_BYTES = 64 * 10**6   # all files --dump-outputs writes, together


def dump_outputs(path, arrays):
    """float64 .npy files of what the timed path returned; a vector beyond its share of DUMP_BYTES is cut to a fixed, seeded,
    sorted sample of its entries (the same for every run with the same arguments)."""
    os.makedirs(path, exist_ok=True)
    cap = (DUMP_BYTES // len(arrays) - 4096) // 8
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def workload_label(config, m, n):
    """one string, byte-identical in both arms"""
    return "%s m=%d sweep-midpoint superblock H*psi, D=%d" % (config, m, n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per apply from the committed ncu capture of this build's kernels
    (profiles/r2_traffic.json: written by hand from `ncu --set full` of the same bench command); None when no capture names
    this workload — the number is never invented."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None, "no ncu capture committed for this build"
    t = json.load(open(p))
    e = t.get(kernel_key)
    if not e:
        return None, "profiles/r2_traffic.json has no entry for %s" % kernel_key
    return e["dram_bytes_per_apply"], e["source"]


def fp64_peak_tflops(torch, dev):
    """FP64 peak is not in MEASURED_PEAKS.json (BASELINE.md §2): measure a cuBLAS DGEMM here, as a measurement tool."""
    n = 6144
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    torch.cuda.synchronize()
    best = 1e9
    for _ in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


class HostWorkload:
    """The synthetic blocks and term lists of a workload WITHOUT the product library: term lists from the oracle's own
    restatement of Hamiltonians::J1J2XXZModel_SquareLattice::H (src/Hamiltonians.cpp:73-122).  Used by the reference arm."""

    def __init__(self, O, config, m):
        import bench_workload as W
        ham = W.CONFIGS[config]
        N = ham["Lx"] * ham["Ly"]
        self.nsites_blk = N // 2 - 1
        T = lambda n: O.ham_terms(ham["Lx"], ham["Ly"], ham["J1"], ham["Jz1"], ham["J2"], ham["Jz2"], n, ham["bcx"], ham["bcy"])
        self.terms_enl, self.terms = T(N // 2), T(N)
        self.host = W.synth_block_host(m, self.nsites_blk, W.used_sites(self.terms_enl, self.terms, self.nsites_blk))


def oracle_rows(O, kb, terms, x, r0, r1, cores):
    """y[r0:r1] of the reference's loop nest (KronSumSetUpShellTerms + MatMult_KronSumShell restated) and the time it took"""
    sh = O.Shell(kb, terms, rows=(r0, r1))
    t = time.time()
    y = sh.apply(x, cores)
    return y, time.time() - t, sh.fmas()


def cpu_baseline(O, kb, wl, x, seconds, alg_bytes, alg_flops):
    """The reference's algorithm (oracle restatement of MatMult_KronSumShell + KronSumSetUpShellTerms) on the host
    cores, on a bounded sample of superblock rows, rows split over threads like PreSplitOwnership over MPI ranks.
    Returns the baseline record and (r0, r1, y_ref) so that the GPU result can be checked on the same rows."""
    cores = os.cpu_count() or 1
    t0 = time.time()
    n = kb.num_states()
    mid = n // 2
    probe = max(8 * cores, 64)
    _, dt, _ = oracle_rows(O, kb, wl.terms, x, mid, min(n, mid + probe), cores)
    per_row = max(dt / probe, 1e-9)
    rows = int(max(probe, min(n, seconds / per_row)))
    # sample = `rows` consecutive rows centred in the vector (covers the heavy pairs); scale by D / rows
    r0 = max(0, mid - rows // 2); r1 = min(n, r0 + rows)
    y_ref, dt, fmas = oracle_rows(O, kb, wl.terms, x, r0, r1, cores)
    full_seconds = dt * n / (r1 - r0)
    rec = {"value": alg_bytes / full_seconds / 1e9, "unit": "GB/s", "cores": cores, "kind": "port", "extrapolated": True,
           "sampled_fraction": (r1 - r0) / float(n),
           "sample": "rows [%d,%d) of %d (%.3g%% of the superblock), %.2f s measured, scaled by rows; unfactored FMAs/row %.3g; setup %.1f s"
                     % (r0, r1, n, 100.0 * (r1 - r0) / n, dt, fmas / (r1 - r0), time.time() - t0 - dt),
           "seconds_per_apply_extrapolated": full_seconds,
           # the reference's unfactored loop nest pays nz_L*nz_R multiply-adds per row per term (src/DMRGKron.cpp:1844-1864):
           # its flop count per apply next to the factored count of our arm separates the algorithmic from the hardware speed-up
           "unfactored_flops_per_apply": 2.0 * fmas / (r1 - r0) * n, "factored_flops_per_apply": alg_flops,
           "gflops": 2.0 * fmas / dt / 1e9}
    return rec, (r0, r1, y_ref)


def parity_windows(n, cuts, pair_offsets, rows_per_window):
    """Row windows the oracle is run on: one straddling every rank boundary (N > 1), one straddling the start of the largest
    sector pair (a ragged edge tile next to full tiles), one in the middle of it (full 64x64 tiles, split stage-2 chains)."""
    w = []
    h = rows_per_window // 2
    for c in list(cuts[1:-1]):
        w.append((max(0, int(c) - h), min(n, int(c) + h)))
    sizes = np.diff(pair_offsets)
    big = int(np.argmax(sizes))
    a = int(pair_offsets[big])
    w.append((max(0, a - h), min(n, a + h)))
    mid = a + int(sizes[big]) // 2
    w.append((max(0, mid - h), min(n, mid + h)))
    e = int(pair_offsets[big + 1])
    w.append((max(0, e - h), min(n, e + h)))
    return sorted(set(x for x in w if x[1] > x[0]))


def reference_arm(args, rank):
    """bench.py --impl reference: the reference's own CPU algorithm for this path on the box's host cores (rank 0 only).
    Nothing of the product is imported or loaded here: blocks from bench_workload (numpy), terms and the timed loop from
    oracle/ (the PETSc/SLEPc build cannot be produced in this image, DESIGN.md §7)."""
    if rank != 0:
        return
    import bench_workload as W
    from oracle import oracle as O
    wl = HostWorkload(O, args.config, args.m)
    _, kb = W.oracle_side(O, wl)
    n = kb.num_states()
    cores = os.cpu_count() or 1
    x = np.random.default_rng(1).standard_normal(n); x /= np.linalg.norm(x)
    mid = n // 2
    probe = max(8 * cores, 64)
    sh = O.Shell(kb, wl.terms, rows=(mid, min(n, mid + probe)))
    t = time.time(); sh.apply(x, cores); per_row = max((time.time() - t) / sh.lrows, 1e-9)
    budget = 120.0 / max(1, args.steps + args.warmup)
    rows = int(max(probe, min(n, budget / per_row)))
    r0 = max(0, mid - rows // 2); r1 = min(n, r0 + rows)
    sh = O.Shell(kb, wl.terms, rows=(r0, r1))
    # algorithmic bytes of the same workload, same definition as our arm (SURVEY.md §8d), computed without the library
    alg_bytes = float(W.algorithmic_bytes(wl.host, wl.terms, wl.nsites_blk, n))
    for _ in range(args.warmup):
        sh.apply(x, cores)
    t = time.time()
    for _ in range(args.steps):
        sh.apply(x, cores)
    dt = (time.time() - t) / max(1, args.steps)
    full = dt * n / (r1 - r0)
    val = alg_bytes / full / 1e9
    line = {"impl": "reference", "metric": "superblock H*psi algorithmic GB/s", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": full * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_label(args.config, args.m, n)},
            "extrapolated": True, "sampled_fraction": (r1 - r0) / float(n),
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": "port", "extrapolated": True, "sampled_fraction": (r1 - r0) / float(n),
                             "sample": "each step = rows [%d,%d) of %d (%.3g%%) of one apply, %.3f s per step measured, scaled by rows to a full apply "
                                       "(reference PETSc/SLEPc build impossible here: oracle restatement of MatMult_KronSumShell)"
                                       % (r0, r1, n, 100.0 * (r1 - r0) / n, dt)},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_sweep(args, rank, world, local, predict=False):
    """Seconds per sweep (the metric's second half) through the reference-named executable on the metric's own config
    (BASELINE configs[2]: 12x6 J1-J2 cylinder, -msweeps 512,1024,2048); at N > 1 every rank starts its own process of the
    executable on its GPU (the executable's ranks find each other through DMRGX_ID_FILE).  predict: the same run with
    -wavefunction_prediction 1 (extension: every sweep step's eigen-solve starts from the transformed previous ground state; the
    reference — and the plain `sweep` section — start from a random vector)."""
    import bench_workload as W
    import tempfile
    exe = os.path.join(ROOT, "dmrg.x_b200", "DMRG-SquareLattice.x")
    if not os.path.exists(exe):
        return {"error": "DMRG-SquareLattice.x not built"}
    ham = W.CONFIGS[args.config]
    td = os.environ.get("DMRGX_BENCH_SWEEP_DIR") or os.path.join(tempfile.gettempdir(), "dmrgx_bench_sweep_%s" % os.environ.get("MASTER_PORT", str(os.getpid())))
    os.makedirs(td, exist_ok=True)
    msw = args.sweep_msweeps
    cmd = [exe, "-Lx", str(ham["Lx"]), "-Ly", str(ham["Ly"]), "-J1", repr(ham["J1"]), "-Jz1", repr(ham["Jz1"]), "-J2", repr(ham["J2"]), "-Jz2", repr(ham["Jz2"]),
           "-mwarmup", "128", "-msweeps", msw, "-data_dir", td + "/", "-do_correlators", "0", "-device", str(local)]
    if ham.get("bcx", 0) == 0 and ham.get("bcy", 1) == 0:
        cmd.append("-BCopen")
    if predict:
        cmd += ["-wavefunction_prediction", "1"]
    env = dict(os.environ)
    env["DMRGX_ID_FILE"] = os.path.join(td, "nccl_id_%s%s" % (os.environ.get("DMRGX_BENCH_NONCE", "0"), "p" if predict else ""))
    t0 = time.time()
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=1500, env=env)
    wall = time.time() - t0
    if rank != 0:
        return {}
    if r.returncode != 0:
        return {"error": "rc=%d %s" % (r.returncode, r.stderr[-400:])}
    run = json.load(open(os.path.join(td, "DMRGRun.json")))
    steps = json.load(open(os.path.join(td, "DMRGSteps.json")))
    tim = json.load(open(os.path.join(td, "Timings.json")))
    hs = steps["headers"]
    loop = hs.index("LoopIdx"); ns, ne = hs.index("NSites_Sys"), hs.index("NSites_Env")
    lastloop = max(row[loop] for row in steps["table"])
    last = [(t, srow) for t, srow in zip(tim["table"], steps["table"]) if srow[loop] == lastloop]
    names = tim["headers"][1:]
    mid = [srow for _, srow in last if srow[ns] == srow[ne]]
    m_last = int(msw.split(",")[-1])
    return {"config": "%s (BASELINE configs[2]) -mwarmup 128 -msweeps %s, %d GPU(s), default -H_eps_tol 1e-8, correlators off%s" % (
                args.config, msw, world, ", -wavefunction_prediction 1 (extension: not the reference's random start)" if predict else ""),
            "steps_with_predicted_start": run.get("StepsWithPredictedStart", 0),
            "m": m_last, "seconds_per_sweep": run["Sweeps"]["Seconds"][-1], "all_sweeps_seconds": run["Sweeps"]["Seconds"], "steps_per_sweep": len(last),
            "phases_s": {nm: float(sum(t[i + 1] for t, _ in last)) for i, nm in enumerate(names)},
            "energy_midpoint": mid[0][hs.index("GSEnergy")] if mid else None, "energy_last_step": steps["table"][-1][hs.index("GSEnergy")],
            "max_trunc_err": max(max(srow[hs.index("TruncErr_Sys")], srow[hs.index("TruncErr_Env")]) for _, srow in last),
            "largest_D": max(srow[hs.index("NumStates_H")] for _, srow in last), "matvecs_total": run["NumMatVecs"], "process_wall_s": wall}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return reference_arm(args, rank)

    # ------------------------------------------------------------------ our arm
    import torch
    import dmrgx_loader
    import bench_workload as W
    P = dmrgx_loader.load_package()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    uid = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        # rank 0 creates the communicator id of the library's own NCCL communicator; torch.distributed is only the courier
        box = [P.dist_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        uid = box[0]
    # a dedicated torch stream: the library launches on it and torch.cuda.Event records on it (the legacy default
    # stream has handle 0, which the C ABI reads as "create a private stream" — events would then miss the kernels)
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    assert tstream.cuda_stream != 0
    ctx = P.Context(local, tstream.cuda_stream, rank, world, uid)
    wl = W.DiskWorkload(P, ctx, args.config, args.from_disk) if args.from_disk else W.Workload(P, ctx, args.config, m=args.m)
    if args.from_disk:
        args.m = wl.m
    H = wl.shell
    st = H.stats()
    n = wl.n
    rb, re_, cuts = H.row_range()
    # the superblock vector is sharded by row ranges: every rank holds its own rows, an apply all-gathers x over NVLink
    xfull = wl.random_state()
    xin = np.zeros(n); xin[rb:re_] = xfull[rb:re_]
    x = ctx.vec(n, xin)
    y = ctx.vec(n)
    apply_fn = (lambda: H.MatMult_sharded(x, y)) if world > 1 else (lambda: H.MatMult(x, y))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        apply_fn()
    peak_fp64 = fp64_peak_tflops(torch, dev)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    # the timed region lasts a few milliseconds, nvidia-smi samples every 100 ms: the same applies run (untimed) for 0.4 s
    # before and after it, so that the clocks / throttle reasons reported are those of this load
    t_probe = time.time()
    for _ in range(5):
        apply_fn()
    torch.cuda.synchronize()
    est = torch.tensor([(time.time() - t_probe) / 5], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(est, op=dist.ReduceOp.MAX)   # the same number of (collective) applies on every rank
    n_soak = int(min(5000, max(10, 0.4 / max(float(est.item()), 1e-6))))

    def soak():
        for _ in range(n_soak):
            apply_fn()
        torch.cuda.synchronize()
    soak()
    barrier()
    l0 = P.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # L2 hygiene: a rank's apply streams through `workspace + panels` bytes.  When that exceeds twice the 126 MB L2 nothing of
    # one iteration survives to the next; otherwise (small m, or the superblock sharded over many GPUs) a 256 MB buffer is
    # overwritten between iterations and every iteration is timed by its own event pair (the flush stays outside).
    per_rank_bytes = st["workspace_bytes"] + (st["alg_bytes"] - 16 * n)
    flush_l2 = per_rank_bytes < 2 * 126e6
    if world > 1:
        fl = torch.tensor([1.0 if flush_l2 else 0.0], device=dev)
        dist.all_reduce(fl, op=dist.ReduceOp.MAX)   # one policy for all ranks
        flush_l2 = bool(fl.item() > 0)
    if flush_l2:
        scratch = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        for a, b in evs:
            scratch.zero_()
            if world > 1:
                dist.barrier()
            a.record(); apply_fn(); b.record()
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        del scratch
    else:
        e0.record()
        for _ in range(args.steps):
            apply_fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
    launches = P.launch_count() - l0
    # the result of the last timed apply, whole vector on rank 0 (each rank computed its own rows)
    yh = y.get()
    if world > 1:
        ymask = np.zeros(n); ymask[rb:re_] = yh[rb:re_]
        yt = torch.from_numpy(ymask).to(dev)
        dist.all_reduce(yt)
        yh = yt.cpu().numpy()
        del yt
    soak()
    clocks = sampler.stop()
    t_local = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
    ms = float(t_local.item())
    ms_step = ms / args.steps
    value = st["alg_bytes_global"] / (ms_step * 1e-3) / 1e9  # one H*psi of the whole superblock, sharded over the ranks
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"hpsi": yh})

    # per-stage timing of the dominant kernel (chain_kernel) for the roofline
    f1, f2 = H.stage_flops()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    t1 = t2 = 0.0
    reps = max(5, min(args.steps, 20))
    for _ in range(reps):
        ev[0].record(); H.MatMult_stage(1, x, y); ev[1].record(); H.MatMult_stage(2, x, y); ev[2].record()
        torch.cuda.synchronize()
        t1 += ev[0].elapsed_time(ev[1]); t2 += ev[1].elapsed_time(ev[2])
    t1 /= reps; t2 /= reps
    achieved = (f1 + f2) / ((t1 + t2) * 1e-3) / 1e12
    peaks, peaks_kind = measured_peaks()

    lz, sparse, sweep = {}, {}, {}
    if not args.no_extras:
        # the eigen-solve around the matvec (EPSSolve call site): time per Lanczos iteration = matvec + orthogonalisation
        try:
            H.EPSSolve(tol=1e-30, ncv=16, max_it=1)
            ev[0].record()
            _, _, stl = H.EPSSolve(tol=1e-30, ncv=16, max_it=3)
            ev[1].record()
            torch.cuda.synchronize()
            lz = {"ms_per_iteration": ev[0].elapsed_time(ev[1]) / max(1, stl["nmatvec"]), "nmatvec": stl["nmatvec"], "ncv": 16,
                  "matvec_share": ms_step / (ev[0].elapsed_time(ev[1]) / max(1, stl["nmatvec"]))}
        except Exception as exc:
            lz = {"error": repr(exc)}

        # the sparse-sector case (un-truncated blocks, CSR / identity tiles, HBM-bound): the dedicated SpMM kernel
        if world == 1:
            try:
                sparse = sparse_sector_section(P, W, ctx, torch, peaks, peaks_kind)
            except Exception as exc:
                sparse = {"error": repr(exc)}

    # e2e: the reference-facing call with HOST buffers, copies inside the timed region
    hx = torch.from_numpy(wl.random_state(2)[rb:re_].copy()).pin_memory()   # this rank's local rows, like VecGetArray
    hy = torch.empty(re_ - rb, dtype=torch.float64).pin_memory()
    hxn, hyn = hx.numpy(), hy.numpy()
    for _ in range(3):
        H.MatMult_host(hxn, hyn)
    barrier()
    e0.record()
    for _ in range(args.steps):
        H.MatMult_host(hxn, hyn)
    e1.record()
    barrier()
    t_e2e = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    ms_e2e = float(t_e2e.item()) / args.steps
    e2e_val = st["alg_bytes_global"] / (ms_e2e * 1e-3) / 1e9

    traffic, traffic_src = ncu_traffic("%s_m%d_hpsi" % (args.config, args.m)) if world == 1 else (None, "not captured for sharded runs (ncu is single-GPU only)")
    tflops = st["alg_flops_global"] / (ms_step * 1e-3) / 1e12
    line = {
        "metric": "superblock H*psi algorithmic GB/s", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "blocks read from disk (InitializeFromDisk layout)" if args.from_disk else "synthetic",
        # what bounds this workload is the FP64 tensor pipe, not HBM (420 flop per algorithmic byte): read these two beside `value`
        "tflops": tflops, "roofline_frac": achieved / peak_fp64,
        "config": {"workload": workload_label(args.config, args.m, n), "shell_terms": st["nterms"],
                   "l2": ("L2 flushed (256 MB overwritten) between iterations, each iteration timed by its own event pair: one apply streams through "
                          "only %.0f MB on a rank" % (per_rank_bytes / 1e6)) if flush_l2 else
                         ("no flush needed: one apply streams through %.0f MB on this rank (V workspace + pre-summed factors + psi, plus %.0f MB of "
                          "operator panels), more than twice the 126 MB L2" % (st["workspace_bytes"] / 1e6, (st["alg_bytes"] - 16 * n) / 1e6)),
                   "parallelism": ("superblock rows sharded over %d GPUs (cuts %s), NCCL sector-halo exchange of psi per apply: rank 0 receives %.1f MB "
                                   "(an all-gather would bring %.1f MB)" % ((world, cuts.tolist()) + tuple(v / 1e6 for v in H.halo_bytes())))
                   if world > 1 else "single"},
        "e2e": {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": 8 * (re_ - rb), "d2h_bytes_per_step": 8 * (re_ - rb), "ms_per_step": ms_e2e},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_fp64, "unit": "TFLOP/s", "frac": achieved / peak_fp64,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": "chain_kernel (FP64 DMMA), 2 launches per apply",
                     "peak_source": "cuBLAS DGEMM %d^3 measured in this run (FP64 is not in MEASURED_PEAKS.json); 148 SM x 128 flop/clk x 1.965 GHz = 37.2" % 6144,
                     "stage_ms": [t1, t2], "stage_flops": [f1, f2],
                     "hbm_frac_of_%s_peak" % peaks_kind: (st["alg_bytes"] / (ms_step * 1e-3) / 1e9) / peaks["hbm_gbs"]},
        "lanczos": lz,
        "sparse_sector": sparse,
        "alg": {"bytes_per_apply": st["alg_bytes_global"], "flops_per_apply": st["alg_flops_global"], "rank0_flops": st["alg_flops"], "D": n,
                "tiles": [st["tiles_stage1"], st["tiles_stage2"]]},
    }

    # ---- parity on the timed result + CPU baseline (rank 0; the oracle is the checker, never the thing measured) ----
    if rank == 0 and not args.from_disk and not (args.no_parity and (args.no_cpu_baseline or world > 1)):
        try:
            from oracle import oracle as O
            _, kb = W.oracle_side(O, wl)
            cores = os.cpu_count() or 1
            tol = 1e-13 * st["nterms"]
            scale = float(np.abs(yh).max())
            checked, worst = [], 0.0
            if world == 1 and not args.no_cpu_baseline:
                rec, (r0, r1, y_ref) = cpu_baseline(O, kb, wl, xfull, args.cpu_baseline_seconds, st["alg_bytes_global"], st["alg_flops_global"])
                line["cpu_baseline"] = rec
                err = float(np.abs(yh[r0:r1] - y_ref).max() / scale)
                checked.append([r0, r1]); worst = max(worst, err)
            if not args.no_parity:
                _, _, _, _, poff = wl.kron.data()
                for (r0, r1) in parity_windows(n, cuts, poff, 768 if world > 1 else 1024):
                    y_ref, _, _ = oracle_rows(O, kb, wl.terms, xfull, r0, r1, cores)
                    err = float(np.abs(yh[r0:r1] - y_ref).max() / scale)
                    checked.append([r0, r1]); worst = max(worst, err)
            line["parity"] = {"rows": checked, "rows_checked": int(sum(b - a for a, b in checked)), "max_rel_err": worst, "tol": tol,
                              "against": "oracle restatement of MatMult_KronSumShell (src/DMRGKron.cpp:1844-1864) on the same x, y of the timed applies",
                              "ok": bool(worst <= tol)}
        except Exception as exc:  # the baseline is reported, never required for the GPU number
            line["cpu_baseline"] = line.get("cpu_baseline", {"error": repr(exc)})
            line["parity"] = {"error": repr(exc), "ok": False}

    # ---- seconds per sweep on the metric's config (all ranks take part at N > 1) ----
    if not args.no_sweep and not args.no_extras and not args.from_disk:
        del x, y
        if world > 1:   # a fresh rendezvous file name per run: a stale id file of a crashed run must never be read
            box = [str(time.time_ns()) if rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            os.environ["DMRGX_BENCH_NONCE"] = box[0]
        try:
            sweep = run_sweep(args, rank, world, local)
        except Exception as exc:
            sweep = {"error": repr(exc)}
        if world > 1:
            dist.barrier()
        try:
            sweep_pred = run_sweep(args, rank, world, local, predict=True)
        except Exception as exc:
            sweep_pred = {"error": repr(exc)}
        if world > 1:
            dist.barrier()
        line["sweep_wavefunction_prediction"] = sweep_pred
    line["sweep"] = sweep
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and "parity" in line and not line["parity"].get("ok", False):
        raise SystemExit("bench.py: GPU result differs from the oracle: %r" % (line["parity"],))


def sparse_sector_section(P, W, ctx, torch, peaks, peaks_kind):
    """north_star: ">= 60 % of HBM roofline on the sparse-sector matvec".  Un-truncated 12-site halves of the 24-site chain
    (CSR upload); x and y (21.6 MB each) fit in L2, so a 256 MB buffer is overwritten before every timed apply and each
    apply is timed by its own event pair."""
    sw = W.ExactChainWorkload(P, ctx, 12)
    sst = sw.shell.stats()
    sx = ctx.vec(sw.n, sw.random_state()); sy = ctx.vec(sw.n)
    for _ in range(5):
        sw.shell.MatMult(sx, sy)
    l0 = P.launch_count()
    sw.shell.MatMult(sx, sy)
    nl = P.launch_count() - l0
    reps = 20
    scratch = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=sx_device(torch))
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        scratch.zero_()
        a.record(); sw.shell.MatMult(sx, sy); b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in evs)
    sms = float(np.median(t))
    # back-to-back (x, y and the operators L2-resident between applies), for comparison
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        sw.shell.MatMult(sx, sy)
    e1.record()
    torch.cuda.synchronize()
    warm = e0.elapsed_time(e1) / reps
    sgb = sst["alg_bytes"] / (sms * 1e-3) / 1e9
    traffic, src = ncu_traffic("exact_chain12_sparse")
    return {"workload": "Heisenberg chain 24 sites, exact 12-site halves (4096 states each, CSR upload), D=%d, H nnz/row %.1f" % (sw.n, sw.h_nnz_per_row),
            "ms_per_apply": sms, "ms_per_apply_l2_warm": warm, "launches_per_apply": int(nl), "alg_bytes": sst["alg_bytes"], "achieved_gbs": sgb,
            "achieved_gbs_l2_warm": sst["alg_bytes"] / (warm * 1e-3) / 1e9, "bound": "hbm",
            "peak_gbs": peaks["hbm_gbs"], "frac": sgb / peaks["hbm_gbs"], "peak_source": peaks_kind, "traffic": traffic, "traffic_source": src,
            "l2": "256 MB overwritten before every timed apply (median of %d event pairs)" % reps,
            "tiles": [sst["tiles_stage1"], sst["tiles_stage2"]]}


def sx_device(torch):
    return torch.device("cuda", torch.cuda.current_device())


if __name__ == "__main__":
    main()
