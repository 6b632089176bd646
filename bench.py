#!/usr/bin/env python
"""Benchmark of the mixemt hot path on B200 (contract: see DESIGN.md, Measurement).

    python bench.py --gpus N --steps K --warmup W            # this framework
    python bench.py --impl reference --steps K --warmup W    # CPU reference arm

A *step* is one EM iteration (E-step + M-step + convergence test) over the
resident read-signature x haplotype matrix of BASELINE.json config 2: a 3-way
synthetic mixture (H1 50% / L3e 30% / U5a1 20%), 1M fragments of 300 bp reduced
to unique signatures in the reference's row order (string-sorted,
preprocess.py:219), against all 5408 Phylotree Build 17 haplotypes.  Under
torchrun every rank builds its own 1M-fragment shard (weak scaling) and the H
column sums are exchanged once per iteration by peer stores inside the tail
kernel (ncclAllReduce when peer access is missing).

One JSON line is printed by rank 0:
  value     matrix cells per second through EM iterations, inputs resident in HBM
  e2e       same metric through the drop-in call mixemt_b200.run_em(pageable host
            ndarray, weights, args) run to convergence with the reference's default
            options: host->device copy of the matrix, class tiles, all iterations,
            read-matrix kernel and the device->host copy of the N x H result inside
            the timed region (after one short untimed call); e2e.breakdown_ms
  roofline  the dominant kernel against the measured HBM copy bandwidth, two readings
            (frac_contract: 8 B per matrix cell, SURVEY 8d; frac_traffic: the bytes of
            the kernel's own data layout), roofline.per_kernel for every kernel of an
            iteration, the fp64-row pass of the same matrix and the build kernel
  restart_sweep  BASELINE.json config 4: --restarts (100) random-init runs to
            convergence on the config-2 matrix; under torchrun the matrix is
            replicated and the restarts are dealt over the GPUs
  parity    (N > 1) the multi-GPU path -- class tiles per shard + peer exchange --
            against the CPU oracle on the whole matrix
  strong_scaling  (N > 1) one config-2 matrix row-split over the N GPUs
  config3   (N = 8, or --config3) BASELINE.json config 3: 5-way mixture, 1.25 M
            signature rows per GPU (10 M rows x 5408 on eight)
  cpu_baseline  the CPU oracle port (C + OpenMP, all host threads) on a row sample
--impl reference times the UNMODIFIED reference's em_step (staged copy oracle/_ref,
see oracle/stage_ref.py) on one core.  --rows N replaces the workload by N
undeduplicated rows per GPU (config-3 shard sizes).  --dump-outputs DIR writes the
log-proportions of the last timed step to DIR/lnprops.npy (bench_outputs/ in the tree is
git-ignored for this); the workload and the start are seeded, so two builds run with the
same arguments can be compared on it.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "em_matrix_cells_per_s"
UNIT = "cells/s"
MIXTURE = [("H1", 0.5), ("L3e", 0.3), ("U5a1", 0.2)]
GOLDEN = os.path.join(ROOT, "tests", "golden")


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--fragments", type=int, default=1000000,
                    help="fragments per GPU (config 2: 1M)")
    ap.add_argument("--rows", type=int, default=0,
                    help="signature rows per GPU drawn without dedupe (config-3 shard sizes, "
                         "e.g. 1250000); 0 = the config-2 workload of --fragments")
    ap.add_argument("--seed", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the restart-sweep leg")
    ap.add_argument("--restarts", type=int, default=100,
                    help="restarts of the config-4 leg (BASELINE.json: 100)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (N > 1)")
    ap.add_argument("--no-config3", action="store_true", help="skip the config-3 leg (N = 8)")
    ap.add_argument("--config3", action="store_true", help="run the config-3 leg at any N > 1")
    ap.add_argument("--config3-rows", type=int, default=1250000,
                    help="signature rows per GPU of the config-3 leg")
    ap.add_argument("--pageable-result", action="store_true",
                    help="e2e: leave the result in pageable memory (no pinned pool)")
    ap.add_argument("--cpu-rows", type=int, default=0, help="row sample of the CPU legs (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed EM iterations computed in their last step to "
                         "DIR/<name>.npy, to compare two builds output for output (e.g. "
                         "bench_outputs, which git ignores)")
    opts = ap.parse_args()
    if opts.dump_outputs and opts.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return opts


MIXTURE5 = [("H1", 0.6), ("L3e", 0.25), ("U5a1", 0.1), ("M7", 0.04), ("D4a", 0.01)]


def load_workload(fragments, seed, strings=False, rows=0):
    from mixemt_b200.phylo_tables import PhyloTables
    from mixemt_b200 import synth
    phylo = PhyloTables.load(os.path.join(GOLDEN, "phylotree17.npz"))
    haps = sorted(phylo.hap_var)
    if rows > 0:
        mix = synth.random_rows(phylo, phylo.refseq, MIXTURE5, rows, seed=seed)
    else:
        mix = synth.make_mixture(phylo, phylo.refseq, MIXTURE, fragments, seed=seed,
                                 strings=strings)
    return phylo, haps, mix


def workload_name(fragments, n_rows, n_hap, rows=0):
    if rows > 0:
        return ("config3 shard: 5-way mixture H1/L3e/U5a1/M7/D4a 60/25/10/4/1, %d signature rows "
                "per GPU x %d Phylotree-17 haplotypes (fp64 matrix %.2f GB per GPU)"
                % (n_rows, n_hap, n_rows * n_hap * 8 / 1e9))
    return ("config2: 3-way mixture H1/L3e/U5a1 50/30/20, %d fragments x 300bp -> %d unique "
            "signatures x %d Phylotree-17 haplotypes (fp64 matrix %.2f GB)"
            % (fragments, n_rows, n_hap, n_rows * n_hap * 8 / 1e9))


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler(object):
    """Samples SM clock and throttle reasons of one GPU while a region runs."""

    def __init__(self, index, period=0.1):
        # NVML queries take the driver's global lock: polling much faster than this slows
        # the cudaMalloc / copy calls of the region being sampled (measured: 20 ms polling
        # turned an 8 ms em_create into 120-630 ms)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = [("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"),
                 ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                 ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"),
                 ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap"),
                 ("hw_power_brake", "nvmlClocksThrottleReasonHwPowerBrakeSlowdown")]
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for label, attr in names:
                    bit = getattr(nv, attr, 0)
                    if bit and (mask & bit):
                        self.reasons.add(label)
            except Exception:
                pass
            time.sleep(self.period)

    def __enter__(self):
        if self.nv is not None and not os.environ.get("BENCH_NO_SAMPLER"):
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def ncu_traffic():
    """dram bytes per launch of the pass kernel from the committed ncu capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return None


# ---------------------------------------------------------------------------
# CPU legs (the only places bench.py may touch oracle/)
# ---------------------------------------------------------------------------
def cpu_sample_matrix(rows, seed):
    """A row sample of the config-2 matrix, built by the CPU oracle itself."""
    from mixemt_b200.preprocess import HapVarBaseMatrix
    from oracle import oracle_c
    phylo, haps, mix = load_workload(max(4000, rows * 8), seed)
    tables = HapVarBaseMatrix(phylo.refseq, phylo, haps).pack()
    csr = mix.csr(tables)
    rows = min(rows, csr.n_rows)
    from mixemt_b200.preprocess import SignatureCSR
    sub = SignatureCSR(csr.row_ptr[:rows + 1].copy(), csr.pos_idx[:csr.row_ptr[rows]],
                       csr.base_code[:csr.row_ptr[rows]])
    t0 = time.perf_counter()
    mat, _ = oracle_c.build_matrix(tables, sub, want_counts=False)
    build_s = time.perf_counter() - t0
    return mat, mix.weights[:rows].astype(np.float64), len(haps), build_s


def cpu_baseline_port(budget_s=15.0):
    """C/OpenMP oracle em_step on a row sample, all host threads."""
    from oracle import oracle_c
    cores = os.cpu_count() or 1
    rows = 2048
    mat, wts, h, build_s = cpu_sample_matrix(rows, seed=2)
    lnp = np.log(np.random.RandomState(0).dirichlet([1.0] * h))
    oracle_c.em_step(mat, wts, lnp)  # warm-up
    times = []
    t_end = time.perf_counter() + budget_s
    while len(times) < 3 or (time.perf_counter() < t_end and len(times) < 20):
        t0 = time.perf_counter()
        oracle_c.em_step(mat, wts, lnp)
        times.append(time.perf_counter() - t0)
    best = min(times)
    return {"value": mat.size / best, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "oracle.c em_step (OpenMP, %d threads) on %d rows x %d haplotypes of the "
                      "config-2 matrix, best of %d" % (cores, mat.shape[0], h, len(times)),
            "build_cells_per_s": mat.size / build_s}


def run_reference(opts):
    """CPU reference arm: the UNMODIFIED reference's own ``mixemt.em.em_step``
    (em.py:57-91), one core like the reference (SURVEY F10), on a bounded row
    sample of the config-2 workload.  The reference is imported from
    /root/reference when mounted, else from the copy oracle/stage_ref.py staged
    under oracle/_ref (git-ignored; travels to the GPU box).  Nothing of
    mixemt_b200 is imported on this path: the sample comes from oracle/workload.py
    (reference Phylotree + reduce_reads, matrix by the numpy restatement).  Only
    when no reference is reachable the numpy/scipy restatement is timed instead
    (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import scipy
    from oracle import refload, workload, oracle_np
    assert "mixemt_b200" not in sys.modules
    have_ref = refload.available()
    if have_ref:
        _, ref_pre, ref_em = refload.load()
        step = ref_em.em_step
        kind = "reference"
        what = ("unmodified mixemt.em.em_step (%s)"
                % ("staged copy oracle/_ref" if refload.staged() else refload.REFERENCE_ROOT))
    else:
        step = oracle_np.em_step_scipy
        kind = "port"
        what = "numpy/scipy restatement of em.em_step (oracle_np.em_step_scipy; no reference found)"
    if not have_ref:
        raise SystemExit(json.dumps({"impl": "reference", "unavailable":
                                     "reference neither mounted nor staged (oracle/stage_ref.py)"}))
    budget = 100.0
    rows = opts.cpu_rows or 256
    phylo, refseq, reads, haps, wts, mat = workload.sample_matrix(rows, seed=opts.seed)
    h = len(haps)
    lnp = np.log(np.random.RandomState(0).dirichlet([1.0] * h))
    if not opts.cpu_rows:
        t0 = time.perf_counter()
        step(mat, wts, lnp, np.empty_like(mat))
        per_row = (time.perf_counter() - t0) / mat.shape[0]
        rows = int(max(128, min(8192, budget / ((opts.steps + opts.warmup) * per_row))))
        phylo, refseq, reads, haps, wts, mat = workload.sample_matrix(rows, seed=opts.seed)
    mix = np.empty_like(mat)
    for _ in range(opts.warmup):
        step(mat, wts, lnp, mix)
    t0 = time.perf_counter()
    for _ in range(opts.steps):
        step(mat, wts, lnp, mix)
    total = time.perf_counter() - t0
    value = mat.size * opts.steps / total
    # kernel 1 of the reference: its own build_em_matrix on a few rows (SURVEY 8d: >= 40 rows)
    build = None
    if have_ref:
        nb = min(40, len(reads))
        t0 = time.perf_counter()
        ref_mat = ref_pre.build_em_matrix(refseq, phylo, reads[:nb], haps,
                                          argparse.Namespace(verbose=False))
        build_s = time.perf_counter() - t0
        build = {"cells_per_s": ref_mat.size / build_s, "rows": nb, "seconds": build_s,
                 "call": "unmodified mixemt.preprocess.build_em_matrix",
                 "sample_matrix_bit_identical": bool(np.array_equal(ref_mat, mat[:nb]))}
    sample = ("%s on %d rows x %d haplotypes of the config-2 matrix, numpy %s scipy %s, 1 thread "
              "of %d cores" % (what, mat.shape[0], h, np.__version__, scipy.__version__,
                               os.cpu_count() or 1))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
            "n_gpus": opts.gpus, "steps": opts.steps, "warmup": opts.warmup,
            "ms_per_step": 1e3 * total / opts.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "config2: 3-way mixture H1/L3e/U5a1 50/30/20, 1M fragments x "
                       "300bp x %d Phylotree-17 haplotypes [CPU arm: bounded sample of %d "
                       "signature rows of it per step]" % (h, mat.shape[0])},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind,
                             "sample": sample, "build": build},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------
def csr_rows(csr, lo, hi):
    """Rows [lo, hi) of a SignatureCSR."""
    from mixemt_b200.preprocess import SignatureCSR
    a, b = int(csr.row_ptr[lo]), int(csr.row_ptr[hi])
    return SignatureCSR(csr.row_ptr[lo:hi + 1] - csr.row_ptr[lo], csr.pos_idx[a:b],
                        csr.base_code[a:b])


def run_b200(opts):
    import ctypes
    import torch
    import torch.distributed as dist
    import mixemt_b200
    from mixemt_b200 import _lib, em as b200_em, sharding
    from mixemt_b200._lib import lib, check, ptr
    from mixemt_b200.preprocess import HapVarBaseMatrix, build_matrix_from_csr
    from mixemt_b200.runtime import get_context

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    ctx = get_context()
    if world > 1:
        ctx.init_comm_from_torch()

    def barrier():
        torch.cuda.synchronize()
        ctx.synchronize()
        if world > 1:
            dist.barrier()

    def reduce_ranks(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce_ranks(x, dist.ReduceOp.MAX if world > 1 else None)

    def sum_over_ranks(x):
        return reduce_ranks(x, dist.ReduceOp.SUM if world > 1 else None)

    def guarded(name, fn, *fargs):
        """An optional leg must not take the bench line down: its error is reported under its
        key.  (The kernels of the peer exchange time out instead of hanging, so a rank that
        fails alone costs the others a bounded wait.)"""
        try:
            return fn(*fargs)
        except Exception as exc:
            sys.stderr.write("[bench] rank %d: leg %s failed: %r\n" % (rank, name, exc))
            return {"error": "%s: %s" % (type(exc).__name__, exc)}

    def new_session(dmat, weights, sharded):
        sess = ctypes.c_void_p()
        check(lib.mxb_em_create(ctx.handle, dmat.handle, ptr(weights), 1 if sharded else 0,
                                ctypes.byref(sess)))
        nbytes, flag = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nbytes), ctypes.byref(flag)))
        return sess, int(nbytes.value), flag.value == 0     # flag 0: class tiles, -1: fp64 rows

    def profile(sess, iters):
        ms = (ctypes.c_float * 4)()
        check(lib.mxb_em_profile(sess, iters, ms))
        return {"class_sums": ms[0], "pass": ms[1], "gather": ms[2], "tail": ms[3]}

    peak, peak_src = measured_peak()
    sharded = world > 1

    # ---- workload: every rank its own shard (weak scaling) ---------------------------
    phylo, haps, mix = load_workload(opts.fragments, opts.seed + rank, rows=opts.rows)
    if opts.rows > 400000:
        opts.no_e2e = True      # the drop-in call needs two N x H host arrays
    tables = HapVarBaseMatrix(phylo.refseq, phylo, haps).pack()
    csr = mix.csr(tables)
    n, h = csr.n_rows, len(haps)
    ld = ((h + 15) // 16) * 16
    weights = mix.weights.astype(np.float64)

    # ---- kernel 1: build (device resident) --------------------------------------------
    build_ms = []
    dmat = None
    for _ in range(3):
        if dmat is not None:
            dmat.free()
        _, _, dmat, ms = build_matrix_from_csr(tables, csr, ctx=ctx, want_host=False,
                                               keep_device=True)
        build_ms.append(ms)
    build_best = min(build_ms)

    # ---- kernel 2: EM iterations, inputs resident ---------------------------------------
    sess, pass_bytes, tiled = new_session(dmat, weights, sharded)
    lnp0 = np.log(np.random.RandomState(1).dirichlet([1.0] * h))
    check(lib.mxb_em_set_lnprops(sess, ptr(lnp0)))
    el = ctypes.c_float()
    if opts.warmup > 0:
        check(lib.mxb_em_iterate_fixed(sess, opts.warmup, ctypes.byref(el), None))
    with ClockSampler(local) as clocks:
        barrier()
        l0 = ctx.launch_count
        t0 = time.perf_counter()
        check(lib.mxb_em_iterate_fixed(sess, opts.steps, ctypes.byref(el), None))
        barrier()
        wall = time.perf_counter() - t0
        launches = ctx.launch_count - l0
        dev_s = max_over_ranks(el.value / 1e3)
        # what the last timed step handed back, read before profile() iterates on
        # (mxb_em_iterate_fixed fails unless all opts.steps iterations ran)
        if opts.dump_outputs and rank == 0:
            lnprops = np.empty(h)
            check(lib.mxb_em_get_lnprops(sess, 0, ptr(lnprops)))
        # per-kernel attribution (an event between the kernels of every iteration), rank-local
        kern = profile(sess, min(opts.steps, 100))
    cells_total = sum_over_ranks(float(n) * h)
    value = cells_total * opts.steps / dev_s
    lib.mxb_em_destroy(sess)

    # the same iterations over plain fp64 rows (MXB_EM_NO_PACK=1): the pass that sits at the HBM
    # roofline on the 8 bytes per cell of SURVEY section 8(d)
    fp64_bytes = float(n) * ld * 8
    os.environ["MXB_EM_NO_PACK"] = "1"
    try:
        sess2, bytes2, _ = new_session(dmat, weights, sharded)
        check(lib.mxb_em_set_lnprops(sess2, ptr(lnp0)))
        check(lib.mxb_em_iterate_fixed(sess2, max(3, opts.warmup), ctypes.byref(el), None))
        barrier()
        k2 = min(opts.steps, 50)
        check(lib.mxb_em_iterate_fixed(sess2, k2, ctypes.byref(el), None))
        fp64_step_ms = el.value / k2
        kern64 = profile(sess2, k2)
        lib.mxb_em_destroy(sess2)
    finally:
        os.environ.pop("MXB_EM_NO_PACK", None)

    # ---- roofline: both readings, per kernel (VERDICT r1 item 7) ---------------------
    # frac_contract: SURVEY 8(d)'s 8 bytes per matrix cell over the kernel's time and the
    # measured HBM peak; frac_traffic: the bytes the kernel actually has to read (its data
    # layout, = ncu dram bytes where a capture is committed) over the same.
    traffic = ncu_traffic() or {}
    on_cfg2 = opts.rows == 0 and opts.fragments == 1000000

    def entry(name, ms, layout_bytes, traffic_key=None, contract_bytes=fp64_bytes):
        if not ms:
            return None
        t = ms / 1e3
        e = {"kernel": name, "ms_per_launch": ms,
             "contract_bytes_per_launch": contract_bytes,
             "layout_bytes_per_launch": layout_bytes,
             "frac_contract": contract_bytes / t / 1e9 / peak if contract_bytes else None,
             "frac_traffic": layout_bytes / t / 1e9 / peak,
             "achieved_GBs": layout_bytes / t / 1e9}
        if traffic_key and on_cfg2:
            e["ncu_dram_bytes_per_launch"] = traffic.get(traffic_key)
        return e

    n_batches = (n + 127) // 128
    map_bytes = float(n_batches) * ((h + 7) // 8 * 8) * 2
    tile_pass_bytes = pass_bytes - 3 * map_bytes if tiled else pass_bytes
    pass_name = ("tile_pass_kernel (class tiles: rows x column classes per 128-row batch)"
                 if tiled else "em_pass_fast_kernel (fp64 rows)")
    kernels = [entry(pass_name, kern["pass"], tile_pass_bytes,
                     "tile_pass_kernel_bytes_per_launch" if tiled
                     else "em_pass_fast_kernel_bytes_per_launch"),
               entry("tile_pi_kernel (class sums of the proportions)", kern["class_sums"],
                     2 * map_bytes, "tile_pi_kernel_bytes_per_launch", 0.0),
               entry("tile_gather_kernel (class sums back to columns)", kern["gather"],
                     map_bytes, "tile_gather_kernel_bytes_per_launch", 0.0),
               entry("em_finish_kernel (M-step, convergence test%s)"
                     % (", peer exchange" if sharded else ""), kern["tail"],
                     (32 if tiled else 148) * ld * 8.0, None, 0.0),
               entry("em_pass_fast_kernel (same matrix as fp64 rows, MXB_EM_NO_PACK=1)",
                     kern64["pass"], fp64_bytes, "em_pass_fast_kernel_bytes_per_launch"),
               entry("build_matrix_kernel (kernel 1, N x H x 8 B written once)", build_best,
                     fp64_bytes, "build_matrix_kernel_bytes_per_launch")]
    kernels = [k for k in kernels if k]
    step_ms = 1e3 * dev_s / opts.steps
    dom = kernels[0]
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "unit": "GB/s", "peak": peak,
                "peak_source": peak_src,
                # the dominant kernel on the bytes its layout holds (what it must read)
                "achieved": dom["achieved_GBs"], "frac": dom["frac_traffic"],
                "frac_traffic": dom["frac_traffic"], "frac_contract": dom["frac_contract"],
                "algorithmic_bytes_per_launch": dom["layout_bytes_per_launch"],
                "contract_bytes_per_launch": fp64_bytes,
                "ms_per_launch": dom["ms_per_launch"],
                "traffic": dom.get("ncu_dram_bytes_per_launch"),
                # the whole iteration against the contract bytes (8 B x N x H per iteration)
                "iteration": {"ms": step_ms, "frac_contract": fp64_bytes / (step_ms / 1e3) / 1e9 / peak,
                              "layout_bytes": float(pass_bytes),
                              "frac_traffic": pass_bytes / (step_ms / 1e3) / 1e9 / peak},
                "fp64_rows_iteration_ms": fp64_step_ms,
                "per_kernel": kernels,
                "note": "frac_contract = 8 B x cells / time / peak (SURVEY 8d); frac_traffic = "
                        "bytes of the kernel's own data layout / time / peak; every frac can be "
                        "recomputed from *_bytes_per_launch, ms_per_launch and peak"}

    # ---- multi-GPU legs ------------------------------------------------------------------
    parity = strong = config3 = None
    if world > 1:
        parity = guarded("parity", parity_leg, ctx, tables, phylo, haps, rank, world, barrier)
        if not opts.no_strong and opts.rows == 0:
            strong = guarded("strong_scaling", strong_leg, ctx, tables, phylo, haps, opts, rank,
                             world, barrier, max_over_ranks, lnp0)
        if (world == 8 or opts.config3) and opts.rows == 0 and not opts.no_config3:
            dmat.free()
            dmat = None
            ctx.trim()
            config3 = guarded("config3", config3_leg, ctx, tables, phylo, haps, opts, rank, world,
                              barrier, max_over_ranks, sum_over_ranks, peak)
            ctx.trim()
            _, _, dmat, _ = build_matrix_from_csr(tables, csr, ctx=ctx, want_host=False,
                                                  keep_device=True)

    # ---- config 4: restart sweep to convergence ------------------------------------------
    # n_multi random-init restarts (default 100, fixed seed) on the config-2 matrix; under
    # torchrun the matrix of rank 0's seed is replicated, the restarts are dealt in contiguous
    # blocks (args.b200_shard = "restarts") and combined like em.py:145-163 combines them.
    def sweep_leg():
        n_multi = opts.restarts
        inits = np.log(np.random.RandomState(3).dirichlet([1.0] * h, size=n_multi))
        sargs = argparse.Namespace(verbose=False, init_alpha=1.0, tolerance=1e-4, max_iter=10000,
                                   n_multi=n_multi, b200_shard="restarts" if world > 1 else None)
        smat, swts = dmat, weights
        if world > 1 and rank != 0:
            _, _, mix0 = load_workload(opts.fragments, opts.seed)
            _, _, smat, _ = build_matrix_from_csr(tables, mix0.csr(tables), ctx=ctx,
                                                  want_host=False, keep_device=True)
            swts = mix0.weights.astype(np.float64)
        wargs = argparse.Namespace(**vars(sargs))
        wargs.max_iter, wargs.n_multi = 3, 2 * world      # first-use costs of the restart path
        b200_em.run_em_device(smat, swts, wargs, want_host=False, inits=inits[:2 * world])
        barrier()
        t0 = time.perf_counter()
        s_props, _, s_info, _ = b200_em.run_em_device(smat, swts, sargs, want_host=False,
                                                      inits=inits)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        iters_total = sum_over_ranks(float(sum(s_info["iterations"])))
        out = {"n_multi": n_multi, "seconds": dt, "restarts_per_s": n_multi / dt,
               "iterations_total": iters_total,
               "cell_updates_per_s": float(smat.shape[0]) * h * iters_total / dt,
               "props_sum": float(s_props.sum()),
               "top_haplogroups": [[haps[i], float(s_props[i])]
                                   for i in np.argsort(s_props)[::-1][:3]],
               "call": "run_em(config-2 matrix, n_multi=%d, tolerance 1e-4, fixed seed) to "
                       "convergence, read matrices folded on the device" % n_multi,
               "parallelism": ("matrix replicated, restarts in contiguous blocks over %d GPUs, "
                               "read matrices combined by an all-to-all of row shards + local "
                               "logaddexp fold" % world) if world > 1 else "single GPU"}
        if smat is not dmat:
            smat.free()
        return out

    sweep = None
    if not opts.no_sweep and opts.rows == 0 and opts.restarts > 0:
        sweep = guarded("restart_sweep", sweep_leg)

    # ---- e2e: the drop-in call with host buffers -----------------------------------------
    # Input: an ordinary (pageable) numpy array, like a caller of the reference API holds.
    # Result: pooled pinned host memory, reserved before the untimed warm-up call (what a
    # service does once; MIXEMT_B200_PINNED / reserve_pinned, INTEGRATION.md).
    def e2e_leg():
        host = np.empty((n, h), dtype=np.float64)      # pageable
        dmat.to_host(out=host)
        if not opts.pageable_result:
            _lib.reserve_pinned(host.nbytes, 1)
        args = argparse.Namespace(verbose=False, init_alpha=1.0, tolerance=1e-4, max_iter=10000,
                                  n_multi=1, b200_shard="rows" if world > 1 else None)
        import io
        import re
        import contextlib
        warm = argparse.Namespace(**vars(args))
        warm.max_iter = 20
        np.random.seed(opts.seed)
        mixemt_b200.run_em(host, weights, warm)
        np.random.seed(opts.seed)
        args.verbose = True
        buf = io.StringIO()
        check(lib.mxb_stage_timing(1))
        with ClockSampler(local) as clocks_e2e:
            barrier()
            t0 = time.perf_counter()
            with contextlib.redirect_stderr(buf):
                props, read_mix = mixemt_b200.run_em(host, weights, args)
            barrier()
            e2e_s = max_over_ranks(time.perf_counter() - t0)
        stage = (ctypes.c_double * 6)()
        check(lib.mxb_stage_times(stage, 6))
        check(lib.mxb_stage_timing(0))
        found = re.findall(r"Converged! \((\d+)\)", buf.getvalue())
        iters = int(found[0]) if found else args.max_iter
        top = np.argsort(props)[::-1][:3]
        out = {"value": cells_total * iters / e2e_s, "unit": UNIT,
               "h2d_bytes_per_step": (host.nbytes + weights.nbytes + 8 * h) / iters,
               "d2h_bytes_per_step": (read_mix.nbytes + 8 * h) / iters,
               "call": "mixemt_b200.run_em(pageable host ndarray, weights, args) to convergence "
                       "(tolerance 1e-4, Dirichlet(1) start, seed %d)" % opts.seed,
               "input_memory": "pageable numpy array",
               "result_memory": ("pooled pinned block (reserved before the warm-up call)"
                                 if read_mix.base is not None else "pageable numpy array"),
               "iterations": iters, "seconds": e2e_s,
               "breakdown_ms": {"h2d": stage[0], "setup_tiles": stage[1], "iterate": stage[2],
                                "read_mix": stage[3], "d2h": stage[4], "release": stage[5],
                                "note": "rank 0, wall clock between stream synchronisations"},
               "h2d_bytes": host.nbytes + weights.nbytes, "d2h_bytes": read_mix.nbytes,
               "em_iters_per_s": iters / e2e_s,
               "top_haplogroups": [[haps[i], float(props[i])] for i in top],
               "clocks": clocks_e2e.summary()}
        del host, read_mix
        return out

    e2e = None
    if not opts.no_e2e:
        e2e = guarded("e2e", e2e_leg)
    dmat.free()

    # ---- e2e of kernel 1: the drop-in build_em_matrix(signature strings) -> host ndarray ----
    def build_e2e_leg():
        _, _, smix = load_workload(opts.fragments, opts.seed, strings=True)
        bargs = argparse.Namespace(verbose=False)
        mixemt_b200.build_em_matrix(phylo.refseq, phylo, smix.signatures[:2000], haps, bargs)
        barrier()
        t0 = time.perf_counter()
        mat = mixemt_b200.build_em_matrix(phylo.refseq, phylo, smix.signatures, haps, bargs)
        barrier()
        dt = time.perf_counter() - t0
        out = {"seconds": dt, "cells_per_s": mat.size / dt, "d2h_bytes": mat.nbytes,
               "result_memory": "pooled pinned block" if mat.base is not None
               else "pageable numpy array",
               "call": "mixemt_b200.build_em_matrix(refseq, phylo, %d signature strings, "
                       "%d haplogroups, args) -> host ndarray: table packing, string "
                       "parsing, kernel 1 and the %.2f GB device->host copy inside"
                       % (len(smix.signatures), h, mat.nbytes / 1e9)}
        del mat
        return out

    build_e2e = None
    if not opts.no_e2e and world == 1 and opts.rows == 0:
        build_e2e = guarded("build.e2e", build_e2e_leg)

    cpu = None
    if rank == 0 and world == 1 and not opts.no_cpu:
        try:
            cpu = cpu_baseline_port()
        except Exception as exc:  # the baseline must not take the bench down
            cpu = {"error": repr(exc)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world,
                "steps": opts.steps, "warmup": opts.warmup,
                "ms_per_step": step_ms, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_name(opts.fragments, n, h, opts.rows),
                           "rows_per_gpu": n, "haplotypes": h,
                           "row_order": "string-sorted signatures, as build_em_input hands them "
                                        "over (preprocess.py:219)",
                           "layout": "class tiles" if tiled else "fp64 rows",
                           "parallelism":
                           ("rows sharded x%d, H column sums exchanged per iteration by %s"
                            % (world, "peer stores inside the EM tail kernel (CUDA IPC over NVLink)"
                               if lib.mxb_comm_p2p_enabled(ctx.handle) else "ncclAllReduce(fp64)"))
                           if world > 1 else "single GPU",
                           "l2_policy": ("%.3f GB read per iteration, larger than the 126 MB L2: "
                                         "no flush needed" % (pass_bytes / 1e9))},
                "em_iters_per_s": opts.steps / dev_s,
                "wall_ms_per_step": 1e3 * wall / opts.steps,
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "restart_sweep": sweep, "parity": parity, "strong_scaling": strong,
                "config3": config3,
                "gpu_launches": int(launches), "clocks": clocks.summary(),
                "build": {"ms": build_best, "cells_per_s": float(n) * h / (build_best / 1e3),
                          "write_GBs": float(n) * h * 8 / (build_best / 1e3) / 1e9,
                          "frac_of_hbm_peak": float(n) * h * 8 / (build_best / 1e3) / 1e9 / peak,
                          "e2e": build_e2e},
                "versions": {"numpy": np.__version__, "torch": torch.__version__}}
        print(json.dumps(line))
        if opts.dump_outputs:
            # the H log-proportions (float64) the last timed step produced, as
            # mxb_em_get_lnprops hands them to a caller of the session
            os.makedirs(opts.dump_outputs, exist_ok=True)
            np.save(os.path.join(opts.dump_outputs, "lnprops.npy"), lnprops)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def parity_leg(ctx, tables, phylo, haps, rank, world, barrier):
    """The path the multi-GPU numbers run on -- class tiles on every rank's row shard, column
    sums exchanged inside the tail kernel -- against the CPU oracle on the whole matrix
    (oracle/ as the checker, rank 0; VERDICT r1 item 1c)."""
    import ctypes
    from mixemt_b200 import em as b200_em, sharding, synth
    from mixemt_b200._lib import lib, check, ptr
    from mixemt_b200.preprocess import build_matrix_from_csr
    mix = synth.make_mixture(phylo, phylo.refseq, MIXTURE, 6000, seed=11, strings=False)
    csr = mix.csr(tables)
    n, h = csr.n_rows, len(haps)
    lo, hi = sharding.row_shard(n, rank, world)
    _, _, shard, _ = build_matrix_from_csr(tables, csr_rows(csr, lo, hi), ctx=ctx,
                                           want_host=False, keep_device=True)
    wts = mix.weights.astype(np.float64)
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, shard.handle, ptr(wts[lo:hi]), 1, ctypes.byref(sess)))
    nb, flag = ctypes.c_int64(), ctypes.c_int64()
    check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nb), ctypes.byref(flag)))
    lib.mxb_em_destroy(sess)
    inits = np.log(np.random.RandomState(12).dirichlet([1.0] * h, size=1))
    args = argparse.Namespace(verbose=False, init_alpha=1.0, tolerance=1e-7, max_iter=120,
                              n_multi=1, b200_shard="rows")
    props, _, info, mix_dev = b200_em.run_em_device(shard, wts[lo:hi], args, inits=inits,
                                                    want_host=False, keep_device=True)
    votes = mix_dev.argmax_rows()
    mix_dev.free()
    shard.free()
    out = None
    if rank == 0:
        from oracle import oracle_c
        full, _ = oracle_c.build_matrix(tables, csr, want_counts=False)
        o_props, o_mix, o_iters = oracle_c.run_em(full, wts, inits, args.max_iter, args.tolerance)
        d = float(np.abs(props - o_props).max())
        same_votes = bool(np.array_equal(votes, np.argmax(o_mix[lo:hi], 1)))
        it_equal = list(o_iters) == info["iterations"]
        out = {"ok": bool(d < 1e-6 and it_equal and same_votes), "max_abs_dprops": d,
               "iterations_equal": it_equal, "iterations": info["iterations"],
               "argmax_votes_equal_rank0_shard": same_votes,
               "layout": "class tiles" if flag.value == 0 else "fp64 rows",
               "rows": n, "checker": "oracle.c run_em on the whole matrix (CPU, rank 0)"}
    barrier()
    return out


def strong_leg(ctx, tables, phylo, haps, opts, rank, world, barrier, max_over_ranks, lnp0):
    """One sample (the config-2 matrix of --seed) row-split over the ranks: what a user with
    one BAM gets from N GPUs."""
    import ctypes
    from mixemt_b200 import sharding
    from mixemt_b200._lib import lib, check, ptr
    from mixemt_b200.preprocess import build_matrix_from_csr
    _, _, mix = load_workload(opts.fragments, opts.seed)
    csr = mix.csr(tables)
    n, h = csr.n_rows, len(haps)
    lo, hi = sharding.row_shard(n, rank, world)
    _, _, shard, _ = build_matrix_from_csr(tables, csr_rows(csr, lo, hi), ctx=ctx,
                                           want_host=False, keep_device=True)
    wts = mix.weights.astype(np.float64)[lo:hi].copy()
    sess = ctypes.c_void_p()
    check(lib.mxb_em_create(ctx.handle, shard.handle, ptr(wts), 1, ctypes.byref(sess)))
    check(lib.mxb_em_set_lnprops(sess, ptr(lnp0)))
    el = ctypes.c_float()
    check(lib.mxb_em_iterate_fixed(sess, max(3, opts.warmup), ctypes.byref(el), None))
    barrier()
    check(lib.mxb_em_iterate_fixed(sess, opts.steps, ctypes.byref(el), None))
    barrier()
    ms = max_over_ranks(el.value) / opts.steps
    lib.mxb_em_destroy(sess)
    shard.free()
    return {"rows_total": n, "rows_per_gpu": hi - lo, "ms_per_iteration": ms,
            "em_iters_per_s": 1e3 / ms, "cells_per_s": float(n) * h * 1e3 / ms,
            "workload": "the config-2 matrix of one sample row-split over %d GPUs" % world}


def config3_leg(ctx, tables, phylo, haps, opts, rank, world, barrier, max_over_ranks,
                sum_over_ranks, peak):
    """BASELINE.json configs[2]: 5-way low-fraction mixture, 10 M signature rows row-sharded
    over 8 GPUs (1.25 M rows x 5408 per GPU, rows grouped like the reference orders them)."""
    import ctypes
    import torch
    from mixemt_b200 import synth
    from mixemt_b200._lib import lib, check, ptr
    from mixemt_b200.preprocess import build_matrix_from_csr
    rows = opts.config3_rows
    mix = synth.random_rows(phylo, phylo.refseq, MIXTURE5, rows, seed=100 + rank)
    csr = mix.csr(tables)
    n, h = csr.n_rows, len(haps)
    _, _, dmat, build_ms = build_matrix_from_csr(tables, csr, ctx=ctx, want_host=False,
                                                 keep_device=True)
    wts = mix.weights.astype(np.float64)
    sess = ctypes.c_void_p()
    try:
        t0 = time.perf_counter()
        check(lib.mxb_em_create(ctx.handle, dmat.handle, ptr(wts), 1, ctypes.byref(sess)))
        ctx.synchronize()
        setup_s = time.perf_counter() - t0
        nb, flag = ctypes.c_int64(), ctypes.c_int64()
        check(lib.mxb_em_pass_bytes(sess, ctypes.byref(nb), ctypes.byref(flag)))
        lnp0 = np.log(np.random.RandomState(1).dirichlet([1.0] * h))
        check(lib.mxb_em_set_lnprops(sess, ptr(lnp0)))
        el = ctypes.c_float()
        check(lib.mxb_em_iterate_fixed(sess, 3, ctypes.byref(el), None))
        barrier()
        steps = min(opts.steps, 50)
        check(lib.mxb_em_iterate_fixed(sess, steps, ctypes.byref(el), None))
        barrier()
        ms = max_over_ranks(el.value) / steps
        free_b, total_b = torch.cuda.mem_get_info()
    finally:                    # a shard is 54 GB: give it back also when the leg fails
        if sess:
            lib.mxb_em_destroy(sess)
        dmat.free()
        ctx.trim()
    ld = ((h + 15) // 16) * 16
    cells = sum_over_ranks(float(n) * h)
    contract = float(n) * ld * 8
    return {"workload": "config3: 5-way mixture H1/L3e/U5a1/M7/D4a 60/25/10/4/1, %d signature "
                        "rows per GPU x %d haplogroups on %d GPUs (%.0f GB of fp64 cells in all)"
                        % (n, h, world, cells * 8 / 1e9),
            "rows_per_gpu": n, "layout": "class tiles" if flag.value == 0 else "fp64 rows",
            "ms_per_iteration": ms, "cells_per_s": cells * 1e3 / ms,
            "bytes_read_per_iteration_per_gpu": float(nb.value),
            "frac_contract": contract / (ms / 1e3) / 1e9 / peak,
            "frac_traffic": nb.value / (ms / 1e3) / 1e9 / peak,
            "build_ms": build_ms, "session_setup_s": setup_s,
            "hbm_free_GB_during_iterations": free_b / 1e9, "hbm_total_GB": total_b / 1e9}


def main():
    opts = parse_args()
    if opts.impl == "reference":
        run_reference(opts)
    else:
        run_b200(opts)


if __name__ == "__main__":
    main()
