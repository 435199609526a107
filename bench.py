#!/usr/bin/env python
"""bench.py -- headline benchmark of the packed-genotype hot path (BASELINE.json metric:
"genotypes/sec in bed_prodVec").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step is one bed_prodVec (X~ . y, binomial center/scale, all rows, all columns) over the resident synthetic
.bed.  Workload (default, `cfg5`) = BASELINE.json configs[4], the matrix the metric is quoted on: UKBB-shaped
487,000 samples x 1,100,000 SNPs (134 GB packed, SNP-major copy only: it fits one 180 GB GPU), SNP columns split
over the N ranks (STRONG scaling), every step ending in one all-reduce of the n-vector of partial products; the
same line carries the second headline, bed_randomSVD(k = 20) wall time.  `--workload cfg2` is configs[1]
(50,000 x 500,000 per GPU, weak scaling, SVD k = 10); at N = 1 the default run appends it as `extra.cfg2`.

Printed JSON (one line, rank 0): the base contract + `roofline`, `cpu_baseline`, `e2e`, `clocks`,
`gpu_launches`.  `value` has inputs resident in HBM; `e2e` goes through the 9-argument C-ABI call
(bsg_prodvec) with pinned HOST buffers, H2D/D2H inside the timed region.

`parity` = max relative error of bed_prodVec / bed_cprodVec against the CPU oracle on a bounded column sample of the
same matrix (rank 0), so the timed path is checked against the reference's arithmetic in the run that times it.

`--impl reference` times the reference's CPU implementation of the same call on the host cores: the literal
C/OpenMP port in oracle/ (the reference needs R + Rcpp + bigstatsr and cannot be built here), all host
threads, on a bounded column sample of the same synthetic matrix.

`--dump-outputs DIR` writes, after the timed steps, the n-vector the last timed bed_prodVec step returned as
DIR/<workload>_prodvec.npy (float64; with the default N = 1 run also cfg2_prodvec.npy of the extra leg).  The matrix
and the vector are generated from fixed seeds, so two builds run with the same arguments can be compared file by file.

bench.py writes nothing into the tree: it uses the CUDA library and the CPU oracle that `python __graft_entry__.py`
built, and stops if either is missing or older than its sources.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the tree: the benchmark may run from a read-only checkout

import numpy as np  # noqa: E402

SEED = 20250924 + 1  # SURVEY.md section 8d: 20250924 + config index
WORKLOADS = {
    "cfg2": dict(n=50_000, m=500_000, scaling="weak", svd_k=10,
                 name="configs[1]: bed_prodVec on synthetic 50,000 x 500,000 2-bit .bed per GPU (binomial center/scale)"),
    "cfg5": dict(n=487_000, m=1_100_000, scaling="strong", svd_k=20,
                 name="configs[4]: bed_prodVec on UKBB-shaped synthetic 487,000 x 1,100,000 .bed, SNP columns sharded over the GPUs"),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.err = None

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {
                getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
                getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
                getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            }
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(
                nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = get_reasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(self.period)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), **({"error": self.err} if self.err else {})}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


_CANDS = None


def host_thread_candidates():
    """Cached at the first call: once libgomp has bound the main thread to its place (OMP_PROC_BIND) the process
    affinity mask no longer says how many CPUs the job may use."""
    global _CANDS
    if _CANDS is None:
        _CANDS = _host_thread_candidates()
    return _CANDS


def _host_thread_candidates():
    """Thread counts worth trying for the CPU port: every CPU this process may run on and one per physical core.
    Taken from the OS, not from OMP_NUM_THREADS (torchrun exports OMP_NUM_THREADS=1 to its workers); the oracle's
    loops take the count as their `ncores` argument, like the reference's."""
    try:
        logical = len(os.sched_getaffinity(0))
    except Exception:
        logical = os.cpu_count() or 1
    cands = {max(1, logical)}
    try:
        import psutil

        phys = psutil.cpu_count(logical=False)
        if phys:
            cands.add(max(1, min(logical, phys)))
    except Exception:
        pass
    return sorted(cands)


def pin_cpu_threads():
    """The CPU arm must be reproducible from box to box (VERDICT r1 weak #8): one OpenMP thread per core, bound, before
    libgomp is loaded (it reads the environment once).  torchrun exports OMP_NUM_THREADS=1 to its workers -- override."""
    os.environ["OMP_NUM_THREADS"] = str(max(host_thread_candidates()))
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")


class CpuSample:
    """The oracle's bed_pMatVec4 / bed_cpMatVec4 port on a bounded column sample (the first m_s SNPs) of the synthetic
    matrix.  The sample is generated in parallel by the oracle's own generator, so its pages are first-touched by the
    threads that later read them (the NUMA-interleaved allocation asked for in VERDICT r1)."""

    def __init__(self, n, m_cols, seed, na_rate=0.0):
        from oracle import ref

        self.ref, self.n, self.m = ref, n, m_cols
        self.o = ref.synth_bed(n, m_cols, seed=seed, na_rate=na_rate)
        self.threads = ref.max_threads()
        self.sc = ref.bed_scaleBinom(self.o, ncores=self.threads)
        self.y = np.random.default_rng(seed + 1).normal(size=m_cols)
        self.yr = np.random.default_rng(seed + 2).normal(size=n)
        self.ir, self.ic = self.o.rows_along(), self.o.cols_along()

    def prodvec(self, threads=None):
        return self.ref.bed_pMatVec4(self.o, self.ir, self.ic, self.sc["center"], self.sc["scale"], self.y,
                                     threads or self.threads)

    def cprodvec(self, threads=None):
        return self.ref.bed_cpMatVec4(self.o, self.ir, self.ic, self.sc["center"], self.sc["scale"], self.yr,
                                      threads or self.threads)

    def rate(self, steps=1, warmup=0, threads=None):
        for _ in range(warmup):
            self.prodvec(threads)
        t0 = time.perf_counter()
        for _ in range(steps):
            out = self.prodvec(threads)
        dt = time.perf_counter() - t0
        return float(self.n) * self.m * steps / dt, dt / steps, out


def best_threads(n, seed):
    """Calibrate warm on a small sample: every logical CPU vs one thread per physical core (SMT oversubscription halves
    this loop's rate on some hosts); returns (threads, genotypes/s)."""
    cal = CpuSample(n, max(256, int(2e9 // n)), seed)
    best, rate0 = 1, 0.0
    for t in host_thread_candidates():
        r, _, _ = cal.rate(steps=2, warmup=2, threads=t)
        if r > rate0:
            rate0, best = r, t
    return best, rate0


def sample_columns(n, m_avail, rate, seconds, cap_bytes=6e9):
    """Columns of a CPU step: ~`seconds` of work at `rate`, at most `cap_bytes` of packed host memory, at most m_avail."""
    n_byte = (n + 3) // 4
    return int(max(256, min(m_avail, rate * seconds / n, cap_bytes / n_byte)))


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    pin_cpu_threads()
    n = wl["n"]
    threads, rate0 = best_threads(n, SEED)
    # one step = the port's bed_pMatVec4 on the sample; sized so K + W steps end within ~2.5 minutes
    per_step = max(0.5, min(4.0, 150.0 / max(1, args.steps + args.warmup)))
    m_s = sample_columns(n, wl["m"], rate0, per_step)
    smp = CpuSample(n, m_s, SEED)
    rate, sec_step, _ = smp.rate(steps=args.steps, warmup=args.warmup, threads=threads)
    sample = "bed_pMatVec4 port (oracle/bsg_oracle.c, -O2 -fopenmp, OMP_PROC_BIND=%s) on the first %d of %d SNP columns " \
             "of the synthetic %d-sample matrix (%.2e genotypes per step)" % (
                 os.environ.get("OMP_PROC_BIND"), m_s, wl["m"], n, float(n) * m_s)
    line = {
        "impl": "reference", "metric": "genotypes/sec in bed_prodVec", "value": rate, "unit": "genotypes/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_step * 1e3,
        "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": {"workload": wl["name"], "n": n, "m_total": wl["m"], "m_sample": m_s},
        "cpu_baseline": {"value": rate, "unit": "genotypes/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "genotypes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


def traffic_for(kernel, alg_bytes):
    """DRAM bytes per launch of the dominant kernel: the ratio (dram read + write) / algorithmic bytes measured by the
    committed ncu --set full captures of the same kernel (bench.py cannot run under ncu and report a number), applied to
    this launch's algorithmic bytes; the source file is named beside the value."""
    tp = os.path.join(ROOT, "profiles", "r02_pmv_traffic.json")
    try:
        d = json.load(open(tp))
        r = d["ratio_vs_algorithmic"].get(kernel)
        if r:
            return float(r) * alg_bytes, "profiles/r02_pmv_traffic.json: measured ratio %.4f x algorithmic bytes; %s" % (r, d["source"])
    except Exception:
        pass
    return None, None


def run_workload(args, wl_key, torch, dist, B, L, rank, world, local, with_cpu, layout):
    """One workload on this process group: timed products, roofline, e2e (pinned and pageable host buffers), parity
    against the oracle on a bounded sample, bed_randomSVD wall time.  Returns the JSON pieces (rank 0) or None."""
    import ctypes as C

    from bigsnpr_b200 import _lib

    wl = WORKLOADS[wl_key]
    n = wl["n"]
    if wl["scaling"] == "weak":
        m_loc, col0 = wl["m"], rank * wl["m"]
    else:
        from bigsnpr_b200.dist import shard_bounds

        col0, col1 = shard_bounds(wl["m"], world, rank)
        m_loc = col1 - col0
    seed = SEED if wl_key == "cfg2" else 20250924 + 4
    lay = B.LAYOUT_SNP_MAJOR if layout == "snp" else (B.LAYOUT_SNP_MAJOR | B.LAYOUT_SAMPLE_MAJOR)
    g = B.Bed.synthetic(n, m_loc, seed=seed, na_rate=args.na_rate, col_offset=col0, device=local, layouts=lay)
    layouts = g.layouts
    sc = B.bed_scaleBinom(g)
    view = B.View(g, center=sc["center"], scale=sc["scale"])
    dev = torch.device("cuda", local)
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed + 17 + rank)
    x = torch.randn(m_loc, dtype=torch.float64, device=dev, generator=gen)
    out = torch.zeros(n, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    assert stream != 0

    comm = None
    if world > 1 and not args.nccl:
        from bigsnpr_b200.dist import Comm

        comm = Comm(n, device=local)  # NVLink peer-memory communicator of the library: reduction fused into the epilogue

    def step():
        if comm is not None:
            comm.prodvec_allreduce(view, x.data_ptr(), out.data_ptr(), stream)
        else:
            view.prodvec_dev(x.data_ptr(), out.data_ptr(), stream)
            if world > 1:
                dist.all_reduce(out)

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()

    # ---------------- timed region: K steps, inputs resident in HBM ----------------
    sampler = ClockSampler(physical_gpu_index(local))
    L.bsg_set_kernel_timing(1)
    launches0 = L.bsg_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    # the result of the last timed step, copied before the later legs run the product again
    last_out = out.cpu().numpy() if args.dump_outputs else None
    launches = int(L.bsg_launch_count() - launches0)
    cnt, tot = C.c_int(0), C.c_double(0)
    _lib.check(L.bsg_kernel_time_stats(C.byref(cnt), C.byref(tot)))
    L.bsg_set_kernel_timing(0)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    tg = torch.tensor([float(n) * float(m_loc)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tg)
    geno_total = float(tg.item())
    m_total = int(round(geno_total / n))
    value = geno_total * args.steps / (ms / 1e3)

    # roofline of the dominant kernel: algorithmic bytes = ceil(n/4) * m per launch (SURVEY.md 8d)
    alg_bytes = float((n + 3) // 4) * m_loc
    kern_ms = tot.value / max(cnt.value, 1)
    peak, peak_src = measured_peaks()
    achieved = alg_bytes / (kern_ms / 1e3) / 1e9 if kern_ms > 0 else None
    # with missing values the product kernel runs in its no-missing mode and bsg::naell::k_corr adds the list sums
    # (bigsnpr_b200/csrc/bsg_naell.cu); kernel_ms is the product kernel alone, ms_per_step the whole step
    kernel = "bsg::pmv::k_pmv" if (layouts & 2) else "bsg::pmvt::k_pmvT"
    traffic, traffic_src = traffic_for(kernel, alg_bytes)
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": kernel, "kernel_ms": kern_ms, "launches_timed": cnt.value,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "kernel_share_of_step": (kern_ms * args.steps / ms) if ms > 0 else None}
    if world > 1:
        # the step ends in a collective, so it runs at the pace of the slowest GPU: show every rank's kernel time and clock
        mine = torch.tensor([kern_ms, float(clocks.get("sm_mhz") or 0.0)], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        roofline["kernel_ms_per_rank"] = [round(float(t[0]), 4) for t in allr]
        roofline["kernel_ms_max_over_ranks"] = max(float(t[0]) for t in allr)
        roofline["sm_mhz_per_rank"] = [float(t[1]) for t in allr]
        roofline["kernel_share_of_step"] = (roofline["kernel_ms_max_over_ranks"] * args.steps / ms) if ms > 0 else None

    # ---------------- e2e: the 9-argument C-ABI call with HOST buffers (H2D / D2H inside the timed region) --------
    e2e_steps = max(3, min(args.steps, 50))
    pd = lambda tns: C.cast(tns.data_ptr(), _lib.c_dbl_p)  # noqa: E731
    xh = x.cpu()

    def e2e_leg(pinned):
        mk = (lambda a: a.pin_memory()) if pinned else (lambda a: a)
        xc = mk(xh.clone())
        cen = mk(torch.from_numpy(np.ascontiguousarray(sc["center"])).clone())
        sca = mk(torch.from_numpy(np.ascontiguousarray(sc["scale"])).clone())
        outh = mk(torch.empty(n, dtype=torch.float64))

        def e2e_step():
            _lib.check(L.bsg_prodvec(g._h, None, n, None, m_loc, pd(cen), pd(sca), pd(xc), pd(outh)))
            if world > 1:
                od = outh.to(dev, non_blocking=True)
                dist.all_reduce(od)
                outh.copy_(od)

        for _ in range(3):
            e2e_step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return geno_total * e2e_steps / float(te.item()), outh

    e2e_val, outh = e2e_leg(True)
    e2e_pageable, _ = e2e_leg(False)
    same = bool(torch.equal(out.cpu(), outh)) if world == 1 else None
    _lib.check(L.bsg_set_scaling_reuse(1))  # opt-in: an unchanged scaling is not uploaded again (include/bsgpu.h)
    try:
        r_pin, outr = e2e_leg(True)
        r_page, _ = e2e_leg(False)
        e2e_reuse = {"value": r_pin, "pageable_value": r_page, "h2d_bytes_per_step": 8 * m_loc,
                     "bit_equal_to_resident_path": bool(torch.equal(out.cpu(), outr)) if world == 1 else None}
    finally:
        _lib.check(L.bsg_set_scaling_reuse(0))

    # ---------------- parity against the oracle (rank 0, bounded column sample of ITS shard) and cpu_baseline --------
    parity, cpu_baseline = None, None
    if rank == 0 and with_cpu:
        try:
            pin_cpu_threads()
            threads, rate0 = best_threads(n, seed)
            m_s = sample_columns(n, m_loc, rate0, 3.0)
            smp = CpuSample(n, m_s, seed, na_rate=args.na_rate)
            reps = int(max(1, min(8, 12.0 / max(1e-3, float(n) * m_s / rate0))))
            r1, sec, a0 = smp.rate(steps=reps, warmup=1, threads=threads)
            b0 = smp.cprodvec(threads)
            cpu_baseline = {"value": r1, "unit": "genotypes/s", "cores": threads, "kind": "port",
                            "sample": "bed_pMatVec4 port (oracle/bsg_oracle.c, -O2 -fopenmp, threads bound to cores) on "
                                      "the first %d of %d columns, %d samples: %d x %.2f s" % (m_s, m_loc, n, reps, sec)}
            ic = np.arange(1, m_s + 1, dtype=np.int32)
            cen, sca = sc["center"][:m_s], sc["scale"][:m_s]
            assert np.array_equal(cen, smp.sc["center"]) and np.array_equal(sca, smp.sc["scale"]), "scaling differs"
            a = B.bed_prodVec(g, smp.y, ind_col=ic, center=cen, scale=sca)
            b = B.bed_cprodVec(g, smp.yr, ind_col=ic, center=cen, scale=sca)
            ea = float(np.max(np.abs(a - a0)) / np.max(np.abs(a0)))
            eb = float(np.max(np.abs(b - b0)) / np.max(np.abs(b0)))
            parity = {"max_rel_err_vs_oracle": max(ea, eb), "prodvec": ea, "cprodvec": eb, "scaling_bit_equal": True,
                      "config": "%s: first %d columns x %d samples of this run's matrix, bed_prodVec and bed_cprodVec "
                                "with binomial scaling vs the oracle port" % (wl_key, m_s, n)}
            del smp
        except Exception as e:  # pragma: no cover
            cpu_baseline = cpu_baseline or {"value": None, "error": repr(e)}
            parity = {"max_rel_err_vs_oracle": None, "error": repr(e)}

    # ---------------- extra leg: the same product from the SNP-major copy alone (k_pmvT) ----------------
    single_copy = None
    if (layouts & 2) and not args.no_single_copy:
        _lib.check(L.bsg_set_prodvec_path(1))
        try:
            for _ in range(3):
                step()
            torch.cuda.synchronize()
            L.bsg_set_kernel_timing(1)
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ksc = max(3, min(args.steps, 20))
            s0.record()
            for _ in range(ksc):
                step()
            s1.record()
            torch.cuda.synchronize()
            c2, t2 = C.c_int(0), C.c_double(0)
            _lib.check(L.bsg_kernel_time_stats(C.byref(c2), C.byref(t2)))
            L.bsg_set_kernel_timing(0)
            kms = t2.value / max(c2.value, 1)
            single_copy = {"kernel": "bsg::pmvt::k_pmvT", "steps": ksc, "ms_per_step": s0.elapsed_time(s1) / ksc,
                           "kernel_ms": kms, "achieved": alg_bytes / (kms / 1e3) / 1e9 if kms > 0 else None,
                           "frac": (alg_bytes / (kms / 1e3) / 1e9 / peak) if kms > 0 else None,
                           "note": "X.y read from the SNP-major copy only (no sample-major copy needed); this rank"}
        finally:
            _lib.check(L.bsg_set_prodvec_path(0))

    # ---------------- second headline metric: bed_randomSVD wall time (not part of `value`) ----------------
    svd_info = None
    if not args.no_svd:
        k = wl["svd_k"]
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        if comm is not None:
            from bigsnpr_b200.dist import randomsvd_comm

            sv = randomsvd_comm(g, comm, m_total, k=k)
        elif world > 1:
            from bigsnpr_b200.dist import randomsvd_sharded

            sv = randomsvd_sharded(g, m_total, k=k)
        else:
            sv = B.bed_randomSVD(g, k=k)
        tsvd = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tsvd, op=dist.ReduceOp.MAX)
        wall = float(tsvd.item())
        bytes_read = float((n + 3) // 4) * m_total * (2 * sv["nops"] + k + 1)
        svd_info = {"k": k, "tol": 1e-4, "wall_s": wall, "nops": sv["nops"], "niter": sv["niter"],
                    "d_top3": [float(v) for v in sv["d"][:3]], "packed_bytes_read": bytes_read,
                    "hbm_frac_over_wall": bytes_read / wall / 1e9 / (peak * world),
                    "note": "bed_randomSVD(fun.scaling = bed_scaleBinom, k = %d), Lanczos on the device; wall time includes "
                            "the scaling pass, the iteration and the k products for v" % k}

    if comm is not None:
        comm.check()
        torch.cuda.synchronize()
        dist.barrier()
        comm.close()
    view.close()
    g.close()
    if rank != 0:
        return None
    par = "1 GPU" if world == 1 else (
        "snp-column shards over %d GPUs; per step the n-vector of partial products is summed %s" % (
            world, "inside the X.y epilogue kernel over NVLink peer memory (k_ar_oneshot, no NCCL, no host hop)"
            if comm is not None else "by one NCCL all-reduce"))
    return {
        "value": value, "ms_per_step": ms / args.steps, "scaling": wl["scaling"],
        "config": {"workload": wl["name"], "n": n, "m_total": m_total, "m_per_gpu": m_loc, "na_rate": args.na_rate,
                   "layouts": layouts,
                   "l2": "inputs larger than L2: %.2f GB of packed genotypes per pass per GPU vs 126 MB L2" % (alg_bytes / 1e9),
                   "arithmetic": "exact int8 x uint2 on the integer tensor pipe, 61-bit fixed-point vector, fp64 epilogue",
                   "parallelism": par},
        "roofline": roofline, "cpu_baseline": cpu_baseline, "parity": parity,
        "e2e": {"value": e2e_val, "unit": "genotypes/s", "h2d_bytes_per_step": 3 * 8 * m_loc, "d2h_bytes_per_step": 8 * n,
                "steps": e2e_steps, "host_buffers": "pinned", "pageable_value": e2e_pageable,
                "bit_equal_to_resident_path": same,
                "with_scaling_reuse": e2e_reuse,
                "note": "bsg_prodvec(h, NULL, n, NULL, m, center, scale, x, out) with host buffers: x, center and scale go "
                        "up and the result comes back every step (the reference re-reads center / scale on every call).  "
                        "with_scaling_reuse: the same after bsg_set_scaling_reuse(1) -- an unchanged scaling (address, "
                        "length, strided sample of the values) is not uploaded again: 8 m bytes up per step"},
        "clocks": clocks, "gpu_launches": launches, "svd": svd_info, "single_copy": single_copy,
        "outputs": {wl_key + "_prodvec": last_out} if last_out is not None else {},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS))
    ap.add_argument("--na-rate", type=float, default=0.0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity leg")
    ap.add_argument("--no-svd", action="store_true", help="skip the bed_randomSVD wall-time leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[1] extra leg of the default N = 1 run")
    ap.add_argument("--layout", choices=("auto", "both", "snp"), default="auto",
                    help="snp: the SNP-major copy only (the library's default; X.y on k_pmvT); both: also the sample-major "
                         "copy (X.y on k_pmv); auto: snp for cfg5 (134 GB), both for cfg2")
    ap.add_argument("--nccl", action="store_true", help="N > 1: reduce with torch.distributed / NCCL instead of the library's "
                                                       "own peer-memory communicator (the baseline it is measured against)")
    ap.add_argument("--no-single-copy", action="store_true", help="skip the extra leg timing X.y on the SNP-major copy alone")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm sizes its column sample from a timing, so its inputs vary by run")
    from bigsnpr_b200 import build
    from oracle import ref

    for so, old in ((build.OUT, build.stale()), (ref._SO, ref.stale())):
        if old:
            raise SystemExit("%s is missing or older than its sources: build first (python __graft_entry__.py)" % so)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, wl)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local)
    if world > 1:
        # rank 0 prints exactly one line on stdout: keep NCCL's own "NCCL version ..." banner (NCCL_DEBUG=VERSION,
        # which some launch environments export) out of it; INFO / TRACE requests are respected
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION", "WARN"):
            os.environ["NCCL_DEBUG"] = "NONE"  # WARN still prints the banner (VERSION < WARN in NCCL's levels)
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # whatever NCCL does print stays off stdout
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import bigsnpr_b200 as B
    from bigsnpr_b200 import _lib

    L = _lib.lib()
    dev = torch.device("cuda", local)
    # a dedicated (non-default) stream: the library enqueues on the stream it is handed, and the CUDA events that time
    # the region are recorded on the same stream
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)

    layout = args.layout if args.layout != "auto" else ("snp" if args.workload == "cfg5" else "both")
    res = run_workload(args, args.workload, torch, dist, B, L, rank, world, local, not args.no_cpu, layout)
    extra = None
    if args.workload == "cfg5" and world == 1 and not args.no_extra:
        torch.cuda.empty_cache()
        r2 = run_workload(args, "cfg2", torch, dist, B, L, rank, world, local, False, "both")
        extra = {"cfg2": {k: r2[k] for k in ("value", "ms_per_step", "config", "roofline", "e2e", "svd", "single_copy")}}

    if rank == 0:
        line = {
            "metric": "genotypes/sec in bed_prodVec", "value": res["value"], "unit": "genotypes/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": res["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": res["config"], "roofline": res["roofline"], "cpu_baseline": res["cpu_baseline"],
            "parity": res["parity"], "e2e": res["e2e"], "clocks": res["clocks"], "gpu_launches": res["gpu_launches"],
            "svd": res["svd"], "single_copy": res["single_copy"], "extra": extra,
        }
        if args.dump_outputs:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in {**res["outputs"], **(r2["outputs"] if extra else {})}.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
