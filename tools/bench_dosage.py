"""Centi-dosage matrix-vector products on one GPU: X.y and Xt.y over value bytes (bsg_pmv8.cu) against the same shape
as hard calls (2-bit), plus one bed_randomSVD(k = 10).

    python tools/bench_dosage.py [--n 100000] [--m 200000] [--steps 20] [--warmup 3] [--out FILE]

The matrix is seeded CODE_DOSAGE code bytes built on the host (n x m bytes: 20 GB at the default shape, far beyond the
126 MB of L2) and staged once.  Products are timed with CUDA events over device-resident vectors after warm-up; GB/s is
over the n x m bytes one product reads (n x m / 4 for hard calls), reported as a share of the 6.57 TB/s HBM read rate
measured on this project's B200 (DESIGN.md) and, separately, of the 7.7 TB/s data-sheet figure.  The GPU name and
power limit are read in the same run.  Parity: Xt.y on a sample of columns against fp64 on the host."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
MEASURED_TBS, DATASHEET_TBS = 6.57, 7.7


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power = [t.strip() for t in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power}


def time_products(B, torch, g, n, m, steps, warmup, center, scale):
    v = B.View(g, np.arange(1, n + 1), np.arange(1, m + 1), center, scale)
    x = torch.randn(m, dtype=torch.float64, device="cuda")
    y = torch.randn(n, dtype=torch.float64, device="cuda")
    out_n = torch.empty(n, dtype=torch.float64, device="cuda")
    out_m = torch.empty(m, dtype=torch.float64, device="cuda")
    res = {}
    for name, call in (("prodvec", lambda: v.prodvec_dev(x.data_ptr(), out_n.data_ptr())),
                       ("cprodvec", lambda: v.cprodvec_dev(y.data_ptr(), out_m.data_ptr()))):
        for _ in range(warmup):
            call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            call()
        e1.record()
        torch.cuda.synchronize()
        res[name + "_ms"] = e0.elapsed_time(e1) / steps
    v.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--m", type=int, default=200_000)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    import bigsnpr_b200 as B

    if not torch.cuda.is_available():
        sys.exit("bench_dosage: no CUDA device")
    n, m = a.n, a.m
    rng = np.random.default_rng(20251017)
    G = np.empty((n, m), dtype=np.uint8, order="F")
    blk = max(1, (1 << 28) // n)
    for j in range(0, m, blk):
        G[:, j:j + blk] = rng.integers(7, 208, size=(n, min(blk, m - j)), dtype=np.uint8)
    code = B.CODE_DOSAGE
    t0 = time.perf_counter()
    g = B.Bed.from_fbm(G, code256=code)
    stage_s = time.perf_counter() - t0
    center, scale = np.full(m, 1.0), np.full(m, 0.6)
    res = {"shape": [n, m], "steps": a.steps, "warmup": a.warmup, **gpu_info(), "stage_s": stage_s}
    dos = time_products(B, torch, g, n, m, a.steps, a.warmup, center, scale)
    nbytes = n * m
    for k in ("prodvec", "cprodvec"):
        gbs = nbytes / (dos[k + "_ms"] * 1e-3) / 1e9
        res["dosage_" + k] = {"ms": dos[k + "_ms"], "GB_per_s": gbs, "share_of_measured_6.57TBs": gbs / (MEASURED_TBS * 1e3),
                              "share_of_datasheet_7.7TBs": gbs / (DATASHEET_TBS * 1e3)}
    # parity of Xt.y on a column sample (fp64 on the host)
    cols = np.sort(rng.choice(m, 64, replace=False)) + 1
    yr = rng.normal(size=n)
    got = B.bed_cprodVec(g, yr, np.arange(1, n + 1), cols, center[cols - 1], scale[cols - 1])
    want = np.array([np.dot(yr.astype(np.longdouble), ((code[G[:, j - 1]] - 1.0) / 0.6).astype(np.longdouble))
                     for j in cols], dtype=np.float64)
    res["parity_cprodvec_rel_err"] = float(np.max(np.abs(got - want)) / np.max(np.abs(want)))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    svd = B.bed_randomSVD(g, fun_scaling=lambda X, **kw: {"center": center, "scale": scale}, k=10)
    res["randomSVD_k10_s"] = time.perf_counter() - t0
    res["randomSVD_nops"] = svd["nops"]
    g.close()
    del G
    # the same shape as hard calls (2-bit, a quarter of the bytes)
    h = B.Bed.synthetic(n, m, seed=5)
    hc = time_products(B, torch, h, n, m, a.steps, a.warmup, center, scale)
    for k in ("prodvec", "cprodvec"):
        gbs = nbytes / 4 / (hc[k + "_ms"] * 1e-3) / 1e9
        res["hardcall_" + k] = {"ms": hc[k + "_ms"], "GB_per_s": gbs,
                                "share_of_measured_6.57TBs": gbs / (MEASURED_TBS * 1e3)}
    h.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
