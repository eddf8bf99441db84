"""Baum-Welch (cv_baum_welch) at the POS shape on one GPU: time per EM iteration, the kernel split, FP64 and HBM use
against rates measured in the same run, a parity check against the threaded C oracle, and the oracle's own rate.

  python tools/bw_bench.py [--seqs 1000000] [--iters 5] [--parity-seqs 100000] [--out bw_bench.json]

Prints one JSON document.  The workload is bench.workload_pos (K = 45, M = 20 000, Zipf words, gamma lengths)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import consistent_viterbi_b200 as cv  # noqa: E402


def model(w):
    """A model of its own: training updates the HMM's arrays in place, and HMM does not copy contiguous f64 input."""
    return cv.HMM(w["A"].copy(), w["B"].copy(), w["pi"].copy())


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def hbm_bandwidth():
    """Device-to-device copy of 4 GB, CUDA events: (read + write) bytes / time."""
    import torch
    x = torch.empty(1 << 29, dtype=torch.float64, device="cuda")
    y = torch.empty_like(x)
    y.copy_(x)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        y.copy_(x)
    e1.record()
    torch.cuda.synchronize()
    return 5 * 2 * x.numel() * 8 / (e0.elapsed_time(e1) * 1e-3)


def kernel_split(w):
    """torch.profiler over one 2-iteration call: device time per kernel family, per iteration."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        model(w).train_arrays(w["obs"], w["off"], n_iter=2, device=0)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        name = ev.key
        if "bw_" not in name:
            continue
        fam = "forward" if "bw_fwd" in name else "backward" if "bw_bwd" in name else "emission_mstep"
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        out[fam] = out.get(fam, 0.0) + t / 1e3 / 2
    return out


def rel_err(got, ref):
    f = ~np.isneginf(ref)
    if not (np.isneginf(got) == np.isneginf(ref)).all():
        return float("inf")
    g, r = 10.0 ** got[f], 10.0 ** ref[f]
    keep = r >= 1e-250
    return float(np.max(np.abs(g[keep] - r[keep]) / r[keep])) if keep.any() else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=1_000_000)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--parity-seqs", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "bw_bench needs a CUDA device"
    from oracle import bw_oracle as bwo

    res = dict(card=card())
    w = bench.workload_pos(0, args.seqs)
    K, N = w["K"], int(w["off"][-1])
    # warm-up (module load, allocations), then the timed call
    model(w).train_arrays(w["obs"][: int(w["off"][1000])], w["off"][:1001], n_iter=1, device=0)
    h = model(w)
    t0 = time.perf_counter()
    r = h.train_arrays(w["obs"], w["off"], n_iter=args.iters, device=0)
    wall = time.perf_counter() - t0
    ms_it = r["device_ms"] / r["iters"]
    fmas = 3.0 * K * K * N
    L = cv._lib.lib()
    import ctypes as C
    rate, pms = C.c_double(0.0), C.c_double(0.0)
    cv._lib.check(L.cv_debug_probe_fp64(0, 25, 20000, C.byref(rate), C.byref(pms)))
    bw = hbm_bandwidth()
    # history bytes: tiles of 64 sequences (longest first) x their longest length x K x 8 B; written by the forward
    # pass, read and rewritten (gamma) by the backward pass, read by the emission pass: 4 passes over it
    lens = np.sort(np.diff(w["off"]))[::-1]
    slabs = int(lens[::64].sum())
    slabs_bytes = slabs * K * 64 * 8
    hbm_bytes = 4.0 * slabs_bytes
    res["pos"] = dict(workload=w["desc"], sequences=args.seqs, positions=N, iters=r["iters"], ms_per_iter=ms_it,
                      call_wall_s=wall, positions_per_s=N / (ms_it * 1e-3), loglik=list(r["loglik"]), skipped=r["skipped"],
                      fp64_fma_per_iter=fmas, dfma_probe_per_s=rate.value,
                      fp64_fraction_of_probe=(fmas / (ms_it * 1e-3)) / rate.value,
                      history_bytes=slabs_bytes, hbm_bytes_per_iter_model=hbm_bytes, hbm_copy_bw_bytes_per_s=bw,
                      hbm_fraction_of_copy_bw=(hbm_bytes / (ms_it * 1e-3)) / bw,
                      kernel_ms_per_iter=kernel_split(w))
    # parity on a slice, and the oracle's own rate on all host threads
    P = min(args.parity_seqs, args.seqs)
    so, sf = w["off"][: P + 1], w["obs"][: int(w["off"][P])]
    hp = model(w)
    rp = hp.train_arrays(sf, so, n_iter=1, device=0)
    nth = os.cpu_count() or 1
    t0 = time.perf_counter()
    ro = bwo.baum_welch(w["A"], w["B"], w["pi"], sf, so, n_iter=1, nthreads=nth)
    t_or = time.perf_counter() - t0
    errs = dict(a=rel_err(hp.a, ro["a"]), b=rel_err(hp.b, ro["b"]), pi=rel_err(hp.pi, ro["pi"]))
    ll_err = abs(rp["loglik"][0] - ro["loglik"][0]) / abs(ro["loglik"][0])
    fails = sum(e > 1e-9 for e in errs.values()) + (ll_err > 1e-12) + (rp["skipped"] != ro["skipped"])
    res["parity"] = dict(sequences=P, max_rel_err=errs, loglik_rel_err=ll_err, skipped_gpu=rp["skipped"],
                         skipped_oracle=ro["skipped"], failures=int(fails))
    res["cpu_oracle"] = dict(threads=nth, sequences=P, positions=int(so[-1]), seconds=t_or,
                             positions_per_s=int(so[-1]) / t_or)
    # datasets/ar houses: a few long sequences (the small-batch case)
    ar = []
    for wa in bench.workload_ar():
        ha = model(wa)
        ra = ha.train_arrays(wa["obs"], wa["off"], n_iter=3, device=0)
        ar.append(dict(name=wa["name"], K=wa["K"], sequences=len(wa["off"]) - 1, positions=int(wa["off"][-1]),
                       ms_per_iter=ra["device_ms"] / ra["iters"], skipped=ra["skipped"]))
    res["ar_houses"] = ar
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
