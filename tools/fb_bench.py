"""Forward-backward inference (cv_loglik_batch / cv_posterior_batch) at the POS shape on one GPU: device and wall time
of the three call shapes, the kernel split, FP64 use against the DFMA rate measured in the same run, and a parity
block against the threaded C oracle.

  python tools/fb_bench.py [--seqs 1000000] [--reps 3] [--parity-seqs 100000] [--out fb_bench.json]

Prints one JSON document.  The workload is bench.workload_pos (K = 45, M = 20 000, Zipf words, gamma lengths)."""
from __future__ import annotations

import argparse
import ctypes as C
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


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def calls(h, w):
    """the three call shapes: name -> function running one call"""
    obs, off = w["obs"], w["off"]
    return {
        "loglik": lambda: cv.loglik_batch(h, obs, off, device=0),
        "posterior_no_post": lambda: cv.posterior_batch(h, obs, off, device=0),
        "posterior_with_post": lambda: cv.posterior_batch(h, obs, off, device=0, want_posteriors=True),
    }


def profile_call(fn):
    """torch.profiler over one call: device time per kernel and of the host<->device copies (ms)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        name = ev.key
        if "bw_fwd_kernel" in name:
            fam = "forward"
        elif "fb_bwd_kernel" in name:
            fam = "backward"
        elif "fb_out_kernel" in name or "fb_ll_kernel" in name:
            fam = "output"
        elif "bw_prep_kernel" in name:
            fam = "prep"
        elif "Memcpy HtoD" in name:
            fam = "copy_h2d"
        elif "Memcpy DtoH" in name:
            fam = "copy_d2h"
        else:
            continue
        out[fam] = out.get(fam, 0.0) + t / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parity-seqs", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "fb_bench needs a CUDA device"
    from oracle import fb_oracle as fbo

    res = dict(card=card())
    w = bench.workload_pos(0, args.seqs)
    K, N, B = w["K"], int(w["off"][-1]), args.seqs
    h = cv.HMM(w["A"], w["B"], w["pi"])
    small = dict(obs=w["obs"][: int(w["off"][1000])], off=w["off"][:1001])
    for fn in calls(h, small).values():            # module load, layouts of the handle, allocations
        fn()
    L = cv._lib.lib()
    rate, pms = C.c_double(0.0), C.c_double(0.0)
    cv._lib.check(L.cv_debug_probe_fp64(0, 25, 20000, C.byref(rate), C.byref(pms)))
    lens = np.sort(np.diff(w["off"]))[::-1]
    slabs = int(lens[::64].sum())
    shapes = {}
    for name, fn in calls(h, w).items():
        fn()                                        # warm-up at full size
        walls = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            fn()
            walls.append(time.perf_counter() - t0)
        split = profile_call(fn)
        kern = sum(v for k, v in split.items() if not k.startswith("copy"))
        copies = split.get("copy_h2d", 0.0) + split.get("copy_d2h", 0.0)
        wall_ms = float(np.median(walls)) * 1e3
        fmas = (1.0 if name == "loglik" else 2.0) * K * K * N      # forward K^2 per position, backward (a u) K^2
        shapes[name] = dict(wall_ms_median=wall_ms, wall_ms_all=[x * 1e3 for x in walls], device_kernel_ms=kern,
                            copy_ms=copies, kernel_and_copy_ms=split, host_ms_outside_device=wall_ms - kern - copies,
                            fp64_fma_per_position=fmas / N, fp64_fma=fmas,
                            fp64_fraction_of_dfma_probe=(fmas / (kern * 1e-3)) / rate.value if kern > 0 else None)
    res["pos"] = dict(workload=w["desc"], sequences=B, positions=N, history_slabs=slabs,
                      history_bytes=slabs * 64 * K * 8, posterior_bytes=N * K * 8, dfma_probe_per_s=rate.value,
                      calls=shapes)
    # parity against the oracle on a slice
    P = min(args.parity_seqs, B)
    so, sf = w["off"][: P + 1], w["obs"][: int(w["off"][P])]
    r = cv.posterior_batch(h, sf, so, device=0, want_posteriors=True)
    nth = os.cpu_count() or 1
    t0 = time.perf_counter()
    ro = fbo.forward_backward(w["A"], w["B"], w["pi"], sf, so, nthreads=nth)
    t_or = time.perf_counter() - t0
    f = np.isfinite(ro["loglik"])
    ll_err = float(np.max(np.abs(r["loglik"][f] - ro["loglik"][f]) / np.maximum(1.0, np.abs(ro["loglik"][f]))))
    post_err = float(np.max(np.abs(r["post"] - ro["post"])))
    top2 = np.sort(ro["post"], axis=1)[:, -2:]
    clear = top2[:, 1] - top2[:, 0] > 1e-9
    mism = int((r["path"][clear] != ro["post"].argmax(axis=1)[clear]).sum())
    res["parity"] = dict(sequences=P, positions=int(so[-1]), max_loglik_err_rel=ll_err, max_posterior_abs_err=post_err,
                         neg_inf_pattern_equal=bool((np.isneginf(r["loglik"]) == ~f).all()),
                         mpm_positions_margin_gt_1e9=int(clear.sum()), mpm_mismatches=mism,
                         failures=int((ll_err > 1e-12) + (post_err > 1e-12) + (mism > 0)),
                         oracle_threads=nth, oracle_seconds=t_or)
    h.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write(txt + "\n")


if __name__ == "__main__":
    main()
