"""k-best Viterbi (cv_decode_batch_kbest) at the POS shape on one GPU: wall and device time per call for k in
{1, 2, 8, 32}, the split between the kernel and the copies, candidates per second, the ratio to cv_decode_batch on the
same batch, and a parity block against the threaded C oracle.

  python tools/kbest_bench.py [--seqs 1000000] [--reps 3] [--parity-seqs 100000] [--out kbest_bench.json]

Prints one JSON document.  The workload is bench.workload_pos (K = 45, M = 20 000, Zipf words, gamma lengths).  The
forward pass, the end selection and the backtrace run in one kernel (kbest_kernel), so the profiler split is kernel /
host-to-device copies / device-to-host copies."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
import consistent_viterbi_b200 as cv  # noqa: E402
from fb_bench import card  # noqa: E402


def profile_call(fn):
    """torch.profiler over one call: device time of the k-best kernel and of the host<->device copies (ms)"""
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
        fam = ("kernel" if "kbest_kernel" in name else "copy_h2d" if "Memcpy HtoD" in name else
               "copy_d2h" if "Memcpy DtoH" in name else None)
        if fam:
            out[fam] = out.get(fam, 0.0) + t / 1e3
    return out


def timed(fn, reps):
    fn()                                            # warm-up at full size
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        walls.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(walls)), walls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seqs", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--ks", default="1,2,8,32")
    ap.add_argument("--parity-seqs", type=int, default=100_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "kbest_bench needs a CUDA device"
    from oracle import kbest_oracle as kbo

    res = dict(card=card())
    w = bench.workload_pos(0, args.seqs)
    K, N, B = w["K"], int(w["off"][-1]), args.seqs
    steps = N - B                                   # positions t >= 1: the ones with a list to build
    h = cv.HMM(w["A"], w["B"], w["pi"])
    obs, off = w["obs"], w["off"]
    cv.decode_batch_kbest(h, obs[: int(off[1000])], off[:1001], 2, device=0)   # module load, allocations
    dec_ms, dec_all = timed(lambda: cv.decode_batch(h, obs, off, device=0), args.reps)
    runs = {}
    for k in (int(x) for x in args.ks.split(",")):
        fn = lambda: cv.decode_batch_kbest(h, obs, off, k, device=0)  # noqa: E731
        wall, walls = timed(fn, args.reps)
        split = profile_call(fn)
        kern = split.get("kernel", 0.0)
        copies = split.get("copy_h2d", 0.0) + split.get("copy_d2h", 0.0)
        cands = float(steps) * K * K * k            # every (j, r) candidate of every (t, i), the early exit ignored
        runs[str(k)] = dict(wall_ms_median=wall, wall_ms_all=walls, kernel_ms=kern, copy_ms=copies,
                            device_split_ms=split, host_ms_outside_device=wall - kern - copies,
                            candidates_full=cands, candidates_per_s_full=cands / (kern * 1e-3) if kern > 0 else None,
                            candidates_skipped="not counted: the kernel keeps no counter",
                            ratio_to_decode_batch_wall=wall / dec_ms,
                            backpointer_bytes=2 * (8 * ((K + 7) // 8)) * (1 << (k - 1).bit_length()) * N,   # u16 [N][Kp][capacity]
                            path_bytes_d2h=4 * k * N)
    res["pos"] = dict(workload=w["desc"], sequences=B, positions=N, steps=steps,
                      decode_batch_wall_ms_median=dec_ms, decode_batch_wall_ms_all=dec_all, kbest=runs)
    # parity against the oracle on a slice
    P = min(args.parity_seqs, B)
    so, sf = off[: P + 1], obs[: int(off[P])]
    nth = os.cpu_count() or 1
    got = cv.decode_batch_kbest(h, sf, so, 8, device=0)
    t0 = time.perf_counter()
    ref = kbo.decode_batch_kbest(w["A"], w["B"], sf, so, 8, nthreads=nth)
    t_or = time.perf_counter() - t0
    dp, ds = cv.decode_batch(h, sf, so, device=0)
    res["parity"] = dict(sequences=P, positions=int(so[-1]), k=8,
                         paths_equal=got[0].tobytes() == ref[0].tobytes(),
                         scores_equal=got[1].tobytes() == ref[1].tobytes(),
                         rank0_equals_decode_batch=got[0][0].tobytes() == dp.tobytes() and got[1][0].tobytes() == ds.tobytes(),
                         mismatched_sequences=int((got[1] != ref[1]).any(axis=0).sum()),
                         oracle_threads=nth, oracle_seconds=t_or)
    res["parity"]["failures"] = int(not (res["parity"]["paths_equal"] and res["parity"]["scores_equal"]
                                         and res["parity"]["rank0_equals_decode_batch"]))
    h.close()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fo:
            fo.write(txt + "\n")


if __name__ == "__main__":
    main()
