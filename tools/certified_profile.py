"""Where the time of the certified exact decode goes (K <= 64, cv_decode_batch_dev): f32 forward kernel, backtrace with
certification, how many sequences were flagged and what their f64 re-decode costs; the device step against the forced
f64 path; the results checked byte for byte against that path.

  python tools/certified_profile.py [--nseq 1000000 125000] [--steps 10] [--out profile.json]
                                    [--routes tile chain 1184 2368 4736 ...]

--routes also times the step with the fallback's route forced (cv_debug_set_fallback): `tile`, `chain`, or a number of
the longest flagged sequences given to the warp-per-sequence kernel beside the tile path (route_step_ms).

Per workload (the POS shape of bench.py at each size, and the POS lengths on a tie-heavy model of dyadic values with
+-0.0, where most decisions are exact ties):
  fwd_ms        f32 forward kernel alone (CUDA events, cv_set_timing: backtrace after the forward kernel)
  bt_ms         backtrace + certification, bound scaled to 0 (nothing flagged, no fallback)
  bt_fb_ms      backtrace + certification + host round trip + fallback, default bound
  fallback_ms   bt_fb_ms - bt_ms
  flagged       sequences re-decoded in f64
  fallback_chain  of those, the ones the warp-per-sequence kernel decoded (the rest went to the f64 tile path)
  step_ms       device step as bench.py times it (concurrent backtrace), certified / forced f64
The forward kernel's bound is its issue rate, not bench.py's FP64 peak (bench.py's roofline.frac still divides by the
FP64 DADD+DSETP rate): a cell is one FADD2 or FMNMX3 issue slot (two cells each for an add and a max), so at most
128 cells per SM per clock; fwd_issue_frac = cells / (SMs x 128 x clocks.max.sm) / fwd_ms.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit_w": float(plim), "clocks_max_sm_mhz": float(clk)}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


def profile(cv, torch, wl, steps, routes=()):
    L = cv._lib.lib()
    K = wl["K"]
    hmm = cv.HMM(wl["A"], wl["B"], np.zeros(K))
    h = hmm.device_handle(0)
    obs, off = wl["obs"], wl["off"]
    Bn, N = len(off) - 1, len(obs)
    max_len = int(np.diff(off).max())
    d_obs = torch.from_numpy(obs.view(np.int32)).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_path = torch.empty(N, dtype=torch.int32, device="cuda")
    d_score = torch.empty(Bn, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()

    def call():
        cv._lib.check(L.cv_decode_batch_dev(h, d_obs.data_ptr(), d_off.data_ptr(), Bn, N, max_len, d_path.data_ptr(),
                                            d_score.data_ptr(), stream.cuda_stream, 0))

    def step_ms():
        for _ in range(2):
            call()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            call()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def timed(n=5):
        L.cv_set_timing(1)
        f, b = [], []
        try:
            for _ in range(n):
                call()
                torch.cuda.synchronize()
                f.append(L.cv_last_kernel_ms(h)); b.append(L.cv_last_backtrace_ms(h))
        finally:
            L.cv_set_timing(0)
        return float(np.median(f)), float(np.median(b))

    r = {"workload": wl["name"], "sequences": Bn, "elements": N, "cells": wl["cells"]}
    L.cv_debug_set_certified(0)
    try:
        r["step_ms_f64"] = step_ms()
        ref_p, ref_s = d_path.cpu().numpy(), d_score.cpu().numpy()
        r["f64_fwd_ms"], r["f64_bt_ms"] = timed()
    finally:
        L.cv_debug_set_certified(1)
    r["step_ms"] = step_ms()
    r["flagged"] = int(L.cv_debug_last_flagged(h))
    r["fallback_chain"] = int(L.cv_debug_last_fallback_chain(h))
    r["paths_equal_f64"] = bool((d_path.cpu().numpy() == ref_p).all())
    r["score_bits_equal_f64"] = d_score.cpu().numpy().tobytes() == ref_s.tobytes()
    r["fwd_ms"], r["bt_fb_ms"] = timed()
    L.cv_debug_set_cert_tolerance(0.0)
    try:
        _, r["bt_ms"] = timed()
    finally:
        L.cv_debug_set_cert_tolerance(1.0)
    r["fallback_ms"] = r["bt_fb_ms"] - r["bt_ms"]
    if routes:
        r["route_step_ms"], r["route_fallback_ms"] = {}, {}
        for rt in routes:
            route, k = {"tile": (1, 0), "chain": (2, 0)}.get(rt, (3, int(rt) if rt.isdigit() else 0))
            L.cv_debug_set_fallback(route, k)
            try:
                ms = step_ms()
                same = bool((d_path.cpu().numpy() == ref_p).all()) and d_score.cpu().numpy().tobytes() == ref_s.tobytes()
                _, bt_fb = timed()
            finally:
                L.cv_debug_set_fallback(0, 0)
            r["route_step_ms"][rt] = ms
            r["route_fallback_ms"][rt] = bt_fb - r["bt_ms"]
            r["paths_equal_f64"] = r["paths_equal_f64"] and same
    hmm.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nseq", type=int, nargs="+", default=[1_000_000, 125_000])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--routes", nargs="*", default=[])
    args = ap.parse_args()
    import torch

    import consistent_viterbi_b200 as cv
    from bench import workload_pos
    from util import random_hmm

    assert torch.cuda.is_available(), "needs a CUDA device"
    info = gpu_info()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = {"gpu": info, "sms": sms, "runs": []}
    for n in args.nseq:
        res["runs"].append(profile(cv, torch, workload_pos(0, n), args.steps, args.routes))
    wl = workload_pos(0, args.nseq[-1])
    wl["A"], wl["B"], _ = random_hmm(np.random.default_rng(3019), wl["K"], wl["M"], ties=True)
    wl["name"] = "pos_lengths_tie_heavy_model"
    res["runs"].append(profile(cv, torch, wl, args.steps, args.routes))
    clk = info.get("clocks_max_sm_mhz")
    for r in res["runs"]:
        if clk:
            r["fwd_issue_frac"] = r["cells"] / (sms * 128 * clk * 1e6) / (r["fwd_ms"] * 1e-3)
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
