#!/usr/bin/env python
"""bench.py -- Viterbi cells/s of the B200 hot path, one JSON line (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload pos|large] [--impl ours|reference]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic input.  Default workload = BASELINE.json
configs[2], the POS-tagging shape (K=45 tags, 20k vocab, 1M sentences, avg T=25): the batched, sharding
configuration the metric "cells/s at 1/2/4/8 B200" is quoted on (configs[1], datasets/ar, is 60 sequences /
1.5e7 cells, latency bound and unshardable -- it is reported under "other" together with the constrained-decode
configs and a reduced large-state run).
N > 1: launched by torchrun, one rank per GPU, every rank decodes its own shard of 1M sentences (weak
scaling, no data-path collective), max-over-ranks timing.

value    cells/s with inputs resident in HBM (cv_decode_batch_dev on torch's current stream)
e2e      cells/s through the C ABI call a user makes (cv_decode_batch, pinned HOST buffers, H2D + D2H inside)
roofline dominant kernel (forward recurrence) vs the FP64 issue peak measured in the same run, plus HBM view
cpu_baseline  the C oracle (port of the reference loops) on this box's cores, bounded sample
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree the bench runs from may be read-only; it writes nothing there

METRIC = "viterbi_cells_per_s"
UNIT = "cells/s"


# ----------------------------------------------------------------------------------------------
# synthetic workloads (SURVEY.md section 8d), seeded
# ----------------------------------------------------------------------------------------------
def _log_dirichlet_rows(rng, n, m, alpha, zero_frac):
    # gamma draws normalised per row = Dirichlet(alpha); chunked to bound memory
    out = np.empty((n, m), dtype=np.float64)
    for r0 in range(0, n, 64):
        r1 = min(n, r0 + 64)
        g = rng.standard_gamma(alpha, size=(r1 - r0, m))
        g[g == 0.0] = np.finfo(np.float64).tiny
        p = g / g.sum(axis=1, keepdims=True)
        p[rng.random((r1 - r0, m)) < zero_frac] = 0.0
        with np.errstate(divide="ignore"):
            out[r0:r1] = np.log10(p)
    return out


def make_hmm(seed, K, M, alpha, zero_frac):
    rng = np.random.default_rng(seed)
    A = _log_dirichlet_rows(rng, K, K, alpha, zero_frac)
    B = _log_dirichlet_rows(rng, K, M, alpha, zero_frac)
    pi = _log_dirichlet_rows(rng, 1, K, alpha, zero_frac)[0]
    return A, B, pi


def workload_pos(rank, nseq):
    """K=45, V=20000, T = clamp(round(Gamma(2.5, 10)), 1, 200), Zipf(1.1) word ids; seed 3019 (+rank)."""
    K, M = 45, 20000
    A, B, pi = make_hmm(3019, K, M, 0.1, 0.05)
    rng = np.random.default_rng(3019 + 1000 * (rank + 1))
    lens = np.clip(np.rint(rng.gamma(2.5, 10.0, size=nseq)), 1, 200).astype(np.int64)
    off = np.zeros(nseq + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    obs = (rng.zipf(1.1, size=int(off[-1])) % M).astype(np.uint32)
    cells = float(((lens - 1) * K * K).sum())
    return dict(name="pos_K45_V20k", K=K, M=M, A=A, B=B, pi=pi, obs=obs, off=off, cells=cells,
                steps=float((lens - 1).sum()), desc=f"POS shape K=45 V=20000 B={nseq} avgT=25 (configs[2])")


def workload_large(rank, nseq, T, K=1024, M=4096):
    A, B, pi = make_hmm(3019, K, M, 0.05, 0.0)
    rng = np.random.default_rng(3019 + 1000 * (rank + 1))
    off = np.arange(nseq + 1, dtype=np.int64) * T
    obs = rng.integers(0, M, size=nseq * T).astype(np.uint32)
    cells = float(nseq) * (T - 1) * K * K
    return dict(name=f"large_K{K}", K=K, M=M, A=A, B=B, pi=pi, obs=obs, off=off, cells=cells,
                steps=float(nseq) * (T - 1), desc=f"large-state K={K} M={M} T={T} B={nseq} (configs[3])")


def workload_ar():
    """BASELINE configs[1]: datasets/ar houses A/B/C as committed fixtures (tests/golden/ar_house_*.npz, made by
    tools/make_golden.py from the reference's CSVs; the reference has no preprocessing of its own)."""
    out = []
    for hname in "ABC":
        z = np.load(os.path.join(ROOT, "tests", "golden", f"ar_house_{hname}.npz"))
        K = int(z["n_activities"])
        off = z["seq_off"]
        out.append(dict(name=f"ar_house_{hname}", K=K, M=int(z["n_sensors"]), A=z["logA"], B=z["logB"], pi=z["logPi"],
                        obs=z["obs"], off=off, cells=float(((np.diff(off) - 1) * K * K).sum()), golden=z["paths"]))
    return out


def workload_cp(kind):
    """Constrained decode inputs, sampled from the model itself so that the constraints are satisfiable (as in the
    reference's pipeline, where control tags are true tags): hidden paths and observations are drawn from the HMM,
    four states are "control" states and a position carrying one of them is tagged with that state with some
    probability; component = tag value (Constraints::from_tags), prop = 1.
    trucks: BASELINE configs[0] stand-in (real datasets/trucks is absent): D=2 bdims [16,8] (M=128), K=12, 200
    sequences T~U[50,400], ~10 % of the positions clamped.  (With zero probabilities in the model the reference's
    bound -- stale backpointers into fresh rows, SURVEY Q5 -- is -inf at depth 2 and the search ends after 2K nodes.)
    heavy: configs[4]: K=16, M=64, 64 sequences x T=10000, ~20 % of the positions clamped."""
    rng = np.random.default_rng(3019)
    if kind == "trucks":
        K, M, nseq, pact, tlo, thi, zf = 12, 128, 200, 0.30, 50, 400, 0.0
    elif kind == "heavy10":                                   # configs[4] with ten times the sequences (N = 6.4M)
        K, M, nseq, pact, tlo, thi, zf = 16, 64, 640, 0.80, 10000, 10000, 0.0
    else:
        K, M, nseq, pact, tlo, thi, zf = 16, 64, 64, 0.80, 10000, 10000, 0.0
    A, B, pi = make_hmm(3019, K, M, 0.5, zf)
    PA, PB, Ppi = 10.0 ** A, 10.0 ** B, 10.0 ** pi
    PA /= PA.sum(1, keepdims=True); PB /= PB.sum(1, keepdims=True); Ppi /= Ppi.sum()
    cA, cB = np.cumsum(PA, axis=1), np.cumsum(PB, axis=1)
    lens = rng.integers(tlo, thi + 1, size=nseq)
    N = int(lens.sum())
    start = np.zeros(N, dtype=np.uint8)
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    start[starts] = 1
    states = np.zeros(N, dtype=np.int64)
    u = rng.random(N)
    cur = np.minimum((np.cumsum(Ppi)[None, :] < u[starts][:, None]).sum(1), K - 1)   # first state of every sequence
    pos = starts.copy()
    alive = np.ones(nseq, dtype=bool)
    for t in range(int(lens.max())):                       # all sequences advance together (vectorised over sequences)
        idx = pos[alive]
        states[idx] = cur[alive]
        nxt = np.minimum((cA[cur[alive]] < u[np.minimum(idx + 1, N - 1)][:, None]).sum(1), K - 1)
        cur[alive] = nxt
        pos[alive] += 1
        alive = (pos - starts) < lens
        if not alive.any():
            break
    obs = np.minimum((cB[states] < rng.random(N)[:, None]).sum(1), M - 1).astype(np.uint32)
    control = rng.choice(K, size=4, replace=False)
    comp = np.full(N, -1, dtype=np.int32)
    tagged = rng.random(N) < pact
    for c, st in enumerate(control):
        comp[(states == st) & tagged] = c
    used = sorted(set(int(c) for c in comp if c >= 0))
    remap = {c: i for i, c in enumerate(used)}
    comp = np.array([remap[int(c)] if c >= 0 else -1 for c in comp], dtype=np.int32)
    return dict(name=f"cp_{kind}", K=K, M=M, A=A, B=B, pi=pi, obs=obs, start=start, comp=comp, ncomp=len(used), N=N,
                clamped=float((comp >= 0).mean()))


# ----------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi fields via NVML) during the timed region
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.samples, self.reasons, self.stop = [], set(), False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.max = None

    def _run(self):
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self.stop:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.02)

    def __enter__(self):
        if self.ok:
            self.t = threading.Thread(target=self._run, daemon=True)
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.ok:
            self.t.join()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max, "reasons": sorted(self.reasons)}


# ----------------------------------------------------------------------------------------------
# CPU baseline: the C oracle (port of the reference loops), bounded sample
# ----------------------------------------------------------------------------------------------
def cpu_sample(wl, threads):
    """The bounded sample both CPU legs (cpu_baseline of the GPU arm and --impl reference) run per pass:
    (obs, off, cells, description).  K <= 64: the WHOLE batch when one pass takes a few seconds on this host
    (it does at the POS shape on the GPU boxes), else the longest prefix that does.  K > 64: `threads` sequences x
    the first 64 steps (one full sequence already costs seconds)."""
    from oracle import pyoracle as po

    off, obs, K = wl["off"], wl["obs"], wl["K"]
    B = len(off) - 1
    if K > 64:
        T = int(off[1] - off[0])
        Tc, nb = min(T, 64), min(B, threads)
        o = np.arange(nb + 1, dtype=np.int64) * Tc
        ob = np.concatenate([obs[off[b]: off[b] + Tc] for b in range(nb)])
        return ob, o, float(nb) * (Tc - 1) * K * K, f"{nb} sequences x first {Tc} steps of the workload"
    nb = max(1, min(B, 2000))
    t0 = time.perf_counter()
    po.decode_batch(wl["A"], wl["B"], obs[: off[nb]], off[: nb + 1], nthreads=threads)
    dt = max(time.perf_counter() - t0, 1e-4)
    per_seq = dt / nb
    nb2 = B if per_seq * B <= 8.0 else int(max(nb, min(B, 6.0 / per_seq)))
    o = off[: nb2 + 1]
    desc = f"all {B} sequences of the workload" if nb2 == B else f"first {nb2} of {B} sequences of the workload"
    return obs[: o[-1]], o, float(((np.diff(o) - 1) * K * K).sum()), desc


def cpu_baseline(wl, budget_s=12.0, threads=None):
    """Times the oracle on the sample and RETURNS its output so that the caller can compare the GPU result with it
    (bench.py "parity")."""
    from oracle import pyoracle as po

    threads = threads or (os.cpu_count() or 1)
    ob, o, cells, desc = cpu_sample(wl, threads)
    tot_t, reps, paths, scores = 0.0, 0, None, None
    while tot_t < budget_s and reps < 4:          # ~10-30 s of CPU work in total
        t0 = time.perf_counter()
        paths, scores = po.decode_batch(wl["A"], wl["B"], ob, o, nthreads=threads)
        tot_t += time.perf_counter() - t0
        reps += 1
    line = {"value": cells * reps / tot_t, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{desc} x {reps} passes, {tot_t:.1f} s, C oracle (port of viterbi.rs:5-32), {threads} OpenMP threads"}
    return line, (paths, scores, o)


def parity_block(ref, got_paths, got_scores, off_full):
    """GPU result vs the oracle output of cpu_baseline on the same sequences (bit patterns for the scores)."""
    rp, rs, o = ref
    nb, ne = len(o) - 1, int(o[-1])
    same_layout = bool((np.asarray(off_full[: nb + 1]) == o).all())
    if not same_layout:                            # K > 64 sample: truncated sequences, not comparable element-wise
        return None
    mism = int((got_paths[:ne] != rp).sum())
    return {"sequences": nb, "elements": ne, "path_mismatches": mism,
            "score_bits_equal": bool(got_scores[:nb].tobytes() == rs.tobytes()),
            "against": "C oracle (oracle/cv_oracle.c, restatement of viterbi.rs:5-32), same inputs, same run"}


# ----------------------------------------------------------------------------------------------
def _roof(cells, ms, peak_mix, bytes_moved, hbm_peak, note=""):
    """Both SURVEY 8(d) views for a secondary leg: FP64 add+compare issue (2 per cell) and HBM bytes."""
    alu = 2.0 * cells / (ms * 1e-3)
    hbm = bytes_moved / (ms * 1e-3) / 1e9
    r = {"fp64": {"achieved": alu / 1e12, "peak": peak_mix / 1e12, "unit": "TFLOP/s", "frac": alu / peak_mix},
         "hbm": {"achieved": hbm, "peak": hbm_peak, "unit": "GB/s", "frac": hbm / hbm_peak}, "ms": ms}
    r["bound"] = "latency (neither roofline above 10 %)" if max(r["fp64"]["frac"], r["hbm"]["frac"]) < 0.10 else \
                 ("fp64_alu" if r["fp64"]["frac"] >= r["hbm"]["frac"] else "hbm")
    if note:
        r["note"] = note
    return r


def run_other(cv, L, device, peak_mix, hbm_peak, large_full=True):
    """Short, bounded runs of the other BASELINE configs (reported under "other"; parity for each is in tests/ and,
    where the CPU leg runs the same work, asserted here as well)."""
    from oracle import pyoracle as po
    other = {}
    nthreads = os.cpu_count() or 1
    # configs[1]: datasets/ar, full data set, batched decode (three models, 60 day-sequences in total)
    ar, t_gpu, t_cpu, cells, steps, kbytes = workload_ar(), 0.0, 0.0, 0.0, 0.0, 0.0
    for w in ar:
        hm = cv.HMM(w["A"], w["B"], w["pi"])
        cv.decode_batch(hm, w["obs"], w["off"], device=device)
        t0 = time.perf_counter()
        for _ in range(5):
            paths, _ = cv.decode_batch(hm, w["obs"], w["off"], device=device)
        t_gpu += (time.perf_counter() - t0) / 5
        assert (paths == w["golden"]).all()
        t0 = time.perf_counter()
        rp, _ = po.decode_batch(w["A"], w["B"], w["obs"], w["off"], nthreads=nthreads)
        t_cpu += time.perf_counter() - t0
        assert (paths == rp).all()
        cells += w["cells"]
        nst = float((np.diff(w["off"]) - 1).sum())
        kbytes += nst * (4 + 8 * w["K"] + 2 * w["K"] + 4)       # obs + logB^T row + u8 psi row written and read + path
        hm.close()
    other["ar_full_dataset"] = {"cells": cells, "e2e_ms": 1e3 * t_gpu, "e2e_cells_per_s": cells / t_gpu,
                                "cpu_port_cells_per_s": cells / t_cpu, "paths_equal_oracle_and_golden": True,
                                "roofline": _roof(cells, 1e3 * t_gpu, peak_mix, kbytes, hbm_peak,
                                                  "60 sequences, 1.5e7 cells, serial in t: step latency x longest sequence bounds it; "
                                                  "time is the whole host call (copies and three launches included)"),
                                "note": "60 sequences, 1.5e7 cells: latency bound (serial in t), paths equal the golden fixture"}
    # configs[3] shape at reduced batch/length, and (large_full) the full B=4096, T=4096 pass
    w = workload_large(0, 2048, 64)
    hm = cv.HMM(w["A"], w["B"], w["pi"])
    cv.decode_batch(hm, w["obs"], w["off"], device=device)
    t0 = time.perf_counter()
    cv.decode_batch(hm, w["obs"], w["off"], device=device)
    dt = time.perf_counter() - t0
    other["large_K1024_B2048_T64"] = {"cells": w["cells"], "e2e_ms": 1e3 * dt, "e2e_cells_per_s": w["cells"] / dt}
    if large_full:
        try:
            other["large_full"] = run_large_full(cv, L, device, hm, peak_mix, hbm_peak)
        except Exception as e:  # noqa: BLE001
            other["large_full"] = {"error": repr(e)}
    hm.close()
    # SURVEY 8f N3: supervised MLE event counts (hmm.rs:35-48) at the POS shape, 1M sentences, random tags
    w = workload_pos(0, 1000000)
    tg = np.random.default_rng(3019).integers(0, w["K"], len(w["obs"])).astype(np.int32)
    hm = cv.HMM.new(w["K"], (w["B"].shape[1],))
    hm.mle_arrays(w["obs"], tg, w["off"], device=device)
    hm2 = cv.HMM.new(w["K"], (w["B"].shape[1],))
    t0 = time.perf_counter()
    cms = hm2.mle_arrays(w["obs"], tg, w["off"], device=device)
    dt = time.perf_counter() - t0
    nel = len(w["obs"])
    other["mle_counts_pos_1M"] = {"elements": nel, "count_kernels_ms": cms, "count_GBps": 10.0 * nel / (cms * 1e-3) / 1e9,
                                    "e2e_ms": 1e3 * dt, "bytes_per_element": 10,
                                    "note": "cv_mle: device event counts (u64 atomics; 10 B/element: obs u32, tag i32, start flag written + read) + host replay of the "
                                            "reference's += 1.0 / divide / ln(x)/ln(10); e2e includes H2D of obs+tags and the K*M finalisation"}
    # SURVEY 8f N4: CFN cost tables (cfn.rs:82-167) on the configs[4] super-sequence; CPU port on a prefix
    w = workload_cp("heavy")
    hm = cv.HMM(w["A"], w["B"], w["pi"])
    cv.cfn_tables(hm, w["obs"][:5000], w["start"][:5000], w["comp"][:5000], w["ncomp"], device=device)
    t0 = time.perf_counter()
    r = cv.cfn_tables(hm, w["obs"], w["start"], w["comp"], w["ncomp"], device=device)
    dt = time.perf_counter() - t0
    act = np.flatnonzero(w["comp"] >= 0)
    chg = np.concatenate([[True], w["comp"][act][1:] != w["comp"][act][:-1]])
    bnd = act[chg]
    K = w["K"]
    cells = float(np.diff(bnd).sum()) * K ** 3
    npre = 40000
    t0 = time.perf_counter()
    rc = po.cfn_tables(w["A"], w["B"], w["pi"], w["obs"][:npre], w["start"][:npre], w["comp"][:npre], w["ncomp"])
    dtc = time.perf_counter() - t0
    bpre = bnd[bnd < npre]
    other["cfn_tables_heavy"] = {"N": w["N"], "K": K, "boundaries": int(r["nboundaries"]), "cells": cells,
                                 "device_ms": r["device_ms"], "device_cells_per_s": cells / (r["device_ms"] * 1e-3),
                                 "e2e_ms": 1e3 * dt, "cpu_port_cells_per_s": float(np.diff(bpre).sum()) * K ** 3 / dtc * 1.0,
                                 "cpu_sample": f"first {npre} elements, single thread; the literal port runs K*K sweeps per pair "
                                               "(K-fold the device's work for the same tables), cells counted as K sweeps per pair",
                                 "lower_bound": r["lower_bound"]}
    hm.close()
    # configs[0] stand-in and configs[4]: constrained decode.  First GPU and CPU at the SAME small node budget, every
    # result compared (objective bits, solution, nodes, steps, per-node bounds); then the GPU at the full budget.
    for kind, budget, cpu_budget in (("trucks", 0, 150), ("heavy", 2000, 20)):    # trucks-like: complete search
        w = workload_cp(kind)
        hm = cv.HMM(w["A"], w["B"], w["pi"])
        args = (w["obs"], w["start"], w["comp"], w["ncomp"])
        cv.cp_solve_arrays(hm, *args, max_nodes=3, device=device)
        t0 = time.perf_counter()
        rc = po.cp_solve(w["A"], w["B"], w["pi"], *args, max_nodes=cpu_budget, trace_nodes=cpu_budget)
        dtc = time.perf_counter() - t0
        g = cv.cp_solve_arrays(hm, *args, max_nodes=cpu_budget, device=device, want_ub=cpu_budget)
        n = min(len(g["ub"]), int(rc["explored"]))
        same = bool(g["explored"] == rc["explored"] and g["steps"] == rc["steps"] and (g["sol"] == rc["sol"]).all()
                    and np.float64(g["obj"]).tobytes() == np.float64(rc["obj"]).tobytes()
                    and g["ub"][:n].tobytes() == rc["ub"][:n].tobytes())
        assert same, f"{kind}: GPU and oracle differ at max_nodes={cpu_budget}"
        L.cv_set_timing(1)
        t0 = time.perf_counter()
        r = cv.cp_solve_arrays(hm, *args, max_nodes=budget, device=device)
        dt = time.perf_counter() - t0
        loop_ms = L.cv_last_kernel_ms(hm.device_handle(device))
        L.cv_set_timing(0)
        K = w["K"]
        cells = float(r["steps"]) * K * K
        # per sweep step: delta row written (8K) + psi row written (2K, u16) + previous delta row read (8K) + obs (4)
        other[w["name"]] = {"N": w["N"], "K": K, "nodes": int(r["explored"]), "sweep_steps": int(r["steps"]),
                            "cells": cells, "e2e_ms": 1e3 * dt,
                            "e2e_cells_per_s": cells / dt, "ms_per_node": 1e3 * dt / max(1, r["explored"]),
                            "device_loop_ms_per_node": loop_ms / max(1, r["explored"]),
                            "cpu_port_cells_per_s": float(rc["steps"]) * K * K / dtc, "cpu_nodes": int(rc["explored"]),
                            "cpu_ms_per_node": 1e3 * dtc / max(1, rc["explored"]), "objective": r["obj"],
                            "max_nodes": budget, "clamped_fraction": w["clamped"],
                            "parity": {"max_nodes": cpu_budget, "identical_to_oracle": same,
                                       "compared": "objective bits, solution, explored nodes, sweep steps, every node's bound"},
                            "roofline": _roof(cells, loop_ms, peak_mix, float(r["steps"]) * (18 * K + 4), hbm_peak,
                                              "device loop of the whole search (CUDA events); a node is a chain of short "
                                              "dependent launches, so step latency, not a pipe, bounds it"),
                            "note": "max_nodes = 0: complete branch and bound; the CPU port (single thread, like the "
                                    "reference) runs a node-budgeted prefix of the same search"}
        hm.close()
    return other


def run_large_full(cv, L, device, hm, peak_mix, hbm_peak):
    """BASELINE configs[3] at full size: K = 1024, M = 4096, T = 4096, B = 4096 (1.76e13 cells, 137 GB of delta
    history).  One warm-up pass at reduced batch (kernels and model already warm), one timed full pass with the
    forward/backtrace kernels timed by CUDA events, and 8 sequences checked against the oracle."""
    import torch
    from oracle import pyoracle as po

    w = workload_large(0, 4096, 4096)
    K = w["K"]
    h = hm.device_handle(device)
    N, B = len(w["obs"]), len(w["off"]) - 1
    d_obs = torch.from_numpy(w["obs"].view(np.int32)).cuda()
    d_off = torch.from_numpy(w["off"]).cuda()
    d_path = torch.empty(N, dtype=torch.int32, device="cuda")
    d_score = torch.empty(B, dtype=torch.float64, device="cuda")
    st = torch.cuda.current_stream()
    L.cv_set_timing(1)
    try:
        t0 = time.perf_counter()
        cv._lib.check(L.cv_decode_batch_dev(h, d_obs.data_ptr(), d_off.data_ptr(), B, N, 4096, d_path.data_ptr(),
                                            d_score.data_ptr(), st.cuda_stream, 1))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        fwd, bt = L.cv_last_kernel_ms(h), L.cv_last_backtrace_ms(h)
    finally:
        L.cv_set_timing(0)
    paths = d_path.cpu().numpy().view(np.uint32)
    scores = d_score.cpu().numpy()
    sel = [0, 511, 1024, 1777, 2048, 3000, 3583, 4095]
    off = w["off"]
    sub_obs = np.concatenate([w["obs"][off[b]:off[b + 1]] for b in sel])
    sub_off = np.arange(len(sel) + 1, dtype=np.int64) * 4096
    t0 = time.perf_counter()
    rp, rs = po.decode_batch(w["A"], w["B"], sub_obs, sub_off, nthreads=os.cpu_count() or 1)
    dtc = time.perf_counter() - t0
    got_p = np.concatenate([paths[off[b]:off[b + 1]] for b in sel])
    mism = int((got_p != rp).sum())
    bits = bool(scores[sel].tobytes() == rs.tobytes())
    steps = float(B) * 4095
    kl = ((K + 127) // 128) * 128
    # the delta history is what moves: one [Kl] f64 row per (sequence, step) written by the forward pass, read by the backtrace
    out = {"cells": w["cells"], "B": B, "T": 4096, "K": K, "kernel_ms": fwd, "backtrace_ms": bt, "wall_ms": 1e3 * wall,
           "cells_per_s": w["cells"] / (fwd * 1e-3), "cells_per_s_wall": w["cells"] / wall,
           "roofline": _roof(w["cells"], fwd, peak_mix, steps * (4 + 8 * K + 8 * kl), hbm_peak,
                             "forward kernel(s) alone, CUDA events on the launching stream; FP64 peak from this run's probe"),
           "parity": {"sequences": len(sel), "path_mismatches": mism, "score_bits_equal": bits,
                      "against": f"C oracle on sequences {sel} ({dtc:.1f} s)"},
           "cpu_port_cells_per_s": len(sel) * 4095.0 * K * K / dtc}
    assert mism == 0 and bits, "large_full: GPU and oracle differ"
    del d_obs, d_off, d_path, d_score
    torch.cuda.empty_cache()
    return out


def run_cp_sharded(cv, L, spec, local, rank, world, dist, torch):
    """Constrained decode sharded over the ranks (NVLink peer stores, no NCCL on the data path) next to the same
    solve on one GPU; every rank must return the single-GPU result bit for bit.  Device-loop times (CUDA events,
    set-up and copies excluded), max over ranks."""
    kind, _, budget = spec.partition(":")
    budget = int(budget or 0)
    w = workload_cp(kind)
    hm = cv.HMM(w["A"], w["B"], w["pi"])
    args = (w["obs"], w["start"], w["comp"], w["ncomp"])
    h = hm.device_handle(local)
    L.cv_set_timing(1)
    cv.cp_solve_arrays(hm, *args, max_nodes=3, device=local)
    single = cv.cp_solve_arrays(hm, *args, max_nodes=budget, device=local)
    ms_single = L.cv_last_kernel_ms(h)
    grp = cv.CpDistGroup(hm, cap_N=w["N"], cap_terms=int((w["comp"] >= 0).sum()), device=local)
    grp.solve(*args, max_nodes=3)
    dist.barrier()
    t0 = time.perf_counter()
    r = grp.solve(*args, max_nodes=budget)
    wall = time.perf_counter() - t0
    ms_sharded = L.cv_last_kernel_ms(h)
    L.cv_set_timing(0)
    same = bool((r["sol"] == single["sol"]).all() and r["obj"] == single["obj"] and r["explored"] == single["explored"])
    t = torch.tensor([ms_sharded, ms_single, 1e3 * wall, 0.0 if same else 1.0], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    cuts = cv.plan_cuts(w["comp"], world).tolist()
    grp.close()
    hm.close()
    nodes = max(1, int(r["explored"]))
    return {"workload": w["name"], "N": w["N"], "K": w["K"], "nodes": nodes, "row_cuts": cuts,
            "identical_to_single_gpu_on_every_rank": bool(t[3].item() == 0.0),
            "sharded_ms_per_node": t[0].item() / nodes, "single_gpu_ms_per_node": t[1].item() / nodes,
            "sharded_wall_ms": t[2].item(),
            "exchange": "bound terms, backtrack maps and solution rows by NVLink peer stores + flags (CUDA IPC); no NCCL"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pos", choices=["pos", "large"])
    ap.add_argument("--nseq", type=int, default=0, help="sequences of the batch (0 = the config's size)")
    ap.add_argument("--seqlen", type=int, default=0, help="T for --workload large (0 = 4096)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-other", action="store_true", help="skip the short runs of the other configs")
    ap.add_argument("--no-large-full", action="store_true", help="skip the full-size configs[3] pass of the `other` legs")
    ap.add_argument("--cp-sharded", default="heavy:2000", metavar="KIND:NODES",
                    help="with --gpus > 1: the constrained decode sharded over the ranks (csrc/cp_dist.cuh) next to the "
                         "single-GPU solve, e.g. heavy:2000 (configs[4], the default) or trucks:0; 'off' skips it")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the decoded scores and paths of the last step as DIR/<name>.npy "
                         "(see dump_outputs) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_SCORES_MAX = 1 << 21      # 16 MiB of f64
DUMP_PATHS_MAX = 1 << 22       # 16 MiB of f32
DUMP_PATHS_SAMPLE = 1 << 21


def dump_outputs(out_dir, paths, scores):
    """The batch-ordered results of the last timed step (what a caller of the decode receives) as .npy files:
    scores.npy (f64, one per sequence) and paths.npy (f32 states, one per observation).  An array larger than its cap
    is replaced by a fixed, seeded sample at sorted positions, stored next to it as <name>_index.npy (f64); the
    sample depends only on the array's length, so runs with the same arguments dump the same positions.  At most
    56 MiB in all."""
    os.makedirs(out_dir, exist_ok=True)
    for name, x, cap, n_sample, dtype in (("scores", scores, DUMP_SCORES_MAX, DUMP_SCORES_MAX, np.float64),
                                          ("paths", paths, DUMP_PATHS_MAX, DUMP_PATHS_SAMPLE, np.float32)):
        if len(x) > cap:
            idx = np.sort(np.random.default_rng(3019).choice(len(x), n_sample, replace=False))
            x = x[idx]
            np.save(os.path.join(out_dir, f"{name}_index.npy"), idx.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), x.astype(dtype))


def build_workload(args, rank=0):
    if args.workload == "pos":
        return workload_pos(rank, args.nseq or 1_000_000)
    return workload_large(rank, args.nseq or 4096, args.seqlen or 4096)


def config_block(wl, world):
    """Identical in both arms (`--impl ours` / `--impl reference`): the driver compares it."""
    B, N = len(wl["off"]) - 1, int(wl["off"][-1])
    return {"workload": wl["name"], "desc": wl["desc"], "sequences": B, "elements": N, "cells_per_step": wl["cells"],
            "sharding": f"the batch cut into {world} contiguous slices by forward steps, one per GPU; decoded paths and "
                        "scores all-gathered (ncclAllGather) inside the timed region" if world > 1 else "1 GPU, whole batch",

            "l2": "inputs + delta history per step >> 126 MB L2 (no flush needed)"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (C oracle port; the Rust binary cannot be built here)
    with all host threads; each step one pass over the same bounded sample cpu_baseline uses (the whole batch at the
    POS shape on the GPU boxes)."""
    if rank != 0:
        return
    from oracle import pyoracle as po

    wl = build_workload(args)
    threads = os.cpu_count() or 1
    ob, o, cells, desc = cpu_sample(wl, threads)
    for _ in range(args.warmup):
        po.decode_batch(wl["A"], wl["B"], ob, o, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        paths, scores = po.decode_batch(wl["A"], wl["B"], ob, o, nthreads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, paths, scores)
    v = cells * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_block(wl, world),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{desc} per step, C oracle (port of viterbi.rs:5-32), {threads} OpenMP threads"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def pin_rank_to_gpu_cpus(local, world):
    """Keep this rank's host threads on its own share of the CPUs NVML lists as local to its GPU (its NUMA node);
    pinned buffers allocated afterwards are first-touched there.  Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1 and 64 * i + b < ncpu]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return "unchanged (NVML lists no usable CPUs)"
        n_local = max(1, world)
        share = [c for i, c in enumerate(allowed) if i * n_local // len(allowed) == local % n_local] or allowed
        os.sched_setaffinity(0, share)
        return f"{len(share)} of the {len(allowed)} CPUs local to GPU {local}"
    except Exception as e:  # noqa: BLE001
        return f"unchanged ({type(e).__name__})"


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import consistent_viterbi_b200 as cv
    from consistent_viterbi_b200.dist import ShardedDecoder

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    affinity = pin_rank_to_gpu_cpus(local, world) if world > 1 else "not pinned (1 rank)"
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    L = cv._lib.lib()
    wl = build_workload(args)                      # the SAME batch on every rank; rank r decodes slice r of it
    hmm = cv.HMM(wl["A"], wl["B"], wl["pi"])
    h = hmm.device_handle(local)
    obs_np, off_np = wl["obs"], wl["off"]
    B, N = len(off_np) - 1, int(off_np[-1])
    K = wl["K"]

    # ---- FP64 issue peak of this GPU, measured now (roofline denominator) ----
    ops, ms = C.c_double(), C.c_double()
    cv._lib.check(L.cv_debug_probe_fp64(local, 0, 20000, C.byref(ops), C.byref(ms)))
    peak_dadd = ops.value
    cv._lib.check(L.cv_debug_probe_fp64(local, 1, 20000, C.byref(ops), C.byref(ms)))
    peak_mix = ops.value

    # ---- this rank's slice, device resident; results land in the padded all-gather buffers ----
    sd = ShardedDecoder(hmm, off_np, device=local)
    sd.load_obs(obs_np)
    my_cells = float(((np.diff(sd.off_l_np) - 1) * K * K).sum())
    stream = torch.cuda.current_stream()

    def step_dev():
        sd.step()      # cv_decode_batch_dev(_u8) into this rank's row of the gather buffer (+ one in-place ncclAllGather when world > 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_dev()
    barrier()
    launches0 = L.cv_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        e0.record(stream)
        for _ in range(args.steps):
            step_dev()
        e1.record(stream)
        barrier()
    launches = L.cv_launch_count() - launches0
    dev_ms = e0.elapsed_time(e1)
    full_paths = sd.paths().cpu().numpy()
    full_paths = full_paths.astype(np.uint32) if sd.narrow_paths else full_paths.view(np.uint32)
    full_scores = sd.scores().cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, full_paths, full_scores)

    # ---- share of the collective: the same steps without / with only the all-gather ----
    gather_ms = 0.0
    if world > 1:
        g0, g1, g2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        barrier()
        g0.record(stream)
        for _ in range(args.steps):
            sd.decode_local()
        g1.record(stream)
        for _ in range(args.steps):
            sd.gather()
        g2.record(stream)
        barrier()
        local_ms, gather_ms = g0.elapsed_time(g1) / args.steps, g1.elapsed_time(g2) / args.steps

    # ---- dominant-kernel duration: CUDA events on the launching stream around the forward kernel ----
    L.cv_set_timing(1)
    fwd_ms, bt_ms = [], []
    n_el, n_sq = sd.n_el[rank], sd.n_sq[rank]
    dec_fn = L.cv_decode_batch_dev_u8 if sd.narrow_paths else L.cv_decode_batch_dev
    for _ in range(max(3, min(args.steps, 5))):
        rc = dec_fn(h, sd.obs_l.data_ptr(), sd.off_l.data_ptr(), n_sq, n_el, sd.max_len,
                    sd.gpaths[rank].data_ptr(), sd.gscores[rank].data_ptr(), stream.cuda_stream, 1)
        cv._lib.check(rc)
        fwd_ms.append(L.cv_last_kernel_ms(h))
        bt_ms.append(L.cv_last_backtrace_ms(h))
    L.cv_set_timing(0)
    fwd, bt = float(np.mean(fwd_ms)), float(np.mean(bt_ms))

    # ---- end to end through the C ABI with pinned host buffers: this rank's slice in, its results out ----
    e0_, e1_ = sd.e0, sd.e1
    off_l = sd.off_l_np

    def pinned(arr):
        p = L.cv_host_alloc(max(arr.nbytes, 1))
        assert p, "cv_host_alloc failed"
        buf = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(arr.nbytes, 1),))
        buf[: arr.nbytes] = arr.view(np.uint8).reshape(-1)
        return p
    p_obs = pinned(np.ascontiguousarray(obs_np[e0_:e1_]))
    p_off = pinned(np.ascontiguousarray(off_l))
    p_path = L.cv_host_alloc(max(4 * n_el, 1))
    p_score = L.cv_host_alloc(max(8 * n_sq, 1))

    keep_path = torch.empty(max(n_el, 1), dtype=torch.int32, device="cuda") if world > 1 else None

    def step_e2e():
        # H2D of the slice, decode, D2H of its paths / scores: one C-ABI call with host pointers
        if world == 1:
            cv._lib.check(L.cv_decode_batch(h, p_obs, p_off, n_sq, p_path, p_score))
        else:
            # every rank also needs the others' paths on its device (north_star): the device copies of this rank's
            # results stay in its row of the gather buffers (cv_decode_batch_keep), then the all-gather on device
            cv._lib.check(L.cv_decode_batch_keep(h, p_obs, p_off, n_sq, p_path, p_score, keep_path.data_ptr(),
                                                 sd.gscores[rank].data_ptr()))
            sd.gpaths[rank, :n_el].copy_(keep_path[:n_el])            # u32 -> the gather buffer's element type (u8 for K <= 64)
            sd.gather()
            torch.cuda.current_stream().synchronize()
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    n_e2e = max(2, min(args.steps, 5))
    for _ in range(n_e2e):
        step_e2e()
    barrier()
    e2e_s = (time.perf_counter() - t0) / n_e2e
    # check the end-to-end result against the device-resident one
    host_paths = np.ctypeslib.as_array(C.cast(p_path, C.POINTER(C.c_uint32)), shape=(max(n_el, 1),))[:n_el]
    assert (host_paths == full_paths[e0_:e1_]).all(), "e2e and device-resident paths differ"

    # ---- the same call with narrow host formats (u16 observations in, u8 states out): a third of the PCIe bytes ----
    narrow_s = None
    if K <= 64 and wl["M"] <= 65536:
        p_obs16 = pinned(np.ascontiguousarray(obs_np[e0_:e1_].astype(np.uint16)))
        p_path8 = L.cv_host_alloc(max(n_el, 1))

        def step_narrow():
            cv._lib.check(L.cv_decode_batch_u16u8(h, p_obs16, p_off, n_sq, p_path8, p_score))
        for _ in range(2):
            step_narrow()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            step_narrow()
        barrier()
        narrow_s = (time.perf_counter() - t0) / n_e2e
        host_paths8 = np.ctypeslib.as_array(C.cast(p_path8, C.POINTER(C.c_uint8)), shape=(max(n_el, 1),))[:n_el]
        assert (host_paths8 == full_paths[e0_:e1_]).all(), "narrow-format and device-resident paths differ"
        L.cv_host_free(p_obs16); L.cv_host_free(p_path8)

    # ---- optional f32 mode (cv_decode_batch_dev_f32; not the parity path): throughput and distance from the exact result ----
    f32_mode = None
    if world == 1 and K <= 64:
        d_p32 = torch.empty(max(n_el, 1), dtype=torch.int32, device="cuda")
        d_s32 = torch.empty(max(n_sq, 1), dtype=torch.float64, device="cuda")

        def step_f32():
            cv._lib.check(L.cv_decode_batch_dev_f32(h, sd.obs_l.data_ptr(), sd.off_l.data_ptr(), n_sq, n_el, sd.max_len,
                                                    d_p32.data_ptr(), d_s32.data_ptr(), stream.cuda_stream, 0))
        for _ in range(3):
            step_f32()
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(args.steps):
            step_f32()
        f1.record(stream)
        torch.cuda.synchronize()
        f32_ms = f0.elapsed_time(f1) / args.steps
        s32, p32 = d_s32.cpu().numpy(), d_p32.cpu().numpy().view(np.uint32)
        fin = np.isfinite(full_scores)
        rel = np.abs(s32[fin] - full_scores[fin]) / np.maximum(np.abs(full_scores[fin]), 1.0)
        same_el = float((p32 == full_paths).mean())
        f32_mode = {"ms_per_step": f32_ms, "value": wl["cells"] / (f32_ms * 1e-3), "unit": UNIT, "dtype": "f32",
                    "max_rel_score_error_vs_f64": float(rel.max()) if rel.size else 0.0, "tolerance": 1e-5,
                    "neg_inf_scores_match": bool((np.isneginf(s32) == np.isneginf(full_scores)).all()),
                    "path_elements_equal_to_f64": same_el,
                    "note": "optional mode of BASELINE.json's north_star (f32 recurrence, FADD2 + FMNMX3); NOT the parity path -- "
                            "the headline value / parity / roofline above are the exact f64 mode"}
        del d_p32, d_s32

    # ---- reduce over ranks ----
    def allred(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=op)
        return float(t.item())

    def allgather_vals(xs):
        t = torch.tensor(xs, dtype=torch.float64, device="cuda")
        if world == 1:
            return [xs]
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [o.tolist() for o in out]

    MAX, SUM = (dist.ReduceOp.MAX, dist.ReduceOp.SUM) if world > 1 else (None, None)

    # ---- secondary: weak scaling (every rank decodes its OWN full-size batch, no collective), as round 1 measured ----
    weak = None
    if world > 1 and args.workload == "pos":
        wlw = workload_pos(rank + 1, args.nseq or 1_000_000)
        d_obs = torch.from_numpy(wlw["obs"].view(np.int32)).cuda()
        d_off = torch.from_numpy(wlw["off"]).cuda()
        Bw, Nw = len(wlw["off"]) - 1, int(wlw["off"][-1])
        d_path = torch.empty(Nw, dtype=torch.int32, device="cuda")
        d_score = torch.empty(Bw, dtype=torch.float64, device="cuda")
        mlw = int(np.diff(wlw["off"]).max())

        def step_weak():
            cv._lib.check(L.cv_decode_batch_dev(h, d_obs.data_ptr(), d_off.data_ptr(), Bw, Nw, mlw, d_path.data_ptr(),
                                                d_score.data_ptr(), stream.cuda_stream, 0))
        for _ in range(args.warmup):
            step_weak()
        barrier()
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record(stream)
        for _ in range(args.steps):
            step_weak()
        w1.record(stream)
        barrier()
        wms = allred(w0.elapsed_time(w1), MAX)
        wcells = allred(wlw["cells"], SUM)
        weak = {"scaling": "weak", "value": wcells * args.steps / (wms * 1e-3), "unit": UNIT, "ms_per_step": wms / args.steps,
                "per_gpu_sequences": Bw, "note": "every rank decodes its own batch of the config's size; no data-path collective"}
        del d_obs, d_off, d_path, d_score

    cp_sharded = None
    if args.cp_sharded and args.cp_sharded != "off" and world > 1:
        try:
            cp_sharded = run_cp_sharded(cv, L, args.cp_sharded, local, rank, world, dist, torch)
        except Exception as e:  # noqa: BLE001
            cp_sharded = {"error": repr(e)}

    per_rank = allgather_vals([dev_ms / args.steps, 1e3 * e2e_s, fwd, bt, gather_ms, float(n_sq), my_cells])
    dev_ms = allred(dev_ms, MAX)
    e2e_s = allred(e2e_s, MAX)
    if narrow_s is not None:
        narrow_s = allred(narrow_s, MAX)
    launches = int(allred(float(launches), SUM))
    fwd_max = allred(fwd, MAX)
    bt_max = allred(bt, MAX)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        # algorithmic HBM bytes per step of one sequence (DESIGN.md "Roofline"): obs u32 + logB^T row +
        # delta-history row written by the forward kernel and read back by the backtrace + path u32
        if K <= 64:
            bytes_per_step = 4 + 8 * K + 8 * K + 8 * K + 4
        else:
            w = 1 if ((K + 127) // 128) * 128 <= 256 else 2
            bytes_per_step = 4 + 8 * K + w * K + w + 4
        my_steps = float((np.diff(off_l) - 1).sum())
        achieved_alu = 2.0 * my_cells / (fwd * 1e-3)                 # 1 DADD + 1 compare per cell, rank 0's slice
        step_ms = dev_ms / args.steps
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if world == 1 and wl["name"] in tj:
                traffic, traffic_src = tj[wl["name"]], tj.get("_source")
        except Exception:
            pass
        hbm_ach = my_steps * bytes_per_step / ((fwd + bt) * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": wl["cells"] * args.steps / (dev_ms * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(wl, world),
            "e2e": {"value": wl["cells"] / e2e_s, "unit": UNIT,
                    "h2d_bytes_per_step": int(4 * n_el + 8 * (n_sq + 1)),
                    "d2h_bytes_per_step": int(4 * n_el + 8 * n_sq), "ms_per_step": 1e3 * e2e_s,
                    "bytes_note": "rank 0's slice; every rank moves its own slice",
                    "api": "cv_decode_batch (C ABI, pinned host buffers)" if world == 1 else
                           "cv_decode_batch_keep (C ABI, pinned host buffers; device copies kept) per rank + ncclAllGather"},
            "gpu_launches": launches,
            "clocks": clk.summary(),
            "roofline": {
                "bound": "fp64_alu", "kernel": "decode_small_fwd_kernel" if K <= 64 else "decode_large_kernel",
                "achieved": achieved_alu / 1e12, "peak": peak_mix / 1e12, "unit": "TFLOP/s",
                "unit_note": "FP64 add+compare operations (2 per cell, SURVEY 8d), not tensor FLOPs",
                "frac": achieved_alu / peak_mix,
                "frac_on_step": 2.0 * wl["cells"] / world / (step_ms * 1e-3) / peak_mix,
                "frac_note": "frac = the forward kernel timed alone (CUDA events on its stream); frac_on_step = the same "
                             "algorithmic operations over the whole driver-timed step (forward + concurrent backtrace"
                             + (" + all-gather" if world > 1 else "") + ")",
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "measured in this run: DADD+DSETP issue rate over all SMs (cv_debug_probe_fp64 mode 1); "
                               f"DADD alone {peak_dadd / 1e12:.2f}",
                "kernel_ms": fwd, "backtrace_ms": bt, "kernel_ms_max_over_ranks": fwd_max, "backtrace_ms_max_over_ranks": bt_max,
                "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "bytes_per_step": bytes_per_step,
                        "frac": hbm_ach / hbm_peak,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s"},
            },
        }
        if f32_mode is not None:
            line["f32_mode"] = f32_mode
        if narrow_s is not None:
            line["e2e_narrow"] = {"value": wl["cells"] / narrow_s, "unit": UNIT, "ms_per_step": 1e3 * narrow_s,
                                  "h2d_bytes_per_step": int(2 * n_el + 8 * (n_sq + 1)), "d2h_bytes_per_step": int(n_el + 8 * n_sq),
                                  "api": "cv_decode_batch_u16u8 (u16 observations, u8 states; per rank, no collective)",
                                  "note": "secondary: the reference-shaped u32 call above is the headline e2e"}
        if world > 1:
            line["collective"] = {"name": "one in-place ncclAllGather (torch.distributed.all_gather_into_tensor) of the [world][scores f64 | "
                                          "paths u8 (K <= 64, else u32)] buffer, rows padded to the largest slice",
                                  "ms_per_step": gather_ms, "local_decode_ms_per_step": local_ms,
                                  "share_of_step": gather_ms / max(step_ms, 1e-9),
                                  "path_element_bytes": int(sd.gpaths.element_size()),
                                  "bytes_received_per_rank": int((world - 1) * sd.gbuf.shape[1])}
            line["per_rank"] = {"columns": ["step_ms", "e2e_ms", "fwd_kernel_ms", "backtrace_ms", "gather_ms", "sequences", "cells"],
                                "rows": per_rank, "host_affinity": affinity}
            if weak is not None:
                line["weak_scaling"] = weak
        if not args.no_cpu and world == 1:
            line["cpu_baseline"], ref = cpu_baseline(wl)
            par = parity_block(ref, full_paths, full_scores, off_np)
            if par is not None:
                line["parity"] = par
        if not args.no_other and world == 1 and args.workload == "pos":
            hmm.close()                                   # free the POS workspaces (9 GB of history) first
            del sd
            torch.cuda.empty_cache()
            try:
                line["other"] = run_other(cv, L, local, peak_mix, hbm_peak, large_full=not args.no_large_full)
            except Exception as e:  # the headline numbers stand on their own
                line["other"] = {"error": repr(e)}
        if cp_sharded is not None:
            line["cp_sharded"] = cp_sharded
        print(json.dumps(line), flush=True)
    for p in (p_obs, p_off, p_path, p_score):
        L.cv_host_free(p)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
