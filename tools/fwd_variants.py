"""Times the forward tile kernel variants on the POS shape (BASELINE configs[2]) and checks each against variant 0.

    python tools/fwd_variants.py [nseq] [variants...]        e.g.  python tools/fwd_variants.py 1000000 1 0

variant: 1 = balanced state split (default), 0 = groups of 8 states (last one padded), 3 = the optional f32 mode (cv_decode_batch_dev_f32; results differ by design), 4 = default but
run-time row pitches in the forward kernel (cv_debug_set_fwd_ldc(0)), 5 = default but every warp fetches emission rows
(cv_debug_set_em_light(0)), 6 = default but the one-thread-per-sequence backtrace (cv_debug_set_bt_split(0)), 7 = the four-lane backtrace at
every batch size (cv_debug_set_bt_split(2); the default uses it up to ~1300 sequences per SM).  Prints the forward kernel alone (CUDA events, timing mode), and the device-resident step (forward +
concurrent backtrace) for each variant, plus the extra `CV_*` settings given in the environment."""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import consistent_viterbi_b200 as cv  # noqa: E402

nseq = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
variants = [int(v) for v in sys.argv[2:]] or [1, 0]
assert all(v in (0, 1, 3, 4, 5, 6, 7) for v in variants), "unknown variant"
wl = bench.workload_pos(0, nseq)
L = cv._lib.lib()
hmm = cv.HMM(wl["A"], wl["B"], wl["pi"])
h = hmm.device_handle(0)
N, B = len(wl["obs"]), len(wl["off"]) - 1
d_obs = torch.from_numpy(wl["obs"].view(np.int32)).cuda()
d_off = torch.from_numpy(wl["off"]).cuda()
d_path = torch.empty(N, dtype=torch.int32, device="cuda")
d_score = torch.empty(B, dtype=torch.float64, device="cuda")
ml = int(np.diff(wl["off"]).max())
st = torch.cuda.current_stream()
ops, ms = C.c_double(), C.c_double()
cv._lib.check(L.cv_debug_probe_fp64(0, 1, 20000, C.byref(ops), C.byref(ms)))
peak = ops.value


FN = [L.cv_decode_batch_dev]


def run(sync):
    cv._lib.check(FN[0](h, d_obs.data_ptr(), d_off.data_ptr(), B, N, ml, d_path.data_ptr(),
                        d_score.data_ptr(), st.cuda_stream, sync))


ref = None
out = []
for v in variants:
    L.cv_debug_set_balanced_split(1 if v else 0)
    L.cv_debug_set_fwd_ldc(0 if v == 4 else 1)
    L.cv_debug_set_em_light(0 if v == 5 else 1)
    L.cv_debug_set_bt_split(0 if v == 6 else 2 if v == 7 else 1)
    FN[0] = L.cv_decode_batch_dev_f32 if v == 3 else L.cv_decode_batch_dev        # 3 = the optional f32 mode
    for _ in range(3):
        run(0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(8):
        run(0)
    e1.record(st)
    torch.cuda.synchronize()
    step = e0.elapsed_time(e1) / 8
    p, s = d_path.cpu().numpy().copy(), d_score.cpu().numpy().copy()
    if ref is None:
        ref = (p, s)
    same = bool((p == ref[0]).all() and s.tobytes() == ref[1].tobytes())
    L.cv_set_timing(1)
    f, b = [], []
    for _ in range(4):
        run(1)
        f.append(L.cv_last_kernel_ms(h)); b.append(L.cv_last_backtrace_ms(h))
    L.cv_set_timing(0)
    rec = {"variant": v, "fwd_ms": float(np.mean(f)), "bt_ms": float(np.mean(b)), "step_ms": step,
           "frac_fwd": 2 * wl["cells"] / (np.mean(f) * 1e-3) / peak, "frac_step": 2 * wl["cells"] / (step * 1e-3) / peak,
           "same_as_first": same}
    out.append(rec)
    print(json.dumps(rec), flush=True)
L.cv_debug_set_balanced_split(1)
L.cv_debug_set_fwd_ldc(1)
L.cv_debug_set_em_light(1)
L.cv_debug_set_bt_split(1)
print(json.dumps({"peak_fp64_ops": peak, "env": {k: v for k, v in os.environ.items() if k.startswith("CV_")}}))
