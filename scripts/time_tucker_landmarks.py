"""Device-resident cost of the raw-landmark Tucker entry points against their feature twins.

Usage: python scripts/time_tucker_landmarks.py [--n 1000000] [--rounds 5] [--out result.json]

1 M synthetic faces (shipped W and cosine rows) are turned into raw MediaPipe-style landmarks by a per-face scale and
shift (as tests/golden/make_golden_prepost.py does); their IPD-normalised twins are computed here in float64 on the
device.  fit (T = 3000) and the converged solve run on the raw rows (landmarks=True) and on the twins, alternately, timed
with CUDA events; the card's name and power limit are read in the same run.  The outputs of the two inputs are checked
bit for bit before anything is timed.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from nlml_hpe_b200 import synthetic  # noqa: E402
from nlml_hpe_b200.tucker import TuckerFitter  # noqa: E402

T_ITERS = 3000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "unavailable"}


def make_inputs(n, art, rows, chunk=65536):
    feats = synthetic.make_features_torch(n, art["W"], *rows, U_id=art["U_id"], seed=1234, device="cuda")
    raw = torch.empty_like(feats)
    norm = torch.empty_like(feats)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(99)
    for s0 in range(0, n, chunk):
        m = min(chunk, n - s0)
        f = feats[s0:s0 + m].double().view(m, 468, 3)
        scale = torch.rand(m, 1, 1, generator=gen, device="cuda", dtype=torch.float64) * 0.25 + 0.05
        shift = torch.rand(m, 1, 3, generator=gen, device="cuda", dtype=torch.float64) * 0.4 + 0.3
        r = (f * scale + shift).float()
        raw[s0:s0 + m] = r.view(m, -1)
        # the reference's arithmetic (FeatureExtractor.py:30-66): float64, ((dx*dx + dy*dy) + dz*dz), 1e-6 when zero
        r64 = r.double()
        d = r64[:, 33] - r64[:, 263]
        ipd = torch.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
        ipd = torch.where(ipd == 0, torch.full_like(ipd, 1e-6), ipd)
        norm[s0:s0 + m] = ((r64 - r64[:, 1:2]) / ipd[:, None, None]).float().view(m, -1)
    del feats
    return raw, norm


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this script measures on the GPU only")
    n = args.n
    art, rows = bench.load_artifacts()
    fit = TuckerFitter(art["W"], *rows, device="cuda:0")
    raw, norm = make_inputs(n, art, rows)
    P = torch.empty((n, fit.n_params), device="cuda")

    # same bits first (fit at a short T over the whole batch, the solve with its evaluation counts)
    a = fit.fit(raw, 20, landmarks=True).cpu().numpy().view(np.uint32)
    b = fit.fit(norm, 20).cpu().numpy().view(np.uint32)
    sa, ea = fit.solve(raw, return_evals=True, landmarks=True)
    sb, eb = fit.solve(norm, return_evals=True)
    same = bool(np.array_equal(a, b) and torch.equal(sa.view(torch.int32), sb.view(torch.int32)) and torch.equal(ea, eb))
    del sa, sb, ea, eb

    calls = {
        "fit_landmarks": lambda: fit.fit(raw, T_ITERS, out=P, landmarks=True),
        "fit_features": lambda: fit.fit(norm, T_ITERS, out=P),
        "solve_landmarks": lambda: fit.solve(raw, out=P, landmarks=True),
        "solve_features": lambda: fit.solve(norm, out=P),
    }
    for fn in calls.values():   # warm-up of every shape
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in calls}
    for _ in range(args.rounds):   # alternate the two inputs so drift hits both alike
        for k, fn in calls.items():
            ms[k].append(timed(fn))
    res = {"n": n, "T": T_ITERS, "rounds": args.rounds, "device": card(), "bit_identical": same, "ms": ms}
    for k, v in ms.items():
        res[f"{k}_median_ms"] = statistics.median(v)
        res[f"{k}_poses_per_s"] = n / statistics.median(v) * 1e3
    res["fit_ratio_landmarks_over_features"] = res["fit_landmarks_median_ms"] / res["fit_features_median_ms"]
    res["solve_ratio_landmarks_over_features"] = res["solve_landmarks_median_ms"] / res["solve_features_median_ms"]
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
