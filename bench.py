#!/usr/bin/env python
"""bench.py -- poses/sec of the NLML_HPE inference hot path on B200 (one process per GPU).

Contract (task statement): `python bench.py --gpus N --steps K --warmup W` (under torchrun for N>1)
prints ONE JSON line on rank 0.  A "step" is one pass of the hot path over one batch of synthetic
feature vectors per GPU.  Headline = the Tucker-fit half (BASELINE.json configs[3]: 1M synthetic
samples per GPU, shipped W, ranks (5,3,3,3), T=3000); the Encoder+heads half (configs[2]) is reported in
the same line under "mlp".  `--impl reference` times the CPU port of the reference (oracle/) instead.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F = 1404
RANKS = (5, 3, 3, 3)
T_ITERS, LR, CLIP = 3000, 1e-3, 1.0

# executed FP32 work of the folded-Gram iteration, per sample (DESIGN.md section 3):
#   quadratic pass 216*(15+15+3)+36*3 FMA, back-substitution 52, linear term 351, features/clip ~60
TUCKER_FMA_PER_ITER = 216 * 33 + 36 * 3 + 52 + 351 + 60
TUCKER_FLOP_PER_POSE = 2 * (135 * F + T_ITERS * TUCKER_FMA_PER_ITER)
TUCKER_FLOP_PER_POSE_GRAM = 2 * 135 * F + T_ITERS * (2 * 135 * 135 + 2000)      # SURVEY.md section 8d
TUCKER_FLOP_PER_POSE_REFERENCE = T_ITERS * 2 * 2 * 135 * F                        # SURVEY.md section 8d
# tensor-core kernel: issued FP16 flops per pose (two GEMMs per iteration, three hi/lo passes per MAC)
# one Newton evaluation: per S row (216) 15 FMA for T + 4x15 FMA for GU/HY/HP/HR + 20 for the scalar sums,
# linear term 5*3*(6*9) FMA + assembly
SOLVE_FLOP_PER_EVAL = 2 * (216 * (15 + 60 + 20) + 5 * 3 * 54 + 400)
TUCKER_TC_FLOP_PER_POSE = T_ITERS * 2 * 3 * (224 * 16 + 96 * 48) + 2 * 3 * 144 * 1408   # ISSUED: three FP16 hi/lo passes and padding
                                                                                          # (+ phase A: 3xTF32 projection, 144 x 1408 padded)
TUCKER_TC_USEFUL_FLOP_PER_POSE = T_ITERS * 2 * (2 * 15 * 216) + 2 * 135 * F   # USEFUL: the two contractions with the folded Gram tensor + q = W2 x
TUCKER_BYTES_PER_POSE = F * 4 + 8 * 4
# DRAM traffic of the fit (projection GEMM + iteration kernel) per sample, from the committed `ncu --set full` capture of a
# 37 888-sample batch; scaled to the bench launch
TUCKER_TC_NCU_SOURCE = "profiles/r02_tucker_tc_final_ncu.txt"
TUCKER_TC_NCU_DRAM_BYTES_PER_POSE = (222.596608e6 + 14.701824e6 + 20.696064e6 + 0.0) / 37888   # projection read + write, fit read + write
# DRAM traffic of the Encoder+heads chain per sample: ncu dram__bytes_read.sum + dram__bytes_write.sum over the nine launches of
# one 151 552-sample chunk (profiles/r02_mlp_launches.txt: 3915.8 MB read + 2593.0 MB written)
MLP_NCU_DRAM_BYTES_PER_POSE = (3897.6e6 + 2588.9e6) / 151552   # profiles/r02_mlp_launches.txt: DRAM read + write of one chunk's nine launches
MLP_FLOP_PER_POSE = 4_714_240                                                     # SURVEY.md section 8a (a10)
MLP_BYTES_PER_POSE = F * 4 + 3 * 4

# --dump-outputs: outputs longer than DUMP_ROWS rows keep the same seeded sample of DUMP_ROWS rows, which holds the
# 1M-row default run's dump to 27 MB
DUMP_ROWS = 1 << 18
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each output as out_dir/<name>.npy.  With the same arguments the inputs and the sampled rows are the same
    from run to run, so two builds of the project can be compared array for array."""
    picked = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"{name}: {a.dtype} output")
        if a.shape[0] > DUMP_ROWS:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], DUMP_ROWS, replace=False))]
        picked[name] = a
    total = sum(a.nbytes for a in picked.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes, more than {DUMP_MAX_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in picked.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def load_artifacts():
    art = dict(np.load(os.path.join(ROOT, "tests", "golden", "shipped_artifacts.npz")))
    rows = tuple(np.ascontiguousarray(art[f"optimized_{k}"][0:3, :]) for k in ("yaw", "pitch", "roll"))
    return art, rows


def state_dicts(art):
    from nlml_hpe_b200 import synthetic
    enc = synthetic.synthetic_encoder_state_dict(art["W"], art["optimized_yaw"], art["optimized_pitch"],
                                                 art["optimized_roll"], U_id=art["U_id"], seed=0)
    heads = [{k.split(".", 1)[1]: v for k, v in art.items() if k.startswith(f"{h}_network.")}
             for h in ("yaw", "pitch", "roll")]
    return enc, heads[0], heads[1], heads[2]


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.path = gpu_index, None, None

    def __enter__(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(5)
            except Exception:
                self.proc.kill()

    def summary(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.path or not os.path.exists(self.path):
            return out
        sm, mx, reasons = [], [], set()
        for line in open(self.path):
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            busy = [s for s in sm if s > 0.5 * max(sm)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
def time_steps(fn, steps, warmup, torch, dist, world):
    """W warm-ups, then exactly K steps between barrier+synchronize, CUDA events, max over ranks."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = e0.elapsed_time(e1)
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms, wall_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall_ms = t.tolist()
    return ms, wall_ms


def time_host_steps(fn, steps, warmup, torch, dist, world):
    """Same for a host-buffer call (synchronous): wall clock around K calls, max over ranks."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    return ms


def cpu_baseline_tucker(art, rows, cores, seconds_cap=40.0):
    """oracle port of TD_Tester.optimize_with_sgd (autograd form, as the reference runs it), one sample per
    worker process with 1 torch thread each, `cores` workers, T=3000."""
    from concurrent.futures import ProcessPoolExecutor
    from nlml_hpe_b200 import synthetic
    cores = physical_cores(cores)
    X = synthetic.make_features(cores, art["W"], *rows, U_id=art["U_id"], seed=1234)
    with ProcessPoolExecutor(max_workers=cores, initializer=_pin_worker, initargs=(cores,)) as pool:
        list(pool.map(_cpu_warm_worker, range(cores)))          # interpreter + torch import stay outside the timing
        t0 = time.perf_counter()
        list(pool.map(_cpu_tucker_worker, [(art["W"], X[i], rows) for i in range(cores)]))
        dt = time.perf_counter() - t0
    return {"value": cores / dt, "unit": "poses/s", "cores": cores, "kind": "port", "s_per_sample_per_core": dt, "seconds": dt,
            "sample": f"{cores} samples (one per worker process pinned to its own physical core, 1 thread each), T={T_ITERS}, "
                      f"oracle.tucker_oracle.sgd_reference_form = autograd restatement of TD_Tester.py:127-159; {dt:.1f} s"}


def cpu_baseline_powell(art, rows, cores):
    """What TD_Tester.Test runs by default: scipy Powell over the float64 objective (oracle.tucker_oracle.powell_fit =
    restatement of TD_Tester.py:162-199), one sample per worker process."""
    from concurrent.futures import ProcessPoolExecutor
    from nlml_hpe_b200 import synthetic
    cores = physical_cores(cores)
    X = synthetic.make_features(cores, art["W"], *rows, U_id=art["U_id"], seed=1234)
    with ProcessPoolExecutor(max_workers=cores, initializer=_pin_worker, initargs=(cores,)) as pool:
        list(pool.map(_cpu_warm_worker, range(cores)))
        t0 = time.perf_counter()
        list(pool.map(_cpu_powell_worker, [(art["W"], X[i], rows) for i in range(cores)]))
        dt = time.perf_counter() - t0
    return {"value": cores / dt, "unit": "poses/s", "cores": cores, "kind": "port",
            "sample": f"{cores} samples (one per worker process), scipy Powell as TD_Tester.Test (TD_Tester.py:191-199); {dt:.1f} s"}


def physical_cores(logical):
    """One worker per PHYSICAL core (hyper-thread siblings share an FP unit: oversubscribing them made the two CPU legs of
    round 1 disagree by 2x).  Falls back to the logical count when /sys is not readable."""
    try:
        seen = set()
        for cpu in sorted(os.sched_getaffinity(0)):
            with open(f"/sys/devices/system/cpu/cpu{cpu}/topology/thread_siblings_list") as f:
                seen.add(f.read().strip())
        return max(1, min(logical, len(seen)))
    except Exception:
        return logical


def _cpu_powell_worker(args):
    import torch
    torch.set_num_threads(1)
    from oracle import tucker_oracle
    W, x, rows = args
    return tucker_oracle.powell_fit(W, x, *rows)[0]


def _cpu_warm_worker(_):
    import torch
    torch.set_num_threads(1)
    from oracle import tucker_oracle  # noqa: F401
    time.sleep(0.2)
    return 0


def _cpu_tucker_worker(args):
    import torch
    torch.set_num_threads(1)
    from oracle import tucker_oracle
    W, x, rows = args
    return tucker_oracle.sgd_reference_form(W, x, *rows, lr=LR, iters=T_ITERS, clip=CLIP)


def cpu_baseline_mlp(art, cores, n=16384, reps=3):
    import torch
    from nlml_hpe_b200 import synthetic
    from oracle import mlp_oracle
    sds = state_dicts(art)
    rows = tuple(art[f"optimized_{k}"][0:3] for k in ("yaw", "pitch", "roll"))
    X = synthetic.make_features(n, art["W"], *rows, U_id=art["U_id"], seed=1234)
    torch.set_num_threads(cores)
    mlp_oracle.forward(*sds, X[:1024], threads=cores)
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        mlp_oracle.forward(*sds, X, threads=cores)
        best = min(best, time.perf_counter() - t0)
    return {"value": n / best, "unit": "poses/s", "cores": cores, "kind": "port",
            "sample": f"{n} vectors in one batched call, best of {reps}, torch CPU f32 ({cores} threads), "
                      "oracle.mlp_oracle.forward = restatement of NLML_HPE_Model_Builder.py:115-126"}


ENLARGED = [  # BASELINE.json configs[4]: enlarged synthetic cores (higher rank), full feature count, T = 3000
    {"ranks": (8, 5, 5, 5), "waves": 4, "steps": 2, "cpu_iters": 3000},
    {"ranks": (16, 8, 8, 8), "waves": 1, "steps": 1, "cpu_iters": 100},
]


def tri(r):
    return r * (r + 1) // 2


def enlarged_problem(ranks, seed=11):
    from nlml_hpe_b200 import synthetic
    G = synthetic.synthetic_core(ranks, F, seed=seed, std=1.0)
    rws = [synthetic.synthetic_cos_params(r, 21 + i) for i, r in enumerate(ranks[1:])]
    return G, rws


def cpu_baseline_enlarged(ranks, cores, iters):
    """oracle port of TD_Tester.optimize_with_sgd on the enlarged core, one sample per worker process (1 thread each),
    `iters` iterations timed and scaled to T = 3000 (every iteration costs the same: two einsums over the core)."""
    from concurrent.futures import ProcessPoolExecutor
    from nlml_hpe_b200 import synthetic
    G, rws = enlarged_problem(ranks)
    n = min(cores, 16)
    X = synthetic.make_features(n, G, *rws, U_id=None, seed=1234)
    with ProcessPoolExecutor(max_workers=n, initializer=_pin_worker, initargs=(n,)) as pool:
        list(pool.map(_cpu_warm_worker, range(n)))
        t0 = time.perf_counter()
        list(pool.map(_cpu_tucker_worker_iters, [(G, X[i], rws, iters) for i in range(n)]))
        dt = time.perf_counter() - t0
    per_pose = dt * T_ITERS / iters
    return {"value": n / per_pose, "unit": "poses/s", "cores": n, "kind": "port",
            "s_per_sample_per_core": per_pose,
            "sample": f"{n} samples (one per pinned worker process, 1 thread each), {iters} of T={T_ITERS} iterations timed "
                      f"({dt:.1f} s) and scaled; oracle.tucker_oracle.sgd_reference_form on the ranks {ranks} core"}


def _cpu_tucker_worker_iters(args):
    import torch
    torch.set_num_threads(1)
    from oracle import tucker_oracle
    W, x, rows, iters = args
    return tucker_oracle.sgd_reference_form(W, x, *rows, lr=LR, iters=iters, clip=CLIP)


_PIN_COUNTER = None


def _pin_worker(n_workers):
    """ProcessPoolExecutor initializer: pin each worker to its own CPU (one worker per core, no migration), so the two
    CPU legs of a run agree (VERDICT r1: 1.70 vs 3.72 poses/s for the same leg minutes apart, unpinned)."""
    try:
        import multiprocessing as mp
        firsts = []
        seen = set()
        for cpu in sorted(os.sched_getaffinity(0)):
            try:
                with open(f"/sys/devices/system/cpu/cpu{cpu}/topology/thread_siblings_list") as f:
                    sib = f.read().strip()
            except Exception:
                sib = str(cpu)
            if sib not in seen:
                seen.add(sib)
                firsts.append(cpu)            # first hardware thread of every physical core
        ident = mp.current_process()._identity
        k = (ident[0] - 1) if ident else 0
        os.sched_setaffinity(0, {firsts[k % len(firsts)]})
    except Exception:
        pass


def bench_enlarged(spec, fitter_cls, torch, dist, world, rank, dev, num_sms, tf32_peak, peaks, with_cpu, outputs=None):
    """One enlarged-core record: device-resident value, host-buffer e2e, tensor roofline (useful and issued), CPU port.
    With `outputs` (a dict), the device-resident fit's last result goes there too."""
    from nlml_hpe_b200 import synthetic
    ranks = spec["ranks"]
    G, rws = enlarged_problem(ranks)
    n = spec["waves"] * num_sms * 128
    t0 = time.perf_counter()
    fit = fitter_cls(G, *rws, device=dev)
    torch.cuda.synchronize()
    plan_s = time.perf_counter() - t0
    X = synthetic.make_features_torch(n, G, *rws, U_id=None, seed=77 + rank, device=dev, chunk=8192)
    Xh = torch.empty((n, F), dtype=torch.float32, pin_memory=True)
    Xh.copy_(X)
    np_ = 3 + ranks[0]
    P = torch.empty((n, np_), dtype=torch.float32, device=dev)
    Ph = np.empty((n, np_), dtype=np.float32)
    fit.fit(X, 3, LR, CLIP, out=P)                       # warm-up: first launch, q workspace
    fit.fit_host(Xh.numpy()[: 2 * 128], 3, LR, CLIP)
    l0 = fit.launches
    ms, _ = time_steps(lambda: fit.fit(X, T_ITERS, LR, CLIP, out=P), spec["steps"], 0, torch, dist, world)
    launches = fit.launches - l0
    ms /= spec["steps"]
    if outputs is not None:
        outputs["enlarged_" + "x".join(map(str, ranks)) + "_fit"] = P.cpu().numpy()
    ms_e = time_host_steps(lambda: fit.fit_host(Xh.numpy(), T_ITERS, LR, CLIP, out=Ph), 1, 1, torch, dist, world)   # one warm-up: staging buffers
    fit.close()
    del X, Xh, P
    torch.cuda.empty_cache()
    ri, ry, rp, rr = ranks
    nA, nBCD, R = tri(ri), tri(ry) * tri(rp) * tri(rr), ri * ry * rp * rr
    useful = T_ITERS * 2 * (2 * nA * nBCD)                       # the two contractions with the folded Gram tensor, per pose
    # issued: padded columns x (KA + NA16) x 3 passes (the kernel's configuration is re-derived as in choose_gen_config)
    rrmax = 5 if rr <= 5 else 8
    ndp = (tri(rrmax) + 7) // 8 * 8
    KA = NA16 = (nA + 15) // 16 * 16
    issued_lo = T_ITERS * 2 * 3 * (tri(ry) * tri(rp) * ndp) * (KA + NA16)
    peak16 = peaks["bf16_tflops_sustained"]
    per_gpu = n / (ms * 1e-3)
    rec = {
        "ranks": list(ranks), "R": R, "F": F, "T": T_ITERS,
        "metric": "poses/sec (Tucker-fit, enlarged core, run-time-rank tensor-core kernel)",
        "value": n * world / (ms * 1e-3), "unit": "poses/s", "ms_per_step": ms, "steps": spec["steps"], "dtype": "f32",
        "config": {"workload": f"BASELINE.json configs[4]: synthetic core ranks {ranks} (W {R}x{F} f32 = {R * F * 4 / 1e6:.1f} MB, folded Gram tensor "
                               f"{nA}x{nBCD} = {nA * nBCD * 4 / 1e6:.1f} MB), {n} synthetic feature vectors per GPU, T={T_ITERS}",
                   "samples_per_gpu": n, "plan_create_s": plan_s},
        "e2e": {"value": n * world / (ms_e * 1e-3), "unit": "poses/s", "h2d_bytes_per_step": n * F * 4, "d2h_bytes_per_step": n * np_ * 4,
                "steps": 1, "api": "nlml_tucker_fit_host_f32 (pinned host X -> host P)"},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "unit": "TFLOP/s", "peak": peak16,
                     "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']}): kind::f16 MMAs (FP16 hi/lo operand split, FP32 accumulate)",
                     "achieved": per_gpu * useful / 1e12, "frac": per_gpu * useful / 1e12 / peak16,
                     "issued_frac": per_gpu * issued_lo / 1e12 / peak16, "mma_passes": 3, "traffic": None,
                     "kernel": "tucker_fit_gen_kernel",
                     "note": f"useful = T x 2 x (2 x {nA} x {nBCD}) flop per pose (both contractions with the folded Gram tensor); "
                             "issued counts the three hi/lo passes and the padding of the pair / roll-pair axes"},
        "roofline_hbm": {"bound": "hbm", "unit": "GB/s", "peak": peaks["hbm_gbs"], "achieved": per_gpu * (F * 4 + np_ * 4) / 1e9,
                         "frac": per_gpu * (F * 4 + np_ * 4) / 1e9 / peaks["hbm_gbs"]},
    }
    if with_cpu:
        rec["cpu_baseline"] = cpu_baseline_enlarged(ranks, os.cpu_count() or 1, spec["cpu_iters"])
    return rec


def bind_to_gpu_numa(local_rank):
    """Pin this rank's host threads to the CPUs nvidia-smi reports as local to its GPU (`nvidia-smi topo -m`, CPU Affinity
    column) BEFORE any pinned host buffer is allocated, so staging memory is first-touched on the GPU's NUMA node."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        header = None
        for line in out.splitlines():
            cols = [c.strip() for c in line.split("\t") if c.strip()]
            if not cols:
                continue
            if header is None and any("CPU Affinity" in c for c in cols):
                header = cols
                continue
            if header is not None and cols[0] == f"GPU{local_rank}":
                idx = [i for i, c in enumerate(header) if "CPU Affinity" in c][0] + 1   # data rows start with the row label
                spec = cols[idx]
                cpus = set()
                for part in spec.split(","):
                    lo, _, hi = part.partition("-")
                    cpus.update(range(int(lo), int(hi or lo) + 1))
                cpus &= set(os.sched_getaffinity(0))
                if cpus:
                    os.sched_setaffinity(0, cpus)
                    return {"cpus": spec, "bound": True}
        return {"bound": False, "why": "no CPU Affinity entry for this GPU"}
    except Exception as e:   # noqa: BLE001
        return {"bound": False, "why": str(e)[:80]}


def h2d_probe(torch, dist, world, dev, seconds=0.6, chunk_bytes=850_000_000):
    """Concurrent host->device bandwidth of the box: every rank streams a pinned buffer to its GPU with plain
    cudaMemcpyAsync (one copy per chunk, as the host-buffer entry points do) at the same time; per-rank GB/s by CUDA
    events, aggregate = sum over ranks.  The ceiling the PCIe-bound end-to-end paths can reach at this GPU count."""
    n = chunk_bytes // 4
    host = torch.empty(n, dtype=torch.float32, pin_memory=True)
    host.fill_(1.0)
    devb = torch.empty(n, dtype=torch.float32, device=dev)
    devb.copy_(host, non_blocking=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 0
    t0 = time.perf_counter()
    e0.record()
    while time.perf_counter() - t0 < seconds:
        devb.copy_(host, non_blocking=True)
        reps += 1
    e1.record()
    torch.cuda.synchronize()
    gbs = reps * n * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    t = torch.tensor([gbs], device=dev, dtype=torch.float64)
    lo = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    del host, devb
    return {"aggregate_gbs": t.item(), "min_rank_gbs": lo.item(), "ranks": world, "chunk_bytes": n * 4,
            "how": "pinned -> device cudaMemcpyAsync, all ranks at once, CUDA events"}


def strong_record(fn_device, make_slice, n_total, width, torch, dist, world, rank, dev, steps, warmup):
    """One batch of n_total rows cut by sample index across the ranks (sharding.shard_bounds), run through
    sharding.run_sharded and gathered with sharding.gather_rows (one NCCL all_gather of the ragged shards at the end):
    barrier + synchronize on both sides, CUDA events, max over ranks.  Returns (rows per second, ms per step)."""
    from nlml_hpe_b200 import sharding
    lo, hi = sharding.shard_bounds(n_total, world, rank)
    Xs = make_slice(lo, hi)
    out = {}

    def step():
        out["y"] = sharding.run_sharded(fn_device, lambda a, b: Xs, n_total)
    ms, _ = time_steps(step, steps, warmup, torch, dist, world)
    y = out["y"]
    assert y.shape[0] == n_total and y.shape[1] == width
    ok = bool(torch.isfinite(y).all().item())
    del Xs
    return n_total / (ms / steps * 1e-3), ms / steps, ok


def run_b200(args):
    import torch
    import torch.distributed as dist
    from nlml_hpe_b200 import NLML_HPE_Model_Builder as MB
    from nlml_hpe_b200 import _lib, synthetic
    from nlml_hpe_b200.tucker import TuckerFitter

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: nlml_hpe_b200 has no CPU fallback")
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa(local) if not args.no_numa_bind else {"bound": False, "why": "--no-numa-bind"}
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    art, rows = load_artifacts()
    peaks = measured_peaks()
    n = args.samples
    steps, warmup = args.steps, args.warmup

    # ---- inputs: resident in HBM (value) and in pinned host memory (e2e) ----
    X = synthetic.make_features_torch(n, art["W"], *rows, U_id=art["U_id"], seed=1234 + rank, device=dev)
    X_host = torch.empty((n, F), dtype=torch.float32, pin_memory=True)
    X_host.copy_(X)
    torch.cuda.synchronize()

    fitter = TuckerFitter(art["W"], *rows, device=dev)
    model = MB.build_combined_model(*state_dicts(art))
    P = torch.empty((n, 8), dtype=torch.float32, device=dev)
    P_host = np.empty((n, 8), dtype=np.float32)
    Y_host = np.empty((n, 3), dtype=np.float32)

    import ctypes
    fp32_peak, fp32_peak_3reg = ctypes.c_double(), ctypes.c_double()
    _lib.check(lib.nlml_measure_fp32_tflops(local, ctypes.byref(fp32_peak)))
    _lib.check(lib.nlml_measure_fp32_tflops_3reg(local, ctypes.byref(fp32_peak_3reg)))
    fp32_peak, fp32_peak_3reg = fp32_peak.value, fp32_peak_3reg.value
    tf32_peak = ctypes.c_double()
    _lib.check(lib.nlml_measure_tf32_tflops(local, ctypes.byref(tf32_peak)))
    tf32_peak = tf32_peak.value
    num_sms = torch.cuda.get_device_properties(dev).multi_processor_count

    # --dump-outputs: what each timed device-resident call returned in its last step, copied to the host after timing
    outputs = {} if args.dump_outputs else None
    last = {}

    def keep(name, fn):
        def step():
            last[name] = fn()
        return step

    result = {}
    with ClockSampler(local) as clocks:
        # Tucker fit, device-resident
        l0 = fitter.launches
        ms, wall = time_steps(lambda: fitter.fit(X, T_ITERS, LR, CLIP, out=P), steps, warmup, torch, dist, world)
        t_launches = (fitter.launches - l0) * steps // (steps + warmup)
        tucker_ms = ms / steps
        if outputs is not None:
            outputs["tucker_fit"] = P.cpu().numpy()
        # Tucker fit, host buffers through the C ABI (H2D + fit + D2H inside the timed region)
        e2e_steps = max(1, min(steps, args.e2e_steps))
        ms_e2e = time_host_steps(lambda: fitter.fit_host(X_host, T_ITERS, LR, CLIP, out=P_host), e2e_steps, 1, torch, dist, world)
        tucker_e2e_ms = ms_e2e / e2e_steps
        # converged fit (SURVEY.md section 8f row 1): what TD_Tester.Test computes with scipy Powell
        l0 = fitter.launches
        ms_s, _ = time_steps(lambda: fitter.solve(X, out=P), steps, warmup, torch, dist, world)
        s_launches = (fitter.launches - l0) * steps // (steps + warmup)
        solve_ms = ms_s / steps
        if outputs is not None:
            outputs["tucker_solve"] = P.cpu().numpy()
        ms_se = time_host_steps(lambda: fitter.solve_host(X_host.numpy(), out=P_host), e2e_steps, 1, torch, dist, world)
        solve_e2e_ms = ms_se / e2e_steps
        _, ev = fitter.solve(X[:65536], return_evals=True)
        solve_evals = float(ev.float().mean().item())
    clk = clocks.summary()

    with ClockSampler(local) as clocks2:
        l0 = model.launches
        model.predict(X[:1024])
        ms_m, _ = time_steps(keep("mlp", lambda: model.predict(X)), steps, warmup, torch, dist, world)
        m_launches = (model.launches - l0) * steps // (steps + warmup)
        mlp_ms = ms_m / steps
        # the same forward fed RAW landmarks, IPD normalisation fused into the load stage (SURVEY.md section 8f row 3)
        ms_lm, _ = time_steps(keep("mlp_landmarks", lambda: model.predict_landmarks(X)), steps, warmup, torch, dist, world)
        if outputs is not None:
            outputs.update((k, v.cpu().numpy()) for k, v in last.items())
        last.clear()
        ms_me = time_host_steps(lambda: model.predict_host(X_host.numpy()), e2e_steps, 1, torch, dist, world)
        mlp_e2e_ms = ms_me / e2e_steps
    clk2 = clocks2.summary()

    # the same end-to-end calls fed PAGEABLE host memory (what the reference hands over: plain numpy arrays)
    n_pg = min(n, 262144)
    X_page = np.array(X_host.numpy()[:n_pg], copy=True)
    ms_pg_t = time_host_steps(lambda: fitter.fit_host(X_page, T_ITERS, LR, CLIP, out=P_host[:n_pg]), 1, 1, torch, dist, world)
    ms_pg_m = time_host_steps(lambda: model.predict_host(X_page), 2, 1, torch, dist, world) / 2
    del X_page

    # concurrent host->device bandwidth at this GPU count (the ceiling of the PCIe-bound end-to-end paths)
    probe = h2d_probe(torch, dist, world, dev)

    # strong scaling: ONE n-row batch cut by sample index across the ranks, gathered at the end (NCCL all_gather)
    strong = {}
    if not args.no_strong:
        def make_slice(lo, hi):
            return synthetic.make_features_torch(hi - lo, art["W"], *rows, U_id=art["U_id"], seed=4242 + rank, device=dev)
        st_steps = max(1, min(steps, 3))
        v, ms_s, ok = strong_record(lambda x: fitter.fit(x, T_ITERS, LR, CLIP), make_slice, n, 8, torch, dist, world, rank, dev, st_steps, 1)
        strong["tucker"] = {"value": v, "unit": "poses/s", "ms_per_step": ms_s, "rows_total": n, "finite": ok}
        v, ms_s, ok = strong_record(lambda x: model.predict(x), make_slice, n, 3, torch, dist, world, rank, dev, st_steps, 1)
        strong["mlp"] = {"value": v, "unit": "poses/s", "ms_per_step": ms_s, "rows_total": n, "finite": ok}
        v, ms_s, ok = strong_record(lambda x: fitter.solve(x), make_slice, n, 8, torch, dist, world, rank, dev, st_steps, 1)
        strong["converged"] = {"value": v, "unit": "poses/s", "ms_per_step": ms_s, "rows_total": n, "finite": ok}
        strong["scaling"] = "strong"
        strong["how"] = (f"one batch of {n} rows cut with sharding.shard_bounds over {world} rank(s), each rank runs its slice "
                         "(device-resident), sharding.gather_rows all-gathers the ragged [rows, k] results over NCCL; "
                         "barrier + synchronize on both sides, CUDA events, max over ranks; efficiency = value(N) / (N x value(1))")

    enlarged = []
    if not args.no_enlarged:
        del model
        torch.cuda.empty_cache()
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)
        for spec in ENLARGED:
            enlarged.append(bench_enlarged(spec, TuckerFitter, torch, dist, world, rank, dev, num_sms, tf32_peak, peaks,
                                           with_cpu=(world == 1 and rank == 0 and not args.no_cpu_baseline), outputs=outputs))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    total = n * world
    tucker_pps = total / (tucker_ms * 1e-3)
    mlp_pps = total / (mlp_ms * 1e-3)
    per_gpu_t = n / (tucker_ms * 1e-3)
    per_gpu_m = n / (mlp_ms * 1e-3)
    cores = os.cpu_count() or 1
    line = {
        "metric": "poses/sec (Tucker-fit, fixed T=3000 iterations; Encoder+MLP heads under 'mlp')",
        "value": tucker_pps, "unit": "poses/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": tucker_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"TD_Inference batched Tucker-fit (BASELINE.json configs[3]): {n} synthetic on-manifold+noise "
                               f"feature vectors per GPU, shipped W ranks {RANKS}, F={F}, T={T_ITERS}, lr={LR}, clip={CLIP}",
                   "samples_per_gpu": n, "sharding": f"sample-index, {world} rank(s), no collective on the compute path",
                   "l2": f"inputs {n * F * 4 / 1e9:.2f} GB per GPU, larger than the 126 MB L2 (no flush needed)"},
        "e2e": {"value": total / (tucker_e2e_ms * 1e-3), "unit": "poses/s", "h2d_bytes_per_step": n * F * 4,
                "d2h_bytes_per_step": n * 8 * 4, "steps": e2e_steps,
                "api": "nlml_tucker_fit_host_f32 (TuckerFitter.fit_host), pinned host X -> host P"},
        "gpu_launches": int(t_launches),
        "roofline": {"bound": "tensor", "achieved": per_gpu_t * TUCKER_TC_USEFUL_FLOP_PER_POSE / 1e12,
                     "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": per_gpu_t * TUCKER_TC_USEFUL_FLOP_PER_POSE / 1e12 / peaks["bf16_tflops_sustained"],
                     "issued_frac": per_gpu_t * TUCKER_TC_FLOP_PER_POSE / 1e12 / peaks["bf16_tflops_sustained"], "mma_passes": 3,
                     "traffic": TUCKER_TC_NCU_DRAM_BYTES_PER_POSE * n,
                     "traffic_note": "bytes per launch = ncu dram__bytes_read+write of tucker_project_tc_kernel + tucker_fit_tc_kernel on a "
                                     f"37 888-sample batch ({TUCKER_TC_NCU_SOURCE}), {TUCKER_TC_NCU_DRAM_BYTES_PER_POSE:.0f} B/sample against "
                                     f"{TUCKER_BYTES_PER_POSE} algorithmic (q = 136 floats per sample crosses HBM between the two kernels), x samples per launch",
                     "kernel": "tucker_fit_tc_kernel (+ tucker_project_tc_kernel for phase A)",
                     "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']}): the iteration's MMAs are kind::f16 "
                                    "(FP16 hi/lo operand split, FP32 accumulate), same tensor rate as bf16",
                     "note": f"frac = USEFUL flops ({TUCKER_TC_USEFUL_FLOP_PER_POSE / 1e6:.1f} MFLOP/pose: T x 2 x (2 x 15 x 216), the two contractions "
                             "with the folded Gram tensor, + the projection q = W2 x) / sustained dense 16-bit tensor peak -- the same convention as "
                             "mlp.roofline.frac; issued_frac counts the three hi/lo passes and the operand padding (per iteration 128x224x16 and "
                             f"128x96x48 per 128 samples, 3 MMAs per MAC = {TUCKER_TC_FLOP_PER_POSE / 1e6:.1f} MFLOP/pose). The tensor pipe is NOT "
                             "the binding unit of this kernel (ncu: tensor pipe ~31 % active): each iteration is a serial chain "
                             "features -> operand rows -> GEMMs -> tcgen05.ld -> gradient -> step on two warps per SM sub-partition, and the "
                             "kernel is bound by that chain's latency plus the FP32 work left on the CUDA cores (roofline_fp32; DESIGN.md 3a)."},
        "roofline_fp32": {"bound": "fp32_fma", "achieved": per_gpu_t * TUCKER_FLOP_PER_POSE / 1e12, "peak": fp32_peak,
                          "unit": "TFLOP/s", "frac": per_gpu_t * TUCKER_FLOP_PER_POSE / 1e12 / fp32_peak,
                          "peak_3reg": fp32_peak_3reg, "frac_3reg": per_gpu_t * TUCKER_FLOP_PER_POSE / 1e12 / fp32_peak_3reg,
                          "note": "folded-Gram algorithmic flops (46.6 MFLOP/pose; Gram form "
                                  f"{TUCKER_FLOP_PER_POSE_GRAM / 1e6:.1f}, reference einsum form {TUCKER_FLOP_PER_POSE_REFERENCE / 1e6:.0f}) "
                                  "against the FFMA rates measured live (immediate-operand form / three-register form). The FP32-only "
                                  "kernel (kernel_hint 1) reaches frac_3reg 0.87; values above 1 here mean the tensor cores took the "
                                  "two big contractions off the FP32 pipe."},
        "roofline_hbm": {"bound": "hbm", "achieved": per_gpu_t * TUCKER_BYTES_PER_POSE / 1e9, "peak": peaks["hbm_gbs"],
                         "unit": "GB/s", "frac": per_gpu_t * TUCKER_BYTES_PER_POSE / 1e9 / peaks["hbm_gbs"],
                         "traffic": TUCKER_TC_NCU_DRAM_BYTES_PER_POSE * n,
                         "peak_source": peaks["source"]},
        "clocks": {"sm_mhz": clk["sm_mhz"], "sm_max_mhz": clk["sm_max_mhz"], "reasons": clk["reasons"]},
        "converged": {
            "metric": "poses/sec (Tucker-fit to convergence: damped Newton from p=0, the optimum TD_Tester.Test searches with scipy Powell)",
            "value": total / (solve_ms * 1e-3), "unit": "poses/s", "ms_per_step": solve_ms, "dtype": "f32",
            "e2e": {"value": total / (solve_e2e_ms * 1e-3), "unit": "poses/s", "h2d_bytes_per_step": n * F * 4,
                    "d2h_bytes_per_step": n * 8 * 4, "steps": e2e_steps, "api": "nlml_tucker_solve_host_f32"},
            "gpu_launches": int(s_launches), "mean_evaluations_per_pose": solve_evals,
            "roofline_fp32": {"bound": "fp32_fma", "unit": "TFLOP/s", "peak_3reg": fp32_peak_3reg,
                              "achieved": n / (solve_ms * 1e-3) * (2 * 135 * F + solve_evals * SOLVE_FLOP_PER_EVAL) / 1e12,
                              "frac_3reg": n / (solve_ms * 1e-3) * (2 * 135 * F + solve_evals * SOLVE_FLOP_PER_EVAL) / 1e12 / fp32_peak_3reg,
                              "note": f"2*R*F projection + mean evaluations x {SOLVE_FLOP_PER_EVAL} flop (value+gradient+Hessian from one "
                                      "pass over the folded Gram tensor); warps run until their slowest sample converges"},
            "roofline_hbm": {"bound": "hbm", "achieved": n / (solve_ms * 1e-3) * TUCKER_BYTES_PER_POSE / 1e9, "peak": peaks["hbm_gbs"],
                             "unit": "GB/s", "frac": n / (solve_ms * 1e-3) * TUCKER_BYTES_PER_POSE / 1e9 / peaks["hbm_gbs"]},
        },
        "mlp": {
            "metric": "poses/sec (Encoder + yaw/pitch/roll MLP heads forward)", "value": mlp_pps, "unit": "poses/s",
            "ms_per_step": mlp_ms, "dtype": "f32",
            "config": {"workload": f"BASELINE.json configs[2]: {n} synthetic feature vectors per GPU, shipped heads + synthetic encoder"},
            "e2e": {"value": total / (mlp_e2e_ms * 1e-3), "unit": "poses/s", "h2d_bytes_per_step": n * F * 4,
                    "d2h_bytes_per_step": n * 3 * 4, "steps": e2e_steps, "api": "nlml_mlp_forward_host_f32"},
            "gpu_launches": int(m_launches),
            "from_raw_landmarks": {"value": total / (ms_lm / steps * 1e-3), "unit": "poses/s", "ms_per_step": ms_lm / steps,
                                   "note": "nlml_mlp_forward_landmarks_f32: float64 IPD normalisation fused into the operand split"},
            "roofline": {"bound": "tensor", "achieved": per_gpu_m * MLP_FLOP_PER_POSE / 1e12, "peak": peaks["bf16_tflops_sustained"],
                         "unit": "TFLOP/s", "frac": per_gpu_m * MLP_FLOP_PER_POSE / 1e12 / peaks["bf16_tflops_sustained"],
                         "traffic": MLP_NCU_DRAM_BYTES_PER_POSE * n, "peak_source": peaks["source"], "mma_passes": 3,
                         "traffic_note": "bytes per 1M-sample forward = ncu dram__bytes_read+write summed over the nine launches of one 151 552-sample "
                                         f"chunk (profiles/r02_mlp_launches.txt): {MLP_NCU_DRAM_BYTES_PER_POSE:.0f} B/sample against {MLP_BYTES_PER_POSE} "
                                         "algorithmic -- the FP16 hi/lo activation planes of every layer round-trip HBM (see DESIGN.md section 4)",
                         "issued_frac": 3 * per_gpu_m * MLP_FLOP_PER_POSE / 1e12 / peaks["bf16_tflops_sustained"],
                         "note": "algorithmic 4.714 MFLOP/pose against the sustained bf16 tensor peak; every MAC is three "
                                 "FP16 MMAs (hi/lo operand split needed for the 1e-3 deg budget), issued_frac counts them"},
            "roofline_hbm": {"bound": "hbm", "achieved": per_gpu_m * MLP_BYTES_PER_POSE / 1e9, "peak": peaks["hbm_gbs"],
                             "unit": "GB/s", "frac": per_gpu_m * MLP_BYTES_PER_POSE / 1e9 / peaks["hbm_gbs"]},
            "clocks": {"sm_mhz": clk2["sm_mhz"], "sm_max_mhz": clk2["sm_max_mhz"], "reasons": clk2["reasons"]},
        },
        "enlarged": enlarged,
        "strong": strong,
        "h2d_probe": probe,
        "numa": numa,
        "e2e_pageable": {"tucker": {"value": n_pg * world / (ms_pg_t * 1e-3), "unit": "poses/s", "rows": n_pg},
                         "mlp": {"value": n_pg * world / (ms_pg_m * 1e-3), "unit": "poses/s", "rows": n_pg},
                         "note": "same host-buffer C-ABI calls fed pageable numpy arrays (the reference's callers hand over "
                                 "plain numpy / torch CPU tensors); the driver stages pageable copies through its own pinned buffers"},
        "fp32_fma_peak_tflops_measured": fp32_peak, "fp32_fma_3reg_peak_tflops_measured": fp32_peak_3reg,
        "tf32_tensor_peak_tflops_measured": tf32_peak,
    }
    if world == 1 and not args.no_cpu_baseline:
        os.sched_setaffinity(0, all_cpus)   # the CPU legs use every host core again
        line["cpu_baseline"] = cpu_baseline_tucker(art, rows, cores)
        line["converged"]["cpu_baseline"] = cpu_baseline_powell(art, rows, cores)
        line["mlp"]["cpu_baseline"] = cpu_baseline_mlp(art, cores)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------
# reference arm: the CPU port of the reference's own path, all host threads
# ---------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    art, rows = load_artifacts()
    cores = os.cpu_count() or 1
    for _ in range(min(args.warmup, 1)):
        cpu_baseline_tucker(art, rows, cores)
    vals, t0 = [], time.perf_counter()
    for _ in range(args.steps):
        vals.append(cpu_baseline_tucker(art, rows, cores))
        if time.perf_counter() - t0 > 150:
            break
    dt = time.perf_counter() - t0
    # samples fitted (one per pinned physical core per step) / time inside the fits (worker start-up and imports excluded,
    # exactly as in the b200 arm's cpu_baseline leg, so the two CPU figures of a run agree)
    value = sum(v["cores"] for v in vals) / sum(v["seconds"] for v in vals)
    base = dict(vals[-1], value=value)
    mlp = cpu_baseline_mlp(art, cores)
    line = {
        "impl": "reference",
        "metric": "poses/sec (Tucker-fit, fixed T=3000 iterations; Encoder+MLP heads under 'mlp')",
        "value": value, "unit": "poses/s", "n_gpus": args.gpus, "steps": len(vals), "warmup": min(args.warmup, 1),
        "ms_per_step": sum(v["seconds"] for v in vals) / len(vals) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"TD_Inference Tucker-fit, CPU port of the reference (TD_Tester.optimize_with_sgd), shipped W ranks {RANKS}, "
                               f"F={F}, T={T_ITERS}; each step = {vals[-1]['cores']} samples, one per physical host core (pinned)"},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "mlp": {"value": mlp["value"], "unit": "poses/s", "cpu_baseline": mlp,
                "e2e": {"value": mlp["value"], "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
    }
    print(json.dumps(line), flush=True)


def _count(least):
    def parse(s):
        v = int(s)
        if v < least:
            raise argparse.ArgumentTypeError(f"{v} < {least}")
        return v
    return parse


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_count(1), default=5,
                    help="timed steps of the device-resident Tucker fit (headline), converged fit and Encoder+heads forwards")
    ap.add_argument("--warmup", type=_count(0), default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples", type=int, default=1_000_000, help="feature vectors per GPU per step")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-enlarged", action="store_true", help="skip the enlarged-core records (BASELINE.json configs[4])")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling records")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the rank to its GPU's NUMA-local CPUs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after timing, write what the device-resident Tucker fit, converged fit, Encoder+heads forward (on "
                         "features and on raw landmarks) and enlarged-core fits returned in their last step as DIR/<name>.npy "
                         f"(float32; a fixed seeded sample of {DUMP_ROWS} rows of longer outputs)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
