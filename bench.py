#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 HOP horizon-selection path.

Metric (BASELINE.json): horizon-selection solves/sec, batched HOP-LQR, quadrotor n=12, N=128.
Workload "S1" (SURVEY.md s.8d): `batch` quadrotor instances per GPU, x0_b = x0 + sigma*xi_b,
U = tile(u_ref), T in [40, 128].  One *solve* = augmented embedding + LFT stage/prefix/query sweep +
argmin for one instance (reference: augmented.py:10-87 + horizon_selection.py:36-86 + solver.py:522).

  value : fused selection kernel on HBM-resident (A, B, X, U), CUDA-event timed, max over ranks.
  e2e   : the public host-buffer call (hop.api.select_horizon_host): pinned-host x0 -> device,
          rollout + FD linearisation + fused selection on device, T*/J*/status/J(T) back to host.
  --impl reference : the same x0 -> T* pipeline on the host cores through the REFERENCE ITSELF (the unmodified Python
          modules staged in oracle/_ref by __graft_entry__.build(), one process per core); the plain-C port
          (oracle/hop_oracle.c, all host threads) is timed beside it and is the fallback when oracle/_ref is absent
          (`--ref-kind port` forces it).

Launch: `python bench.py --gpus 1 --steps K --warmup W`, or under torchrun for N > 1 (one rank per
GPU; the batch is sharded, no collective on the solve path, a final all_gather of T*/J*).
`--dump-outputs DIR` writes what the last timed kernel step returned (rank 0's shard) as float64 .npy files, so that two
builds can be compared output for output: the inputs depend only on --batch and the rank.
The benchmark writes nothing into the source tree (which may be read-only): the libraries are built by
__graft_entry__.build() beforehand.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True                          # no __pycache__ in the source tree
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "time-opt-ilqr_b200"))
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")

import numpy as np  # noqa: E402

METRIC = "horizon-selection solves/sec (batched HOP-LQR, quadrotor n=12, N=128)"
WORKLOAD = ("S1 quadrotor n=12 m=4 d=13 N=128 T in [40,128]: iteration-0 HOP horizon selection per initial state "
            "(rollout + forward-FD linearisation -> augmented embedding + LFT stage/prefix/query sweep + argmin)")
UNIT = "solves/s"
N_HORIZON, D_AUG, M_CTRL = 128, 13, 4
DUMP_INSTANCES = 1 << 20     # --dump-outputs: per-instance arrays in full up to this batch (8 MiB each)
DUMP_J_ROWS = 16384          # --dump-outputs: rows of the J(T) curves (16 MiB at T_max = 128; all of them are 64 MiB at the default batch)


def f_alg(N, d, m):
    """Algorithmic FLOPs per solve (SURVEY.md s.8d)."""
    return N * (5 * d**3 + 2 * d * m * m + 2 * d * d * m) + (N - 1) * (11 * d**3 + 3 * d * d) + N * (7 * d**3 + 4 * d * d)


def b_alg_fused(N, n, m):
    """Algorithmic HBM bytes per solve of the fused kernel: reads A, B, X, U(shared: not counted), xg, w; writes J, T*, J*, status."""
    return 8 * (N * (n * n + n * m) + (N + 1) * n + n + 1) + 8 * N + 4 + 8 + 4


def s1_x0(B, seed):
    x0 = np.zeros(12); x0[:3] = 2.0
    sigma = np.array([0.4, 0.4, 0.4] + [0.0] * 9)
    return x0[None] + sigma[None] * np.random.default_rng(seed).standard_normal((B, 12))


def dump_outputs(out_dir, res):
    """Write a Selection as float64 DIR/<name>.npy: T_star, J_star, status per instance and J, the curves J(T) of a fixed,
    seeded sample of instances; instances.npy and J_rows.npy hold the batch indices of those rows (at most 48.1 MiB)."""
    os.makedirs(out_dir, exist_ok=True)
    B = res.T_star.shape[0]

    def sample(k):
        return np.arange(B) if B <= k else np.sort(np.random.default_rng(0).choice(B, k, replace=False))

    inst, rows = sample(DUMP_INSTANCES), sample(DUMP_J_ROWS)
    host = {k: getattr(res, k).cpu().numpy() for k in ("J", "T_star", "J_star", "status")}
    arrays = {"T_star": host["T_star"][inst], "J_star": host["J_star"][inst], "status": host["status"][inst],
              "instances": inst, "J": host["J"][rows], "J_rows": rows}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [t.strip() for t in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.2] or [r for (_, r) in self.rows]
        sm, mx, reasons, pw = [], [], set(), []
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_from_x0(case, x0, nthreads):
    import oracle as O
    F, _x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    U = np.tile(u_ref, (N, 1))
    t = time.perf_counter()
    J, T, st = O.select_from_x0_batch(F.hop_sys, F.hop_params, N, T_min, T_max, x0, U, xg, u_ref, Q, R, alpha, w, wrap_idx,
                                      nthreads=nthreads)
    return time.perf_counter() - t, J, T, st


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the x0 -> T* pipeline on all host cores, a bounded
    sample per step.  kind "reference" = the unmodified Python modules from oracle/_ref (one process per core);
    kind "port" = oracle/hop_oracle.c on one pthread per core (timed in both cases, reported beside it)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_py
    from hop import cases
    case = cases.make_case("Quadrotor", N=N_HORIZON)
    cores = os.cpu_count() or 1
    # ---- the C port: calibrate, then ~2 s of CPU work
    dt, *_ = cpu_from_x0(case, s1_x0(4 * cores, 1), cores)
    rate = 4 * cores / dt
    psample = int(max(cores, min(args.batch, round(rate * 2.0 / cores) * cores)))
    dtp, Jp, Tp, _ = cpu_from_x0(case, s1_x0(psample, 0), cores)
    port = {"value": psample / dtp, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{psample} instances, oracle/hop_oracle.c on {cores} pthreads"}
    use_py = ref_py.available() and args.ref_kind != "port"
    if use_py:
        pool = ref_py.Pool(cores)
        sample = 4 * cores                                                  # ~0.45 s per instance and core: ~2 s per step
        x0 = s1_x0(sample, 0)
        step = lambda: pool.s1_select(x0)                                   # noqa: E731
        kind = "reference"
        what = (f"{sample} instances per step through the unmodified reference modules (oracle/_ref: solver.rollout, "
                f"linearization.linearize_forward_diff_traj, augmented.*, horizon_selection.propagator_all_Jt_aug), "
                f"{cores} worker processes, OPENBLAS threads = 1")
    else:
        sample = int(max(cores, min(args.batch, round(rate * 4.0 / cores) * cores)))   # ~4 s of CPU work per step
        x0 = s1_x0(sample, 0)
        step = lambda: cpu_from_x0(case, x0, cores)                         # noqa: E731
        kind = "port"
        what = (f"{sample} instances per step, pthread fan-out of oracle/hop_oracle.c over {cores} host threads "
                "(oracle/_ref not staged: the reference is pure Python and was not copied by build())")
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    el = time.perf_counter() - t0
    val = sample * args.steps / el
    agree = None
    if use_py:
        pool.close()
        agree = bool(np.array_equal(out[0], Tp[:sample])) if sample <= psample else None
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_step": sample, "threads": cores,
                       "timed": "whole x0 -> T* pipeline on the host cores (the e2e definition of the hop arm)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": what,
                             "port": port, "T_star_reference_equals_port_on_sample": agree},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_hop(args):
    import torch
    import torch.distributed as dist

    from hop import _cabi, api, cases

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the HOP B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _cabi.require_device()

    case = cases.make_case("Quadrotor", N=N_HORIZON)
    F, x0c, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    B = args.batch
    n, m = 12, 4
    x0_host = torch.empty((B, n), dtype=torch.float64).pin_memory()
    x0_host.copy_(torch.from_numpy(s1_x0(B, seed=rank)))

    # ---- resident inputs for the kernel-only number: rollout + linearisation done once, on device
    mode = {"fast": api.MODE_FAST, "exact": api.MODE_EXACT, "gj": api.MODE_GJ}[args.mode]
    sel = api.HorizonSelector(case, B, device=dev, mode=mode)
    x0_dev = x0_host.to(dev)
    res = sel(x0_dev)                                   # also warms everything up
    X, A, Bm = sel.views()   # (X, A, Bm) stay resident in the selector's workspace
    xg_dev = torch.from_numpy(np.broadcast_to(xg, (B, n)).copy()).to(dev)
    w_dev = torch.full((B,), float(w), dtype=torch.float64, device=dev)
    T_ref = res.T_star.clone()
    del A, Bm, X
    gath_T = torch.empty(world * B, dtype=torch.int32, device=dev) if world > 1 else None
    gath_J = torch.empty(world * B, dtype=torch.float64, device=dev) if world > 1 else None

    def kernel_step():
        return sel.select_resident(xg_dev, w_dev)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        r = kernel_step()
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    sync_all()
    tw0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        r = kernel_step()
        if world > 1:                                   # final gather of the per-instance results
            dist.all_gather_into_tensor(gath_T, r.T_star)
            dist.all_gather_into_tensor(gath_J, r.J_star)
    e1.record()
    sync_all()
    tw1 = time.perf_counter()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    clocks = sampler.stop(tw0, tw1) if rank == 0 else None
    assert torch.equal(r.T_star, T_ref), "kernel-only and from-x0 selections disagree"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, r)
    value = world * B * args.steps / (ms_total * 1e-3)

    # ---- end-to-end through the public host-buffer API
    T_h = torch.empty(B, dtype=torch.int32).pin_memory().numpy()
    Js_h = torch.empty(B, dtype=torch.float64).pin_memory().numpy()
    st_h = torch.empty(B, dtype=torch.int32).pin_memory().numpy()
    J_h = torch.empty((B, T_max), dtype=torch.float64).pin_memory().numpy()
    x0_np = x0_host.numpy()
    for _ in range(max(args.warmup, 3)):
        api.select_horizon_host(case, x0_np, mode=mode, out=(J_h, T_h, Js_h, st_h))
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        api.select_horizon_host(case, x0_np, mode=mode, out=(J_h, T_h, Js_h, st_h))
    torch.cuda.synchronize(dev)
    el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    e2e_val = world * B * args.steps / float(el.item())
    assert np.array_equal(T_h, T_ref.cpu().numpy()), "host-buffer path disagrees with the device path"
    h2d = 8 * (B * n + B * n + B + N * m + m + 2 * n * n + m * m)
    d2h = B * (8 * T_max + 4 + 8 + 4)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (k_select_fused), against a DFMA peak measured in this run
    tf, pms = C.c_double(0), C.c_double(0)
    _cabi.check(lib.hop_probe_fp64_tflops(4096, C.byref(tf), C.byref(pms)), "hop_probe_fp64_tflops")
    ms_launch = ms_total / args.steps
    flop_launch = f_alg(N_HORIZON, D_AUG, M_CTRL) * B
    byte_launch = b_alg_fused(N_HORIZON, n, m) * B
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    traffic = None                                      # dram bytes per launch of the same kernel from the committed ncu capture
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if tr.get("batch") == B and tr.get("mode") == args.mode:
            traffic = tr["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    ach_tf = flop_launch / (ms_launch * 1e-3) / 1e12
    ach_gb = byte_launch / (ms_launch * 1e-3) / 1e9
    roofline = {"bound": "fp64", "achieved": ach_tf, "peak": tf.value, "unit": "TFLOP/s", "frac": ach_tf / tf.value,
                "traffic": traffic, "kernel": {"fast": "k_select_fused_mma<13,4,pipelined>", "gj": "k_select_fused_mma<13,4,materialised>",
                                                        "exact": "k_select_ref_fused"}[args.mode],
                "peak_source": "DFMA microbenchmark in this run (hop_probe_fp64_tflops); nominal 37.2 TFLOP/s",
                "algorithmic_flop_per_solve": f_alg(N_HORIZON, D_AUG, M_CTRL),
                "hbm": {"achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gb / hbm_peak,
                        "algorithmic_bytes_per_solve": b_alg_fused(N_HORIZON, n, m),
                        "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"}}

    cpu_baseline = None
    if not args.no_cpu_legs:
        # ---- CPU baseline + parity census (outside every timed region)
        #  * the C port on ALL B instances of rank 0 (all host cores): throughput + the three-number census of oracle/census.py
        #    (|gpu-oracle|, |oracle-fp80|, |gpu-fp80|, argmin gaps, ill-posed instances; a T* mismatch must be explained by it)
        #  * HOP_MODE_EXACT on the same batch on the device: the measured mode against the parity mode
        #  * the REAL reference (oracle/_ref, unmodified Python) on the first instances: T* equality and solves/s per core
        #  * the committed reference-generated golden (first 4096 instances of this very batch, tests/golden)
        from oracle import census, ref_py
        cores = os.cpu_count() or 1
        t0c = time.perf_counter()
        rep = census.census_from_x0(case, x0_np, J_h, T_h, nthreads=cores, fp80_stride=8)
        t_census = time.perf_counter() - t0c
        dtc, Jc, Tc, stc = cpu_from_x0(case, x0_np[:min(B, 16384)], cores)          # timed alone (the census also runs fp80 sweeps)
        sample = min(B, 16384)
        ex = api.select_horizon_batched(case, x0_dev, mode=api.MODE_EXACT)
        T_ex = ex.T_star.cpu().numpy().astype(np.int64); J_ex = ex.J.cpu().numpy()
        Tg = T_h.astype(np.int64)
        dmode = np.abs(J_h[:, T_min - 1:] - J_ex[:, T_min - 1:]) / np.abs(J_ex[:, T_min - 1:])
        mm = np.nonzero(T_ex != Tg)[0]
        unexpl = 0
        for i in mm:
            gap = abs(J_ex[i, T_ex[i] - 1] - J_ex[i, Tg[i] - 1]) / abs(J_ex[i, T_ex[i] - 1])
            noise = max(abs(J_h[i, t - 1] - J_ex[i, t - 1]) / abs(J_ex[i, t - 1]) for t in (T_ex[i], Tg[i]))
            unexpl += int(not gap < 10.0 * noise)
        rep_ex = census.census_from_x0(case, x0_np[:sample], J_ex[:sample], T_ex[:sample], nthreads=cores, fp80_stride=8)
        vs_exact = {"checked": int(B), "T_star_mismatches": int(mm.size), "T_star_mismatches_unexplained": unexpl,
                    "rule": "gap between the two candidates (EXACT curve) < 10 x distance between the two curves at those horizons",
                    "max_rel_J_window": float(dmode.max()), "p99_rel_J_window": float(np.percentile(dmode.max(axis=1), 99)),
                    "exact_mode_vs_oracle": {k: rep_ex[k] for k in ("checked", "T_star_mismatches", "T_star_mismatches_unexplained",
                                                                     "rel_J_window", "rel_J_at_Tstar")}}
        golden_chk = None
        try:
            g = np.load(os.path.join(ROOT, "tests", "golden", "s1_quadrotor_ref4096.npz"))
            if rank == 0 and int(g["seed"]) == 0 and B >= g["T"].shape[0]:
                ng = g["T"].shape[0]
                Tr = g["T"].astype(np.int64)
                cols = np.clip(Tr[:, None] + np.arange(-2, 3)[None, :], 1, T_max)
                J5 = J_h[np.arange(ng)[:, None], cols - 1]
                golden_chk = {"instances": int(ng), "T_star_mismatches": int((Tg[:ng] != Tr).sum()),
                              "max_rel_J_at_Tstar_pm2": float(np.nanmax(np.abs(J5 - g["J_pm2"]) / np.abs(g["J_pm2"]))),
                              "what": "first 4096 instances of this batch computed by the REAL reference in the build container "
                                      "(tests/golden/make_golden.py s1_ref4096)"}
        except OSError:
            pass
        ref_leg = {"available": False, "why": "oracle/_ref not staged"}
        if ref_py.available():
            nref = 8 * cores
            pool = ref_py.Pool(cores)
            Tpy, Jpy, dpy = pool.s1_select(x0_np[:nref])
            pool.close()
            ref_leg = {"available": True, "kind": "reference", "instances": int(nref), "value": nref / dpy, "unit": UNIT,
                       "cores": cores, "per_core": nref / dpy / cores,
                       "T_star_equal_gpu": int((Tpy == T_h[:nref]).sum()), "T_star_equal_port": int((Tpy == Tc[:nref]).sum()),
                       "max_rel_J_window_gpu_vs_reference": float(np.max(np.abs(J_h[:nref, T_min - 1:] - Jpy[:, T_min - 1:]) / np.abs(Jpy[:, T_min - 1:]))),
                       "max_rel_J_window_port_vs_reference": float(np.max(np.abs(Jc[:nref, T_min - 1:] - Jpy[:, T_min - 1:]) / np.abs(Jpy[:, T_min - 1:]))),
                       "what": "the unmodified reference modules (oracle/_ref) on the first instances of this batch, one process per core"}
        cpu_baseline = {"value": sample / dtc, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"first {sample} instances of rank 0's batch, x0 -> T* pipeline, oracle/hop_oracle.c on {cores} "
                                  "pthreads",
                        "reference_python": ref_leg,
                        "parity_on_sample": dict(rep, census_seconds=t_census, mode_checked=args.mode),
                        "fast_vs_exact_mode_on_device": vs_exact, "reference_golden": golden_chk}


    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_launch, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "timed": "value: fused selection kernel on HBM-resident linearisation; e2e: whole x0 -> T* pipeline from pinned host buffers",
                       "batch_per_gpu": B, "global_batch": world * B,
                       "mode": args.mode + {"fast": " (sequential in the horizon; software-pipelined pivot sweeps; checked against HOP_MODE_EXACT "
                                                    "and the oracle on every instance: cpu_baseline.parity_on_sample / fast_vs_exact_mode_on_device)",
                                            "gj": " (materialised blocks, Gauss-Jordan inverse)",
                                            "exact": " (reference operation order, bit-identical to the oracle on identical inputs)"}[args.mode],
                       "l2": "inputs (A,B,X = %.1f GB per GPU) exceed the 126 MB L2" % (byte_launch / 1e9),
                       "parallelism": f"batch-sharded x{world}, final all_gather of T*/J*" if world > 1 else "single GPU"},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "api": "hop.api.select_horizon_host -> hop_select_from_x0_host_f64 (pinned host x0; rollout + "
                           "forward-FD linearisation + fused selection on device, in up to four chunks on two streams so that copies overlap kernels; J(T), T*, J*, status back to host)"},
            "gpu_launches": args.steps, "gpu_launches_e2e": 3 * args.steps * min(4, max(1, -(-B // 16384))),   # e2e: rollout + linearise + select per chunk (hop_cabi.cu: kHostChunkMin / kHostChunksMax)
            "roofline": roofline, "cpu_baseline": cpu_baseline}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["hop", "reference"], default="hop")
    ap.add_argument("--batch", type=int, default=65536, help="instances per GPU (weak scaling)")
    ap.add_argument("--mode", choices=["exact", "fast", "gj"], default="fast",
                    help="selection variant (include/hop_b200.h HOP_MODE_*); all compute the same function")
    ap.add_argument("--no-cpu-legs", action="store_true",
                    help="skip the CPU baseline / parity census (they fork worker processes); only for the ncu launch list")
    ap.add_argument("--ref-kind", choices=["auto", "port"], default="auto",
                    help="--impl reference: auto = the Python reference from oracle/_ref when staged, else the C port")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's T*, J*, status and a seeded sample of J(T) rows to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "hop":
        ap.error("--dump-outputs applies to --impl hop (the reference arm's sample size is calibrated per run)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_hop(args)


if __name__ == "__main__":
    main()
