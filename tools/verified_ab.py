#!/usr/bin/env python
"""HOP_MODE_VERIFIED against FAST and EXACT: device time, re-evaluated share and T* agreement, one JSON line per workload.

  python tools/verified_ab.py [--rounds 5] [--out DIR]

Workloads: S1 (65 536 quadrotor selections, N = 128, the benchmark's seeding; selection on resident device inputs), the
HOP-DDP configurations 2-4 of tests/run_configs.py, and a calibration pass of the small systems (DI, Segway, Cartpole through
the three FAST routing branches) and, with --parts lqr, hop_select_verified_f64 at the LQR boundary (S2 as configuration 5
generates it, and the quadrotor embedding materialised at the boundary): FAST's relative distance to EXACT at its two best horizons, and what the near-tie scan
would decide at several tolerances (numpy restatement of include/hop_b200.h, HOP_MODE_VERIFIED step 2).  The modes are timed
alternately (FAST, VERIFIED, EXACT per round) with CUDA events; the card's name and power limit are printed first.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "time-opt-ilqr_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from hop import api, cases  # noqa: E402
from oracle import census  # noqa: E402
from _common import s1_x0  # noqa: E402

DEV = "cuda:0"
MODES = {"fast": api.MODE_FAST, "verified": api.MODE_VERIFIED, "exact": api.MODE_EXACT}


def emit(out, rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(os.path.join(out, "verified_ab.jsonl"), "a") as fh:
            fh.write(line + "\n")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def alternate(fns, rounds):
    """{name: fn} -> {name: [seconds per call]}, the names interleaved within every round (after one warm-up call each)."""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts[k].append(e0.elapsed_time(e1) * 1e-3)
    return ts


def summary(ts, B):
    return {k: {"median_s": float(np.median(v)), "min_s": float(np.min(v)), "max_s": float(np.max(v)),
                "solves_per_s": B / float(np.median(v))} for k, v in ts.items()}


def resident(case, x0s):
    sel = api.HorizonSelector(case, len(x0s), device=DEV, mode=api.MODE_FAST)
    sel(torch.as_tensor(x0s, device=DEV))
    X, A, Bm = sel.views()
    F, _x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    T_max = min(T_max, N)
    return lambda mode: api.select_fused_batched(A, Bm, X, sel.U, xg, w, u_ref, Q, R, alpha, T_min, T_max, wrap_idx, mode=mode)


def scan_decision(J, T, st, T_min, T_max, tol):
    W = J[:, T_min - 1:T_max]
    Ts = np.argmin(W, axis=1) + T_min
    with np.errstate(invalid="ignore", divide="ignore"):
        gap, _ = census.argmin_gap(J, Ts, T_min, T_max)
        return (gap < tol) | ~np.isfinite(W).all(axis=1) | (st != 0) | (Ts != T)


def distances(case, f, e):
    """FAST's relative distance to EXACT at FAST's two best horizons and at EXACT's T*, and FAST's own argmin gap."""
    T_min, T_max = case[9], min(case[10], case[8])
    Jf, Tf, Je, Te = f.J.cpu().numpy(), f.T_star.cpu().numpy().astype(np.int64), e.J.cpu().numpy(), e.T_star.cpu().numpy().astype(np.int64)
    rows = np.arange(len(Tf))
    gap, second = census.argmin_gap(Jf, Tf, T_min, T_max)
    r = lambda t: np.abs(Jf[rows, t - 1] - Je[rows, t - 1]) / np.abs(Je[rows, t - 1])  # noqa: E731
    return Jf, Tf, Te, gap, np.maximum.reduce([r(Tf), r(second), r(Te)]), T_min, T_max


def s1(args):
    case = cases.make_case("Quadrotor", N=128)
    B = 65536
    run = resident(case, s1_x0(B, seed=0))
    ts = alternate({k: (lambda m=m: run(m)) for k, m in MODES.items()}, args.rounds)
    out = {k: run(m) for k, m in MODES.items()}
    torch.cuda.synchronize()
    re = (out["verified"].status.cpu().numpy() & api.ST_FLAG_REEVALUATED) != 0
    Jf, Tf, Te, gap, dist, *_ = distances(case, out["fast"], out["exact"])
    s = summary(ts, B)
    emit(args.out, {"workload": "S1 selection, 65536 quadrotor instances, N=128, resident device inputs", "card": args.card,
                    "timing": s, "verified_over_exact_throughput": s["verified"]["solves_per_s"] / s["exact"]["solves_per_s"],
                    "verified_over_fast_throughput": s["verified"]["solves_per_s"] / s["fast"]["solves_per_s"],
                    "reevaluated": int(re.sum()), "reevaluated_share": float(re.mean()),
                    "T_star_verified_ne_exact": int((out["verified"].T_star != out["exact"].T_star).sum()),
                    "T_star_fast_ne_exact": int((Tf != Te).sum()),
                    "max_rel_fast_vs_exact_at_candidates": float(dist.max()),
                    "min_gap_over_distance_not_reevaluated": float((gap[~re] / np.maximum(dist[~re], 1e-300)).min())})
    # the VERIFIED call split: FAST alone is the first row; the rest is scan + EXACT tail
    emit(args.out, {"workload": "S1 split", "verified_minus_fast_median_s": s["verified"]["median_s"] - s["fast"]["median_s"],
                    "exact_per_instance_tail_s": (s["verified"]["median_s"] - s["fast"]["median_s"]) / max(1, int(re.sum()))})


def small_calibration(args):
    tols = (1e-7, 3e-7, 1e-6, 1e-5, 1e-4)
    for name, sigma in (("DoubleIntegrator", 0.2), ("Segway_Balance", 0.02), ("Cartpole_SwingUp", None)):
        for B in (300, 900, 3000):
            case = cases.make_case(name)
            rng = np.random.default_rng(B)
            if sigma is None:
                x0s = np.array([rng.normal(0, .1, B), rng.normal(0, .1, B), rng.normal(0, .2, B), rng.normal(0, .2, B)]).T
            else:
                x0s = case[1][None] + sigma * rng.standard_normal((B, case[1].size))
            run = resident(case, x0s)
            f, e = run(api.MODE_FAST), run(api.MODE_EXACT)
            Jf, Tf, Te, gap, dist, T_min, T_max = distances(case, f, e)
            st = f.status.cpu().numpy()
            rec = {"workload": f"calibration {name} B={B} N={case[8]}", "T_star_fast_ne_exact": int((Tf != Te).sum()),
                   "max_rel_fast_vs_exact_at_candidates": float(dist.max()),
                   "p99_rel_fast_vs_exact_at_candidates": float(np.percentile(dist, 99)),
                   "max_fast_gap_where_T_differs": float(gap[Tf != Te].max()) if (Tf != Te).any() else None}
            for tol in tols:
                mark = scan_decision(Jf, Tf.astype(np.int32), st, T_min, T_max, tol)
                rec[f"tol_{tol:g}"] = {"share": float(mark.mean()), "T_star_misses": int(((Tf != Te) & ~mark).sum())}
            emit(args.out, rec)


def ddp(args):
    rng = np.random.default_rng(0)
    seg = cases.make_case("Segway_Balance")
    x_seg = seg[1][None] + 0.02 * rng.standard_normal((25, 4)); x_seg[0] = seg[1]
    rng = np.random.default_rng(0)
    x_cp = np.array([rng.normal(0, .1, 4096), rng.normal(0, .1, 4096), rng.normal(0, .2, 4096), rng.normal(0, .2, 4096)]).T
    quad = cases.make_case("Quadrotor", N=128)
    for cfg, case, x0s in ((2, seg, x_seg), (3, cases.make_case("Cartpole_SwingUp"), x_cp), (4, quad, s1_x0(16384, seed=4))):
        xt = torch.as_tensor(x0s, device=DEV)
        modes = dict(MODES)
        n, m = case[1].size, np.asarray(case[3]).size
        if not api._cabi.load().hop_select_supported_mode(n + 1, m, api.MODE_VERIFIED):
            modes.pop("verified")
        run = lambda mode: api.ilqr_timeopt_batched(case, xt, max_iter=12, use_central_diff=False, mode=mode)  # noqa: E731
        ts = alternate({k: (lambda m=m: run(m)) for k, m in modes.items()}, max(2, args.rounds // 2))
        rec = {"workload": f"config {cfg}: HOP-DDP, {len(x0s)} instances, max-iter 12", "timing": summary(ts, len(x0s))}
        if "verified" in modes:
            v, e = run(api.MODE_VERIFIED), run(api.MODE_EXACT)
            rec["identical_to_exact"] = all(np.array_equal(v[k].cpu().numpy(), e[k].cpu().numpy(), equal_nan=True)
                                            for k in ("X", "U", "J_hist", "T_hist", "n_hist", "T_star"))
            rec["instances_with_a_reevaluated_selection"] = int(((v["status"].cpu().numpy() & api.ST_FLAG_REEVALUATED) != 0).sum())
        else:
            rec["verified"] = "refused for this state dimension (include/hop_b200.h)"
        emit(args.out, rec)


LQR_TOLS = (1e-13, 1e-12, 1e-10, 1e-8, 1e-7)


def s2_config5(B, d, m, N, seed=1234):
    """S2 exactly as tests/run_configs.py configuration 5 generates a tile on the device (its first tile: seed 1234)."""
    gen = torch.Generator(device=DEV); gen.manual_seed(seed)
    A = torch.eye(d, dtype=torch.float64, device=DEV).expand(B, N, d, d) + \
        0.05 / np.sqrt(d) * torch.randn((B, N, d, d), dtype=torch.float64, device=DEV, generator=gen)
    Bm = 0.05 * torch.randn((B, N, d, m), dtype=torch.float64, device=DEV, generator=gen)
    Q = torch.diag_embed(0.5 + 1.5 * torch.rand((B, N, d), dtype=torch.float64, device=DEV, generator=gen))
    QT = (50.0 * torch.eye(d, dtype=torch.float64, device=DEV)).expand(B, N, d, d).contiguous()
    Rd = 0.05 + 0.45 * torch.rand((B, m), dtype=torch.float64, device=DEV, generator=gen)
    Rinv = torch.diag_embed(1.0 / (Rd + 1e-9))
    z0 = torch.randn((B, d), dtype=torch.float64, device=DEV, generator=gen)
    w = 0.01 + 0.09 * torch.rand((B,), dtype=torch.float64, device=DEV, generator=gen)
    return (A, Bm, Q, Rinv, z0, QT), w


def quad_embedding(B):
    """S1 linearisations (the benchmark's seeding) materialised at the LQR boundary: hop_build_augmented_f64 /
    hop_build_terminal_f64, R^-1 = chol_inv(sym(R)), z0 = e_d; the time weight is inside the blocks (no w_explicit)."""
    import ctypes as C
    import oracle as O
    case = cases.make_case("Quadrotor", N=128)
    F, x0, xg, u_ref, Q, R, alpha, w, N, T_min, T_max, wrap_idx, _ = case
    n, m, d = 12, 4, 13
    sel = api.HorizonSelector(case, B, device=DEV, mode=api.MODE_FAST)
    sel(torch.as_tensor(s1_x0(B, seed=0), device=DEV))
    X, A, Bm = sel.views()
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device=DEV)  # noqa: E731
    A_aug = torch.empty((B, N, d, d), dtype=torch.float64, device=DEV); Q_aug = torch.empty_like(A_aug)
    QT = torch.empty_like(A_aug); B_aug = torch.empty((B, N, d, m), dtype=torch.float64, device=DEV)
    xg_t, w_t, ur_t, Q_t, Qf_t = t(np.broadcast_to(xg, (B, n))), t(np.full(B, float(w))), t(u_ref), t(Q), t(O.as_terminal_weight(alpha, n))
    p_ = lambda a: C.c_void_p(a.data_ptr())  # noqa: E731
    lib = api._cabi.require_device()
    api._cabi.check(lib.hop_build_augmented_f64(B, N, n, m, p_(A), p_(Bm), None, p_(X), p_(sel.U), sel.ustride, p_(xg_t), p_(w_t),
                                                p_(ur_t), p_(Q_t), O.wrap_mask(wrap_idx), 1e-9, 1e-12, p_(A_aug), p_(B_aug),
                                                p_(Q_aug), None), "hop_build_augmented_f64")
    api._cabi.check(lib.hop_build_terminal_f64(B, N, n, p_(X), p_(xg_t), p_(Qf_t), O.wrap_mask(wrap_idx), 1e-12, p_(QT), None),
                    "hop_build_terminal_f64")
    torch.cuda.synchronize()
    z0 = np.zeros(d); z0[-1] = 1.0
    return (A_aug, B_aug, Q_aug, t(O.chol_inv(0.5 * (R + R.T))), t(z0), QT), None, T_min, min(T_max, N)


def lqr(args):
    """hop_select_verified_f64 against FAST and EXACT at the LQR boundary: S2 as configuration 5 generates it (N = 128, with
    w_explicit) and the quadrotor embedding materialised at the boundary.  Distances and scan shares are on the minimised
    curve v = J + w t (J alone without w_explicit)."""
    work = [("S2 d=4 m=2 N=128, w_explicit (configuration 5 generator)", lambda: (*s2_config5(262144, 4, 2, 128), 1, 128), args.s2_tol),
            ("S2 d=12 m=4 N=128, w_explicit (configuration 5 generator)", lambda: (*s2_config5(65536, 12, 4, 128), 1, 128), args.s2_tol),
            ("S2 d=13 m=4 N=128, w_explicit (configuration 5 generator)", lambda: (*s2_config5(65536, 13, 4, 128), 1, 128), args.s2_tol),
            ("quadrotor embedding at the LQR boundary, 16384 S1 instances, N=128", lambda: quad_embedding(16384), args.quad_tol)]
    for name, make, tol in work:
        blocks, w, T_min, T_max = make()
        B = blocks[0].shape[0]
        def run(mode, blocks=blocks, w=w, T_min=T_min, T_max=T_max, tol=tol):
            kw = {"tie_tol": tol} if mode == api.MODE_VERIFIED else {}
            return api.propagator_all_Jt_aug_batched(*blocks, T_min, T_max, w_explicit=w, mode=mode, **kw)
        ts = alternate({k: (lambda m=m: run(m)) for k, m in MODES.items()}, args.rounds)
        out = {k: run(m) for k, m in MODES.items()}
        torch.cuda.synchronize()
        t = np.arange(1, T_max + 1, dtype=np.float64)
        wn = np.zeros(B) if w is None else w.cpu().numpy()
        V = {k: o.J.cpu().numpy() + wn[:, None] * t[None, :] for k, o in out.items()}       # numpy: two roundings, as the scan
        Tf, Te = out["fast"].T_star.cpu().numpy().astype(np.int64), out["exact"].T_star.cpu().numpy().astype(np.int64)
        rows = np.arange(B)
        gap, second = census.argmin_gap(V["fast"], Tf, T_min, T_max)
        r = lambda tt: np.abs(V["fast"][rows, tt - 1] - V["exact"][rows, tt - 1]) / np.abs(V["exact"][rows, tt - 1])  # noqa: E731
        dist = np.maximum.reduce([r(Tf), r(second), r(Te)])
        re = (out["verified"].status.cpu().numpy() & api.ST_FLAG_REEVALUATED) != 0
        st = out["fast"].status.cpu().numpy()
        s = summary(ts, B)
        rec = {"workload": name, "card": args.card, "batch": B, "tie_tol": tol, "timing": s,
               "verified_over_exact_throughput": s["verified"]["solves_per_s"] / s["exact"]["solves_per_s"],
               "verified_over_fast_throughput": s["verified"]["solves_per_s"] / s["fast"]["solves_per_s"],
               "reevaluated": int(re.sum()), "reevaluated_share": float(re.mean()),
               "T_star_verified_ne_exact": int((out["verified"].T_star.cpu().numpy() != Te).sum()),
               "T_star_fast_ne_exact": int((Tf != Te).sum()),
               "max_rel_fast_vs_exact_at_candidates": float(dist.max()),
               "p99_rel_fast_vs_exact_at_candidates": float(np.percentile(dist, 99)),
               "max_fast_gap_where_T_differs": float(gap[Tf != Te].max()) if (Tf != Te).any() else None}
        for tl in LQR_TOLS:
            mark = scan_decision(V["fast"], Tf.astype(np.int32), st, T_min, T_max, tl)
            rec[f"tol_{tl:g}"] = {"share": float(mark.mean()), "T_star_misses": int(((Tf != Te) & ~mark).sum())}
        emit(args.out, rec)
        del blocks, w, out, V
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to DIR/verified_ab.jsonl")
    ap.add_argument("--parts", default="s1,small,ddp", help="any of s1, small, ddp, lqr")
    ap.add_argument("--s2-tol", type=float, default=1e-10, help="tie_tol of the VERIFIED runs of the lqr part on S2")
    ap.add_argument("--quad-tol", type=float, default=1e-7, help="tie_tol of the lqr part on the quadrotor embedding")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("verified_ab.py measures on the GPU; no CUDA device is visible")
    if args.out:
        os.makedirs(args.out, exist_ok=True)
    args.card = card()
    emit(args.out, {"card (name, power limit, max SM clock)": args.card})
    parts = args.parts.split(",")
    if "s1" in parts:
        s1(args)
    if "small" in parts:
        small_calibration(args)
    if "ddp" in parts:
        ddp(args)
    if "lqr" in parts:
        lqr(args)


if __name__ == "__main__":
    main()
