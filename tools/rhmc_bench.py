"""One-flavour Wilson RHMC on one GPU: the multi-shift CG's vector passes against the copy peak, and the cost of a trajectory.

In one process:
  * mg2d_msc_pass_a (96 B/site with sigma_0 = 0, 128 with sigma_0 != 0) and mg2d_msc_pass_b (32 + 128 N_active B/site; accumulate
    mode 96 + 64 N_active) at --Lk^2, timed with CUDA events (median; every field is larger than the 126 MB L2), as GB/s of
    that algorithmic traffic and as a fraction of a device-to-device copy measured in the same run;
  * at --L^2 on the links of tools/hmc_bench.py (mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)) and the
    benchmark's multigrid parameters, for each mass: the construction (lambda_min estimate, rational approximations), the poles,
    the multi-shift iterations per force evaluation, the time split of each trajectory, dH and acceptance, and one two-flavour
    trajectory with the same tau and n_md.
Writes one JSON file with the GPU name and power limit beside the numbers (rewritten after every section).

    python tools/rhmc_bench.py [--L 1024] [--masses -0.04 0.05] [--tau 0.25] [--n_md 16] [--traj 2] [--Lk 4096] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from clover_bench import gpu_info  # noqa: E402
from measure_bench import copy_peak  # noqa: E402


def _median_ms(fn, reps):
    import torch
    fn()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def pass_rows(L, peak, reps):
    import torch
    from mg2d import _lib
    ctx = _lib.Context(torch.cuda.current_device())
    st = lambda: torch.cuda.current_stream().cuda_stream
    S, Nmax = L * L, 16
    g = torch.Generator(device="cuda").manual_seed(1)
    r = torch.randn((S, 2), generator=g, dtype=torch.complex128, device="cuda")
    w = torch.randn_like(r)
    y = torch.zeros_like(r)
    Pk = torch.randn((Nmax, S, 2), generator=g, dtype=torch.complex128, device="cuda")
    X = torch.zeros_like(Pk)
    dots = torch.tensor([float(S), 0, 0, 0], dtype=torch.float64, device="cuda")

    def sc_for(n):
        # a_k = 0, b_k = 1, zeta_k = 0: pass B rewrites x_k and p_k unchanged, so repeated launches stay finite; NACT_NEXT = 0
        # keeps pass A's scalar tail empty
        sc = torch.zeros(_lib.MSC_SHIFTS + 6 * Nmax + 2 * (reps + 2), dtype=torch.float64, device="cuda")
        o = _lib.MSC_SHIFTS
        sc[_lib.MSC_RR], sc[_lib.MSC_PP], sc[_lib.MSC_NACT] = 1e-30, 1.0, n
        sc[o + 4 * Nmax:o + 5 * Nmax] = 1.0
        return sc
    out = {}
    for sigma0 in (0.0, 0.01):
        sc = sc_for(Nmax)
        ms = _median_ms(lambda: ctx.call("mg2d_msc_pass_a", r.data_ptr(), w.data_ptr(), Pk.data_ptr(), dots.data_ptr(),
                                         sc.data_ptr(), sigma0, Nmax, S, st()), reps)
        bps = 96.0 if sigma0 == 0.0 else 128.0
        out[f"pass_a_sigma0_{sigma0}"] = _row(bps, S, ms, peak, reps)
    for n in (1, 8, 16):
        sc = sc_for(n)
        ms = _median_ms(lambda: ctx.call("mg2d_msc_pass_b", X.data_ptr(), Pk.data_ptr(), None, r.data_ptr(), sc.data_ptr(), 0.0,
                                         Nmax, S, st()), reps)
        out[f"pass_b_nactive_{n}"] = _row(32.0 + 128.0 * n, S, ms, peak, reps)
    for n in (1, 8, 16):
        sc = sc_for(n)
        ms = _median_ms(lambda: ctx.call("mg2d_msc_pass_b", None, Pk.data_ptr(), y.data_ptr(), r.data_ptr(), sc.data_ptr(), 0.0,
                                         Nmax, S, st()), reps)
        out[f"pass_b_accumulate_nactive_{n}"] = _row(96.0 + 64.0 * n, S, ms, peak, reps)
    ctx.close()
    return out


def _row(bps, S, ms, peak, reps):
    gbs = bps * S / (ms * 1e-3) / 1e9
    return {"bytes_per_site": bps, "median_ms": ms, "GBs": gbs, "fraction_of_copy_peak": gbs / peak, "reps": reps}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--L", type=int, default=1024)
    ap.add_argument("--masses", type=float, nargs="+", default=[0.05, -0.04])
    ap.add_argument("--beta", type=float, default=6.0)
    ap.add_argument("--tau", type=float, default=0.25)
    ap.add_argument("--n_md", type=int, default=16)
    ap.add_argument("--traj", type=int, default=2)
    ap.add_argument("--Lk", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rhmc_bench_L1024.json"))
    args = ap.parse_args()
    card = gpu_info()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rhmc_bench: no CUDA device")
    import bench
    import mg2d
    dev = torch.device("cuda", torch.cuda.current_device())
    peak = copy_peak(dev)
    res = {"gpu": card, "copy_peak_gbs": peak, "copy_peak_note": "2 GiB device-to-device copy, bytes read + written, this run"}

    def save():
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    res["passes"] = {"L": args.Lk, "rows": pass_rows(args.Lk, peak, args.reps)}
    print(json.dumps(res["passes"], indent=1), flush=True)
    save()

    L = args.L
    U, theta = mg2d.gauge.quenched_links_device(L, args.beta, sweeps=60, seed=1234, return_phases=True)
    res.update({"L": L, "beta": args.beta, "gauge": "mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)",
                "tau": args.tau, "n_md": args.n_md, "md_tol": 1e-10, "accept_tol": 1e-12, "runs": {}})
    for m in args.masses:
        p = bench.workload_params(mg2d, L, m)
        run = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h = mg2d.HMC(p, theta, args.beta, tau=args.tau, n_md=args.n_md, flavours=1, seed=2024)
        run["construction_s"] = time.perf_counter() - t0
        run.update({"spectrum": h.spectrum, "poles_md": h.r_md.n, "poles_precise": h.r_acc.n, "poles_heatbath": h.r_hb.n,
                    "error_md": h.r_md.error, "error_precise": h.r_acc.error, "error_heatbath": h.r_hb.error})
        rows = []
        for _ in range(args.traj):
            o = h.trajectory()
            rows.append(o)
            print(json.dumps({"mass": m, "flavours": 1, "traj": o["trajectory"], "dH": o["dH"], "acc": o["accepted"],
                              "iters_md": o["iters_md"], "ms": {k: round(v, 1) for k, v in o["times_ms"].items()}}), flush=True)
        run["trajectories"] = rows
        run["acceptance"] = sum(r["accepted"] for r in rows) / len(rows)
        run["mean_multishift_iters_per_force"] = statistics.mean(i for r in rows for i in r["iters_md"])
        h.mg.close()
        del h
        res["runs"][str(m)] = run
        save()
        h2 = mg2d.HMC(p, theta, args.beta, tau=args.tau, n_md=args.n_md, flavours=2, seed=2024)
        o = h2.trajectory()
        run["two_flavour_trajectory"] = o
        print(json.dumps({"mass": m, "flavours": 2, "dH": o["dH"], "iters_md": o["iters_md"],
                          "ms": {k: round(v, 1) for k, v in o["times_ms"].items()}}), flush=True)
        h2.mg.close()
        del h2
        save()


if __name__ == "__main__":
    main()
