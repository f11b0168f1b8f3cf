"""One-flavour RHMC with the smallest MD poles on multigrid (HMC(flavours=1, mg_poles=K)), and the cost of MG.set_twist.

In one process:
  * at --L^2 (1024) on the links and settings of tools/rhmc_bench.py (mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60,
    seed=1234), bench.workload_params, tau 0.25, 16 steps, seed 2024) for each mass and K = 0..5 with the same spectrum and seed:
    the multi-shift iterations per force, the (-mu, +mu) FGCR iterations per MG pole, the time split of each trajectory, dH
    and acceptance;
  * at --Lb^2 (4096) on the benchmark's hierarchy parameters and links at mass --mb: the device time of set_twist (median over
    alternating twists), the memory it keeps, and the solve time of one MD force's shifts for K = 0 and for the K that was
    fastest at --L^2 (its poles are listed; the spectrum's a is 1/4 of the smallest Ritz value of a multi-shift solve).
Writes one JSON file with the GPU name and power limit read in the same run (rewritten after every section).

    python tools/rhmc_mg_bench.py [--L 1024] [--masses -0.04 0.05] [--K 0 1 2 3 4 5] [--traj 1] [--Lb 4096] [--mb 0.05] [--out FILE]
"""
import argparse
import json
import math
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from clover_bench import gpu_info  # noqa: E402


def _events():
    import torch
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def hmc_rows(mg2d, bench, theta, L, m, Ks, args):
    import torch
    p = bench.workload_params(mg2d, L, m)
    h = mg2d.HMC(p, theta, args.beta, tau=args.tau, n_md=args.n_md, flavours=1, seed=2024)
    spec = h.spectrum
    run = {"spectrum": spec, "poles_md": h.r_md.n, "md_shifts": h.r_md.beta, "md_mu": [math.sqrt(b) for b in h.r_md.beta], "K": {}}
    h.mg.close()
    del h
    for K in Ks:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h = mg2d.HMC(p, theta, args.beta, tau=args.tau, n_md=args.n_md, flavours=1, seed=2024, spectrum=spec, mg_poles=K)
        rows = []
        for _ in range(args.traj):
            o = h.trajectory()
            rows.append({k: o[k] for k in ("trajectory", "dH", "accepted", "iters_md", "iters_md_mg", "iters_accept",
                                           "iters_heatbath", "refreshed", "times_ms")})
            print(json.dumps({"mass": m, "K": K, "dH": o["dH"], "acc": o["accepted"], "iters_md": o["iters_md"][:2],
                              "ms": {k: round(v, 1) for k, v in o["times_ms"].items()}}), flush=True)
        mean = lambda key: statistics.mean(r["times_ms"].get(key, 0.0) for r in rows)
        run["K"][str(K)] = {"construction_s": time.perf_counter() - t0, "trajectories": rows,
                            "acceptance": sum(r["accepted"] for r in rows) / len(rows),
                            "mean_multishift_iters_per_force": statistics.mean(i for r in rows for i in r["iters_md"]),
                            "mean_trajectory_ms": mean("total"),
                            "mean_split_ms": {k: mean(k) for k in ("solves", "mg_solves", "twist", "momentum", "refresh",
                                                                   "links", "energies")}}
        h.mg.close()
        del h
    return run


def large_rows(mg2d, bench, L, m, K, args):
    import torch
    from importlib import import_module
    R = import_module("2d_multigrid_b200.rational")
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)
    p = bench.workload_params(mg2d, L, m)
    mg = mg2d.setup(U, p, init="device")
    g = torch.Generator(device="cuda").manual_seed(11)
    phi = torch.randn((L * L, 2), generator=g, dtype=torch.complex128, device="cuda")
    _, info = mg2d.multishift_cg(mg, phi, [0.0], 1e-6, 100000)
    a, b = 0.25 * info["ritz"][0], (abs(2.0 + m) + 2.0 * math.sqrt(2.0)) ** 2
    r = R.rational_approx(-0.5, a, b, R.MD_TOL)
    out = {"L": L, "mass": m, "levels": p.size, "spectrum": (a, b), "md_shifts": r.beta, "md_mu": [math.sqrt(x) for x in r.beta]}
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated()
    mg.set_twist(0.01)
    torch.cuda.synchronize()
    out["set_twist_kept_bytes"] = torch.cuda.memory_allocated() - m0
    ts = []
    for i in range(args.reps):
        e0 = _events()
        mg.set_twist(0.02 if i % 2 == 0 else 0.01)
        e1 = _events()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    out["set_twist_median_ms"] = statistics.median(ts)
    out["set_twist_reps"] = args.reps
    mg.set_twist(0.0)
    solves = {}
    for k in sorted({0, K}):
        for rep in range(2):           # the first pass captures the graphs of every twist
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            it_ms, it_mg = 0, []
            if k < r.n:
                _, im = mg2d.multishift_cg(mg, phi, r.beta[k:], 1e-10, 100000)
                it_ms = im["iters"]
            if k:
                _, ig = mg2d.normal_solve(mg, phi, r.beta[:k], 1e-10, use_graph=True)
                it_mg = ig["iters"]
            torch.cuda.synchronize()
            solves[str(k)] = {"ms": 1e3 * (time.perf_counter() - t0), "multishift_iters": it_ms, "fgcr_iters": it_mg,
                              "twist_ms": ig["twist_ms"] if k else 0.0, "pass": rep}
        print(json.dumps({"L": L, "K": k, **solves[str(k)]}), flush=True)
    out["force_solves"] = solves
    mg.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--L", type=int, default=1024)
    ap.add_argument("--masses", type=float, nargs="+", default=[-0.04, 0.05])
    ap.add_argument("--K", type=int, nargs="+", default=[0, 1, 2, 3, 4, 5])
    ap.add_argument("--beta", type=float, default=6.0)
    ap.add_argument("--tau", type=float, default=0.25)
    ap.add_argument("--n_md", type=int, default=16)
    ap.add_argument("--traj", type=int, default=1)
    ap.add_argument("--Lb", type=int, default=4096)
    ap.add_argument("--mb", type=float, default=0.05)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rhmc_mg_bench_L1024.json"))
    args = ap.parse_args()
    card = gpu_info()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rhmc_mg_bench: no CUDA device")
    import bench
    import mg2d
    res = {"gpu": card, "L": args.L, "beta": args.beta, "tau": args.tau, "n_md": args.n_md, "md_tol": 1e-10, "accept_tol": 1e-12,
           "gauge": "mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)", "seed": 2024, "runs": {}}

    def save():
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    _, theta = mg2d.gauge.quenched_links_device(args.L, args.beta, sweeps=60, seed=1234, return_phases=True)
    best = {}
    for m in args.masses:
        run = hmc_rows(mg2d, bench, theta, args.L, m, args.K, args)
        best[m] = min(run["K"], key=lambda k: run["K"][k]["mean_trajectory_ms"])
        run["fastest_K"] = int(best[m])
        res["runs"][str(m)] = run
        save()
    if args.Lb:
        K = int(best.get(args.mb, best[args.masses[0]]))
        res["large"] = large_rows(mg2d, bench, args.Lb, args.mb, max(K, 1), args)
        save()


if __name__ == "__main__":
    main()
