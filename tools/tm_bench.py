"""Twisted mass on one GPU at the benchmark's size: kernel rooflines against the Wilson kernels and maximal-twist solves.

In one process on the same beta = 6 device links as bench.py and tools/clover_bench.py:
  * the matrix-free level-0 apply and one two-colour red-black sweep (with r), Wilson and twisted-mass entry points on the
    same fields, timed in alternation with L2 flushed before every launch (CUDA events), as GB/s of algorithmic traffic
    (apply 96 B per site, sweep 128 B in complex128: mu is one constant per launch) and as a fraction of the HBM peak
    (MEASURED_PEAKS.json; the fallback figure is marked as such);
  * m_crit of the untwisted operator from critical.estimate_critical_mass;
  * the reference row: the bench workload at m_crit + delta, mu = 0;
  * twisted solves at m = m_crit (maximal twist) for each mu: iterations, time-to-solution and true residual with the
    complex128 V-cycle and with the complex64 preconditioner (bench.workload_params, FGCR(8), tol 1e-10, CUDA graphs).
Writes one JSON file (default profiles/tm_bench_L4096.json) with the GPU name and power limit beside the numbers.

    python tools/tm_bench.py [--L 4096] [--steps 5] [--mu 1e-3 3e-3 1e-2] [--out FILE]
"""
import argparse
import gc
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


def kernel_rows(mg2d, lv0, mu, hbm, flush, rounds, reps):
    """Wilson and twisted apply / rb2 sweep on the same fields, alternating; median over rounds of mean-of-reps times."""
    import bench
    import torch
    mg = lv0.mg
    L, S = lv0.L, lv0.S
    C = mg2d._lib.C128
    st = lambda: torch.cuda.current_stream().cuda_stream
    a, b, r, o = lv0.new_field(), lv0.new_field(), lv0.new_field(), lv0.new_field()
    a.normal_()
    r.normal_()
    row = lambda t, y: t[y * L:].data_ptr()
    U, m = lv0.U, float(mg.p.mass)
    calls = {
        ("apply", "wilson"): lambda: mg.ctx.call("mg2d_wilson_apply", b.data_ptr(), a.data_ptr(), row(a, L - 1), row(a, 0),
                                                 U.data_ptr(), lv0.U_lo_ptr, None, m, L, L, 0, C, None, st()),
        ("apply", "tm"): lambda: mg.ctx.call("mg2d_wilson_tm_apply", b.data_ptr(), a.data_ptr(), row(a, L - 1), row(a, 0),
                                             U.data_ptr(), lv0.U_lo_ptr, None, None, m, mu, L, L, 0, C, None, st()),
        ("rb2_sweep", "wilson"): lambda: mg.ctx.call("mg2d_wilson_relax_rb2", o.data_ptr(), a.data_ptr(), row(a, L - 2), row(a, 0),
                                                     U.data_ptr(), lv0.U_lo2_ptr, lv0.U_hi_ptr, r.data_ptr(), row(r, L - 1),
                                                     row(r, 0), m, L, L, 0, C, None, st()),
        ("rb2_sweep", "tm"): lambda: mg.ctx.call("mg2d_wilson_tm_relax_rb2", o.data_ptr(), a.data_ptr(), row(a, L - 2), row(a, 0),
                                                 U.data_ptr(), lv0.U_lo2_ptr, lv0.U_hi_ptr, None, None, None, r.data_ptr(),
                                                 row(r, L - 1), row(r, 0), m, mu, L, L, 0, C, None, st()),
    }
    nbytes = {"apply": 96.0, "rb2_sweep": 128.0}
    samples = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            samples[k].append(bench.time_kernel(fn, reps, flush))
    out = {}
    for (kern, op), ts in samples.items():
        ms = statistics.median(ts)
        gbs = nbytes[kern] * S / (ms * 1e-3) / 1e9
        out.setdefault(kern, {})[op] = {"ms": ms, "ms_rounds": ts, "bytes_per_site": nbytes[kern], "gbs": gbs,
                                        "frac_of_peak": gbs / hbm}
    del a, b, r, o
    return out


def solve_legs(mg2d, mg, rhs, steps, warmup):
    import bench
    import torch
    legs = {}
    for leg, kw in (("complex128", {}), ("complex64_precond", {"precond_dtype": "complex64"})):
        solve = lambda: mg2d.solve(mg, rhs=rhs, tol=bench.TOL, outer="gcr", restart=8, use_graph=True, check_every=1, **kw)
        for _ in range(max(warmup, 1)):
            x, info = solve()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            x, info = solve()
        e1.record()
        torch.cuda.synchronize()
        legs[leg] = {"ms": e0.elapsed_time(e1) / steps, "iters": info["iters"], "converged": bool(info["converged"]),
                     "true_resnorm": info.get("true_resnorm")}
    return legs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--L", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--delta", type=float, default=1e-3)
    ap.add_argument("--mu", type=float, nargs="+", default=[1e-3, 3e-3, 1e-2])
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tm_bench_L4096.json"))
    args = ap.parse_args()
    card = gpu_info()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("tm_bench: no CUDA device")
    import bench
    import mg2d
    from importlib import import_module
    critical = import_module("2d_multigrid_b200.critical")

    L, dev = args.L, torch.device("cuda", 0)
    pk, pk_src = bench.peaks()
    hbm = float(pk["hbm_gbs"])
    card["torch_name"] = torch.cuda.get_device_name(0)
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)
    flush = torch.zeros(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)      # 256 MiB > 126 MB L2
    rhs = torch.zeros((L * L, 2), dtype=torch.complex128, device=dev)
    rhs[L // 2 + (L // 2) * L, 0] = 1.0
    res = {"L": L, "beta": 6.0, "gauge": "mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)", "delta": args.delta,
           "gpu": card, "hbm_peak_gbs": hbm, "hbm_peak_source": pk_src}

    t0 = time.time()
    mcrit, _ = critical.estimate_critical_mass(U, lambda m: bench.workload_params(mg2d, L, m), iters=4, refine=3)
    res["m_crit"], res["critical_info"], res["t_crit_s"] = mcrit, dict(critical.estimate_critical_mass.info), time.time() - t0
    print("m_crit", mcrit, res["critical_info"], flush=True)
    gc.collect()
    torch.cuda.empty_cache()

    runs = []
    for mu, mass in [(0.0, mcrit + args.delta)] + [(mu, mcrit) for mu in args.mu]:
        p = bench.workload_params(mg2d, L, mass, mu=mu)
        t0 = time.time()
        mg = mg2d.setup(U, p, init="device")
        torch.cuda.synchronize()
        t_setup = time.time() - t0
        lv0 = mg.LVL[0]
        assert lv0.matrix_free and lv0.clover is None and mg.p.mu == mu
        run = {"mu": mu, "mass": mass, "setup_s": t_setup, "levels": p.size, "dof": p.n_dof}
        if mu == args.mu[0]:
            res["kernels"] = kernel_rows(mg2d, lv0, mu, hbm, flush, args.rounds, 20)
            print(json.dumps(res["kernels"]), flush=True)
        run["solve"] = solve_legs(mg2d, mg, rhs, args.steps, args.warmup)
        print(json.dumps(run), flush=True)
        runs.append(run)
        mg.close()
        del mg, lv0
        gc.collect()
        torch.cuda.empty_cache()
    res["runs"] = runs

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
