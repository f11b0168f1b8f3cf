"""Two-flavour Wilson HMC on one GPU: cost of a trajectory, how fast a stale coarse hierarchy degrades, and the MD kernels' rooflines.

In one process, from the benchmark's links (mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)) and the benchmark's
multigrid parameters (bench.workload_params) at a stated mass above m_crit:
  * mg2d_hmc_momentum (with fermion fields, 128 B/site) and mg2d_hmc_links (with the complex64 copy, 96 B/site) timed with
    CUDA events, L2 flushed before every launch, as GB/s of algorithmic traffic and as a fraction of the HBM peak
    (MEASURED_PEAKS.json; the fallback figure is marked as such);
  * a full setup() against MG.refresh(0) and MG.refresh(k) on the same hierarchy;
  * for each refresh policy (never, refresh(0) = Galerkin products only, refresh(k)): the same trajectories (same seed),
    with the iterations of every solve, dH, acceptance and the per-trajectory time split into solves, momentum kernel, link
    kernel, refresh and energies (CUDA events).
Writes one JSON file with the GPU name and power limit beside the numbers.

    python tools/hmc_bench.py [--L 1024] [--mass -0.04] [--tau 0.25] [--n_md 16] [--traj 4] [--k 8] [--out FILE]
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


def kernel_rows(mg2d, h, hbm, flush, reps):
    import torch
    ctx, L, S = h.ctx, h.L, h.L * h.L
    st = lambda: torch.cuda.current_stream().cuda_stream
    U = h.mg.LVL[0].U
    X = torch.randn((S, 2), dtype=torch.complex128, device=U.device)
    Y = torch.randn((S, 2), dtype=torch.complex128, device=U.device)
    P = torch.randn((S, 2), dtype=torch.float64, device=U.device)
    th = h.theta.clone()
    U32 = U.to(torch.complex64)
    calls = {
        "hmc_momentum": (lambda: ctx.call("mg2d_hmc_momentum", P.data_ptr(), U.data_ptr(), X.data_ptr(), Y.data_ptr(), 6.0, 1e-9, L,
                                          st()), 128.0),
        "hmc_momentum_gauge_only": (lambda: ctx.call("mg2d_hmc_momentum", P.data_ptr(), U.data_ptr(), None, None, 6.0, 1e-9, L,
                                                     st()), 64.0),
        "hmc_links": (lambda: ctx.call("mg2d_hmc_links", th.data_ptr(), P.data_ptr(), 0.0, U.data_ptr(), U32.data_ptr(), 2 * S,
                                       st()), 96.0),
    }
    out = {}
    for name, (fn, bps) in calls.items():
        fn()
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = statistics.median(ts)
        gbs = bps * S / (ms * 1e-3) / 1e9
        out[name] = {"bytes_per_site": bps, "median_ms": ms, "GBs": gbs, "fraction_of_hbm_peak": gbs / hbm, "reps": reps}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--L", type=int, default=1024)
    ap.add_argument("--mass", type=float, default=-0.04)
    ap.add_argument("--beta", type=float, default=6.0)
    ap.add_argument("--tau", type=float, default=0.25)
    ap.add_argument("--n_md", type=int, default=16)
    ap.add_argument("--traj", type=int, default=4)
    ap.add_argument("--k", type=int, default=8, help="null-vector sweeps of the refresh(k) policy")
    ap.add_argument("--policies", default="never,0,k")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hmc_bench_L1024.json"))
    args = ap.parse_args()
    card = gpu_info()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("hmc_bench: no CUDA device")
    import bench
    import mg2d
    pk, pk_src = bench.peaks()
    hbm = float(pk["hbm_gbs"])
    L = args.L
    p = bench.workload_params(mg2d, L, args.mass)
    U, theta = mg2d.gauge.quenched_links_device(L, args.beta, sweeps=60, seed=1234, return_phases=True)
    dev = torch.device("cuda", torch.cuda.current_device())
    flush = torch.zeros(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)      # 256 MiB > 126 MB L2
    res = {"L": L, "beta": args.beta, "mass": args.mass,
           "mass_note": "m_crit = -0.0643 at 4096^2 (critical.py, README); this mass is about 0.024 above it",
           "gauge": "mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)",
           "params": "bench.workload_params (rbgs, n_pre 0, n_post %s, %d levels, block 4, n_null 8, null_iters 100)" % (p.post, p.nlevels),
           "tau": args.tau, "n_md": args.n_md, "md_tol": 1e-10, "accept_tol": 1e-12, "solver": "FGCR(8) + V-cycle, CUDA graphs",
           "gpu": card, "hbm_peak_gbs": hbm, "hbm_peak_source": pk_src}

    # ---- setup against refresh -----------------------------------------------------------------------------------
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mg = mg2d.setup(U.clone(), p, init="device")
    torch.cuda.synchronize()
    t_setup = time.perf_counter() - t0
    mg.update_links(U)
    ref = {"setup_s": t_setup}
    for k in (0, args.k, 0, args.k):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mg.refresh(k)
        torch.cuda.synchronize()
        ref.setdefault(f"refresh_{k}_s", []).append(time.perf_counter() - t0)
    res["setup_vs_refresh"] = ref
    mg.close()
    del mg

    # ---- trajectories per policy ------------------------------------------------------------------------------------
    pol = {"never": None, "0": 0, "k": args.k}
    res["policies"] = {}
    kern = None
    for name in args.policies.split(","):
        rn = pol[name]
        h = mg2d.HMC(p, theta, args.beta, tau=args.tau, n_md=args.n_md, seed=2024, md_tol=1e-10, accept_tol=1e-12,
                     refresh_null_iters=rn, use_graph=True)
        if kern is None:
            kern = kernel_rows(mg2d, h, hbm, flush, args.reps)
        rows = []
        for _ in range(args.traj):
            o = h.trajectory()
            rows.append(o)
            print(json.dumps({"policy": name, "traj": o["trajectory"], "dH": o["dH"], "acc": o["accepted"],
                              "iters_md": o["iters_md"], "ms": {k: round(v, 1) for k, v in o["times_ms"].items()}}), flush=True)
        res["policies"][f"refresh_{name}" if name != "k" else f"refresh_{args.k}"] = {
            "refresh_null_iters": rn, "trajectories": rows,
            "acceptance": sum(r["accepted"] for r in rows) / len(rows),
            "mean_iters_per_md_solve": [statistics.mean(r["iters_md"]) for r in rows]}
        h.mg.close()
        del h
    res["kernels"] = kern
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"kernels": kern, "setup_vs_refresh": ref}, indent=1))


if __name__ == "__main__":
    main()
