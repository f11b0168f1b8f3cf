"""Gauge-ensemble measurements on one GPU: the kernels' rooflines, the cost of the fermionic measurements, and a short
two-flavour HMC stream measured after every trajectory.

(a) At L = 4096 on the benchmark's links (mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)):
  * mg2d_meson_contract (64 B/site), mg2d_topo_charge (32 B/site) and mg2d_wilson_loops (r_max = t_max = 4 and 32) timed
    with CUDA events, L2 flushed before every launch, median over --reps launches; bytes over time against the copy peak
    measured in the same run (a 2 GiB device-to-device copy, read + write), and the Wilson loops' fp64 rate (20 flops per
    (site, R, T): three complex products and a complex add);
  * meson_correlators (two solves) and chiral_condensate(n_noise=4) on a hierarchy built with bench.workload_params at
    --mass, with the complex128 and the complex64 preconditioner: wall time (a warm-up call first captures the graphs) and
    iterations.
(b) A two-flavour HMC stream (--hmc_L, beta, mass, tau, n_md): after every trajectory the plaquette, Q, W(R, T <= 4), the
    pion correlator with m_eff and m_pcac from a point source, and the condensate (4 noises) on h.mg, with the time of the
    trajectory and of the measurement.
The GPU name and power limit are read in the same run and written beside the numbers.

    python tools/measure_bench.py [--L 4096] [--mass -0.0633] [--hmc_L 256] [--traj 20] [--out FILE]
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


def _timed(fn, reps, flush):
    import torch
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
    return statistics.median(ts), min(ts)


def copy_peak(dev):
    """GB/s of a 2 GiB device-to-device copy (bytes read + written), median of 10."""
    import torch
    a = torch.empty(1 << 28, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    ms, _ = _timed(lambda: b.copy_(a), 10, torch.zeros(8, device=dev))
    return 2 * a.numel() * 8 / (ms * 1e-3) / 1e9


def kernel_rows(mg2d, U, L, peak, flush, reps):
    import torch
    from mg2d import _lib
    ctx = _lib.Context(torch.cuda.current_device())
    st = lambda: torch.cuda.current_stream().cuda_stream
    S = L * L
    g = torch.Generator(device=U.device).manual_seed(1)
    psi0 = torch.randn((S, 2), generator=g, dtype=torch.complex128, device=U.device)
    psi1 = torch.randn((S, 2), generator=g, dtype=torch.complex128, device=U.device)
    out = torch.zeros(32 * L + 2 * 32 * 32, dtype=torch.float64, device=U.device)     # G [L, 4, 4] or the loops
    calls = {
        "meson_contract": (lambda: ctx.call("mg2d_meson_contract", psi0.data_ptr(), psi1.data_ptr(), L, out.data_ptr(), st()),
                           64.0, 0.0),
        "topo_charge": (lambda: ctx.call("mg2d_topo_charge", U.data_ptr(), L, out.data_ptr(), st()), 32.0, 0.0),
        "wilson_loops_4x4": (lambda: ctx.call("mg2d_wilson_loops", U.data_ptr(), L, 4, 4, out.data_ptr(), st()), 32.0, 20.0 * 16),
        "wilson_loops_32x32": (lambda: ctx.call("mg2d_wilson_loops", U.data_ptr(), L, 32, 32, out.data_ptr(), st()), 32.0,
                               20.0 * 1024),
    }
    rows = {}
    for name, (fn, bps, fps) in calls.items():
        ms, mn = _timed(fn, reps, flush)
        gbs = bps * S / (ms * 1e-3) / 1e9
        rows[name] = {"bytes_per_site": bps, "median_ms": ms, "min_ms": mn, "GBs": gbs, "fraction_of_copy_peak": gbs / peak,
                      "reps": reps}
        if fps:
            rows[name].update(flops_per_site=fps, fp64_TFLOPs=fps * S / (ms * 1e-3) / 1e12)
    ctx.close()
    return rows


def fermion_rows(mg2d, bench, U, L, mass):
    import torch
    p = bench.workload_params(mg2d, L, mass)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mg = mg2d.setup(U.clone(), p, init="device")
    torch.cuda.synchronize()
    res = {"setup_s": time.perf_counter() - t0, "params": "bench.workload_params(L, %g): %d levels, post %s" % (mass, p.nlevels, p.post)}
    for pd in (None, "complex64"):
        row = {}
        for name, fn in (("meson_correlators", lambda: mg2d.meson_correlators(mg, site=(0, 0), precond_dtype=pd)),
                         ("chiral_condensate_4", lambda: mg2d.chiral_condensate(mg, 4, seed=1, precond_dtype=pd))):
            fn()                                        # captures the iteration graphs
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            o = fn()
            torch.cuda.synchronize()
            row[name] = {"s": time.perf_counter() - t0, "iters": o["iters"]}
            if name == "meson_correlators":
                row[name].update(m_pcac_12=float(o["m_pcac"][12]), m_eff_12=float(o["m_eff"][12]))
            else:
                row[name].update(mean=[o["mean"].real, o["mean"].imag], stderr=o["stderr"])
        res["complex128" if pd is None else pd] = row
        print(json.dumps({"precond": pd, **row}), flush=True)
    mg.close()
    return res


def hmc_stream(mg2d, bench, args):
    import torch
    L = args.hmc_L
    p = bench.workload_params(mg2d, L, args.hmc_mass)
    _, theta = mg2d.gauge.quenched_links_device(L, args.hmc_beta, sweeps=60, seed=1234, return_phases=True)
    h = mg2d.HMC(p, theta, args.hmc_beta, tau=args.tau, n_md=args.n_md, seed=2024)
    rows = []
    for _ in range(args.traj):
        o = h.trajectory()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        U = h.mg.LVL[0].U
        q = mg2d.topological_charge(U, L)
        W = mg2d.wilson_loops(U, L, 4, 4)
        mes = mg2d.meson_correlators(h.mg, site=(0, 0))
        cc = mg2d.chiral_condensate(h.mg, 4, seed=1000 + o["trajectory"])
        torch.cuda.synchronize()
        t_meas = time.perf_counter() - t0
        row = {"trajectory": o["trajectory"], "accepted": o["accepted"], "dH": o["dH"], "plaquette": o["plaquette"], "Q": q,
               "W_re": W.real.tolist(), "pp": mes["pp"][:L // 2 + 1].tolist(), "m_eff": mes["m_eff"][1:L // 2].tolist(),
               "m_pcac": mes["m_pcac"][1:L // 2].tolist(), "condensate": [cc["mean"].real, cc["mean"].imag],
               "condensate_stderr": cc["stderr"], "iters_meson": mes["iters"], "iters_condensate": cc["iters"],
               "mean_iters_md": statistics.mean(o["iters_md"]), "trajectory_ms": o["times_ms"]["total"],
               "measurement_ms": 1e3 * t_meas}
        rows.append(row)
        print(json.dumps({k: (round(v, 5) if isinstance(v, float) else v) for k, v in row.items()
                          if k not in ("W_re", "pp", "m_eff", "m_pcac")} | {"m_pcac_L/8": round(mes["m_pcac"][L // 8], 5)}),
              flush=True)
    h.mg.close()
    acc = sum(r["accepted"] for r in rows) / len(rows)
    return {"L": L, "beta": args.hmc_beta, "mass": args.hmc_mass, "tau": args.tau, "n_md": args.n_md, "seed": 2024,
            "params": "bench.workload_params (%d levels)" % p.nlevels, "acceptance": acc,
            "mean_trajectory_ms": statistics.mean(r["trajectory_ms"] for r in rows),
            "mean_measurement_ms": statistics.mean(r["measurement_ms"] for r in rows[1:] or rows),
            "trajectories": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--L", type=int, default=4096)
    ap.add_argument("--mass", type=float, default=-0.0633, help="m_crit + 1e-3 at 4096^2 (m_crit = -0.0643, README)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--hmc_L", type=int, default=256)
    ap.add_argument("--hmc_beta", type=float, default=6.0)
    ap.add_argument("--hmc_mass", type=float, default=-0.04)
    ap.add_argument("--tau", type=float, default=0.5)
    ap.add_argument("--n_md", type=int, default=16)
    ap.add_argument("--traj", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "measure_bench.json"))
    args = ap.parse_args()
    card = gpu_info()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("measure_bench: no CUDA device")
    import bench
    import mg2d
    dev = torch.device("cuda", torch.cuda.current_device())
    L = args.L
    res = {"gpu": card, "L": L, "beta": 6.0, "gauge": "mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)",
           "solver": "FGCR(8) + V-cycle, CUDA graphs, tol 1e-10"}
    peak = copy_peak(dev)
    res["copy_peak_GBs"] = peak
    flush = torch.zeros(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)      # 256 MiB > 126 MB L2
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)
    res["kernels"] = kernel_rows(mg2d, U, L, peak, flush, args.reps)
    print(json.dumps({"copy_peak_GBs": peak, "kernels": res["kernels"]}, indent=1), flush=True)
    res["Q"] = mg2d.topological_charge(U, L)
    res["W_re_4x4"] = mg2d.wilson_loops(U, L, 4, 4).real.tolist()
    del flush
    res["fermion"] = fermion_rows(mg2d, bench, U, L, args.mass)
    del U
    torch.cuda.empty_cache()
    res["hmc_stream"] = hmc_stream(mg2d, bench, args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res["hmc_stream"][k] for k in ("acceptance", "mean_trajectory_ms", "mean_measurement_ms")}))


if __name__ == "__main__":
    main()
