"""Wilson vs Wilson-clover on one GPU at the benchmark's size: kernel rooflines, critical mass and the bench workload.

For c_sw in {0, 1}, in one process on the same beta = 6 device links (bench.py's configuration):
  * the matrix-free level-0 apply and one two-colour red-black sweep, CUDA events with L2 flushed (bench.time_kernel), as
    GB/s of algorithmic traffic (apply 96 / 104 B per site, sweep 128 / 136 B in complex128) and as a fraction of the
    measured HBM peak (MEASURED_PEAKS.json; the fallback figure is marked as such);
  * m_crit from critical.estimate_critical_mass;
  * the bench workload at m_crit + delta (bench.workload_params, FGCR(8), tol 1e-10, CUDA graphs): iterations,
    time-to-solution and true residual, with the complex128 V-cycle and with the complex64 preconditioner.
Writes one JSON file (default profiles/clover_bench_L4096.json) with the GPU name and power limit beside the numbers.

    python tools/clover_bench.py [--L 4096] [--steps 5] [--delta 1e-3] [--out FILE]
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    """name, power limit and max SM clock of GPU 0 (queried before this process creates its CUDA context)."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power, "clocks_max_sm": clock}
    except Exception as e:                          # the numbers stay valid; say that the card could not be identified
        return {"name": None, "power_limit": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--L", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--delta", type=float, default=1e-3)
    ap.add_argument("--csw", type=float, nargs="+", default=[0.0, 1.0])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "clover_bench_L4096.json"))
    args = ap.parse_args()
    card = gpu_info()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("clover_bench: no CUDA device")
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
           "gpu": card, "hbm_peak_gbs": hbm, "hbm_peak_source": pk_src, "runs": []}

    for csw in args.csw:
        t0 = time.time()
        mcrit, _ = critical.estimate_critical_mass(U, lambda m: bench.workload_params(mg2d, L, m, csw=csw), iters=4, refine=3)
        info_c = dict(critical.estimate_critical_mass.info)
        t_crit = time.time() - t0
        gc.collect()
        torch.cuda.empty_cache()
        p = bench.workload_params(mg2d, L, mcrit + args.delta, csw=csw)
        t0 = time.time()
        mg = mg2d.setup(U, p, init="device")
        torch.cuda.synchronize()
        t_setup = time.time() - t0
        lv0 = mg.LVL[0]
        assert lv0.matrix_free and (lv0.clover is not None) == (csw != 0.0)

        # kernels (L2 flushed before every timed launch)
        a, b = lv0.new_field(), lv0.new_field()
        a.normal_()
        bpe = 104.0 if csw != 0.0 else 96.0
        bps = 136.0 if csw != 0.0 else 128.0
        t_apply = bench.time_kernel(lambda: lv0.apply_D(b, a), 20, flush)
        phi0 = lv0.phi.clone()
        lv0.phi.copy_(a)
        t_sweep = bench.time_kernel(lambda: lv0.relax(2, smoother="rbgs"), 10, flush) / 2
        lv0.phi.copy_(phi0)
        del a, b, phi0
        kern = {}
        for name, nbytes, ms in (("apply", bpe * lv0.S, t_apply), ("rb2_sweep", bps * lv0.S, t_sweep)):
            gbs = nbytes / (ms * 1e-3) / 1e9
            kern[name] = {"ms": ms, "bytes_per_site": nbytes / lv0.S, "gbs": gbs, "frac_of_peak": gbs / hbm}

        # the bench workload
        legs = {}
        for leg, kw in (("complex128", {}), ("complex64_precond", {"precond_dtype": "complex64"})):
            solve = lambda: mg2d.solve(mg, rhs=rhs, tol=bench.TOL, outer="gcr", restart=8, use_graph=True, check_every=1, **kw)
            for _ in range(max(args.warmup, 1)):
                x, info = solve()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                x, info = solve()
            e1.record()
            torch.cuda.synchronize()
            legs[leg] = {"ms": e0.elapsed_time(e1) / args.steps, "iters": info["iters"], "converged": bool(info["converged"]),
                         "true_resnorm": info.get("true_resnorm")}
        run = {"csw": csw, "m_crit": mcrit, "mass": mcrit + args.delta, "critical_info": info_c, "t_crit_s": t_crit,
               "setup_s": t_setup, "levels": p.size, "dof": p.n_dof, "kernels": kern, "solve": legs}
        print(json.dumps(run), flush=True)
        res["runs"].append(run)
        mg.close()
        del mg, lv0
        gc.collect()
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
