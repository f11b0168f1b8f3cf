#!/usr/bin/env python
"""bench.py -- 2D Wilson adaptive-MG time-to-solution (1e-10) and D-apply HBM GB/s on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
    python bench.py --impl reference ...                      (reference arm: the CPU path, see below)
    python bench.py --gpus 1 ... --dump-outputs DIR           (also write the last timed solve's results as DIR/*.npy)

A "step" is one full solve of D x = b (point source, x0 = 0) to |r|/|b| < 1e-10 on the workload lattice with
the hierarchy already set up and all inputs resident in HBM.  `value` is the time to solution in ms
(higher_is_better = false); `e2e` is the same solve through the public API with the right-hand side in pinned
HOST memory and the solution copied back to the host inside the timed region.

Workload (config.workload): BASELINE.json configs[4]/[3] -- 2D U(1) Wilson, quenched beta=6 links generated on
the device, mass = m_crit + 1e-3 (near-critical; m_crit located by MG inverse iteration), adaptive MG with
8 null vectors per chirality-pair (16 coarse dof), 4x4 aggregates, levels L/4^k down to 16, red-black GS
smoother (no pre-smoothing; 4 / 2 / 8 / 8 ... post-smoothing sweeps on levels 0 / 1 / 2 / deeper: measured fastest),
flexible GCR(8) outer iteration,
complex128.

Reference arm / cpu_baseline: the reference (single-threaded C++/Eigen) cannot be built for this workload -- Eigen is
absent and its coarse dof count is hard-wired to 4 -- so the CPU side is the oracle PORT running the SAME algorithm: full
solves (to 1e-10, with the iteration count the CPU solve itself needs) by the plain C + OpenMP restatement of the solve
loop (oracle/c_port) with an explicitly set thread count (every host processor; launchers export OMP_NUM_THREADS=1).
  * `--impl reference` (no GPU code on the path): hierarchy of a 512^2 lattice of the workload's shape set up by the numpy
    oracle (not timed); `value` = measured solve time x (L/512)^2 sites, `ms_per_step` = the measured wall time of a step.
  * `cpu_baseline` of the GPU arm (rank 0, N=1): the hierarchy of a 1024^2 near-critical lattice is built by the GPU
    setup, exported to the host and solved by the C port: a MEASURED solve at 1024^2, scaled only x16 sites to 4096^2.
The JSON says all of this in `sample`.  The reference's own binary IS timed on the configuration it can run (BASELINE
configs[1], key `config2_vs_reference_binary`).
"""
from __future__ import annotations

import argparse
import gc
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree (which may be read-only), bytecode caches included

TOL = 1.0e-10
METRIC = "wilson_mg_time_to_solution_1e-10"
UNIT = "ms"


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons during the timed region (the B200_PROFILING.md clocks line), read through NVML
    in-process: forking nvidia-smi from a process that holds a 45 GB CUDA context perturbs the launch thread."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # NVML indices follow CUDA_VISIBLE_DEVICES-less enumeration; map through the UUID of the torch device
            import torch
            uuid = str(torch.cuda.get_device_properties(index).uuid)
            for i in range(pynvml.nvmlDeviceGetCount()):
                h = pynvml.nvmlDeviceGetHandleByIndex(i)
                u = pynvml.nvmlDeviceGetUUID(h)
                u = u.decode() if isinstance(u, bytes) else u
                if uuid in u:
                    self.h = h
            if self.h is None:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None or self.h is None:
            return
        nv = self.nv
        while not self._stop_evt.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, mx, rs))
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=3)
        sm = sorted(r[0] for r in self.rows)
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        reasons = sorted({n for r in self.rows for n, b in bits.items() if r[2] & b})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max((r[1] for r in self.rows), default=None),
                "reasons": reasons, "samples": len(self.rows)}


def workload_params(mg2d, L, mass, **kw):
    nlevels = max(1, int(round(math.log(L / 16, 4))))
    return mg2d.make_params(L, mass, nlevels=nlevels, block=4, n_null=8, n_smooth=4, n_pre=0, n_post=post_sweeps(nlevels),
                            smoother="rbgs", null_iters=100, tol=TOL, max_iters=500, **kw)


def post_sweeps(nlevels):
    """Cycle shape measured fastest at 4096^2 (tools/tune.py): no pre-smoothing, 4 red-black sweeps on the fine lattice,
    2 on level 1 (whose operator dominates the traffic of a cycle), 6 on level 2, 4 on the small levels below (round 2: with
    8/8/8 there the iteration count is the same 21 -- the coarse levels were over-smoothed; 5 or fewer on level 2, 2 on the
    small ones, or 3 on the fine lattice cost an iteration or leave no margin to the tolerance)."""
    return ([4, 2, 6] + [4] * nlevels)[:nlevels + 1]


# ---------------------------------------------------------------------------------------------------------
CPU_SAMPLE_L = int(os.environ.get("MG2D_CPU_SAMPLE_L", "512"))   # lattice of the bounded CPU sample of the reference arm


def oracle_setup(L_cpu: int):
    """Hierarchy of the numpy oracle on a bounded sample of the workload: same shape (block 4, 16 coarse dof,
    rbgs post-only 4/2/8.., GCR(8)), lattice L_cpu.  Not timed."""
    import numpy as np
    from oracle import mg_oracle as O
    nlevels = max(1, int(round(math.log(L_cpu / 16, 4))))
    th = O.gauge_quenched_phases(L_cpu, 6.0, sweeps=20, seed=1234)
    U = O.gauge_from_phases(th)
    po = O.Params(L=L_cpu, num_iters=4, n_pre=0, n_post=post_sweeps(nlevels), block=4, m=-0.05, nlevels=nlevels,
                  stencil="wilson", smoother="rbgs", n_dof_scale=16, null_iters=20)
    LVL, NTL = O.build_reference_problem(po, U)
    O.compute_near_null(LVL, NTL, po, 1)
    b = np.zeros((L_cpu * L_cpu, 2), dtype=complex)
    b[L_cpu // 2 + (L_cpu // 2) * L_cpu, 0] = 1.0
    from oracle import c_port
    return {"levels": c_port.levels_from_oracle(LVL, po), "size": po.size, "n_dof": po.n_dof, "pre": po.pre, "post": po.post,
            "b": b, "L": L_cpu, "how": f"hierarchy of a {L_cpu}^2 lattice (m = -0.05) set up by the numpy oracle"}


def gpu_export_setup(mg2d, critical, L_cpu: int, delta: float):
    """cpu_baseline of the GPU arm: a near-critical L_cpu^2 hierarchy of the workload's shape built by the GPU setup and
    exported to host arrays in the reference's layouts (D[s][k][i][j], dense P) for the C port.  Not timed."""
    import numpy as np
    import torch
    U = mg2d.gauge.quenched_links_device(L_cpu, 6.0, sweeps=60, seed=1234)
    mcrit, _ = critical.estimate_critical_mass(U, lambda m: workload_params(mg2d, L_cpu, m), iters=4, refine=3)
    p = workload_params(mg2d, L_cpu, mcrit + delta, matrix_free=False)
    mg = mg2d.setup(U, p, init="device")
    levels = []
    for l, lv in enumerate(mg.LVL):
        levels.append({"D": mg2d.D_to_reference_layout(lv.D).cpu().numpy(),
                       "P": lv.phi_null.cpu().numpy() if l < p.nlevels else None})
    b = np.zeros((L_cpu * L_cpu, 2), dtype=complex)
    b[L_cpu // 2 + (L_cpu // 2) * L_cpu, 0] = 1.0
    # the GPU's own solve of this problem, for the iteration count the CPU solve is expected to reproduce
    rhs = torch.as_tensor(b).cuda()
    _, info = mg2d.solve(mg, rhs=rhs, tol=TOL, outer="gcr", restart=8)
    out = {"levels": levels, "size": p.size, "n_dof": p.n_dof, "pre": p.pre, "post": p.post, "b": b, "L": L_cpu,
           "gpu_iters": info["iters"],
           "how": f"hierarchy of a near-critical {L_cpu}^2 lattice (m_crit {mcrit:+.5f} + {delta:g}) built by the GPU setup and exported to the host"}
    mg.close()
    return out


def cpu_solves(st, budget_s: float):
    """Full solves (to 1e-10) of the sample problem with the C + OpenMP port of the solve loop on every host processor,
    repeated until `budget_s` seconds of CPU work are accumulated (at least one).  Returns dict(seconds per solve, iters,
    threads, reps, total seconds)."""
    from oracle import c_port
    c_port.build()
    tot_s, its, reps, threads = 0.0, [], 0, 0
    while reps == 0 or (tot_s < budget_s and reps < 200):
        _, info = c_port.gcr_solve_arrays(st["levels"], st["size"], st["n_dof"], st["pre"], st["post"], 4, st["b"], tol=TOL,
                                          max_iters=200, restart=8, threads=None)
        if not info["converged"]:
            raise RuntimeError("CPU port did not converge on the sample problem")
        tot_s += info["seconds"]
        its.append(info["iters"])
        threads = info["threads"]
        reps += 1
    return {"s_per_solve": tot_s / reps, "iters": its[-1], "threads": threads, "reps": reps, "total_s": tot_s}


def run_reference_arm(args):
    """--impl reference: the CPU path (oracle port, see module docstring) on the box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    L = args.L
    t0 = time.perf_counter()
    st = oracle_setup(CPU_SAMPLE_L)
    t_setup = time.perf_counter() - t0
    scale = (L / st["L"]) ** 2
    for _ in range(min(args.warmup, 2)):
        cpu_solves(st, 0.0)
    vals, walls, res = [], [], None
    for _ in range(args.steps):
        t0 = time.perf_counter()
        res = cpu_solves(st, 0.0)                 # one full solve per step
        walls.append((time.perf_counter() - t0) * 1e3)
        vals.append(res["s_per_solve"] * 1e3 * scale)
    v = sum(vals) / len(vals)
    sample = (f"C+OpenMP port (oracle/c_port) on {res['threads']} OpenMP threads (set explicitly): one full solve to {TOL:g} per step "
              f"({res['iters']} iterations, the count the CPU solve itself needs) on the {st['how']} with the workload's hierarchy shape "
              f"(block 4, 16 coarse dof, red-black post-smoothing 4/2/8.., FGCR(8)); oracle setup {t_setup:.0f} s not timed; "
              f"value = measured solve time x {scale:g} sites ({st['L']}^2 -> {L}^2, extrapolated); ms_per_step = measured wall time of a step")
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sum(walls) / len(walls), "higher_is_better": False, "scaling": "strong", "vs_baseline": None,
            "dtype": "c128", "data": "synthetic",
            "config": {"workload": f"wilson{L}_adaptive_mg_near_critical", "L": L, "tol": TOL, "iters": res["iters"],
                       "sample_L": st["L"], "extrapolated": True, "site_scale": scale},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": res["threads"], "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def reference_binary_config2(mg2d=None):
    """BASELINE configs[1] (2D U(1) Wilson 64x64, adaptive 3-level MG, the reference's Gauss-Seidel smoother, fp64) run by
    the reference's OWN program -- the unmodified S6 source compiled against oracle/eigen_shim (oracle/_ref/s6_mgrid_ntl),
    wall time of the whole process (setup, 500-sweep near-null generation, solve, its per-iteration text output) -- and by
    this package on the same links with the same algorithm (exact lexicographic GS, stationary cycle, tol 1e-13).
    Returns None when the binary is not present."""
    import re
    import subprocess
    import tempfile
    import numpy as np
    from oracle import mg_oracle as O
    exe = os.path.join(ROOT, "oracle", "_ref", "s6_mgrid_ntl")
    if not os.path.exists(exe):
        return None
    L, m, nl = 64, -0.01, 2
    theta = O.gauge_quenched_phases(L, 32.0, sweeps=30, seed=1234)
    with tempfile.TemporaryDirectory() as d:
        os.makedirs(os.path.join(d, "run"))
        os.makedirs(os.path.join(d, "gauge_config_files"))
        O.write_phase_file(os.path.join(d, "gauge_config_files", f"phase_{L}_b32.0.dat"), theta, L)
        t0 = time.perf_counter()
        out = subprocess.run([exe, str(L), "3", "2", "1", repr(m), str(nl), "0", "1"], cwd=os.path.join(d, "run"),
                             capture_output=True, text=True, timeout=900).stdout
        t_ref = time.perf_counter() - t0
    it_ref = int(re.search(r"Ans (\d+)", out).group(1))
    res = {"config": "wilson64_adaptive_3level_gs (BASELINE configs[1]): L=64 m=-0.01 beta=32 block 2, 3 GS sweeps, tol 1e-13",
           "reference_binary_s": t_ref, "reference_iters": it_ref, "cores": 1,
           "note": "reference = unmodified S6 source + oracle/eigen_shim (Eigen absent); wall time of the whole program"}
    if mg2d is not None:
        import torch
        U = torch.as_tensor(O.gauge_from_phases(theta)).cuda()
        p = mg2d.make_params(L, m, nlevels=nl, block=2, n_smooth=3, smoother="gs")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        mg = mg2d.setup(U, p, init="reference")
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        x, info = mg2d.solve(mg)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        res.update({"gpu_setup_s": t1 - t0, "gpu_solve_s": t2 - t1, "gpu_iters": info["iters"],
                    "gpu_final_residual": info["resnorms"][-1], "iters_identical": info["iters"] == it_ref})
        mg.close()
    return res


# ---------------------------------------------------------------------------------------------------------
def time_kernel(fn, reps, flush=None):
    import torch
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tot = 0.0
    for _ in range(reps):
        if flush is not None:
            flush.add_(1.0)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / reps


DUMP_WINDOW = 256            # side of the block of sites around the point source stored in full
DUMP_SAMPLE = 1 << 19        # sites of the fixed, seeded sample of the rest of the lattice
DUMP_SEED = 20240601


def dump_outputs(out_dir: str, x, info: dict, L: int):
    """--dump-outputs: what the timed solve returned in its last step, as float64 .npy files, so that two builds can be
    compared output for output.  The solution x [L*L, 2] complex128 (537 MB at 4096^2) is stored as (re, im) pairs on the
    DUMP_WINDOW^2 sites around the point source (where it is large) and on a seeded sample of DUMP_SAMPLE sites (sorted site
    indices, site = x + L*y, in x_sample_site.npy); the residual history and the recomputed true residual come from info."""
    import numpy as np
    import torch
    w = min(L, DUMP_WINDOW)
    rows = (L // 2 - w // 2 + np.arange(w)) % L
    window = (rows[:, None] * L + rows[None, :]).reshape(-1)
    sample = np.sort(np.random.default_rng(DUMP_SEED).choice(L * L, size=min(L * L, DUMP_SAMPLE), replace=False))

    def pairs(sites):
        v = x[torch.as_tensor(sites, device=x.device)].cpu().numpy()
        return np.stack([v.real, v.imag], axis=-1).astype(np.float64)
    out = {"x_window": pairs(window).reshape(w, w, 2, 2), "x_sample": pairs(sample), "x_sample_site": sample.astype(np.float64),
           "resnorms": np.asarray(info["resnorms"], dtype=np.float64),
           "true_resnorm": np.asarray([info["true_resnorm"]], dtype=np.float64)}
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bind_to_gpu_numa_node(local: int):
    """Pin this process (and with it its first-touch / pinned host allocations) to the CPUs of the NUMA node the GPU hangs off:
    with 8 ranks copying their strips at the same time, host buffers on the wrong socket halve the copy bandwidth.
    Returns the node (or None when the topology cannot be read); never fatal."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else local
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(idx)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bdf = bus.lower()[-12:]                                   # 0000:xx:yy.z
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        orig = os.sched_getaffinity(0)
        allowed = cpus & orig
        if allowed:
            bind_to_gpu_numa_node.orig = orig
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--L", type=int, default=4096)
    ap.add_argument("--delta", type=float, default=1e-3, help="mass offset above the estimated critical mass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-step", action="store_true",
                    help="bracket ONE extra solve (+ one D-apply) with cudaProfilerStart/Stop for `ncu --profile-from-start off`; "
                         "numbers printed by such a run are not bench values")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed solve returned to DIR/<name>.npy (see dump_outputs; one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is supported for the GPU solve on one GPU")
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch
    import mg2d
    from importlib import import_module
    critical = import_module("2d_multigrid_b200.critical")
    dist_mod = import_module("2d_multigrid_b200.dist")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)      # before any pinned allocation: the e2e leg moves 2 x 537 MB through host memory
    comm = dist_mod.init(world, rank, local) if world > 1 else None
    L = args.L
    pk, pk_src = peaks()

    def log(msg):
        if rank == 0:
            print(f"# [{time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)

    # ---- inputs (not timed): links, critical mass, hierarchy ---------------------------------------------
    t0 = time.time()
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234, device=local)     # Metropolis + plaquette kernels (N1)
    plaq = mg2d.gauge.plaquette_device(U, L).real
    if rank == 0:
        print(f"# links {L}^2 beta=6 plaquette {plaq:.4f} ({time.time()-t0:.1f}s)", file=sys.stderr)
    t0 = time.time()
    if comm is None:
        mcrit, _ = critical.estimate_critical_mass(U, lambda m: workload_params(mg2d, L, m), iters=4, refine=3)
    else:
        mcrit = dist_mod.bcast_float(comm, critical.estimate_critical_mass(
            U, lambda m: workload_params(mg2d, L, m), iters=4, refine=3)[0] if rank == 0 else 0.0)
    mass = mcrit + args.delta
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    t_crit = time.time() - t0
    p = workload_params(mg2d, L, mass)
    # N > 1: rank 0 first solves the SAME problem on one GPU; the strip solve must need the same number of iterations
    # (the hierarchy is partition-invariant: counter-based near-null seeds keyed on the global site index)
    ref_n1 = None
    if comm is not None:
        t = torch.zeros(3, dtype=torch.float64, device=dev)
        if rank == 0:
            ref = mg2d.setup(U, p, init="device")
            rr = torch.zeros((L * L, 2), dtype=torch.complex128, device=dev)
            rr[L // 2 + (L // 2) * L, 0] = 1.0
            xr, ir = mg2d.solve(ref, rhs=rr, tol=TOL, outer="gcr", restart=8, use_graph=True, check_every=1)
            x_ref_strip = xr[:(L // world) * L].clone()          # rank 0's strip of the single-GPU solution
            x_ref_max = float(xr.abs().max())                    # (normalise by the GLOBAL peak: far from the source
                                                                 # the solution is below the 1e-10 solver tolerance)
            t[0], t[1] = ir["iters"], ir["true_resnorm"]
            ref.close()
            del ref, rr, xr
            gc.collect()
            torch.cuda.empty_cache()
        torch.distributed.broadcast(t, 0)
        ref_n1 = {"iters": int(t[0].item()), "true_resnorm": float(t[1].item())}
    t0 = time.time()
    mg = mg2d.setup(U, p, init="device") if comm is None else dist_mod.setup(U, p, comm)
    torch.cuda.synchronize()
    t_setup = time.time() - t0
    if rank == 0:
        print(f"# m_crit~{mcrit:.5f} ({t_crit:.1f}s)  mass {mass:.5f}  setup {t_setup:.2f}s levels {p.size} dof {p.n_dof}", file=sys.stderr)

    lv0 = mg.LVL[0]
    rhs_host = torch.zeros((L * L, 2), dtype=torch.complex128).pin_memory()
    rhs_host[L // 2 + (L // 2) * L, 0] = 1.0
    rhs = mg.scatter_field(rhs_host) if comm is not None else rhs_host.to(dev)
    x_host = torch.empty((L * L, 2), dtype=torch.complex128).pin_memory()

    def barrier():
        if comm is not None:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def one_solve():
        return mg2d.solve(mg, rhs=rhs, tol=TOL, outer="gcr", restart=8, use_graph=True, check_every=1)

    # ---- device-resident steps ------------------------------------------------------------------------
    log("warm-up solves")
    for _ in range(max(args.warmup, 3)):
        x, info = one_solve()
    barrier()
    log(f"timed solves (iters {info['iters']}, true residual {info.get('true_resnorm')})")
    if ref_n1 is not None:
        ref_n1["iters_match_n1"] = bool(info["iters"] == ref_n1["iters"])
        if rank == 0:
            ref_n1["x_rel_diff_vs_n1"] = float((x[:x_ref_strip.shape[0]] - x_ref_strip).abs().max() / x_ref_max)
            del x_ref_strip
    n0 = mg.launches
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        x, info = one_solve()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.steps
    clocks = sampler.stop()
    launches = mg.launches - n0
    if comm is not None:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    if args.dump_outputs:           # now: x is LVL[0].phi, which the legs below overwrite
        dump_outputs(args.dump_outputs, x, info, L)

    if args.profile_step:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        one_solve()
        tmp_a, tmp_b = lv0.new_field(), lv0.new_field()
        lv0.apply_D(tmp_b, tmp_a)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        del tmp_a, tmp_b

    log(f"c128 {ms:.1f} ms; mixed-precision leg")
    # ---- the same solve with the V-cycle preconditioner in complex64 (outer GCR / residual stay complex128) ----
    def mixed_solve():
        return mg2d.solve(mg, rhs=rhs, tol=TOL, outer="gcr", restart=8, use_graph=True, check_every=1, precond_dtype="complex64")
    for _ in range(3):
        xm, info_m = mixed_solve()
    barrier()
    e0.record()
    for _ in range(args.steps):
        xm, info_m = mixed_solve()
    e1.record()
    barrier()
    ms_mixed = e0.elapsed_time(e1) / args.steps
    if comm is not None:
        t = torch.tensor([ms_mixed], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_mixed = float(t.item())

    log(f"mixed {ms_mixed:.1f} ms; e2e leg")
    # ---- ... and with that copy's coarse operators stored in half precision (fp32 arithmetic) -------------------
    def half_solve():
        return mg2d.solve(mg, rhs=rhs, tol=TOL, outer="gcr", restart=8, use_graph=True, check_every=1, precond_dtype="complex64+half")
    for _ in range(3):
        xh, info_h = half_solve()
    barrier()
    e0.record()
    for _ in range(args.steps):
        xh, info_h = half_solve()
    e1.record()
    barrier()
    ms_half = e0.elapsed_time(e1) / args.steps
    if comm is not None:
        t = torch.tensor([ms_half], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms_half = float(t.item())
    log(f"c64+half {ms_half:.1f} ms ({info_h['iters']} iters, true residual {info_h.get('true_resnorm')})")

    # ---- end to end: host rhs -> H2D -> solve -> D2H solution -----------------------------------------------
    def e2e_solve():
        r = mg.scatter_field(rhs_host) if comm is not None else rhs_host.to(dev, non_blocking=True)
        xx, inf = mg2d.solve(mg, rhs=r, tol=TOL, outer="gcr", restart=8, use_graph=True, check_every=1)
        if comm is not None:
            mg.gather_field(xx, x_host)
        else:
            x_host.copy_(xx, non_blocking=True)
        torch.cuda.synchronize()
        return inf
    e2e_solve()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_solve()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    if comm is not None:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        e2e_ms = float(t.item())
    nbytes = L * L * 2 * 16
    # one more, instrumented pass (not part of any reported number): where does the end-to-end step spend its time?
    barrier()
    t0 = time.perf_counter()
    r_dev = mg.scatter_field(rhs_host) if comm is not None else rhs_host.to(dev, non_blocking=True)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    xx, _ = mg2d.solve(mg, rhs=r_dev, tol=TOL, outer="gcr", restart=8, use_graph=True, check_every=1)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    if comm is not None:
        mg.gather_field(xx, x_host)
    else:
        x_host.copy_(xx, non_blocking=True)
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    e2e_parts = {"h2d_ms": (t1 - t0) * 1e3, "solve_ms": (t2 - t1) * 1e3, "d2h_ms": (t3 - t2) * 1e3}
    log("e2e parts (rank 0, one extra pass): " + ", ".join(f"{k} {v:.2f}" for k, v in e2e_parts.items()))

    log("e2e done; kernel timings")
    # ---- per-kernel rooflines (every rank runs them: strip-level kernels exchange halos; rank 0 reports) -------
    flush = torch.zeros(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)   # 256 MiB > 126 MB L2
    hbm = float(pk["hbm_gbs"])
    kern = []
    a, b_ = lv0.new_field(), lv0.new_field()
    a.normal_()
    S0 = lv0.S            # local sites (strip)
    t_apply = time_kernel(lambda: lv0.apply_D(b_, a), 20, flush)
    kern.append(("wilson_march_kernel<double> (D-apply, matrix-free)", 96.0 * S0, t_apply))
    lv0.phi.copy_(a)
    t_rb0 = time_kernel(lambda: lv0.relax(2, smoother="rbgs"), 10, flush) / 2
    kern.append(("wilson_rb2_kernel<double> (one red-black GS sweep, both colours in one pass, level 0)", 128.0 * S0, t_rb0))
    if p.nlevels >= 1:
        l1 = mg.LVL[1]
        n1 = l1.n
        big = l1.S * n1 * n1 * 96 >= 2e8            # operator >> L2: no explicit flush needed
        t_rb1a = time_kernel(lambda: l1.relax(1, smoother="rbgs"), 10, None if big else flush)
        t_rb1b = time_kernel(lambda: l1.relax(3, smoother="rbgs"), 6, None if big else flush)
        t_rb1 = (t_rb1b - t_rb1a) / 2
        if l1.lr_rank and mg.lowrank:
            R1 = l1.lr_rank      # rank-R factors of the 4 hopping blocks: 2 * 4R * n numbers per site instead of 4 n^2
            kern.append((f"stencil_rb_lr_kernel<double,{n1},{R1},1,2> x2 (one red-black GS sweep on the rank-{R1} factors of the pre-multiplied "
                         f"hopping blocks, level 1)", (8 * R1 * n1 + 3 * n1) * 16.0 * l1.S, t_rb1))
            kern.append((f"stencil_rb_lr_kernel<double,{n1},{R1},1,1> x2 (first sweep of a relax call: also forms c = D0^-1 r, level 1)",
                         (8 * R1 * n1 + n1 * n1 + 4 * n1) * 16.0 * l1.S, t_rb1a))
        else:
            kern.append((f"stencil_rb_pm_kernel<double,{n1},1,2> x2 (one red-black GS sweep on pre-multiplied blocks, level 1)",
                         (4 * n1 * n1 + 3 * n1) * 16.0 * l1.S, t_rb1))
            kern.append((f"stencil_rb_pm_kernel<double,{n1},1,1> x2 (first sweep of a relax call: also forms c = D0^-1 r, level 1)",
                         (5 * n1 * n1 + 4 * n1) * 16.0 * l1.S, t_rb1a))
        c, d_ = l1.new_field(), l1.new_field()
        c.normal_()
        t_ap1 = time_kernel(lambda: l1.apply_D(d_, c), 10, flush if l1.S * n1 * n1 * 80 < 2e8 else None)
        kern.append((f"stencil_kernel<double,{n1}> (coarse D-apply, level 1)", (5 * n1 * n1 + 2 * n1) * 16.0 * l1.S, t_ap1))
        t_res = time_kernel(lambda: lv0.restriction(l1.r, a, 1), 10, flush)
        chiral = lv0.phi_null_c is not None          # compacted projector: nc x nf/2 per fine site
        pb = n1 * (1 if chiral else 2)
        rname = ("restrict_chiral_nf2_nc16_blk4_kernel<double>" if (chiral and n1 == 16 and lv0.block == 4)
                 else f"restrict{'_chiral' if chiral else ''}_kernel<double,2,{n1}>")
        kern.append((f"{rname} (level 0->1)", ((pb + 2) * 16.0 + n1 * 16.0 / 16) * S0, t_res))
        t_pro = time_kernel(lambda: lv0.prolongation(b_, l1.phi, 1), 10, flush)
        kern.append((f"prolong{'_chiral' if chiral else ''}_kernel<double,2,{n1}> (level 1->0, accumulate)", ((pb + 2 * 2) * 16.0 + n1 * 16.0 / 16) * S0, t_pro))
    barrier()
    if rank != 0:
        _finish(comm)
        return
    table = [{"kernel": k, "bytes": by, "ms": t, "gbs": by / t / 1e6, "frac": by / t / 1e6 / hbm} for k, by, t in kern]
    # share of one V-cycle (nu = 4 pre + 4 post sweeps per level) taken by the level-1 smoother, from these timings
    dom = table[2] if len(table) > 2 else table[0]      # level-1 smoother sweep: the largest share of a solve
    dapply = table[0]
    # dram bytes per launch from the committed ncu capture (profiles/traffic_L1024.json) apply to the L=1024 workload
    traffic = None
    traffic_file = os.path.join(ROOT, "profiles", f"traffic_L{L}.json")
    if os.path.exists(traffic_file):
        try:
            tj = {k.replace(" ", "").replace("<unnamed>::", ""): v for k, v in json.load(open(traffic_file)).items() if isinstance(v, (int, float))}
            want = dom["kernel"].split(" ")[0].replace(" ", "")
            traffic = tj.get(want)
            if traffic is None:      # ncu names carry the trailing template arguments (LINK flag ...): match on the prefix
                hits = [v for k, v in tj.items() if k.startswith(want.rstrip(">"))]
                traffic = hits[0] if hits else None
            if traffic is not None and " x2 " in dom["kernel"]:
                traffic *= 2          # the timed unit is a full sweep = two half-sweep launches
        except Exception:
            traffic = None

    # ---- setup on the scoreboard: wall time, device time per phase and level, and the roofline of its dominant kernel
    # (f_near_null, S6/level.h:177-249: null_iters relaxation sweeps of all near-null candidates, batched) ----------
    phases = mg.info.get("setup_phases", [])
    setup_block = {"value": t_setup, "unit": "s", "null_iters": p.null_iters, "phases": phases}
    if phases:
        top = max(phases, key=lambda q: q["near_null_ms"])
        lt = mg.LVL[top["level"]]
        nv = lt.nc // 2
        if top["level"] == 0:       # matrix-free two-colour sweep per vector: 128 B per site and sweep
            by = 128.0 * lt.S * nv * p.null_iters
            kname = "wilson_rb2_kernel<double> (matrix-free sweeps of the 8 near-null candidates, level 0)"
        elif lt.lr_rank and mg.lowrank:   # batched sweep on the rank-R factors: 4 vectors share one stream of them
            by = ((8 * lt.lr_rank * lt.n) * (nv // 4 if nv % 4 == 0 else nv) + 3 * lt.n * nv) * 16.0 * lt.S * p.null_iters
            kname = f"stencil_rb_lr_kernel<double,{lt.n},{lt.lr_rank},4,0> x2 (batched near-null relaxation on the low-rank factors, level {top['level']})"
        else:                       # batched sweep on the dense pre-multiplied blocks: 4 vectors share one stream of M
            by = ((4 * lt.n * lt.n) * (nv // 4 if nv % 4 == 0 else nv) + 3 * lt.n * nv) * 16.0 * lt.S * p.null_iters
            kname = f"stencil_rb_pm_kernel<double,{lt.n},4,0> x2 (batched near-null relaxation, level {top['level']})"
        setup_block["dominant"] = {"phase": f"near_null level {top['level']}", "kernel": kname, "ms": top["near_null_ms"], "bytes": by,
                                   "gbs": by / top["near_null_ms"] / 1e6, "frac": by / top["near_null_ms"] / 1e6 / hbm,
                                   "note": "whole phase (sweeps + renormalisations) over the algorithmic bytes of its sweeps"}

    # ---- CPU baseline (rank 0, N=1 only): bounded oracle sample, scaled ----------------------------------
    if getattr(bind_to_gpu_numa_node, "orig", None):       # the CPU arm gets every core of the host again
        os.sched_setaffinity(0, bind_to_gpu_numa_node.orig)
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        try:
            Lc = min(1024, L)
            stc = gpu_export_setup(mg2d, critical, Lc, args.delta)
            res = cpu_solves(stc, 10.0)
            scale = (L / Lc) ** 2
            cpu = {"value": res["s_per_solve"] * 1e3 * scale, "unit": UNIT, "cores": res["threads"], "kind": "port",
                   "measured_ms": res["s_per_solve"] * 1e3, "measured_L": Lc, "site_scale": scale,
                   "sample": (f"C+OpenMP port (oracle/c_port) on {res['threads']} OpenMP threads (set explicitly): {res['reps']} full solves to "
                              f"{TOL:g} ({res['iters']} iterations each; the GPU needs {stc['gpu_iters']} on the same problem), {res['total_s']:.1f} s of CPU "
                              f"work, on the {stc['how']}: {res['s_per_solve']*1e3:.0f} ms per solve MEASURED at {Lc}^2; value = that x {scale:g} sites "
                              f"({Lc}^2 -> {L}^2)")}
            del stc
        except Exception as e:      # the CPU leg must never break the bench line
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"unavailable: {type(e).__name__}: {e}"[:300]}
    config2 = None
    if not args.no_cpu_baseline and world == 1:
        try:
            config2 = reference_binary_config2(mg2d)
        except Exception as e:      # an extra, never allowed to break the bench line
            config2 = {"error": f"{type(e).__name__}: {e}"[:200]}

    line = {
        "metric": METRIC, "value": ms, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms, "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "c128",
        "data": "synthetic",
        "config": {"workload": f"wilson{L}_adaptive_mg_near_critical", "L": L, "beta": 6.0, "hbm_gb_in_use": round(torch.cuda.max_memory_allocated() / 1e9, 1), "plaquette": plaq, "mass": mass,
                   "m_crit_est": mcrit, "m_crit_quality": getattr(critical.estimate_critical_mass, "info", None), "delta": args.delta, "levels": p.size, "n_dof": p.n_dof, "block": 4, "n_null": 8,
                   "smoother": "rbgs, pre 0, post " + str(p.post), "outer": "fgcr(8)", "tol": TOL, "iters": info["iters"],
                   "executed_iters": info.get("executed_iters"), "n1_reference": ref_n1,
                   "iters_match_n1": (None if ref_n1 is None else ref_n1["iters_match_n1"]),
                   "final_true_residual": info.get("true_resnorm"), "converged": info["converged"],
                   "setup_s": t_setup, "mcrit_s": t_crit, "cache": "working set >> L2 (126 MB); kernel timings flush L2 with a 256 MiB write",
                   "parallelism": f"strip{world}", "numa_node_rank0": numa},
        "clocks": clocks,
        "e2e": {"value": e2e_ms, "unit": UNIT, "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes, "parts_rank0": e2e_parts},
        "gpu_launches": launches,
        "roofline": {"kernel": dom["kernel"], "bound": "hbm", "achieved": dom["gbs"], "peak": hbm, "unit": "GB/s",
                     "frac": dom["frac"], "traffic": traffic, "peak_source": pk_src},
        "dapply": {"kernel": dapply["kernel"], "bound": "hbm", "achieved": dapply["gbs"], "peak": hbm, "unit": "GB/s",
                   "frac": dapply["frac"], "bytes_per_site": 96, "us": dapply["ms"] * 1e3, "target_frac": 0.70},
        "mixed_precision": {"value": ms_mixed, "unit": UNIT, "iters": info_m["iters"], "final_true_residual": info_m.get("true_resnorm"),
                            "note": "same solve, V-cycle preconditioner on a complex64 copy of the hierarchy; outer FGCR, residual and the 1e-10 test in complex128"},
        "mixed_precision_half": {"value": ms_half, "unit": UNIT, "iters": info_h["iters"], "final_true_residual": info_h.get("true_resnorm"),
                                 "note": "as mixed_precision, with the coarse operators of the complex64 copy stored as __half2 (fp32 arithmetic)"},
        "kernels": table,
        "setup": setup_block,
        "cpu_baseline": cpu,
        "config2_vs_reference_binary": config2,
    }
    print(json.dumps(line), flush=True)
    _finish(comm)


def _finish(comm):
    """Leave without tearing NCCL down under live CUDA graphs that captured its kernels (that hangs): all ranks
    synchronise, flush and exit."""
    if comm is None:
        return
    import torch
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


if __name__ == "__main__":
    main()
