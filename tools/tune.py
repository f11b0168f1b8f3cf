"""Cycle-shape tuning on one GPU: pre/post smoothing counts per level, same hierarchy."""
import os, sys, time, math
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mg2d, bench
from importlib import import_module
critical = import_module("2d_multigrid_b200.critical")
torch.cuda.set_device(0); dev = torch.device("cuda", 0)
L = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234)
mcrit = float(os.environ["MG2D_MCRIT"]) if "MG2D_MCRIT" in os.environ else None
if mcrit is None:
    mcrit, _ = critical.estimate_critical_mass(U, lambda m: bench.workload_params(mg2d, L, m))
p = bench.workload_params(mg2d, L, mcrit + 1e-3)
mg = mg2d.setup(U, p, init="device")
rhs = torch.zeros((L * L, 2), dtype=torch.complex128, device=dev); rhs[L // 2 + (L // 2) * L, 0] = 1.0
nl = p.nlevels
def run(pre, post, mixed, restart=8):
    for m in [mg] + ([mg.info["single"]] if "single" in mg.info else []):
        m.p.pre, m.p.post = list(pre), list(post)
        m.info.pop("precond_graph", None); m.info.pop(("cycle_graph", m.p.mu), None)
    kw = dict(rhs=rhs, tol=1e-10, outer="gcr", restart=restart, use_graph=True, check_every=1, max_iters=120)
    if mixed: kw["precond_dtype"] = "complex64"
    x, info = mg2d.solve(mg, **kw)
    if mixed:   # the shadow was created with the default counts on first use: re-apply and re-run
        m = mg.info["single"]; m.p.pre, m.p.post = list(pre), list(post); m.info.pop("precond_graph", None)
        x, info = mg2d.solve(mg, **kw)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(3):
        x, info = mg2d.solve(mg, **kw)
    e1.record(); torch.cuda.synchronize(); return info, e0.elapsed_time(e1) / 3
def configs():
    z = [0] * (nl + 1)
    shapes = os.environ.get("MG2D_TUNE_SHAPES")
    shapes = ([[int(t) for t in sh.split(",")] for sh in shapes.split(";")] if shapes else
              [[4, 2, 8, 8, 8], [4, 2, 8, 4, 8], [4, 2, 8, 4, 4], [4, 2, 8, 8, 4], [4, 2, 6, 4, 4], [4, 2, 8, 6, 6], [3, 2, 8, 8, 8], [4, 3, 8, 8, 8]])
    for post in shapes:
        yield f"post {post[:nl + 1]}", z, post[:nl + 1]


for null_iters in [int(v) for v in os.environ.get("MG2D_TUNE_NULL", "100").split(",")]:
    if null_iters != p.null_iters:
        mg.close(); del mg
        import gc; gc.collect(); torch.cuda.empty_cache()
        p = bench.workload_params(mg2d, L, mcrit + 1e-3)
        p.null_iters = null_iters
        t0 = time.time()
        mg = mg2d.setup(U, p, init="device")
        torch.cuda.synchronize()
        print(f"# null_iters {null_iters}: setup {time.time() - t0:.2f} s", flush=True)
    for name, pre, post in configs():
        info, ms = run(pre, post, False)
        line = f"c128: {info['iters']:3d} it {ms:7.1f} ms conv {info['converged']} true {info['true_resnorm']:.1e}"
        print(f"null {null_iters:4d} {name:28s} | {line}", flush=True)
