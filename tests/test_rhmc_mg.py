"""Multigrid solves of the one-flavour RHMC poles: MG.set_twist, normal_solve and HMC(flavours=1, mg_poles=K).

CPU: the factorisation (D^dag D + sigma)^-1 = D_tm(mu)^-1 g5 D_tm(-mu)^-1 g5 on the oracle's dense Wilson and Wilson-clover
operators; the second-solve tolerance rule on dense solves perturbed to exactly their tolerances; refusals that need no device.
GPU: set_twist against a fresh setup at the new twist (operators, rebuilt buffers, FGCR iterations, solutions), the exact
return to twist 0 here and on the complex64 shadow, the shadow against make_single_precision, graphs kept per twist, refresh
after set_twist, normal_solve against dense and multi-shift solves, and HMC with mg_poles against mg_poles = 0."""
import math
from importlib import import_module

import numpy as np
import pytest
import torch

import mg2d
from mg2d import _lib
from oracle import mg_oracle as O
from test_twisted_mass import G5, _quenched, dense_tm

MGmod = import_module("2d_multigrid_b200.mg")
RH = import_module("2d_multigrid_b200.rhmc")


# ================================================================================================================
# CPU
# ================================================================================================================
@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_normal_factorisation_dense(csw):
    """(D^dag D + sigma)^-1 = D_tm(+mu)^-1 g5 D_tm(-mu)^-1 g5 with mu = sqrt(sigma), to 1e-12 (this pins the signs)."""
    L, m = 16, 0.1
    U = _quenched(L)
    D = dense_tm(U, L, m, csw, 0.0)
    g5 = G5(L)
    n = D.shape[0]
    for sigma in (0.0, 1e-5, 1e-3, 0.3):
        mu = math.sqrt(sigma)
        lhs = np.linalg.inv(D.conj().T @ D + sigma * np.eye(n))
        rhs = np.linalg.solve(dense_tm(U, L, m, csw, mu), g5 @ np.linalg.solve(dense_tm(U, L, m, csw, -mu), g5))
        assert np.max(np.abs(lhs - rhs)) <= 1e-12 * np.max(np.abs(lhs)), sigma


@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_second_solve_tolerance_bounds_the_normal_residual(csw):
    """Both solves perturbed to exactly their tolerances, the second one along the direction D_tm(mu)^dag amplifies most: the
    residual of the normal equations stays <= tol, and the norm bound holds."""
    L, m, tol = 16, 0.1, 1e-6
    U = _quenched(L)
    g5 = G5(L)
    rng = np.random.default_rng(7)
    p = mg2d.make_params(L, m, nlevels=1, block=4, csw=csw, smoother="rbgs")
    for sigma in (0.0, 1e-5, 0.05):
        mu = math.sqrt(sigma)
        Dm, Dp = dense_tm(U, L, m, csw, -mu), dense_tm(U, L, m, csw, mu)
        assert np.linalg.norm(Dp, 2) <= RH.operator_norm_bound(p, mu)
        b = rng.standard_normal(Dp.shape[0]) + 1j * rng.standard_normal(Dp.shape[0])
        g = g5 @ b
        r1 = rng.standard_normal(b.shape) + 1j * rng.standard_normal(b.shape)
        r1 *= 0.5 * tol * np.linalg.norm(g) / np.linalg.norm(r1)
        z = np.linalg.solve(Dm, g - r1)
        t2 = RH.second_solve_tol(tol, np.linalg.norm(b), np.linalg.norm(z), p, mu)
        u, _, _ = np.linalg.svd(Dp)
        r2 = u[:, 0] * t2 * np.linalg.norm(z)                   # |D_tm(mu)^dag r2| = ||D_tm|| |r2|
        x = np.linalg.solve(Dp, g5 @ z - r2)
        res = b - (Dp.conj().T @ Dp) @ x
        assert np.linalg.norm(res) <= tol * np.linalg.norm(b), sigma
        assert np.linalg.norm(res) >= 0.2 * tol * np.linalg.norm(b), sigma      # the rule is not loose by orders of magnitude


def _fake_mg(cls=None, **kw):
    m = object.__new__(cls or MGmod.MG)
    m.comm, m.info = None, {}
    m.p = mg2d.make_params(16, 0.1, **kw)
    return m


@pytest.mark.parametrize("kw,what", [(dict(nlevels=2, block=2, ntl=True, smoother="rbgs"), "non-telescoping"),
                                     (dict(nlevels=1, block=4, stencil="laplace"), "Wilson stencil")])
def test_set_twist_refusals(kw, what):
    with pytest.raises(mg2d.MG2DError, match=what):
        _fake_mg(**kw).set_twist(0.01)


def test_set_twist_refuses_strips_and_non_finite_mu():
    d = _fake_mg(import_module("2d_multigrid_b200.dist").DistMG, nlevels=1, block=4, smoother="rbgs")
    d.comm = object()
    with pytest.raises(mg2d.MG2DError, match="DistMG"):
        d.set_twist(0.01)
    for mu in (float("nan"), float("inf")):
        with pytest.raises(ValueError, match="finite"):
            _fake_mg(nlevels=1, block=4, smoother="rbgs").set_twist(mu)


def test_normal_solve_refusals():
    m = _fake_mg(nlevels=1, block=4, smoother="rbgs", mu=0.01)
    with pytest.raises(ValueError, match="twist 0"):
        mg2d.normal_solve(m, None, [0.1], 1e-10)


@pytest.mark.parametrize("kw,what", [(dict(mg_poles=2, flavours=2), "flavours=1"), (dict(mg_poles=-1, flavours=1), ">= 0"),
                                     (dict(mg_poles=1.5, flavours=1), "integer")])
def test_hmc_mg_poles_refusals(kw, what):
    p = mg2d.make_params(16, 0.1, nlevels=1, block=4, smoother="rbgs")
    with pytest.raises(ValueError, match=what):
        mg2d.HMC(p, np.zeros((256, 2)), 2.0, **kw)


def test_replace_params_keeps_per_level_blocks():
    P = import_module("2d_multigrid_b200.params")
    p = mg2d.make_params(256, 0.1, nlevels=3, block=[4, 2, 2], smoother="rbgs")
    q = P.replace_params(p, dtype="complex64", mu=0.01)
    assert q.blocks == [4, 2, 2] and q.size == [256, 64, 32, 16] and q.n_dof == p.n_dof and q.mu == 0.01
    p1 = mg2d.make_params(64, 0.1, nlevels=2, block=4, smoother="rbgs")
    q1 = P.replace_params(p1, mu=0.02)
    assert q1.size == p1.size and q1.blocks == p1.blocks and q1.block == p1.block


# ================================================================================================================
# GPU
# ================================================================================================================
MU = 0.0173


def _links(L, beta=6.0, sweeps=30):
    return mg2d.gauge.quenched_links_device(L, beta, sweeps=sweeps, seed=1234, return_phases=True)


def _p(L, block, nlevels, m=0.05, **kw):
    return mg2d.make_params(L, m, nlevels=nlevels, block=block, n_null=8, n_smooth=3, n_pre=0, smoother="rbgs", null_iters=40,
                            tol=1e-10, max_iters=400, **kw)


def _bufs(mg):
    """every twist-dependent buffer of the hierarchy (level, name) -> tensor"""
    out = {}
    for lv in mg.LVL:
        for name in ("D", "D0inv", "M", "F", "Dh", "D0inv_h"):
            t = getattr(lv, name)
            if t is not None:
                out[(lv.lvl, name)] = t
    return out


def _snap(mg):
    return {k: v.clone() for k, v in _bufs(mg).items()}


def _rhs(L, seed=3):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((L * L, 2), generator=g, dtype=torch.complex128, device="cuda")


def _solve(mg, b, **kw):
    x, info = mg2d.solve(mg, rhs=b, tol=1e-10, outer="gcr", restart=8, **kw)
    assert info["converged"], info["resnorms"][-3:]
    return x.clone(), info


def _tm_resid(mg, x, b, mu):
    """|b - D_tm(mu) x| / |b| through mg2d_wilson_tm_apply, independent of the hierarchy's p.mu"""
    lv = mg.LVL[0]
    out = torch.empty_like(x)
    lo, hi = lv._halo(x)
    mg.ctx.call("mg2d_wilson_tm_apply", out.data_ptr(), x.data_ptr(), lo, hi, lv.U.data_ptr(), lv.U_lo_ptr, None, b.data_ptr(),
                float(mg.p.mass), float(mu), lv.L, lv.Ly, _lib.MODE_RESID, _lib.C128, None, torch.cuda.current_stream().cuda_stream)
    return float(torch.linalg.vector_norm(out) / torch.linalg.vector_norm(b))


def _compare_to_fresh(mg, fresh, b):
    """D to 1e-12 max|D|; D0^-1, M, F to 1e-10 of their largest entry (one inversion of 16 x 16 blocks whose inputs differ by
    rounding); FGCR iterations identical and solutions within 1e-8."""
    x0, i0 = _solve(fresh, b)
    x1, i1 = _solve(mg, b)
    A, B = _bufs(mg), _bufs(fresh)
    for key in [k for k in B if k[1] in ("D", "D0inv", "M", "F")]:
        assert key in A, key
        tol = 1e-12 if key[1] == "D" else 1e-10
        assert float((A[key] - B[key]).abs().max()) <= tol * float(B[key].abs().max()), key
    assert i1["iters"] == i0["iters"], (i1["iters"], i0["iters"])
    assert float(torch.linalg.vector_norm(x1 - x0)) <= 1e-8 * float(torch.linalg.vector_norm(x0))


def _shadow_equals_fresh_single(mg):
    sh = mg.info["single"]
    fr = MGmod.make_single_precision(mg)
    for l32, f32 in zip(sh.LVL, fr.LVL):
        if l32.D0inv is not None:
            f32._ensure_D0inv()
        if l32.M is not None:
            f32._ensure_M()
        if l32.Dh is not None:
            f32.make_half_blocks()
    A, B = _bufs(sh), _bufs(fr)
    assert set(A) == set(B)
    for k in A:
        assert torch.equal(A[k], B[k]), k
    assert sh.p.mu == mg.p.mu
    fr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L,block,nlevels", [(128, 4, 2), (128, [4, 2, 2], 3)])
def test_set_twist_equals_fresh_setup_and_returns_exactly(L, block, nlevels):
    U, _ = _links(L)
    base = mg2d.setup(U, _p(L, block, nlevels), init="device")
    nulls = [lv.phi_null.clone() for lv in base.LVL[:-1]]
    base.close()
    mg = mg2d.setup(U, _p(L, block, nlevels), null_vectors=nulls)
    b = _rhs(L)
    _solve(mg, b)
    _solve(mg, b, precond_dtype="complex64+half")
    assert mg.LVL[1].F is not None and mg.LVL[1].lr_rank == 4             # low-rank first coarse level
    assert all(mg.LVL[l].M is not None for l in range(2, nlevels + 1))     # pre-multiplied deeper levels
    snap, snap32 = _snap(mg), _snap(mg.info["single"])
    for mu in (MU, -0.05):
        mg.set_twist(mu)
        assert mg.p.mu == mu and mg.p.size == mg.info["single"].p.size == [lv.L for lv in mg.LVL]
        _shadow_equals_fresh_single(mg)
        fresh = mg2d.setup(U, _p(L, block, nlevels, mu=mu), null_vectors=nulls)
        _compare_to_fresh(mg, fresh, b)
        fresh.close()
    mg.set_twist(0.3)
    mg.set_twist(0.0)
    for k, v in _bufs(mg).items():
        assert torch.equal(v, snap[k]), k
    for k, v in _bufs(mg.info["single"]).items():
        assert torch.equal(v, snap32[k]), k
    mg.close()


@pytest.mark.gpu
def test_make_single_precision_keeps_per_level_blocks():
    L = 128
    U, _ = _links(L)
    mg = mg2d.setup(U, _p(L, [4, 2, 2], 3), init="device")
    sh = MGmod.make_single_precision(mg)
    assert sh.p.size == mg.p.size == [128, 32, 16, 8] and sh.p.blocks == [4, 2, 2]
    assert [lv.L for lv in sh.LVL] == [lv.L for lv in mg.LVL]
    assert [lv.n for lv in sh.LVL] == [lv.n for lv in mg.LVL]
    _solve(mg, _rhs(L), precond_dtype="complex64")
    sh.close()
    mg.close()


@pytest.mark.gpu
def test_graphs_are_kept_per_twist():
    L, mu1, mu2 = 128, 0.02, -0.035
    U, _ = _links(L)
    mg = mg2d.setup(U, _p(L, 4, 2), init="device")
    b = _rhs(L)
    mg.set_twist(mu1)
    x1, _ = _solve(mg, b, use_graph=True, precond_dtype="complex64")
    assert _tm_resid(mg, x1, b, mu1) <= 1e-10
    mg.set_twist(mu2)
    x2, _ = _solve(mg, b, use_graph=True, precond_dtype="complex64")
    assert _tm_resid(mg, x2, b, mu2) <= 1e-10
    cap = mg.capture_launches
    mg.set_twist(mu1)
    x3, _ = _solve(mg, b, use_graph=True, precond_dtype="complex64")
    assert mg.capture_launches == cap
    assert torch.equal(x3, x1)
    mg.close()


@pytest.mark.gpu
def test_refresh_after_set_twist_keeps_set_twist_exact():
    L, block, nlevels = 128, 4, 2
    U, _ = _links(L)
    mg = mg2d.setup(U, _p(L, block, nlevels), init="device")
    mg.update_links(U)
    with pytest.raises(mg2d.MG2DError, match="refresh"):      # the kept factors must come from the links of the coarse levels
        mg.set_twist(0.02)
    mg.refresh(0)
    mg.set_twist(0.02)
    mg.refresh(0)                                             # rebuilt at twist 0.02, the state re-taken there
    assert mg.p.mu == 0.02 and mg.info["twist"]["mu_b"] == 0.02
    nulls = [lv.phi_null.clone() for lv in mg.LVL[:-1]]
    mg.set_twist(MU)
    fresh = mg2d.setup(U, _p(L, block, nlevels, mu=MU), null_vectors=nulls)
    _compare_to_fresh(mg, fresh, _rhs(L))
    fresh.close()
    mg.close()


@pytest.mark.gpu
def test_normal_solve_against_dense_32():
    L, m, tol = 32, 0.1, 1e-10
    U, th = _links(L, beta=2.0)
    mg = mg2d.setup(U, _p(L, 4, 1, m=m), init="device")
    b = _rhs(L)
    shifts = [1e-3, 0.0, 1e-5, 0.1]
    X, info = mg2d.normal_solve(mg, b, shifts, tol, use_graph=True)
    assert mg.p.mu == 0.0 and info["converged"] and len(info["iters"]) == len(shifts)
    assert max(info["true_residuals"]) <= tol, info["true_residuals"]
    assert info["twist_ms"] > 0.0
    D = dense_tm(np.exp(1j * th.cpu().numpy()), L, m, 0.0, 0.0)
    M = D.conj().T @ D
    ev = np.linalg.eigvalsh(M)
    bn = b.cpu().numpy().reshape(-1)
    for k, s in enumerate(shifts):
        x = np.linalg.solve(M + s * np.eye(M.shape[0]), bn)
        kappa = (ev[-1] + s) / (ev[0] + s)
        assert np.linalg.norm(X[k].cpu().numpy().reshape(-1) - x) <= tol * kappa * np.linalg.norm(x), s
    y = torch.empty_like(b)
    mg.LVL[0].apply_D(y, b)                                          # the hierarchy is D again
    chk = torch.as_tensor(D @ bn, device="cuda").reshape(y.shape)
    assert float((y - chk).abs().max()) <= 1e-12 * float(chk.abs().max())
    mg.close()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [256, 1024])
def test_normal_solve_against_multishift(L):
    """MD-like shifts: both solvers reach tol on the true residual, so |x_mg - x_ms| <= (r_mg + r_ms) |b| / (lambda_min + s),
    with lambda_min taken as half the smallest Ritz value of the multi-shift solve (Ritz values lie above lambda_min)."""
    m, tol = 0.05, 1e-10
    U, _ = _links(L, beta=2.0, sweeps=60)
    mg = mg2d.setup(U, _p(L, 4, 2 if L >= 256 else 1, m=m), init="device")
    b = _rhs(L)
    shifts = [1.78e-5, 2.08e-4, 9.38e-4, 3.54e-3]
    Xm, im = mg2d.multishift_cg(mg, b, shifts, tol, 20000)
    Xg, ig = mg2d.normal_solve(mg, b, shifts, tol, precond_dtype="complex64", use_graph=True)
    assert mg.p.mu == 0.0 and max(ig["true_residuals"]) <= tol, ig["true_residuals"]
    lam = 0.5 * im["ritz"][0]
    bn = float(torch.linalg.vector_norm(b))
    for k, s in enumerate(shifts):
        d = float(torch.linalg.vector_norm(Xg[k] - Xm[k]))
        assert d <= (ig["true_residuals"][k] + im["true_residuals"][k]) * bn / (lam + s), (s, d)
    mg.close()


def _hmc64(K, **kw):
    from test_rhmc import _params, _quenched_device
    L, beta, m = 64, 2.0, 0.1
    _, th = _quenched_device(L, sweeps=60, beta=beta)
    return mg2d.HMC(_params(L, m), th, beta, n_md=8, flavours=1, seed=3, md_tol=1e-12, accept_tol=1e-12, mg_poles=K, **kw)


@pytest.mark.gpu
def test_hmc_mg_poles_force_reversibility_and_dH():
    h0 = _hmc64(0)
    h3 = _hmc64(3, spectrum=h0.spectrum)
    a, b = h0.spectrum
    forces = []
    for h in (h0, h3):
        h.draw(0)
        h.P.zero_()
        h.force_step(1.0, [])
        forces.append(h.P.clone())
    # each X_k is within md_tol * kappa (kappa <= b / a) of the exact solve, and the force is bilinear in (X_k, D X_k)
    rel = float(torch.linalg.vector_norm(forces[1] - forces[0]) / torch.linalg.vector_norm(forces[0]))
    assert rel <= 4 * h0.md_tol * b / a, rel
    h3.draw(0)
    theta0 = h3.theta.clone()
    h3.leapfrog(1.0 / 8, 8, [])
    assert float((h3.theta - theta0).abs().max()) > 0.1
    h3.P.neg_()
    h3.leapfrog(1.0 / 8, 8, [])
    assert float((h3.theta - theta0).abs().max()) < 1e-9
    assert h3.mg.p.mu == 0.0
    h3.mg.close()
    h0.mg.close()
    o = []
    for K in (0, 3):
        h = _hmc64(K, spectrum=(a, b))
        o.append(h.trajectory())
        h.mg.close()
    assert abs(o[1]["dH"] - o[0]["dH"]) <= 1e-6, (o[0]["dH"], o[1]["dH"])
    assert o[0]["iters_md_mg"] == [] and len(o[1]["iters_md_mg"]) == 9 and all(len(f) == 3 for f in o[1]["iters_md_mg"])
    assert o[1]["times_ms"]["mg_solves"] > 0 and o[1]["times_ms"]["twist"] > 0
    assert o[1]["iters_md"] and min(o[1]["iters_md"]) > 0 and max(o[1]["iters_md"]) < max(o[0]["iters_md"])


@pytest.mark.gpu
def test_hmc_all_poles_on_multigrid_and_refresh():
    h = _hmc64(0)
    n = h.r_md.n
    spec = h.spectrum
    h.mg.close()
    with pytest.raises(ValueError, match="exceeds"):
        _hmc64(n + 1, spectrum=spec)
    h = _hmc64(n, spectrum=spec)
    out = [h.trajectory() for _ in range(2)]
    assert all(i == 0 for i in out[0]["iters_md"])
    assert out[1]["refreshed"] == out[0]["accepted"]
    h.mg.close()


@pytest.mark.gpu
def test_mg_poles_zero_makes_the_same_calls():
    """Traced eagerly (events cannot be recorded into a graph capture): the same entry points, launches and dH."""
    from test_rhmc import _params, _quenched_device
    _, th = _quenched_device(64, sweeps=60, beta=2.0)
    runs = []
    for kw in ({}, {"mg_poles": 0}):
        h = mg2d.HMC(_params(64, 0.1), th, 2.0, n_md=4, flavours=1, seed=3, spectrum=(1e-3, 30.0), use_graph=False, **kw)
        n0 = h.mg.launches
        _lib.trace_begin()
        o = h.trajectory()
        rep = _lib.trace_report()
        runs.append((h.mg.launches - n0, sorted(rep), o["dH"]))
        assert "twist" not in h.mg.info and not any("twist_set" in k or "pack_a" in k for k in rep)
        h.mg.close()
    assert runs[0] == runs[1]
