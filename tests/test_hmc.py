"""Two-flavour Wilson HMC: forces, leapfrog, the Gaussian generator and moving a built hierarchy to a new gauge field.

CPU: a dense fp64 restatement of S_g = beta sum_P (1 - cos theta_P), S_f = phi^dag (D^dag D)^-1 phi on the oracle's Wilson
operator and of both forces (the formula of csrc/hmc.cu) against central finite differences of the actions at every link;
its leapfrog is reversible and its dH scales as eps^2; a numpy mirror of mg2d_fill_gaussian on oracle.counter_uniform; the
refusals that need no device.
GPU: mg2d_fill_gaussian against the mirror, mg2d_hmc_momentum / mg2d_hmc_links against an fp64 torch restatement (ragged,
capped-grid and 4096^2 shapes), MG.refresh / MG.update_links against setup() and eager solves, and HMC trajectories
against the restatement, reversibility, dH scaling, the Creutz equality and the exact pure-gauge plaquette."""
import math

import numpy as np
import pytest
import torch

import mg2d
from mg2d import _lib
from oracle import mg_oracle as O


# ---- the restatement ------------------------------------------------------------------------------------------------
def counter_gaussian(seed, stream, offset, n, variance=1.0):
    """mg2d_fill_gaussian: sqrt(variance) sqrt(-2 ln(1 - u1)) cos(2 pi u2) on the counter numbers 2(offset+e), 2(offset+e)+1."""
    u = O.counter_uniform(seed, stream, 2 * offset, 2 * n)
    return math.sqrt(variance) * np.sqrt(-2.0 * np.log(1.0 - u[0::2])) * np.cos(2.0 * np.pi * u[1::2])


def dense_D(theta, L, m):
    p = O.Params(L=L, num_iters=1, block=2, m=m, nlevels=1)
    lv = O.Level()
    lv.compute_lvl0_matrix(np.exp(1j * theta), p)
    return O.dense_matrix(lv, L, 2)


def im_plaq(U, L):
    xp, _, yp, _ = O.neighbours(L)
    return U[:, 0] * U[xp, 1] * np.conj(U[yp, 0]) * np.conj(U[:, 1])


def S_gauge(theta, L, beta):
    return beta * float(np.sum(1.0 - im_plaq(np.exp(1j * theta), L).real))


def S_fermion(theta, L, m, phi):
    D = dense_D(theta, L, m)
    y = np.linalg.solve(D.conj().T, phi)
    return float(np.vdot(y, y).real)


def forces(theta, L, beta, m=None, phi=None):
    """dS/dtheta[s, mu] as csrc/hmc.cu computes it: gauge part from Im U_P, fermion part from X = (D^dag D)^-1 phi, Y = D X."""
    U = np.exp(1j * theta)
    xp, xm, yp, ym = O.neighbours(L)
    ip = im_plaq(U, L).imag
    F = np.empty_like(theta)
    F[:, 0] = beta * (ip - ip[ym])
    F[:, 1] = beta * (ip[xm] - ip)
    if phi is not None:
        D = dense_D(theta, L, m)
        Y = np.linalg.solve(D.conj().T, phi)
        X = np.linalg.solve(D, Y).reshape(-1, 2)
        Y = Y.reshape(-1, 2)
        h = {("x", -1): lambda v: v[:, 0] - v[:, 1], ("x", 1): lambda v: v[:, 0] + v[:, 1],
             ("y", -1): lambda v: v[:, 0] + 1j * v[:, 1], ("y", 1): lambda v: v[:, 0] - 1j * v[:, 1]}
        for mu, d, nb in ((0, "x", xp), (1, "y", yp)):
            F[:, mu] += (np.imag(U[:, mu] * np.conj(h[d, -1](Y)) * h[d, -1](X[nb]))
                         - np.imag(np.conj(U[:, mu]) * np.conj(h[d, 1](Y[nb])) * h[d, 1](X)))
    return F


def hamiltonian(theta, P, L, beta, m=None, phi=None):
    H = 0.5 * float(np.sum(P * P)) + S_gauge(theta, L, beta)
    return H + (S_fermion(theta, L, m, phi) if phi is not None else 0.0)


def leapfrog(theta, P, eps, n_md, L, beta, m=None, phi=None):
    """P(eps/2) [Q(eps) P(eps)]^(n_md-1) Q(eps) P(eps/2), as HMC.leapfrog."""
    theta, P = theta.copy(), P.copy()
    P -= 0.5 * eps * forces(theta, L, beta, m, phi)
    for i in range(n_md):
        theta += eps * P
        P -= (eps if i < n_md - 1 else 0.5 * eps) * forces(theta, L, beta, m, phi)
    return theta, P


def quenched(L, beta=6.0, sweeps=30):
    return O.gauge_quenched_phases_counter(L, beta, sweeps=sweeps, seed=1234)


# ================================================================================================================
# CPU
# ================================================================================================================
@pytest.mark.parametrize("L", [4, 8])
def test_forces_match_finite_differences(L):
    rng = np.random.default_rng(L)
    theta = quenched(L)
    beta, m = 2.0, 0.1
    phi = (rng.normal(size=2 * L * L) + 1j * rng.normal(size=2 * L * L)) / math.sqrt(2)
    F = forces(theta, L, beta, m, phi)
    Fg = forces(theta, L, beta)
    h = 1e-5
    fd, fdg = np.empty_like(theta), np.empty_like(theta)
    for s in range(L * L):
        for mu in range(2):
            tp, tm = theta.copy(), theta.copy()
            tp[s, mu] += h
            tm[s, mu] -= h
            fdg[s, mu] = (S_gauge(tp, L, beta) - S_gauge(tm, L, beta)) / (2 * h)
            fd[s, mu] = fdg[s, mu] + (S_fermion(tp, L, m, phi) - S_fermion(tm, L, m, phi)) / (2 * h)
    assert np.max(np.abs(Fg - fdg)) <= 1e-7 * np.max(np.abs(fdg))
    assert np.max(np.abs(F - fd)) <= 1e-7 * np.max(np.abs(fd))
    assert np.max(np.abs(F - Fg)) > 0.1 * np.max(np.abs(Fg))         # the fermion force is not negligible here


def test_leapfrog_reversible_and_dH_scales_as_eps2():
    L, beta, m = 4, 2.0, 0.1
    rng = np.random.default_rng(7)
    theta = quenched(L)
    P = rng.normal(size=theta.shape)
    phi = (rng.normal(size=2 * L * L) + 1j * rng.normal(size=2 * L * L)) / math.sqrt(2)
    t1, P1 = leapfrog(theta, P, 0.1, 10, L, beta, m, phi)
    t2, P2 = leapfrog(t1, -P1, 0.1, 10, L, beta, m, phi)
    assert np.max(np.abs(t2 - theta)) < 1e-12 and np.max(np.abs(P2 + P)) < 1e-12
    H0 = hamiltonian(theta, P, L, beta, m, phi)
    dH = []
    for n in (8, 16, 32):
        t, Pn = leapfrog(theta, P, 1.0 / n, n, L, beta, m, phi)
        dH.append(abs(hamiltonian(t, Pn, L, beta, m, phi) - H0))
    for a, b in zip(dH, dH[1:]):
        assert 3.0 < a / b < 5.0, dH


def test_gaussian_mirror():
    """The mirror's statistics, and its sub-ranges: a draw at offset o is element o of the whole draw."""
    z = counter_gaussian(5, 3, 0, 200000, 0.5)
    assert abs(z.mean()) < 5 * math.sqrt(0.5 / z.size)
    assert abs(z.var() - 0.5) < 5 * 0.5 * math.sqrt(2.0 / z.size)
    assert abs(np.mean(z ** 4) / 0.25 - 3.0) < 0.1                       # normal kurtosis
    np.testing.assert_array_equal(counter_gaussian(5, 3, 1234, 100, 0.5), z[1234:1334])
    assert np.all(np.isfinite(z))


@pytest.mark.parametrize("kw,what", [(dict(mu=0.01), "mu"), (dict(csw=1.0), "csw"), (dict(dtype="complex64"), "complex128"),
                                     (dict(smoother="gs"), "matrix-free"), (dict(ntl=True, nlevels=2), "non-telescoping")])
def test_hmc_refusals(kw, what):
    args = dict(nlevels=1, block=4, smoother="rbgs")
    args.update(kw)
    p = mg2d.make_params(16, 0.1, **args)
    with pytest.raises(ValueError, match=what):
        mg2d.HMC(p, np.zeros((256, 2)), 2.0)


def test_distributed_hierarchy_refused():
    from importlib import import_module
    d = object.__new__(import_module("2d_multigrid_b200.dist").DistMG)
    d.comm, d.p = object(), mg2d.make_params(16, 0.1, nlevels=1, block=4, smoother="rbgs")
    for call in (lambda: d.update_links(None), lambda: d.refresh(0)):
        with pytest.raises(mg2d.MG2DError, match="DistMG"):
            call()


# ================================================================================================================
# GPU
# ================================================================================================================
def _ctx():
    return _lib.Context(torch.cuda.current_device())


def _st():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.gpu
@pytest.mark.parametrize("n,offset,var", [(1, 0, 1.0), (1001, 17, 0.5), (3_000_001, 5, 1.0)])
def test_fill_gaussian_matches_mirror(n, offset, var):
    ctx = _ctx()
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    ctx.call("mg2d_fill_gaussian", out.data_ptr(), n, offset, 99, 7, var, _st())
    got = out.cpu().numpy()
    want = counter_gaussian(99, 7, offset, n, var)
    assert np.max(np.abs(got - want)) <= 1e-14 * max(1.0, np.max(np.abs(want)))


def _links_torch(theta):
    return torch.polar(torch.ones_like(theta), theta)


def _force_torch(U, L, beta, X=None, Y=None):
    """fp64 torch restatement of mg2d_hmc_momentum's F = F^g + F^f on [L, L, 2] (y, x, mu) tensors."""
    sh = lambda a, dx, dy: torch.roll(a, shifts=(-dy, -dx), dims=(0, 1))     # value at (x + dx, y + dy)
    ux, uy = U[..., 0], U[..., 1]
    ip = (ux * sh(uy, 1, 0) * sh(ux, 0, 1).conj() * uy.conj()).imag
    F = torch.stack([beta * (ip - sh(ip, 0, -1)), beta * (sh(ip, -1, 0) - ip)], dim=-1)
    if X is not None:
        hm = [lambda v: v[..., 0] - v[..., 1], lambda v: v[..., 0] + 1j * v[..., 1]]
        hp = [lambda v: v[..., 0] + v[..., 1], lambda v: v[..., 0] - 1j * v[..., 1]]
        for mu, (dx, dy) in enumerate(((1, 0), (0, 1))):
            u = U[..., mu]
            F[..., mu] += ((u * hm[mu](Y).conj() * hm[mu](sh(X, dx, dy))).imag
                           - (u.conj() * hp[mu](sh(Y, dx, dy)).conj() * hp[mu](X)).imag)
    return F


@pytest.mark.gpu
@pytest.mark.parametrize("L", [6, 37, 1000, 4096])
@pytest.mark.parametrize("fermions", [False, True])
def test_hmc_momentum_and_links_kernels(L, fermions):
    ctx = _ctx()
    g = torch.Generator(device="cuda").manual_seed(L)
    S = L * L
    theta = (torch.rand((S, 2), generator=g, dtype=torch.float64, device="cuda") * 2 - 1) * math.pi
    U = _links_torch(theta)
    P = torch.randn((S, 2), generator=g, dtype=torch.float64, device="cuda")
    X = Y = None
    if fermions:
        X = torch.randn((S, 2), generator=g, dtype=torch.complex128, device="cuda")
        Y = torch.randn((S, 2), generator=g, dtype=torch.complex128, device="cuda")
    beta, eps = 1.7, 0.03
    want = P - eps * _force_torch(U.view(L, L, 2), L, beta, None if X is None else X.view(L, L, 2),
                                  None if Y is None else Y.view(L, L, 2)).reshape(S, 2)
    got = P.clone()
    ctx.call("mg2d_hmc_momentum", got.data_ptr(), U.data_ptr(), None if X is None else X.data_ptr(),
             None if Y is None else Y.data_ptr(), beta, eps, L, _st())
    assert float((got - want).abs().max()) <= 1e-12 * float((want - P).abs().max())
    if L > 1000 or not fermions:
        # the link update: theta bit for bit as the fp64 restatement, U bit for bit as mg2d_phases_to_links of that theta
        th, U1, U32 = theta.clone(), torch.empty_like(U), torch.empty((S, 2), dtype=torch.complex64, device="cuda")
        ctx.call("mg2d_hmc_links", th.data_ptr(), got.data_ptr(), eps, U1.data_ptr(), U32.data_ptr(), 2 * S, _st())
        assert torch.equal(th, theta + eps * got)
        ref, ref32 = torch.empty_like(U), torch.empty_like(U32)
        ctx.call("mg2d_phases_to_links", ref.data_ptr(), th.data_ptr(), 2 * S, _lib.C128, _st())
        ctx.call("mg2d_phases_to_links", ref32.data_ptr(), th.data_ptr(), 2 * S, _lib.C64, _st())
        assert torch.equal(U1, ref) and torch.equal(U32, ref32)
        assert float((U1 - _links_torch(th)).abs().max()) < 1e-15
        ctx.call("mg2d_hmc_links", th.data_ptr(), got.data_ptr(), -eps, U1.data_ptr(), None, 2 * S, _st())
        assert float((th - theta).abs().max()) < 1e-14
    if L >= 1000:
        assert S > 2 * 148 * 8 * 256               # more sites than the capped grid (8 CTAs of 256 per SM) has threads


def _params(L, m=0.1, **kw):
    args = dict(nlevels=2 if L >= 64 else 1, block=4, n_null=8, n_smooth=4, n_pre=0, smoother="rbgs", null_iters=40, tol=1e-10,
                max_iters=500)
    args.update(kw)
    return mg2d.make_params(L, m, **args)


def _quenched_device(L, sweeps=60, beta=6.0):
    return mg2d.gauge.quenched_links_device(L, beta, sweeps=sweeps, seed=1234, return_phases=True)


@pytest.mark.gpu
def test_refresh0_equals_setup_with_current_vectors():
    L = 64
    p = _params(L)
    U1, th = _quenched_device(L)
    U2 = _links_torch(th + 0.05 * torch.randn(th.shape, dtype=torch.float64, device="cuda"))
    mg = mg2d.setup(U1, p, init="device")
    mg.update_links(U2)
    nv = [lv.phi_null.clone() for lv in mg.LVL[:p.nlevels]]
    mg.refresh(0)
    ref = mg2d.setup(U2.clone(), p, null_vectors=nv, init="device")
    for a, b in zip(mg.LVL, ref.LVL):
        for name in ("D", "phi_null", "phi_null_c", "F", "D0inv", "U"):
            x, y = getattr(a, name), getattr(b, name)
            assert (x is None) == (y is None), (a.lvl, name)
            if x is not None:
                assert torch.equal(x, y), (a.lvl, name)
    mg.refresh(8)           # warm-started relaxation: still a working hierarchy
    rhs = torch.randn((L * L, 2), dtype=torch.complex128, device="cuda")
    _, info = mg2d.solve(mg, rhs=rhs, tol=1e-10, outer="gcr", restart=8)
    assert info["converged"] and info["true_resnorm"] < 1e-9


@pytest.mark.gpu
@pytest.mark.parametrize("precond", [None, "complex64"])
def test_update_links_graph_replay_equals_eager(precond):
    L = 64
    p = _params(L)
    U1, th = _quenched_device(L)
    keep = U1.clone()
    mg = mg2d.setup(U1, p, init="device")
    rhs = torch.randn((L * L, 2), dtype=torch.complex128, device="cuda")
    kw = dict(tol=1e-10, outer="gcr", restart=8, check_every=1, precond_dtype=precond)
    mg.update_links(U1)
    mg2d.solve(mg, rhs=rhs, use_graph=True, **kw)           # captures the iteration graphs on the owned link tensor
    graphs = {k: dict(v) for k, v in mg.info.items() if isinstance(k, tuple) and k[0] == "iter_graphs"}
    U2 = _links_torch(th + 0.1 * torch.randn(th.shape, dtype=torch.float64, device="cuda"))
    mg.update_links(U2)
    n0 = mg.graph_launches
    xg, ig = mg2d.solve(mg, rhs=rhs, use_graph=True, **kw)
    xg = xg.clone()
    assert mg.graph_launches > n0
    for k, v in graphs.items():                              # replayed, not captured again
        assert all(mg.info[k][s] is g for s, g in v.items())
    xe, ie = mg2d.solve(mg, rhs=rhs, use_graph=False, **kw)
    assert ig["iters"] == ie["iters"] and torch.equal(xg, xe)
    assert ie["true_resnorm"] < 1e-9
    assert torch.equal(U1, keep)                             # the caller's tensor was never written


@pytest.mark.gpu
def test_trajectory_matches_restatement():
    L, beta, m = 16, 2.0, 0.1
    th = torch.as_tensor(quenched(L, sweeps=20))
    h = mg2d.HMC(_params(L, m), th, beta, tau=0.5, n_md=5, seed=11, md_tol=1e-13, accept_tol=1e-13)
    # the draws of trajectory 0 by the device generator, fed to the restatement
    S = L * L
    ctx = _ctx()
    P = torch.empty(2 * S, dtype=torch.float64, device="cuda")
    eta = torch.empty(4 * S, dtype=torch.float64, device="cuda")
    ctx.call("mg2d_fill_gaussian", P.data_ptr(), 2 * S, 0, 11, 0, 1.0, _st())
    ctx.call("mg2d_fill_gaussian", eta.data_ptr(), 4 * S, 0, 11, 1, 0.5, _st())
    P, eta = P.cpu().numpy().reshape(S, 2), eta.cpu().numpy()
    eta = eta[0::2] + 1j * eta[1::2]
    theta0 = th.numpy()
    phi = dense_D(theta0, L, m).conj().T @ eta
    t1, P1 = leapfrog(theta0, P, 0.1, 5, L, beta, m, phi)
    dH = hamiltonian(t1, P1, L, beta, m, phi) - hamiltonian(theta0, P, L, beta, m, phi)
    out = h.trajectory()
    assert abs(out["dH"] - dH) < 1e-8, (out["dH"], dH)
    u = O.counter_uniform(11, 2, 0, 1)[0]
    assert out["accepted"] == (u < math.exp(min(0.0, -dH)))
    got = h.theta.cpu().numpy()
    assert np.max(np.abs(got - (t1 if out["accepted"] else theta0))) < 1e-10


@pytest.mark.gpu
def test_reversibility_and_dH_scaling_64():
    L, beta, m = 64, 2.0, 0.1
    _, th = _quenched_device(L, sweeps=60, beta=beta)
    h = mg2d.HMC(_params(L, m), th, beta, n_md=8, seed=3, md_tol=1e-12, accept_tol=1e-12)
    h.draw(0)
    theta0 = h.theta.clone()
    h.leapfrog(1.0 / 8, 8, [])
    assert float((h.theta - theta0).abs().max()) > 0.1
    h.P.neg_()
    h.leapfrog(1.0 / 8, 8, [])
    assert float((h.theta - theta0).abs().max()) < 1e-9
    # rms of dH over four draws (trajectories k = 0..3, each from the same start): the eps^2 term of one draw is a sum of local
    # terms of both signs and can nearly cancel (draw 0 here: |dH| 0.0188, 0.0027, 0.0005, ratios 7.1 and 5.0, the same in the
    # fp64 restatement), while its mean square scales as eps^4
    dH = []
    for n in (8, 16, 32):
        d = []
        for k in range(4):
            hn = mg2d.HMC(_params(L, m), th, beta, tau=0.25, n_md=n, seed=3, md_tol=1e-12, accept_tol=1e-12)
            hn.k = k                        # draw of trajectory k, from the start configuration
            d.append(hn.trajectory()["dH"])
            hn.mg.close()
        dH.append(math.sqrt(np.mean(np.square(d))))
    for a, b in zip(dH, dH[1:]):
        assert 3.0 < a / b < 5.0, dH


def _blocked(x, nb):
    x = np.asarray(x)
    b = x[:len(x) // nb * nb].reshape(nb, -1).mean(axis=1)
    return b.mean(), b.std(ddof=1) / math.sqrt(nb)


@pytest.mark.gpu
def test_creutz_equality_32():
    L, beta, m = 32, 2.0, 0.2
    _, th = _quenched_device(L, sweeps=60, beta=beta)
    h = mg2d.HMC(_params(L, m), th, beta, n_md=16, seed=5)
    out = [h.trajectory() for _ in range(40)]
    e = np.array([o["exp_minus_dH"] for o in out])
    assert abs(e.mean() - 1.0) < 4 * e.std(ddof=1) / math.sqrt(len(e)), e
    assert np.mean([o["accepted"] for o in out]) > 0.5
    assert all(len(o["iters_md"]) == 2 * (16 + 1) for o in out)


@pytest.mark.gpu
def test_pure_gauge_plaquette_exact():
    from scipy.special import i0, i1
    L, beta = 32, 2.0
    h = mg2d.HMC(_params(L), torch.zeros((L * L, 2), dtype=torch.float64), beta, n_md=10, flavours=0, seed=9)
    plaq = [h.trajectory()["plaquette"] for _ in range(800)][100:]
    mean, err = _blocked(plaq, 20)
    assert abs(mean - i1(beta) / i0(beta)) < 4 * err, (mean, err, i1(beta) / i0(beta))


@pytest.mark.gpu
def test_update_refused_on_stored_and_clover():
    L = 16
    U, _ = _quenched_device(L, sweeps=5)
    for kw, what in ((dict(smoother="gs"), "stored"), (dict(csw=1.0), "clover")):
        mg = mg2d.setup(U.clone(), _params(L, **kw), init="device")
        for call in (lambda: mg.update_links(U), lambda: mg.refresh(0)):
            with pytest.raises(mg2d.MG2DError, match=what):
                call()
        mg.close()
