"""One-flavour Wilson RHMC: rational approximations, the multi-shift CG and the pole-summed fermion force.

CPU: the Remez approximations of x^(-1/2) and x^(+1/4) against a dense log grid and Zolotarev's closed form; a numpy
restatement of the multi-shift recurrences (csrc/rhmc.cu) against dense solves; the one-flavour action and force against
central finite differences on the oracle's Wilson operator; the refusal of a bad spectrum.
GPU: the two vector passes against an fp64 torch restatement, multishift_cg against dense solves and its true residuals, the
heat bath identity, a trajectory against the restatement, reversibility, dH scaling, the Creutz equality, the plaquette
against a reweighted pure-gauge stream, and the Ritz check of the accept step."""
import math
from importlib import import_module

import numpy as np
import pytest
import torch

import mg2d
from mg2d import _lib
from oracle import mg_oracle as O

R = import_module("2d_multigrid_b200.rational")


# ---- the restatement ------------------------------------------------------------------------------------------------
def dense_D(theta, L, m):
    p = O.Params(L=L, num_iters=1, block=2, m=m, nlevels=1)
    lv = O.Level()
    lv.compute_lvl0_matrix(np.exp(1j * theta), p)
    return O.dense_matrix(lv, L, 2)


def counter_gaussian(seed, stream, offset, n, variance=1.0):
    u = O.counter_uniform(seed, stream, 2 * offset, 2 * n)
    return math.sqrt(variance) * np.sqrt(-2.0 * np.log(1.0 - u[0::2])) * np.cos(2.0 * np.pi * u[1::2])


def im_plaq(U, L):
    xp, _, yp, _ = O.neighbours(L)
    return U[:, 0] * U[xp, 1] * np.conj(U[yp, 0]) * np.conj(U[:, 1])


def S_gauge(theta, L, beta):
    return beta * float(np.sum(1.0 - im_plaq(np.exp(1j * theta), L).real))


def apply_r(r, M, v):
    """r(M) v = alpha0 v + sum_k alpha_k (M + beta_k)^-1 v, dense."""
    n = M.shape[0]
    out = r.alpha0 * v
    for al, be in zip(r.alpha, r.beta):
        out = out + al * np.linalg.solve(M + be * np.eye(n), v)
    return out


def S_fermion1(theta, L, m, phi, r):
    D = dense_D(theta, L, m)
    return float(np.vdot(phi, apply_r(r, D.conj().T @ D, phi)).real)


def forces1(theta, L, beta, m, phi, r):
    """dS/dtheta of S_g + phi^dag r(M) phi: sum_k alpha_k times the mg2d_hmc_momentum bracket at X_k = (M + beta_k)^-1 phi,
    Y_k = D X_k, plus the gauge force."""
    U = np.exp(1j * theta)
    xp, xm, yp, ym = O.neighbours(L)
    ip = im_plaq(U, L).imag
    F = np.empty_like(theta)
    F[:, 0] = beta * (ip - ip[ym])
    F[:, 1] = beta * (ip[xm] - ip)
    D = dense_D(theta, L, m)
    M = D.conj().T @ D
    h = {("x", -1): lambda v: v[:, 0] - v[:, 1], ("x", 1): lambda v: v[:, 0] + v[:, 1],
         ("y", -1): lambda v: v[:, 0] + 1j * v[:, 1], ("y", 1): lambda v: v[:, 0] - 1j * v[:, 1]}
    for al, be in zip(r.alpha, r.beta):
        X = np.linalg.solve(M + be * np.eye(M.shape[0]), phi)
        Y = (D @ X).reshape(-1, 2)
        X = X.reshape(-1, 2)
        for mu, d, nb in ((0, "x", xp), (1, "y", yp)):
            F[:, mu] += al * (np.imag(U[:, mu] * np.conj(h[d, -1](Y)) * h[d, -1](X[nb]))
                              - np.imag(np.conj(U[:, mu]) * np.conj(h[d, 1](Y[nb])) * h[d, 1](X)))
    return F


def hamiltonian1(theta, P, L, beta, m, phi, r):
    return 0.5 * float(np.sum(P * P)) + S_gauge(theta, L, beta) + S_fermion1(theta, L, m, phi, r)


def leapfrog1(theta, P, eps, n_md, L, beta, m, phi, r):
    theta, P = theta.copy(), P.copy()
    P -= 0.5 * eps * forces1(theta, L, beta, m, phi, r)
    for i in range(n_md):
        theta += eps * P
        P -= (eps if i < n_md - 1 else 0.5 * eps) * forces1(theta, L, beta, m, phi, r)
    return theta, P


def multishift_numpy(M, phi, shifts, tol, max_iters=10000):
    """The recurrences of csrc/rhmc.cu (pass A: alpha, r, |r|^2 and the scalars; pass B: x_k, p_k) in numpy, shifts ascending."""
    N = len(shifts)
    s0 = shifts[0]
    sig = np.array(shifts) - s0
    r = phi.copy()
    P = np.tile(phi, (N, 1))
    X = np.zeros_like(P)
    rr, pp, b2 = [float(np.vdot(phi, phi).real)] * 3
    zeta, zeta_p = np.ones(N), np.ones(N)
    alpha_p, beta_p, nact_next = 1.0, 0.0, N
    for it in range(max_iters):
        t = M @ P[0]
        alpha = rr / (float(np.vdot(P[0], t).real) + s0 * pp)
        r = r - alpha * (t + s0 * P[0])
        rr_new = float(np.vdot(r, r).real)
        beta = rr_new / rr
        nact, nn = nact_next, 0
        a, b = np.zeros(N), np.zeros(N)
        for k in range(nact):
            zn = zeta[k] * zeta_p[k] * alpha_p / (alpha * beta_p * (zeta_p[k] - zeta[k]) + zeta_p[k] * alpha_p * (1 + sig[k] * alpha))
            a[k], b[k] = alpha * zn / zeta[k], beta * (zn / zeta[k]) ** 2
            zeta_p[k], zeta[k] = zeta[k], zn
            if zn * zn * rr_new > tol * tol * b2:
                nn = k + 1
        rr, alpha_p, beta_p, nact_next = rr_new, alpha, beta, nn
        for k in range(nact):
            X[k] += a[k] * P[k]
            P[k] = zeta[k] * r + b[k] * P[k]
        pp = float(np.vdot(P[0], P[0]).real)
        if nact_next == 0:
            return X, it + 1
    raise AssertionError("no convergence")


def quenched(L, beta=2.0, sweeps=30):
    return O.gauge_quenched_phases_counter(L, beta, sweeps=sweeps, seed=1234)


def spectrum_of(theta, L, m):
    D = dense_D(theta, L, m)
    ev = np.linalg.eigvalsh(D.conj().T @ D)
    return ev[0], ev[-1]


# ================================================================================================================
# CPU
# ================================================================================================================
@pytest.mark.parametrize("p", [-0.5, 0.25])
@pytest.mark.parametrize("ratio,tol", [(1e-2, 1e-12), (1e-2, 1e-6), (1e-5, 1e-6), (1e-8, 1e-6)])
def test_rational_error_on_log_grid(p, ratio, tol):
    b = 23.7
    r = mg2d.rational_approx(p, ratio * b, b, tol)
    x = (np.logspace(np.log10(ratio), 0, 40001) * b).astype(np.longdouble)
    err = float(np.max(np.abs(r(x) / x ** np.longdouble(p) - 1)))
    assert err <= r.error <= tol, (err, r.error, tol)
    assert min(r.beta) > 0 and len(set(r.beta)) == r.n
    if p == -0.5:
        assert min(r.alpha) > 0
    if r.n > 1:             # the smallest degree: one pole fewer misses the tolerance
        assert R._scaled(p, r.n - 1, ratio * b, b).error > tol


@pytest.mark.parametrize("n,ratio", [(6, 1e-2), (12, 1e-4), (16, 1e-8)])
def test_remez_equals_zolotarev(n, ratio):
    got = R._scaled(-0.5, n, ratio, 1.0).error
    want = R.zolotarev_error(n, ratio)
    assert abs(got - want) <= 0.01 * want, (got, want)


def test_multishift_restatement_matches_dense():
    L, m = 4, 0.05
    theta = quenched(L)
    D = dense_D(theta, L, m)
    M = D.conj().T @ D
    rng = np.random.default_rng(3)
    phi = rng.normal(size=2 * L * L) + 1j * rng.normal(size=2 * L * L)
    shifts = [0.003, 0.02, 0.4, 1.0, 7.5]
    X, it = multishift_numpy(M, phi, shifts, 1e-13)
    assert it > 5
    for k, s in enumerate(shifts):
        x = np.linalg.solve(M + s * np.eye(M.shape[0]), phi)
        assert np.linalg.norm(X[k] - x) <= 1e-10 * np.linalg.norm(x), k


@pytest.mark.parametrize("L", [4, 8])
def test_one_flavour_force_matches_finite_differences(L):
    beta, m = 2.0, 0.1
    theta = quenched(L)
    lo, hi = spectrum_of(theta, L, m)
    r = mg2d.rational_approx(-0.5, 0.5 * lo, 2 * hi, 1e-6)
    rng = np.random.default_rng(L)
    phi = (rng.normal(size=2 * L * L) + 1j * rng.normal(size=2 * L * L)) / math.sqrt(2)
    F = forces1(theta, L, beta, m, phi, r)
    h = 1e-5
    fd = np.empty_like(theta)
    for s in range(L * L):
        for mu in range(2):
            tp, tm = theta.copy(), theta.copy()
            tp[s, mu] += h
            tm[s, mu] -= h
            fd[s, mu] = (S_gauge(tp, L, beta) + S_fermion1(tp, L, m, phi, r) - S_gauge(tm, L, beta)
                         - S_fermion1(tm, L, m, phi, r)) / (2 * h)
    assert np.max(np.abs(F - fd)) <= 1e-7 * np.max(np.abs(fd))
    # phi^dag r_{-1/2}(M) phi is |D^-1 ...|: the action matches the exact one to the approximation's error
    D = dense_D(theta, L, m)
    w, V = np.linalg.eigh(D.conj().T @ D)
    exact = float(np.vdot(phi, V @ (w ** -0.5 * (V.conj().T @ phi))).real)
    assert abs(S_fermion1(theta, L, m, phi, r) - exact) <= 2 * r.error * exact


@pytest.mark.parametrize("spectrum", [(0.0, 1.0), (-1.0, 2.0), (2.0, 2.0), (3.0, 1.0), (float("nan"), 1.0)])
def test_bad_spectrum_refused(spectrum):
    p = mg2d.make_params(16, 0.1, nlevels=1, block=4, smoother="rbgs")
    with pytest.raises(ValueError, match="spectrum"):
        mg2d.HMC(p, np.zeros((256, 2)), 2.0, flavours=1, spectrum=spectrum)


def test_rational_refusals():
    for args in ((0.5, 1e-3, 1.0, 1e-6), (-0.5, 0.0, 1.0, 1e-6), (-0.5, 2.0, 1.0, 1e-6), (0.25, 1e-3, 1.0, 0.0)):
        with pytest.raises(ValueError):
            mg2d.rational_approx(*args)


# ================================================================================================================
# GPU
# ================================================================================================================
def _ctx():
    return _lib.Context(torch.cuda.current_device())


def _st():
    return torch.cuda.current_stream().cuda_stream


def _sc_init(N, sig, zeta, zeta_p, rr, pp, alpha_p, beta_p, nact_next, thresh, w, hist=8):
    sc = [0.0] * (_lib.MSC_SHIFTS + 6 * N)
    sc[_lib.MSC_RR], sc[_lib.MSC_PP], sc[_lib.MSC_ALPHA_PREV], sc[_lib.MSC_BETA_PREV] = rr, pp, alpha_p, beta_p
    sc[_lib.MSC_NACT_NEXT], sc[_lib.MSC_ITER], sc[_lib.MSC_THRESH] = nact_next, 3, thresh
    o = _lib.MSC_SHIFTS
    sc[o:o + N], sc[o + N:o + 2 * N], sc[o + 2 * N:o + 3 * N], sc[o + 5 * N:o + 6 * N] = sig, zeta, zeta_p, w
    return torch.tensor(sc + [0.0] * (2 * hist), dtype=torch.float64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("L", [6, 37, 1000, 4096])
@pytest.mark.parametrize("N", [1, 7, 16])
@pytest.mark.parametrize("acc", [False, True])
def test_passes_match_torch(L, N, acc):
    ctx = _ctx()
    g = torch.Generator(device="cuda").manual_seed(L * 100 + N)
    S = L * L
    cr = lambda *sh: torch.randn(sh, generator=g, dtype=torch.complex128, device="cuda")
    r, w, Pk = cr(S, 2), cr(S, 2), cr(N, S, 2)
    X = None if acc else cr(N, S, 2)
    y = cr(S, 2) if acc else None
    sigma0 = 0.0 if N == 7 else 0.0137
    sig = sorted(float(v) for v in np.random.default_rng(N).uniform(0, 3, N))
    sig[0] = 0.0
    zeta = [1.0 / (1 + 0.5 * k) for k in range(N)]
    zeta_p = [1.0 / (1 + 0.2 * k) for k in range(N)]
    wts = [0.3 + k for k in range(N)]
    rr, pp, alpha_p, beta_p = 1.3 * S, 0.9 * S, 0.71, 0.23
    dots = torch.tensor([0.8 * S, 0, 0, 0], dtype=torch.float64, device="cuda")
    # N_active = N; with N = 16 the last shifts fall below the threshold and pass B of the next call skips them
    sc = _sc_init(N, sig, zeta, zeta_p, rr, pp, alpha_p, beta_p, N, 0.0 if N != 16 else 0.1 * S, wts)
    alpha = rr / (0.8 * S + sigma0 * pp)
    r_want = r - alpha * (torch.stack([w[:, 0], -w[:, 1]], 1) + sigma0 * Pk[0])
    rr_new = float((r_want.abs() ** 2).sum())
    r0, X0, P0, y0 = r.clone(), None if X is None else X.clone(), Pk.clone(), None if y is None else y.clone()
    ctx.call("mg2d_msc_pass_a", r.data_ptr(), w.data_ptr(), Pk.data_ptr(), dots.data_ptr(), sc.data_ptr(), sigma0, N, S, _st())
    assert float((r - r_want).abs().max()) <= 1e-13 * float(r_want.abs().max())
    h = sc.tolist()
    assert abs(h[_lib.MSC_RR] - rr_new) <= 1e-12 * rr_new
    beta = rr_new / rr
    zn = [zeta[k] * zeta_p[k] * alpha_p / (alpha * beta_p * (zeta_p[k] - zeta[k]) + zeta_p[k] * alpha_p * (1 + sig[k] * alpha))
          for k in range(N)]
    a = [alpha * zn[k] / zeta[k] for k in range(N)]
    b = [beta * (zn[k] / zeta[k]) ** 2 for k in range(N)]
    o = _lib.MSC_SHIFTS
    np.testing.assert_allclose(h[o + N:o + 2 * N], zn, rtol=1e-12)
    np.testing.assert_allclose(h[o + 3 * N:o + 4 * N], a, rtol=1e-12)
    np.testing.assert_allclose(h[o + 4 * N:o + 5 * N], b, rtol=1e-12)
    assert h[_lib.MSC_NACT] == N and h[o + 6 * N + 6] == alpha and abs(h[o + 6 * N + 7] - beta) <= 1e-12 * beta
    want_next = max([k + 1 for k in range(N) if zn[k] ** 2 * rr_new > (0.0 if N != 16 else 0.1 * S)] + [0])
    assert h[_lib.MSC_NACT_NEXT] == want_next
    if N == 16:
        assert 0 < want_next < N
    ctx.call("mg2d_msc_pass_b", None if X is None else X.data_ptr(), Pk.data_ptr(), None if y is None else y.data_ptr(),
             r.data_ptr(), sc.data_ptr(), sigma0, N, S, _st())
    rt = r
    for k in range(N):
        pk = zn[k] * rt + b[k] * P0[k]
        assert float((Pk[k] - pk).abs().max()) <= 1e-13 * float(pk.abs().max()), k
        if not acc:
            xk = X0[k] + a[k] * P0[k]
            assert float((X[k] - xk).abs().max()) <= 1e-13 * float(xk.abs().max()), k
    if acc:
        y_want = y0 + sum(wts[k] * a[k] * P0[k] for k in range(N))
        assert float((y - y_want).abs().max()) <= 1e-13 * float(y_want.abs().max())
    if sigma0 != 0.0:
        pp_want = float((Pk[0].abs() ** 2).sum())
        assert abs(sc[_lib.MSC_PP].item() - pp_want) <= 1e-12 * pp_want
    # a second pass B skips the shifts pass A has dropped (NACT is only moved by pass A)
    ctx.call("mg2d_msc_pass_a", r.data_ptr(), w.data_ptr(), Pk.data_ptr(), dots.data_ptr(), sc.data_ptr(), sigma0, N, S, _st())
    nact = int(sc[_lib.MSC_NACT].item())
    assert nact == want_next
    keep = Pk[nact:].clone()
    ctx.call("mg2d_msc_pass_b", None if X is None else X.data_ptr(), Pk.data_ptr(), None if y is None else y.data_ptr(),
             r.data_ptr(), sc.data_ptr(), sigma0, N, S, _st())
    assert torch.equal(Pk[nact:], keep)


def _params(L, m=0.1, **kw):
    args = dict(nlevels=2 if L >= 64 else (1 if L >= 16 else 0), block=4, n_null=8, n_smooth=4, n_pre=0, smoother="rbgs",
                null_iters=40, tol=1e-10, max_iters=500)
    args.update(kw)
    return mg2d.make_params(L, m, **args)


def _quenched_device(L, sweeps=60, beta=2.0):
    return mg2d.gauge.quenched_links_device(L, beta, sweeps=sweeps, seed=1234, return_phases=True)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [8, 64, 1024])
def test_multishift_cg(L):
    m = 0.05
    U, th = _quenched_device(L)
    mg = mg2d.setup(U, _params(L, m), init="device")
    rhs = torch.randn((L * L, 2), dtype=torch.complex128, device="cuda")
    shifts = [0.7, 0.002, 0.05, 3.0, 0.01]                      # unsorted on purpose
    tol = 1e-10
    X, info = mg2d.multishift_cg(mg, rhs, shifts, tol, 20000)
    assert info["converged"]
    assert max(info["true_residuals"]) <= tol, info["true_residuals"]
    w = [0.3, 1.0, 0.5, 2.0, 0.25]
    y, info2 = mg2d.multishift_cg(mg, rhs, shifts, tol, 20000, weights=w)
    assert info2["iters"] == info["iters"]
    ysum = sum(wk * X[k] for k, wk in enumerate(w))
    assert float((y - ysum).abs().max()) <= 1e-12 * float(ysum.abs().max())
    lo, hi = info["ritz"]
    assert 0 < lo < hi <= (2 + m + 2 * math.sqrt(2)) ** 2
    if L == 8:
        D = dense_D(th.cpu().numpy(), L, m)
        M = D.conj().T @ D
        ev = np.linalg.eigvalsh(M)
        b = rhs.cpu().numpy().reshape(-1)
        for k, s in enumerate(shifts):
            x = np.linalg.solve(M + s * np.eye(M.shape[0]), b)
            assert np.linalg.norm(X[k].cpu().numpy().reshape(-1) - x) <= 10 * tol * np.linalg.norm(b) / (ev[0] + s)
        assert ev[0] * (1 - 1e-6) <= lo and hi <= ev[-1] * (1 + 1e-6)
        assert abs(lo - ev[0]) <= 1e-3 * ev[0]


@pytest.mark.gpu
def test_heatbath_identity_64():
    L = 64
    _, th = _quenched_device(L)
    h = mg2d.HMC(_params(L), th, 2.0, flavours=1, seed=4, md_tol=1e-10, accept_tol=1e-12)
    h.draw(0)
    y, _ = mg2d.multishift_cg(h.mg, h.phi, h.r_acc.beta, 1e-12, 100000, weights=h.r_acc.alpha)
    sf = h.r_acc.alpha0 * float((h.phi.abs() ** 2).sum()) + float(torch.vdot(h.phi.reshape(-1), y.reshape(-1)).real)
    e2 = float((h.eta.abs() ** 2).sum())
    assert abs(sf - e2) <= 1e-9 * e2, (sf, e2)
    a, b = h.spectrum
    assert b == (2.1 + 2 * math.sqrt(2)) ** 2 and 0 < a < b


@pytest.mark.gpu
def test_trajectory_matches_restatement():
    L, beta, m = 8, 2.0, 0.1
    th = quenched(L, beta, sweeps=20)
    lo, hi = spectrum_of(th, L, m)
    h = mg2d.HMC(_params(L, m), torch.as_tensor(th), beta, tau=0.5, n_md=5, flavours=1, seed=11, md_tol=1e-12,
                 accept_tol=1e-12, spectrum=(0.5 * lo, 1.5 * hi))
    S = L * L
    P = counter_gaussian(11, 0, 0, 2 * S).reshape(S, 2)
    eta = counter_gaussian(11, 1, 0, 4 * S, 0.5)
    eta = eta[0::2] + 1j * eta[1::2]
    D = dense_D(th, L, m)
    phi = apply_r(h.r_hb, D.conj().T @ D, eta)
    t1, P1 = leapfrog1(th, P, 0.1, 5, L, beta, m, phi, h.r_md)
    H0 = 0.5 * float(np.sum(P * P)) + S_gauge(th, L, beta) + float(np.vdot(eta, eta).real)
    H1 = 0.5 * float(np.sum(P1 * P1)) + S_gauge(t1, L, beta) + S_fermion1(t1, L, m, phi, h.r_acc)
    out = h.trajectory()
    assert abs(out["dH"] - (H1 - H0)) < 1e-8, (out["dH"], H1 - H0)
    assert out["accepted"] == (O.counter_uniform(11, 2, 0, 1)[0] < math.exp(min(0.0, -(H1 - H0))))
    got = h.theta.cpu().numpy()
    assert np.max(np.abs(got - (t1 if out["accepted"] else th))) < 1e-10
    assert out["poles"] == (h.r_md.n, h.r_acc.n) and len(out["iters_md"]) == 6 and out["iters_heatbath"] > 0


@pytest.mark.gpu
def test_reversibility_and_dH_scaling_64():
    L, beta, m = 64, 2.0, 0.1
    _, th = _quenched_device(L, sweeps=60, beta=beta)
    h = mg2d.HMC(_params(L, m), th, beta, n_md=8, flavours=1, seed=3, md_tol=1e-12, accept_tol=1e-12)
    spec = h.spectrum
    h.draw(0)
    theta0 = h.theta.clone()
    h.leapfrog(1.0 / 8, 8, [])
    assert float((h.theta - theta0).abs().max()) > 0.1
    h.P.neg_()
    h.leapfrog(1.0 / 8, 8, [])
    assert float((h.theta - theta0).abs().max()) < 1e-9
    dH = []
    for n in (8, 16, 32):
        d = []
        for k in range(4):
            hn = mg2d.HMC(_params(L, m), th, beta, tau=0.25, n_md=n, flavours=1, seed=3, md_tol=1e-12, accept_tol=1e-12,
                          spectrum=spec)
            hn.k = k
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
    h = mg2d.HMC(_params(L, m), th, beta, n_md=12, flavours=1, seed=5)
    out = [h.trajectory() for _ in range(40)]
    e = np.array([o["exp_minus_dH"] for o in out])
    assert abs(e.mean() - 1.0) < 4 * e.std(ddof=1) / math.sqrt(len(e)), e
    assert np.mean([o["accepted"] for o in out]) > 0.5
    assert all(len(o["iters_md"]) == 12 + 1 and not o["refreshed"] for o in out)


@pytest.mark.gpu
def test_plaquette_against_reweighted_pure_gauge_L4():
    """<plaquette> of flavours=1 against a flavours=0 stream reweighted by |det D| (dense determinant)."""
    L, beta, m = 4, 1.0, 0.05
    S = L * L
    bmax = (2 + m + 2 * math.sqrt(2)) ** 2
    spec = (1e-4, bmax)
    h1 = mg2d.HMC(_params(L, m), torch.zeros((S, 2), dtype=torch.float64), beta, n_md=8, flavours=1, seed=21, spectrum=spec)
    h0 = mg2d.HMC(_params(L, m), torch.zeros((S, 2), dtype=torch.float64), beta, n_md=8, flavours=0, seed=22)
    n_th, n = 50, 600
    p1 = [h1.trajectory()["plaquette"] for _ in range(n_th + n)][n_th:]
    pw, wts = [], []
    for i in range(n_th + n):
        o = h0.trajectory()
        if i >= n_th:
            th = h0.theta.cpu().numpy()
            ld = np.linalg.slogdet(dense_D(th, L, m))[1]
            pw.append(np.mean(np.cos(np.angle(im_plaq(np.exp(1j * th), L)))))
            wts.append(ld)
    lw = np.array(wts)
    wv = np.exp(lw - lw.max())
    pw = np.array(pw)
    nb = 20
    m1, e1 = _blocked(p1, nb)
    # blocked reweighted ratio: jackknife over blocks
    B = len(pw) // nb
    num = np.array([np.sum((pw * wv)[i * B:(i + 1) * B]) for i in range(nb)])
    den = np.array([np.sum(wv[i * B:(i + 1) * B]) for i in range(nb)])
    m0 = num.sum() / den.sum()
    jk = np.array([(num.sum() - num[i]) / (den.sum() - den[i]) for i in range(nb)])
    e0 = math.sqrt((nb - 1) / nb * np.sum((jk - jk.mean()) ** 2))
    assert abs(m1 - m0) < 4 * math.hypot(e1, e0), (m1, e1, m0, e0)


@pytest.mark.gpu
def test_spectrum_above_lambda_min_raises():
    L, beta, m = 8, 2.0, 0.1
    th = quenched(L, beta, sweeps=20)
    lo, hi = spectrum_of(th, L, m)
    h = mg2d.HMC(_params(L, m), torch.as_tensor(th), beta, tau=0.2, n_md=2, flavours=1, seed=2, spectrum=(3 * lo, 1.5 * hi))
    with pytest.raises(mg2d.MG2DError, match="Ritz"):
        h.trajectory()
