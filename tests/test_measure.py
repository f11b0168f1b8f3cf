"""Gauge-ensemble measurements: topological charge, Wilson loops, meson correlators with the PCAC mass, chiral condensate.

CPU: the restatements the GPU is held to -- the free-field propagator by FFT against the dense inverse of the oracle's Wilson
matrix, with the plateau values of m_pcac and pp pinned at 64^2; the contraction G (gamma5-hermiticity) against
-tr[G S(x,x0) G' S(x0,x)] with the backward propagator read from the dense inverse (Wilson, clover, twisted mass); the
geometric charge; the U(1)-noise condensate estimator against the dense trace.
GPU: the three kernels against fp64 restatements (up to 4096^2, bit-reproducible), the exact uniform-flux values and the
strong-coupling area law; meson_correlators and chiral_condensate against dense solves, the free field through the multigrid,
gauge invariance, translation covariance, and measurements on a hierarchy an HMC has moved in place."""
import math

import numpy as np
import pytest
import torch

import mg2d
from mg2d import _lib
from oracle import mg_oracle as O

SIG = [np.eye(2, dtype=complex), np.array([[0, 1], [1, 0]], complex), np.array([[0, -1j], [1j, 0]]),
       np.diag([1.0, -1.0]).astype(complex)]


# ---- restatements ---------------------------------------------------------------------------------------------------
def G_restate(S):
    """G[y, a, b] = sum_x tr[s_a S s_b s3 S^dag s3] for S[y, x, al, be] (numpy)."""
    Sd = np.conj(np.swapaxes(S, -1, -2))
    G = np.empty((S.shape[0], 4, 4), complex)
    for a in range(4):
        for b in range(4):
            G[:, a, b] = np.einsum("ij,yxjk,kl,lm,yxmn,ni->y", SIG[a], S, SIG[b], SIG[3], Sd, SIG[3])
    return G


def G_restate_torch(psi0, psi1, L):
    """The same on the device in fp64 from the two columns [L*L, 2]."""
    S = torch.stack([psi0.view(L, L, 2), psi1.view(L, L, 2)], dim=-1)          # [y, x, al, be]
    sig = [torch.as_tensor(s, device=S.device) for s in SIG]
    B = sig[3] @ S.conj().transpose(-1, -2) @ sig[3]
    G = torch.empty((L, 4, 4), dtype=torch.complex128, device=S.device)
    for a in range(4):
        A = sig[a] @ S
        for b in range(4):
            G[:, a, b] = torch.einsum("yxij,yxji->y", A @ sig[b], B)
    return G


def derived(G):
    pp = G[:, 3, 3].real
    ap = (1j * G[:, 1, 3]).real
    return pp, ap, (np.roll(ap, -1) - np.roll(ap, 1)) / (4 * pp)


def free_propagator_fft(L, m, sign=1.0, site=(0, 0)):
    """S[y, x] = D^-1(x, site) of the free Wilson operator, D(p) = 2 + m + sign sum_mu (cos p_mu - i s_mu sin p_mu) (sign +1:
    the hopping sign of wilson.cu and the oracle)."""
    p = 2 * np.pi * np.arange(L) / L
    px, py = np.meshgrid(p, p, indexing="xy")                                   # [y, x]
    c = lambda a: a[..., None, None]
    Dp = (2 + m) * SIG[0] + sign * (c(np.cos(px)) * SIG[0] - 1j * c(np.sin(px)) * SIG[1]
                                    + c(np.cos(py)) * SIG[0] - 1j * c(np.sin(py)) * SIG[2])
    S = np.fft.ifft2(np.linalg.inv(Dp), axes=(0, 1))
    return np.roll(S, (site[1], site[0]), axis=(0, 1))


def dense_D(U, L, m, csw=0.0, mu=0.0):
    """The oracle's Wilson matrix + clover (csw/8) sum Im U_P s3 + i mu s3 on the self blocks, site-major spin-minor."""
    lv = O.Level()
    lv.compute_lvl0_matrix(U, O.Params(L=L, num_iters=1, block=2, m=m, nlevels=1))
    xp, xm, yp, ym = O.neighbours(L)
    ip = np.imag(U[:, 0] * U[xp, 1] * np.conj(U[yp, 0]) * np.conj(U[:, 1]))
    f = (csw / 8.0) * (ip + ip[xm] + ip[ym] + ip[xm][ym])
    lv.D[:, 0, 0, 0] += f + 1j * mu
    lv.D[:, 0, 1, 1] -= f + 1j * mu
    return O.dense_matrix(lv, L, 2)


def columns(Dinv, L, site):
    s0 = site[0] + site[1] * L
    return Dinv[:, 2 * s0:2 * s0 + 2].reshape(L, L, 2, 2)                      # [y, x, al, be]


def charge_restate(U, L):
    xp, _, yp, _ = O.neighbours(L)
    return float(np.sum(np.angle(U[:, 0] * U[xp, 1] * np.conj(U[yp, 0]) * np.conj(U[:, 1])))) / (2 * np.pi)


def gauge_uniform_flux(L, Q):
    """Q flux quanta spread uniformly: theta_y(x, y) = 2 pi Q x / L^2, theta_x(L-1, y) = -2 pi Q y / L, other phases 0;
    every plaquette angle is 2 pi Q / L^2 (mod 2 pi)."""
    th = np.zeros((L, L, 2))
    th[:, :, 1] = 2.0 * np.pi * Q * np.arange(L)[None, :] / L ** 2
    th[:, L - 1, 0] = -2.0 * np.pi * Q * np.arange(L) / L
    return np.exp(1j * th.reshape(L * L, 2))


def noise_mirror(seed, k, S):
    """eta of chiral_condensate: e^{i alpha}, alpha = counter_uniform(seed, k) in [-pi, pi) per component."""
    return np.exp(1j * O.counter_uniform(seed, k, 0, 2 * S, -np.pi, np.pi))


def quenched(L, beta=6.0, sweeps=30):
    return O.gauge_from_phases(O.gauge_quenched_phases_counter(L, beta, sweeps=sweeps, seed=1234))


# ================================================================================================================
# CPU
# ================================================================================================================
@pytest.mark.parametrize("m", [0.1, -0.05])
def test_free_fft_restatement_equals_dense_inverse(m):
    L = 8
    Dinv = np.linalg.inv(dense_D(O.gauge_cold(L), L, m))
    for site in ((0, 0), (3, 5)):
        assert np.max(np.abs(free_propagator_fft(L, m, site=site) - columns(Dinv, L, site))) < 1e-13


def test_free_field_pinned_values():
    """m_pcac(12) and pp(t) at 64^2 from the FFT restatement; the other hopping sign ((-1)^{x+y} psi) gives the same."""
    L = 64
    want = {0.1: 0.09627, 0.05: 0.04900, 0.02: 0.01983, -0.02: -0.02021}
    for m, mp in want.items():
        for sign in (1.0, -1.0):
            G = G_restate(free_propagator_fft(L, m, sign))
            pp, ap, m_pcac = derived(G)
            assert abs(m_pcac[12] - mp) < 5e-6, (m, sign, m_pcac[12])
            assert np.all(pp > 0) and np.max(np.abs((1j * G[:, 1, 3]).imag)) < 1e-15
            if m == 0.05:
                np.testing.assert_allclose(pp[[1, 8, 16]], [0.13266, 0.013513, 0.0042989], rtol=4e-5)


@pytest.mark.parametrize("csw,mu", [(0.0, 0.0), (1.0, 0.0), (0.0, 0.05)])
def test_contraction_equals_direct_backward_propagator(csw, mu):
    """-G_ab = -sum_x tr[s_a S_u(x,x0) s_b S_d(x0,x)] with S_d = D(-mu)^-1 read from the dense inverse (no gamma5 trick)."""
    L, m, site = 6, 0.05, (2, 3)
    U = quenched(L)
    Su = np.linalg.inv(dense_D(U, L, m, csw, mu))
    Sd = np.linalg.inv(dense_D(U, L, m, csw, -mu))
    s0 = site[0] + site[1] * L
    fwd = columns(Su, L, site)                                                  # S_u(x, x0)
    bwd = Sd[2 * s0:2 * s0 + 2, :].reshape(2, L, L, 2).transpose(1, 2, 0, 3)   # S_d(x0, x) as [y, x, al, be]
    direct = np.empty((L, 4, 4), complex)
    for a in range(4):
        for b in range(4):
            direct[:, a, b] = np.einsum("ij,yxjk,kl,yxli->y", SIG[a], fwd, SIG[b], bwd)
    G = G_restate(fwd)
    assert np.max(np.abs(G - direct)) < 1e-13 * np.max(np.abs(G))
    assert np.max(np.abs(G)) > 0.1


def test_geometric_charge_restatement():
    rng = np.random.default_rng(3)
    for L in (4, 9, 16):
        th = rng.uniform(-np.pi, np.pi, (L * L, 2))
        q = charge_restate(np.exp(1j * th), L)
        assert abs(q - round(q)) < 1e-12
        assert abs(charge_restate(np.exp(-1j * th), L) + q) < 1e-12
    qs = [round(charge_restate(np.exp(1j * rng.uniform(-np.pi, np.pi, (64, 2))), 8)) for _ in range(50)]
    assert len(set(qs)) > 2                                                     # random phases visit several sectors
    for L, Q in ((8, 1), (16, -2), (16, 3), (24, 5)):
        assert abs(charge_restate(gauge_uniform_flux(L, Q), L) - Q) < 1e-12
        assert abs(charge_restate(np.conj(gauge_uniform_flux(L, Q)), L) + Q) < 1e-12


def test_condensate_estimator_unbiased():
    L, m, seed, n = 8, 0.1, 7, 400
    S = L * L
    Dinv = np.linalg.inv(dense_D(quenched(L), L, m))
    want = np.trace(Dinv) / S
    v = np.array([np.vdot(e, Dinv @ e) / S for e in (noise_mirror(seed, k, S) for k in range(n))])
    assert np.allclose(np.abs(noise_mirror(seed, 0, S)), 1.0)
    for part in (np.real, np.imag):
        err = part(v).std(ddof=1) / math.sqrt(n)
        assert abs(part(v).mean() - part(want)) < 5 * err + 1e-15, (part(v).mean(), part(want), err)


def test_distributed_hierarchy_refused():
    from importlib import import_module
    d = object.__new__(import_module("2d_multigrid_b200.dist").DistMG)
    d.comm, d.p = object(), mg2d.make_params(16, 0.1, nlevels=1, block=4, smoother="rbgs")
    for call in (lambda: mg2d.meson_correlators(d), lambda: mg2d.chiral_condensate(d, 1)):
        with pytest.raises(mg2d.MG2DError, match="DistMG"):
            call()


# ================================================================================================================
# GPU
# ================================================================================================================
def _ctx():
    return _lib.Context(torch.cuda.current_device())


def _st():
    return torch.cuda.current_stream().cuda_stream


def _rel(got, want):
    return float((got - want).abs().max()) / float(want.abs().max())


def _params(L, m=0.1, **kw):
    args = dict(nlevels=2 if L >= 64 else 1, block=4, n_null=8, n_smooth=4, n_pre=0, smoother="rbgs", null_iters=40, tol=1e-10,
                max_iters=500)
    args.update(kw)
    return mg2d.make_params(L, m, **args)


def _random_links(L, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    th = (torch.rand((L * L, 2), generator=g, dtype=torch.float64, device="cuda") * 2 - 1) * math.pi
    return torch.polar(torch.ones_like(th), th)


@pytest.fixture
def gpu_mem():
    torch.cuda.empty_cache()
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("L", [6, 37, 256, 4096])
def test_meson_contract_kernel(L, gpu_mem):
    ctx = _ctx()
    g = torch.Generator(device="cuda").manual_seed(L)
    psi0 = torch.randn((L * L, 2), generator=g, dtype=torch.complex128, device="cuda")
    psi1 = torch.randn((L * L, 2), generator=g, dtype=torch.complex128, device="cuda")
    outs = []
    for _ in range(2):
        out = torch.empty((L, 4, 4, 2), dtype=torch.float64, device="cuda")
        ctx.call("mg2d_meson_contract", psi0.data_ptr(), psi1.data_ptr(), L, out.data_ptr(), _st())
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    got = torch.view_as_complex(outs[0])
    want = G_restate_torch(psi0, psi1, L)
    assert _rel(got, want) < 1e-12
    if L <= 37:
        S = torch.stack([psi0.view(L, L, 2), psi1.view(L, L, 2)], dim=-1).cpu().numpy()
        assert np.max(np.abs(got.cpu().numpy() - G_restate(S))) < 1e-12 * float(want.abs().max())


@pytest.mark.gpu
@pytest.mark.parametrize("L", [4, 37, 256, 4096])
def test_topo_charge_kernel(L, gpu_mem):
    U = _random_links(L, 100 + L)
    q = mg2d.topological_charge(U, L)
    assert abs(q - round(q)) < 1e-9
    assert abs(q - charge_restate(U.cpu().numpy(), L)) < 1e-9
    assert mg2d.topological_charge(U, L) == q                                # bit-reproducible
    for Q in (-2, 1, 3):
        qf = mg2d.topological_charge(torch.as_tensor(gauge_uniform_flux(L, Q)).cuda(), L)
        assert abs(qf - Q) < 1e-9, (Q, qf)


def loops_brute(U, L, r_max, t_max):
    """W[T-1, R-1] = mean over bases of the four sides multiplied out link by link (fp64 torch, on U's device)."""
    ux, uy = U.view(L, L, 2)[..., 0], U.view(L, L, 2)[..., 1]
    at = lambda a, dx, dy: torch.roll(a, shifts=(-dy, -dx), dims=(0, 1))       # value at (x + dx, y + dy)
    H = [torch.ones_like(ux)]
    for i in range(r_max):
        H.append(H[-1] * at(ux, i, 0))
    V = [torch.ones_like(uy)]
    for j in range(t_max):
        V.append(V[-1] * at(uy, 0, j))
    W = torch.empty((t_max, r_max), dtype=torch.complex128, device=U.device)
    for T in range(1, t_max + 1):
        for R in range(1, r_max + 1):
            W[T - 1, R - 1] = (H[R] * at(V[T], R, 0) * at(H[R], 0, T).conj() * V[T].conj()).mean()
    return W.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("L,r_max,t_max", [(16, 15, 15), (37, 7, 12), (37, 32, 3), (256, 32, 32)])
def test_wilson_loops_kernel(L, r_max, t_max):
    U = _random_links(L, 7 * L) if L != 256 else mg2d.gauge.quenched_links_device(L, 6.0, sweeps=20, seed=5)
    W = mg2d.wilson_loops(U, L, r_max, t_max)
    want = loops_brute(U, L, r_max, t_max)
    assert np.max(np.abs(W - want)) < 1e-12, np.max(np.abs(W - want))
    assert np.array_equal(W, mg2d.wilson_loops(U, L, r_max, t_max))         # bit-reproducible
    assert abs(W[0, 0] - mg2d.gauge.plaquette_device(U, L)) < 1e-14


@pytest.mark.gpu
def test_wilson_loops_bounds_refused():
    U = _random_links(8, 1)
    for r, t in ((0, 1), (1, 0), (8, 1), (1, 8), (33, 1)):
        with pytest.raises(mg2d.MG2DError, match="r_max"):
            mg2d.wilson_loops(U, 8, r, t)
    U = _random_links(40, 1)
    with pytest.raises(mg2d.MG2DError, match="r_max"):
        mg2d.wilson_loops(U, 40, 33, 4)
    mg2d.wilson_loops(U, 40, 32, 32)


@pytest.mark.gpu
@pytest.mark.parametrize("L,Q", [(64, 3), (37, -2)])
def test_wilson_loops_uniform_flux(L, Q):
    U = torch.as_tensor(gauge_uniform_flux(L, Q)).cuda()
    W = mg2d.wilson_loops(U, L, 20, 20)
    R, T = np.meshgrid(np.arange(1, 21), np.arange(1, 21), indexing="xy")
    assert np.max(np.abs(W - np.exp(2j * np.pi * Q * R * T / L ** 2))) < 1e-12


@pytest.mark.gpu
def test_wilson_loops_area_law_metropolis():
    """Strong coupling in 2D U(1) is exact: <W(R,T)> = (I1(beta)/I0(beta))^{RT}.  One 1024^2 configuration at beta = 2."""
    from scipy.special import i0, i1
    L, beta = 1024, 2.0
    U = mg2d.gauge.quenched_links_device(L, beta, sweeps=200, seed=77)
    W = mg2d.wilson_loops(U, L, 9, 9)
    w = i1(beta) / i0(beta)
    for T in range(1, 10):
        for R in range(1, 10):
            if R * T <= 9:
                assert abs(W[T - 1, R - 1] - w ** (R * T)) <= 0.01, (R, T, W[T - 1, R - 1], w ** (R * T))


@pytest.mark.gpu
@pytest.mark.parametrize("csw,mu", [(0.0, 0.0), (1.0, 0.0), (0.0, 0.05)])
def test_meson_correlators_against_dense(csw, mu):
    L, m, site = 16, 0.1, (3, 5)
    Un = quenched(L)
    mg = mg2d.setup(torch.as_tensor(Un).cuda(), _params(L, m, csw=csw, mu=mu), init="device")
    out = mg2d.meson_correlators(mg, site=site, tol=1e-12)
    Dinv = np.linalg.inv(dense_D(Un, L, m, csw, mu))
    G = np.roll(G_restate(columns(Dinv, L, site)), -site[1], axis=0)
    assert np.max(np.abs(out["G"] - G)) < 1e-10 * np.max(np.abs(G))
    pp, ap, m_pcac = derived(G)
    np.testing.assert_allclose(out["pp"], pp, rtol=1e-10)
    assert np.max(np.abs(out["m_pcac"] - m_pcac)) < 1e-9
    assert len(out["iters"]) == 2 and all(r < 1e-11 for r in out["true_resnorms"])
    mg.close()


@pytest.mark.gpu
def test_free_field_through_the_multigrid():
    L = 64
    want = {0.1: 0.09627, 0.05: 0.04900, 0.02: 0.01983, -0.02: -0.02021}
    U = torch.ones((L * L, 2), dtype=torch.complex128, device="cuda")
    for m, mp in want.items():
        mg = mg2d.setup(U, _params(L, m), init="device")
        out = mg2d.meson_correlators(mg, site=(5, 9), tol=1e-12)
        G = G_restate(free_propagator_fft(L, m))
        assert np.max(np.abs(out["G"] - G)) < 1e-9 * np.max(np.abs(G)), m
        assert abs(out["m_pcac"][12] - mp) < 5e-6
        if m == 0.05:
            np.testing.assert_allclose(out["pp"][[1, 8, 16]], [0.13266, 0.013513, 0.0042989], rtol=4e-5)
        assert np.all(np.isfinite(out["m_eff"][1:L // 2]))
        mg.close()


@pytest.mark.gpu
def test_gauge_invariance_64():
    L, m = 64, 0.05
    U, _ = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=1234, return_phases=True)
    g = torch.Generator(device="cuda").manual_seed(9)
    w = torch.polar(torch.ones(L * L, dtype=torch.float64, device="cuda"),
                    (torch.rand(L * L, generator=g, dtype=torch.float64, device="cuda") * 2 - 1) * math.pi)
    xp, _, yp, _ = (torch.as_tensor(a, device="cuda") for a in O.neighbours(L))
    Ug = torch.stack([w * U[:, 0] * w[xp].conj(), w * U[:, 1] * w[yp].conj()], dim=1)
    res = []
    for links in (U, Ug):
        mg = mg2d.setup(links.clone(), _params(L, m), init="device")
        res.append((mg2d.meson_correlators(mg, site=(11, 40), tol=1e-12)["G"], mg2d.topological_charge(links, L),
                    mg2d.wilson_loops(links, L, 6, 6)))
        mg.close()
    (G0, q0, W0), (G1, q1, W1) = res
    assert np.max(np.abs(G1 - G0)) < 1e-9 * np.max(np.abs(G0))
    assert abs(q1 - q0) < 1e-9
    assert np.max(np.abs(W1 - W0)) < 1e-12


@pytest.mark.gpu
def test_translation_covariance():
    L, m, site, (dx, dy) = 32, 0.05, (4, 7), (9, 20)
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=60, seed=4)
    Ur = torch.roll(U.view(L, L, 2), shifts=(dy, dx), dims=(0, 1)).reshape(L * L, 2).contiguous()
    Gs = []
    for links, s in ((U, site), (Ur, ((site[0] + dx) % L, (site[1] + dy) % L))):
        mg = mg2d.setup(links.clone(), _params(L, m), init="device")
        Gs.append(mg2d.meson_correlators(mg, site=s, tol=1e-12)["G"])
        mg.close()
    assert np.max(np.abs(Gs[1] - Gs[0])) < 1e-9 * np.max(np.abs(Gs[0]))


@pytest.mark.gpu
def test_condensate_per_noise_against_dense():
    L, m, seed = 16, 0.1, 5
    S = L * L
    Un = quenched(L)
    mg = mg2d.setup(torch.as_tensor(Un).cuda(), _params(L, m), init="device")
    out = mg2d.chiral_condensate(mg, 3, seed=seed, tol=1e-12)
    D = dense_D(Un, L, m)
    want = np.array([np.vdot(e, np.linalg.solve(D, e)) / S for e in (noise_mirror(seed, k, S) for k in range(3))])
    assert np.max(np.abs(out["values"] - want)) < 1e-10 * np.max(np.abs(want))
    assert abs(out["mean"] - want.mean()) < 1e-10 and out["stderr"] > 0
    one = mg2d.chiral_condensate(mg, 1, seed=seed, tol=1e-12)                   # noise 0 alone: the same draw
    assert abs(one["values"][0] - out["values"][0]) < 1e-12 * abs(want[0]) and math.isnan(one["stderr"])
    assert abs(mg2d.chiral_condensate(mg, 1, seed=seed + 1, tol=1e-12)["values"][0] - out["values"][0]) > 1e-6
    mg.close()


@pytest.mark.gpu
def test_measurements_on_hmc_hierarchy_equal_fresh_setup():
    """After two trajectories the hierarchy has been moved in place (and refreshed after an acceptance); measuring on it
    gives what a fresh setup() on the same links gives, to solver tolerance."""
    L, beta, m = 32, 2.0, 0.1
    _, th = mg2d.gauge.quenched_links_device(L, beta, sweeps=60, seed=1234, return_phases=True)
    p = _params(L, m)
    h = mg2d.HMC(p, th, beta, tau=0.5, n_md=8, seed=21)
    for _ in range(2):
        h.trajectory()
    U = h.mg.LVL[0].U
    assert float((U - torch.polar(torch.ones_like(h.theta), th)).abs().max()) > 1e-3     # the links moved
    fresh = mg2d.setup(U.clone(), p, init="device")
    a = mg2d.meson_correlators(h.mg, site=(1, 2), tol=1e-12)
    b = mg2d.meson_correlators(fresh, site=(1, 2), tol=1e-12)
    assert np.max(np.abs(a["G"] - b["G"])) < 1e-9 * np.max(np.abs(b["G"]))
    ca, cb = mg2d.chiral_condensate(h.mg, 2, seed=3, tol=1e-12), mg2d.chiral_condensate(fresh, 2, seed=3, tol=1e-12)
    assert np.max(np.abs(ca["values"] - cb["values"])) < 1e-9 * np.max(np.abs(cb["values"]))
    assert mg2d.topological_charge(U, L) == mg2d.topological_charge(fresh.LVL[0].U, L)
    assert np.array_equal(mg2d.wilson_loops(U, L, 4, 4), mg2d.wilson_loops(fresh.LVL[0].U, L, 4, 4))
    fresh.close()
    h.mg.close()
