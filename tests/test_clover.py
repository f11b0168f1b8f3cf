"""The Wilson-clover (Sheikholeslami-Wohlert) level-0 operator: self block (2+m) 1 + f(s) sigma3 with
f(s) = (c_sw/8) sum of Im U_P over the four plaquettes with a corner at s.

CPU: the oracle's operator -- the O(a) shift of the would-be zero modes of a uniform-flux torus (cancelled at c_sw = 1,
doubled at c_sw = -1), gamma5-hermiticity, gauge covariance, c_sw = 0 is the Wilson operator, the clover term moves the
near-critical spectrum of quenched configurations, and MGParams' checks.
GPU: mg2d_clover_field, mg2d_clover_add and the sw entry points against the oracle / an fp64 torch restatement (ragged,
strip and 4096^2 shapes, complex128 to 1e-12 and complex64 to 2e-5 relative in the max-norm), and solves, the critical-mass
estimate and the strip code with c_sw = 1 against the oracle and the single-GPU solver."""
import math
import os

import numpy as np
import pytest
import torch

import mg2d
from oracle import mg_oracle as O

TOL, TOL32 = 1e-12, 2e-5
C128, C64 = 0, 1
CT = {C128: torch.complex128, C64: torch.complex64}
RT = {C128: torch.float64, C64: torch.float32}


# ---- the clover operator on top of the numpy oracle's Wilson operator --------------------------------------------
def gauge_uniform_flux(L, Q):
    """Links of a torus with Q flux quanta spread uniformly: theta_y(x, y) = 2 pi Q x / L^2, theta_x(L-1, y) = -2 pi Q y / L,
    every other phase 0.  Every plaquette angle is then 2 pi Q / L^2 (mod 2 pi), and D(0) has |Q| real would-be zero modes."""
    th = np.zeros((L, L, 2))  # th[y, x, dir]
    th[:, :, 1] = 2.0 * np.pi * Q * np.arange(L)[None, :] / L ** 2
    th[:, L - 1, 0] = -2.0 * np.pi * Q * np.arange(L) / L
    return O.gauge_from_phases(th.reshape(L * L, 2))


def clover_field(U, L, csw):
    """f(s) = (csw/8) sum over the four plaquettes with a corner at s (bases s, s-x, s-y, s-x-y) of Im U_P, with
    U_P(b) = U_x(b) U_y(b+x) conj(U_x(b+y)) conj(U_y(b)) as in O.plaquette: c_sw (i/4) sigma_xy F_xy with
    sigma_xy = (i/2)[sigma1, sigma2] = -sigma3 for gamma_x = sigma1, gamma_y = sigma2."""
    xp, xm, yp, ym = O.neighbours(L)
    im_p = np.imag(U[:, 0] * U[xp, 1] * np.conj(U[yp, 0]) * np.conj(U[:, 1]))
    return (csw / 8.0) * (im_p + im_p[xm] + im_p[ym] + im_p[xm][ym])


def add_clover(lv, U, L, csw):
    """the oracle's level-0 Wilson operator (reference layout D[s][k][i][j]) -> Wilson-clover: D[s][0] += f(s) sigma3"""
    if csw != 0.0:
        f = clover_field(U, L, csw)
        lv.D[:, 0, 0, 0] += f
        lv.D[:, 0, 1, 1] -= f


def _dense(U, L, m=0.0, csw=0.0):
    p = O.Params(L=L, num_iters=1, block=2, m=m, nlevels=1)
    lv = O.Level()
    lv.compute_lvl0_matrix(U, p)
    add_clover(lv, U, L, csw)
    return lv, O.dense_matrix(lv, L, 2)


# ================================================================================================================
# CPU: the oracle
# ================================================================================================================
@pytest.mark.parametrize("L,Q", [(16, 1), (16, 2), (24, 2)])
def test_uniform_flux_would_be_zero_modes(L, Q):
    """|Q| real eigenvalues of smallest modulus: theta_P/2 without clover, 0 at tree-level c_sw = 1, theta_P at c_sw = -1."""
    U = gauge_uniform_flux(L, Q)
    th = 2 * math.pi * Q / L ** 2
    assert abs(O.plaquette(U, L) - np.exp(1j * th)) < 1e-14
    for csw, want in ((0.0, th / 2), (1.0, 0.0), (-1.0, th)):
        ev = np.linalg.eigvals(_dense(U, L, csw=csw)[1])
        ev = ev[np.argsort(np.abs(ev))]
        assert np.all(np.abs(ev[:Q].imag) < 1e-10) and abs(ev[Q].imag) > 1e-10, (csw, ev[:Q + 1])
        assert np.all(np.abs(ev[:Q].real - want) <= 0.01 * th), (csw, ev[:Q], want)


def test_gamma5_hermiticity():
    L = 12
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    _, M = _dense(U, L, m=0.1, csw=1.3)
    G = np.kron(np.eye(L * L), np.diag([1.0, -1.0]))
    assert np.max(np.abs(G @ M @ G - M.conj().T)) < 1e-14


def test_gauge_covariance():
    """U_mu(s) -> w(s) U_mu(s) conj(w(s+mu)): f is unchanged and D_sw -> W D_sw W^dagger."""
    L = 12
    rng = np.random.default_rng(5)
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    w = np.exp(1j * rng.uniform(-np.pi, np.pi, L * L))
    xp, _, yp, _ = O.neighbours(L)
    Ug = np.stack([w * U[:, 0] * np.conj(w[xp]), w * U[:, 1] * np.conj(w[yp])], axis=1)
    f, fg = clover_field(U, L, 1.0), clover_field(Ug, L, 1.0)
    assert np.max(np.abs(f)) > 0.05 and np.max(np.abs(fg - f)) < 1e-14
    _, M = _dense(U, L, m=0.05, csw=1.0)
    _, Mg = _dense(Ug, L, m=0.05, csw=1.0)
    W = np.kron(np.diag(w), np.eye(2))
    assert np.max(np.abs(Mg - W @ M @ W.conj().T)) < 1e-14


def test_csw0_is_the_wilson_operator():
    """c_sw = 0 gives exactly the operator built without a clover coefficient, and the clover term touches only the
    self blocks, as f sigma3."""
    L = 16
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    lv0 = O.Level()
    lv0.compute_lvl0_matrix(U, O.Params(L=L, num_iters=1, block=2, m=0.07, nlevels=1))
    lvz = _dense(U, L, m=0.07, csw=0.0)[0]
    assert np.array_equal(lvz.D, lv0.D)
    lv1 = _dense(U, L, m=0.07, csw=1.0)[0]
    f = clover_field(U, L, 1.0)
    assert np.array_equal(lv1.D[:, 1:], lv0.D[:, 1:])
    d = lv1.D[:, 0] - lv0.D[:, 0]
    assert np.max(np.abs(d[:, 0, 0] - f)) < 1e-15 and np.max(np.abs(d[:, 1, 1] + f)) < 1e-15
    assert np.all(d[:, 0, 1] == 0) and np.all(d[:, 1, 0] == 0)
    assert np.max(np.abs(f)) <= 0.5


@pytest.mark.parametrize("seed", [1234, 1235])
def test_clover_moves_the_near_critical_spectrum(seed):
    """32^2 quenched beta = 6: the smallest real part of the spectrum of D(0) drops by at least a factor 0.6 at c_sw = 1."""
    L = 32
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=200, seed=seed))
    lo = [np.linalg.eigvals(_dense(U, L, csw=c)[1]).real.min() for c in (0.0, 1.0)]
    assert 0 < lo[1] <= 0.6 * lo[0], lo


def test_params_checks():
    p = mg2d.make_params(32, -0.05, csw=1.0)
    assert p.csw == 1.0 and mg2d.make_params(32, -0.05).csw == 0.0
    with pytest.raises(ValueError):
        mg2d.make_params(32, 0.1, stencil="laplace", csw=1.0)
    mg2d.make_params(32, 0.1, stencil="laplace", csw=0.0)
    with pytest.raises(ValueError):
        mg2d.make_params(32, -1.5, csw=1.0)              # 2 - 1.5 - 0.5 = 0: a self block may be singular
    with pytest.raises(ValueError):
        mg2d.make_params(32, 0.0, csw=-4.5)
    mg2d.make_params(32, -1.4, csw=1.0)


# ================================================================================================================
# GPU
# ================================================================================================================
_CTX = None


def call(name, *args):
    global _CTX
    if _CTX is None:
        _CTX = mg2d._lib.Context(0)
    _CTX.call(name, *args)


def P_(t):
    return None if t is None else t.data_ptr()


def S_():
    return torch.cuda.current_stream().cuda_stream


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def T(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def rel(got, want):
    """max |got - want| / max |want|, fp64, in chunks"""
    g, w = got.reshape(-1), want.reshape(-1)
    num = den = 0.0
    for i in range(0, w.numel(), 1 << 24):
        wi = w[i:i + (1 << 24)].to(torch.complex128)
        num = max(num, float((g[i:i + (1 << 24)].to(torch.complex128) - wi).abs().max()))
        den = max(den, float(wi.abs().max()))
    return num / max(den, 1e-300)


def gen(seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return g


def crandn(g, *shape):
    return torch.randn(shape, dtype=torch.complex128, device="cuda", generator=g)


def rounded(t, dtype):
    return t.to(CT[dtype]).to(torch.complex128)


def links(g, Ly, Lx, dtype=C128, width=0.6):
    """Links near the identity (plaquettes of a rough quenched field) on a [Ly, Lx, 2] grid."""
    th = torch.randn((Ly, Lx, 2), dtype=torch.float64, device="cuda", generator=g) * width
    return rounded(torch.polar(torch.ones_like(th), th), dtype)


@pytest.fixture
def gpu_mem():
    torch.cuda.empty_cache()
    yield
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ---- fp64 restatement (fields [Ly, Lx, 2], x periodic, rows -1 / Ly from halo rows) ----------------------------------
def clover_ref(U, U_lo, U_hi, csw):
    """f of the rows of U [Ly, Lx, 2]; U_lo / U_hi = link rows -1 / Ly."""
    E = torch.cat([U_lo[-1:], U, U_hi[:1]], dim=0)                # rows -1 .. Ly
    Ux, Uy = E[..., 0], E[..., 1]
    P = (Ux[:-1] * Uy[:-1].roll(-1, dims=1) * Ux[1:].conj() * Uy[:-1].conj()).imag   # bases on rows -1 .. Ly-1
    Pb, Pm = P[1:], P[:-1]                                         # bases in rows y and y-1
    return (csw / 8.0) * (Pb + Pb.roll(1, dims=1) + Pm + Pm.roll(1, dims=1))


def _proj(device):
    I = torch.eye(2, dtype=torch.complex128, device=device)
    g1 = torch.tensor([[0, 1], [1, 0]], dtype=torch.complex128, device=device)
    g2 = torch.tensor([[0, -1j], [1j, 0]], dtype=torch.complex128, device=device)
    return [0.5 * (I - g1), 0.5 * (I + g1), 0.5 * (I - g2), 0.5 * (I + g2)]


def hop_ref(f, lo, hi, U, U_lo):
    """sum_k D_k f(s + d_k) of the Wilson stencil; lo / hi: rows below / above f (last / first used), U_lo: link rows below."""
    e = torch.cat([lo[-1:], f, hi[:1]], dim=0)
    nb = (f.roll(-1, dims=1), f.roll(1, dims=1), e[2:], e[:-2])
    Uy_m = torch.cat([U_lo[-1:, :, 1], U[:-1, :, 1]], dim=0)
    coef = (U[..., 0], U[..., 0].roll(1, dims=1).conj(), U[..., 1], Uy_m.conj())
    P = _proj(f.device)
    return sum(coef[k][..., None] * torch.einsum("ij,...j->...i", P[k], nb[k]) for k in range(4))


def self_ref(F, m):
    """the diagonal of the clover self block per site and component, [Ly, Lx, 2]"""
    return torch.stack([2.0 + m + F, 2.0 + m - F], dim=-1).to(torch.complex128)


def half_ref(phi, lo, hi, U, U_lo, F, r, m, colour, yoff):
    new = ((0 if r is None else r) - hop_ref(phi, lo, hi, U, U_lo)) / self_ref(F, m)
    y = torch.arange(phi.shape[0], device=phi.device)[:, None]
    x = torch.arange(phi.shape[1], device=phi.device)[None, :]
    return torch.where(((x + y + yoff) % 2 == colour)[:, :, None], new, phi)


def rb2_ref(phi, lo2, hi2, U, U_lo2, U_hi, F, F_lo, F_hi, r, r_lo, r_hi, m, yoff):
    """colour 0 on rows -1 .. Ly from the old values two rows deep, then colour 1 on rows 0 .. Ly-1 from those."""
    Ly = phi.shape[0]
    E = torch.cat([lo2, phi, hi2], dim=0)
    UE = torch.cat([U_lo2, U, U_hi], dim=0)
    FE = torch.cat([F_lo, F, F_hi], dim=0)
    RE = None if r is None else torch.cat([r_lo, r, r_hi], dim=0)
    red = half_ref(E[1:Ly + 3], E[:1], E[Ly + 3:], UE[1:Ly + 3], UE[:1], FE, RE, m, 0, yoff + 1)
    return half_ref(red[1:Ly + 1], red[:1], red[Ly + 1:], U, U_lo2, F, r, m, 1, yoff)


# ---- mg2d_clover_field -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("L", [4, 6, 10, 32, 130, 256])
def test_clover_field_matches_oracle(L):
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=10))
    for dtype, tol in ((C128, TOL), (C64, TOL32)):
        Ud = T(U).to(CT[dtype])
        F = torch.empty(L * L, dtype=RT[dtype], device="cuda")
        call("mg2d_clover_field", P_(F), P_(Ud), P_(Ud[(L - 1) * L:]), P_(Ud), 1.0, L, L, dtype, S_())
        want = clover_field(U, L, 1.0)
        assert np.max(np.abs(F.double().cpu().numpy() - want)) <= tol * np.max(np.abs(want)), (L, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("Lx,Ly", [(5, 7), (34, 18), (66, 130), (4096, 4096)])
def test_clover_field_ragged_and_strips(Lx, Ly, gpu_mem):
    """Rectangular lattices against the torch restatement; strips (U_lo / U_hi pointing into the whole field, ragged
    cuts included) give the whole field's rows bit for bit.  At 4096^2 the launch grid is capped and every CTA loops."""
    g = gen(Lx + Ly)
    for dtype, tol in ((C128, TOL), (C64, TOL32)):
        U = links(g, Ly, Lx, dtype)
        Uk = U.to(CT[dtype]).contiguous()
        F = torch.empty(Lx * Ly, dtype=RT[dtype], device="cuda")
        flat = Uk.reshape(-1, 2)
        call("mg2d_clover_field", P_(F), P_(flat), P_(flat[(Ly - 1) * Lx:]), P_(flat), -1.7, Lx, Ly, dtype, S_())
        want = clover_ref(U, U[-1:], U[:1], -1.7)
        assert rel(F.reshape(Ly, Lx), want) < tol, (Lx, Ly, dtype)
        cuts = sorted({0, 1, Ly // 3, Ly // 2, Ly - 1, Ly}) if Ly > 2 else [0, Ly]
        for y0, y1 in zip(cuts[:-1], cuts[1:]):
            Fs = torch.empty((y1 - y0) * Lx, dtype=RT[dtype], device="cuda")
            lo, hi = ((y0 - 1) % Ly) * Lx, (y1 % Ly) * Lx
            call("mg2d_clover_field", P_(Fs), P_(flat[y0 * Lx:]), P_(flat[lo:]), P_(flat[hi:]), -1.7, Lx, y1 - y0, dtype, S_())
            assert torch.equal(Fs, F[y0 * Lx:y1 * Lx]), (Lx, Ly, dtype, y0, y1)
        del U, Uk, F, flat, want


# ---- mg2d_clover_add -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_clover_add_gives_the_oracle_operator():
    L, m = 32, -0.04
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    lvo = _dense(U, L, m=m, csw=1.0)[0]
    for dt, tol in (("complex128", TOL), ("complex64", TOL32)):
        p = mg2d.make_params(L, m, nlevels=1, csw=1.0, matrix_free=False, dtype=dt)
        mg = mg2d.MG(p)
        mg.set_gauge(T(U))
        lv = mg.LVL[0]
        assert lv.clover is not None and lv.clover.dtype == (torch.float64 if dt == "complex128" else torch.float32)
        D = mg2d.D_to_reference_layout(lv.D).to(torch.complex128).cpu().numpy()
        assert np.max(np.abs(D - lvo.D)) <= tol * np.max(np.abs(lvo.D)), dt
        mg.close()


# ---- the sw entry points -----------------------------------------------------------------------------------------
def _sw_case(Lx, Ly, dtype, strip, yoff, seed, capped=False):
    m, csw = -0.05, 1.0
    S = Lx * Ly
    g = gen(seed)
    Ug = links(g, Ly, Lx, dtype)
    pg, rg = rounded(crandn(g, Ly, Lx, 2), dtype), rounded(crandn(g, Ly, Lx, 2), dtype)
    if strip:
        lo2, hi2 = rounded(crandn(g, 2, Lx, 2), dtype), rounded(crandn(g, 2, Lx, 2), dtype)
        U_lo2, U_hi = links(g, 2, Lx, dtype), links(g, 1, Lx, dtype)
        r_lo, r_hi = rounded(crandn(g, 1, Lx, 2), dtype), rounded(crandn(g, 1, Lx, 2), dtype)
    else:
        lo2, hi2, U_lo2, U_hi, r_lo, r_hi = pg[-2:], pg[:2], Ug[-2:], Ug[:1], rg[-1:], rg[:1]
    # the clover field of the strip from the kernel (its own test holds it to the reference), halo rows from their links
    k = lambda t: t.to(CT[dtype]).contiguous()
    Uk, pk, rk = k(Ug).reshape(S, 2), k(pg).reshape(S, 2), k(rg).reshape(S, 2)
    lo2k, hi2k, Ulo2k, Uhik, rlok, rhik = k(lo2), k(hi2), k(U_lo2), k(U_hi), k(r_lo), k(r_hi)
    F = torch.empty(S, dtype=RT[dtype], device="cuda")
    call("mg2d_clover_field", P_(F), P_(Uk), P_(Ulo2k[1:]), P_(Uhik), csw, Lx, Ly, dtype, S_())
    if strip:
        F_lo, F_hi = (torch.randn((1, Lx), dtype=torch.float64, device="cuda", generator=g) * 0.3).to(RT[dtype]), \
                     (torch.randn((1, Lx), dtype=torch.float64, device="cuda", generator=g) * 0.3).to(RT[dtype])
    else:
        F_lo, F_hi = F.reshape(Ly, Lx)[-1:].clone(), F.reshape(Ly, Lx)[:1].clone()
    Fg, Flo, Fhi = F.reshape(Ly, Lx).double(), F_lo.double(), F_hi.double()
    tol = TOL if dtype == C128 else TOL32
    if capped:
        # the launchers' formulas (csrc/wilson.cu, csrc/wilson_rb2.cu): every CTA / warp loops, the last pass is partial
        RY = 32
        while RY > 4 and -(-Lx // 128) * -(-Ly // RY) < sms() * 6:
            RY >>= 1
        nwork = -(-Lx // 128) * -(-Ly // RY)
        assert nwork > 4096 and nwork % 4096, "wilson_march_kernel is not in the capped regime"
        ntx, RY2 = -(-Lx // 62), 128
        while RY2 > 8 and ntx * -(-Ly // RY2) < sms() * 12:
            RY2 >>= 1
        nitems = ntx * -(-Ly // RY2)
        assert nitems > sms() * 16 and nitems % (sms() * 16), "wilson_rb2_kernel is not in the capped regime"
    # apply; residual with the fused dots
    want = hop_ref(pg, lo2, hi2, Ug, U_lo2) + self_ref(Fg, m) * pg
    out = torch.empty_like(pk)
    call("mg2d_wilson_sw_apply", P_(out), P_(pk), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(F), None, m, Lx, Ly, 0,
         dtype, None, S_())
    assert rel(out, want) < tol, (Lx, Ly, dtype, "apply")
    d = torch.zeros(4, dtype=torch.float64, device="cuda")
    call("mg2d_wilson_sw_apply", P_(out), P_(pk), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(F), P_(rk), m, Lx, Ly, 1,
         dtype, P_(d), S_())
    res = rg - want
    assert rel(out, res) < tol, (Lx, Ly, dtype, "resid")
    o64 = out.to(torch.complex128).reshape(-1)
    d = d.cpu().numpy()
    n2, ip, b2 = float((o64.abs() ** 2).sum()), complex(torch.vdot(o64, pg.reshape(-1))), float((rg.abs() ** 2).sum())
    assert abs(d[0] / n2 - 1) < TOL and abs(d[3] / b2 - 1) < TOL
    assert abs(complex(d[1], d[2]) - ip) < TOL * math.sqrt(n2 * float((pg.abs() ** 2).sum()))
    del out, o64, res, want
    # the one-pass two-colour sweep, with and without r
    for with_r in (True, False):
        o = torch.empty_like(pk)
        call("mg2d_wilson_sw_relax_rb2", P_(o), P_(pk), P_(lo2k), P_(hi2k), P_(Uk), P_(Ulo2k), P_(Uhik), P_(F), P_(F_lo), P_(F_hi),
             P_(rk if with_r else None), P_(rlok if with_r else None), P_(rhik if with_r else None), m, Lx, Ly, yoff, dtype, None, S_())
        want = rb2_ref(pg, lo2, hi2, Ug, U_lo2, U_hi, Fg, Flo, Fhi, rg if with_r else None, r_lo, r_hi, m, yoff)
        assert rel(o, want) < tol, (Lx, Ly, dtype, "rb2", with_r)
        del o, want
    # the half sweep (in place), both colours in turn
    ph = pk.clone()
    cur = pg
    for colour in (0, 1):
        call("mg2d_wilson_sw_relax_rb", P_(ph), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(F), P_(rk), m, Lx, Ly, colour,
             yoff, dtype, S_())
        cur = half_ref(cur, lo2, hi2, Ug, U_lo2, Fg, rg, m, colour, yoff)
        assert rel(ph, cur) < tol, (Lx, Ly, dtype, "rb", colour)


@pytest.mark.gpu
@pytest.mark.parametrize("Lx,Ly", [(6, 4), (34, 18), (130, 66), (256, 256)])
def test_sw_kernels_small(Lx, Ly):
    for dtype in (C128, C64):
        _sw_case(Lx, Ly, dtype, False, 0, Lx * 7 + Ly)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_sw_kernels_4096(dtype, gpu_mem):
    _sw_case(4096, 4096, dtype, False, 0, 21)


@pytest.mark.gpu
def test_sw_kernels_capped_grid(gpu_mem):
    """A ragged lattice large enough that the apply, the two-colour sweep and the half sweep all run on capped grids."""
    _sw_case(5000, 4128, C128, False, 0, 22, capped=True)


@pytest.mark.gpu
@pytest.mark.parametrize("Ly,yoff,dtype", [(512, 1, C128), (2048, 0, C128), (512, 1, C64), (3, 1, C128)])
def test_sw_kernels_strips(Ly, yoff, dtype, gpu_mem):
    """Strips with explicit halo rows of phi (two deep), links, r and the clover field."""
    _sw_case(4096 if Ly > 3 else 64, Ly, dtype, True, yoff, 23 + Ly)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_sw_entry_points_with_zero_field_equal_wilson(dtype):
    """F = 0 through the sw entry points gives the Wilson entry points' results to rounding.  (Not bit for bit: the complex
    products reach ptxas as separate multiplies and subtractions, and which product it fuses into an FMA is decided per
    kernel.  A hierarchy with csw = 0 never calls the sw entry points.)"""
    Lx, Ly, m = 130, 66, 0.03
    S = Lx * Ly
    tol = 4e-16 * 4 if dtype == C128 else 6e-8 * 8
    g = gen(31)
    U = links(g, Ly, Lx, dtype).to(CT[dtype]).reshape(S, 2).contiguous()
    phi, r = crandn(g, S, 2).to(CT[dtype]), crandn(g, S, 2).to(CT[dtype])
    F0 = torch.zeros(S, dtype=RT[dtype], device="cuda")
    lo2, hi2, Ulo2, Uhi = phi[(Ly - 2) * Lx:], phi, U[(Ly - 2) * Lx:], U
    rlo, rhi = r[(Ly - 1) * Lx:], r
    for mode, b in ((0, None), (1, r)):
        a, c = torch.empty_like(phi), torch.empty_like(phi)
        da, dc = torch.zeros(4, dtype=torch.float64, device="cuda"), torch.zeros(4, dtype=torch.float64, device="cuda")
        call("mg2d_wilson_apply", P_(a), P_(phi), P_(lo2[Lx:]), P_(hi2), P_(U), P_(Ulo2[Lx:]), P_(b), m, Lx, Ly, mode, dtype, P_(da), S_())
        call("mg2d_wilson_sw_apply", P_(c), P_(phi), P_(lo2[Lx:]), P_(hi2), P_(U), P_(Ulo2[Lx:]), P_(F0), P_(b), m, Lx, Ly, mode, dtype,
             P_(dc), S_())
        assert rel(c, a) <= tol, mode
        # the dots sum the outputs' products in fp64: they inherit the outputs' rounding (|out|^2: twice its relative size)
        assert float((dc - da).abs().max()) <= max(1e-13, 2 * tol) * float(da.abs().max()), mode
    for rr in (r, None):
        a, c = torch.empty_like(phi), torch.empty_like(phi)
        rl, rh = (rlo, rhi) if rr is not None else (None, None)
        call("mg2d_wilson_relax_rb2", P_(a), P_(phi), P_(lo2), P_(hi2), P_(U), P_(Ulo2), P_(Uhi), P_(rr), P_(rl), P_(rh), m, Lx, Ly, 1,
             dtype, None, S_())
        call("mg2d_wilson_sw_relax_rb2", P_(c), P_(phi), P_(lo2), P_(hi2), P_(U), P_(Ulo2), P_(Uhi), P_(F0), P_(F0), P_(F0), P_(rr),
             P_(rl), P_(rh), m, Lx, Ly, 1, dtype, None, S_())
        assert rel(c, a) <= 4 * tol                  # (the black stage reads the red stage's values)
        a, c = phi.clone(), phi.clone()
        for colour in (0, 1):
            call("mg2d_wilson_relax_rb", P_(a), P_(a[(Ly - 1) * Lx:]), P_(a), P_(U), P_(Ulo2[Lx:]), P_(rr), m, Lx, Ly, colour, 0,
                 dtype, S_())
            call("mg2d_wilson_sw_relax_rb", P_(c), P_(c[(Ly - 1) * Lx:]), P_(c), P_(U), P_(Ulo2[Lx:]), P_(F0), P_(rr), m, Lx, Ly,
                 colour, 0, dtype, S_())
        assert rel(c, a) <= 4 * tol


@pytest.mark.gpu
@pytest.mark.parametrize("store", [False, True])
def test_uniform_flux_zero_mode_on_the_gpu(store):
    """The oracle's would-be zero mode x of the 16^2, Q = 1 torus at c_sw = 1 is an eigenvector of the device operator
    (matrix-free sw_apply, or the stored operator with mg2d_clover_add) to 1e-12."""
    L = 16
    U = gauge_uniform_flux(L, 1)
    ev, V = np.linalg.eig(_dense(U, L, csw=1.0)[1])
    i = int(np.argmin(np.abs(ev)))
    lam, x = ev[i], V[:, i].reshape(L * L, 2)
    assert abs(lam.imag) < 1e-10 and abs(lam) < 1e-3
    p = mg2d.make_params(L, 0.0, nlevels=0, smoother="rbgs", csw=1.0)
    mg = mg2d.MG(p)
    mg.LVL[0].compute_lvl0_matrix(T(U), store=store)
    xd = T(x)
    Dx = torch.empty_like(xd)
    mg.LVL[0].apply_D(Dx, xd)
    assert float(torch.linalg.vector_norm(Dx - lam * xd) / torch.linalg.vector_norm(xd)) <= 1e-12
    mg.close()


# ---- solves --------------------------------------------------------------------------------------------------------
def _quenched(L, sweeps=30, seed=1234):
    return O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=sweeps, seed=seed))


@pytest.mark.gpu
def test_reference_gs_flow_with_clover():
    """The reference's flow (random start, GS smoother on the stored operator, stationary cycle) with c_sw = 1."""
    L, m = 32, 0.02
    U = _quenched(L)
    po = O.Params(L=L, num_iters=3, block=2, m=m, nlevels=2, null_iters=40, max_iters=300, res_threshold=1e-12)
    LVLo, NTLo = O.build_reference_problem(po, U)          # O.run_reference_flow with the clover term added to level 0
    add_clover(LVLo[0], U, L, 1.0)
    O.compute_near_null(LVLo, NTLo, po, po.quad)
    io = O.perform_MG(LVLo, NTLo, po)
    p = mg2d.make_params(L, m, nlevels=2, n_smooth=3, null_iters=40, max_iters=300, tol=1e-12, csw=1.0)
    mg, ig = mg2d.run_reference_flow(p, T(U))
    assert io["converged"] and ig["converged"] and ig["iters"] == io["iters"], (ig["iters"], io["iters"])
    x = mg.LVL[0].phi.cpu().numpy()
    assert np.max(np.abs(x - LVLo[0].phi)) < 1e-9 * np.max(np.abs(LVLo[0].phi))


@pytest.mark.gpu
def test_matrix_free_rbgs_fgcr_with_clover():
    """Matrix-free red-black smoothing (sw_relax_rb2, sw_apply) inside FGCR against the oracle; then the complex64
    preconditioner reaches a true residual of 1e-10."""
    L, m = 32, 0.0
    U = _quenched(L)
    b = np.zeros((L * L, 2), dtype=complex)
    b[L // 2 + (L // 2) * L, 0] = 1.0
    po = O.Params(L=L, num_iters=2, block=2, m=m, nlevels=2, null_iters=40, smoother="rbgs")
    LVLo, NTLo = O.build_reference_problem(po, U)
    add_clover(LVLo[0], U, L, 1.0)
    O.compute_near_null(LVLo, NTLo, po, 1)
    xo, io = O.gcr_MG(LVLo, NTLo, po, b, tol=1e-10, restart=8)
    p = mg2d.make_params(L, m, nlevels=2, n_smooth=2, smoother="rbgs", null_iters=40, csw=1.0)
    mg = mg2d.setup(T(U), p)
    assert mg.LVL[0].matrix_free and mg.LVL[0].clover is not None
    x, ig = mg2d.solve(mg, rhs=T(b), tol=1e-10, outer="gcr", restart=8)
    assert io["converged"] and ig["iters"] == io["iters"], (ig["iters"], io["iters"])
    assert np.max(np.abs(x.cpu().numpy() - xo)) < 1e-9 * np.max(np.abs(xo))
    xm, im = mg2d.solve(mg, rhs=T(b), tol=1e-10, outer="gcr", restart=8, precond_dtype="complex64", use_graph=True)
    sh = mg.info["single"].LVL[0]
    assert sh.clover is not None and sh.clover.dtype == torch.float32
    assert im["converged"] and im["true_resnorm"] < 1e-10 and abs(im["iters"] - ig["iters"]) <= 2
    chk = torch.empty_like(xm)
    mg.LVL[0].apply_D(chk, xm)
    assert float(torch.linalg.vector_norm(chk - T(b))) < 1e-10
    mg.close()


@pytest.mark.gpu
def test_critical_mass_with_clover_against_dense_spectrum():
    from importlib import import_module
    critical = import_module("2d_multigrid_b200.critical")
    L = 32
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=200, seed=1234))
    ev = np.linalg.eigvals(_dense(U, L, csw=1.0)[1])
    lam = ev[np.argmin(ev.real)]
    assert abs(lam.imag) < 1e-10 and 0.0 < lam.real < 0.05, lam          # the lowest mode is real (a would-be zero mode)
    factory = lambda m: mg2d.make_params(L, m, nlevels=2, block=2, n_null=4, n_smooth=3, smoother="rbgs", null_iters=40,
                                         tol=1e-10, csw=1.0)
    mcrit, _ = critical.estimate_critical_mass(T(U), factory)
    assert abs(mcrit + lam.real) < 1e-4, (mcrit, lam, critical.estimate_critical_mass.info)


def _strip_problem(L, dev):
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=20, seed=1234, device=dev)
    p = mg2d.make_params(L, 0.03, nlevels=2, block=4, n_null=8, n_smooth=3, n_pre=0, n_post=[4, 2, 8], smoother="rbgs",
                         null_iters=40, tol=1e-10, max_iters=100, csw=1.0)
    rhs = torch.zeros((L * L, 2), dtype=torch.complex128, device=f"cuda:{dev}")
    rhs[L // 2 + (L // 2) * L, 0] = 1.0
    return U, p, rhs


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_strip_code_with_clover_equals_single_gpu(fused):
    """The strip code with the rank as its own neighbour (exchanged clover halo rows, fused or standalone smoother halos)."""
    from importlib import import_module
    dmod = import_module("2d_multigrid_b200.dist")
    L = 128
    U, p, rhs = _strip_problem(L, 0)
    ref = mg2d.setup(U, p, init="device")
    x_ref, i_ref = mg2d.solve(ref, rhs=rhs, tol=1e-10, outer="gcr")
    x_ref = x_ref.clone()
    comm = dmod.Comm.single(mg2d.Context(0), torch.device("cuda", 0))
    comm.fused = fused
    dmg = dmod.setup(U, p, comm, min_rows=16)
    lv0 = dmg.LVL[0]
    assert lv0.distributed and lv0._clover_halos is not None
    assert torch.equal(lv0.clover, ref.LVL[0].clover[lv0.y0 * L:(lv0.y0 + lv0.Ly) * L])
    x, info = mg2d.solve(dmg, rhs=rhs, tol=1e-10, outer="gcr")
    assert info["converged"] and info["iters"] == i_ref["iters"], (info["iters"], i_ref["iters"])
    dx = float((x - x_ref[lv0.y0 * L:(lv0.y0 + lv0.Ly) * L]).abs().max() / x_ref.abs().max())
    assert dx < 1e-9 and info["true_resnorm"] < 1e-10, dx
    ref.close()
    dmg.close()


def _two_rank_worker(rank, world, port, L, out):
    from importlib import import_module
    dmod = import_module("2d_multigrid_b200.dist")
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    comm = dmod.init(world, rank, rank)
    U, p, rhs = _strip_problem(L, rank)
    if rank == 0:
        ref = mg2d.setup(U, p, init="device")
        x_ref, i_ref = mg2d.solve(ref, rhs=rhs, tol=1e-10, outer="gcr")
    dmg = dmod.setup(U, p, comm, min_rows=16)
    x, info = mg2d.solve(dmg, rhs=dmg.scatter_field(rhs), tol=1e-10, outer="gcr")
    if rank == 0:
        lv0 = dmg.LVL[0]
        dx = float((x - x_ref[lv0.y0 * L:(lv0.y0 + lv0.Ly) * L]).abs().max() / x_ref.abs().max())
        out.put(dict(iters=info["iters"], ref_iters=i_ref["iters"], dx=dx, true=info["true_resnorm"]))
    torch.cuda.synchronize()
    torch.distributed.barrier()
    os._exit(0)


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_with_clover_equal_single_gpu():
    import torch.multiprocessing as tmp
    ctx = tmp.get_context("spawn")
    out = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, 29541, 256, out)) for r in range(2)]
    for pr in procs:
        pr.start()
    res = out.get(timeout=600)
    for pr in procs:
        pr.join(timeout=120)
    assert res["iters"] == res["ref_iters"] and res["dx"] < 1e-9 and res["true"] < 1e-10, res
