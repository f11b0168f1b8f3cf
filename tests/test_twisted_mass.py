"""Twisted mass on the level-0 Wilson(-clover) operator: D_tm(m, mu) = D_W(m) [+ clover] + i mu gamma5, gamma5 = sigma3,
self block diag(2+m+f+i mu, 2+m-f-i mu).

CPU: a dense restatement on the oracle's Wilson operator (the clover term from test_clover.py): g5 D(mu) g5 = D(-mu)^dag,
D(mu)^dag D(mu) = D(0)^dag D(0) + mu^2, the smallest singular value |mu| on the free field at m = 0 (sign and size of the
term), MGParams' checks and the guard of critical.estimate_critical_mass.
GPU: the tm entry points and mg2d_twist_add against an fp64 torch restatement (ragged, capped, 4096^2 and 8-rank strip
shapes; strips with real neighbour rows equal the whole lattice bit for bit), the norm identity at 4096^2, the Galerkin
identity self(mu) - self(0) = i mu Gamma5_c on every coarse level, the reference GS flow against the oracle, maximal-twist
solves at m_crit on quenched links, and the strip code with its linked sweep."""
import math

import numpy as np
import pytest
import torch

import mg2d
from oracle import mg_oracle as O
from test_clover import (C64, C128, CT, RT, TOL, TOL32, P_, S_, _dense, add_clover, call, crandn, gen, gpu_mem,
                         hop_ref, links, rel, rounded, self_ref, sms)

_ = gpu_mem                                  # the fixture, imported for the GPU tests below


# ---- the twisted operator on top of the oracle's Wilson(-clover) operator -------------------------------------------
def G5(L):
    return np.kron(np.eye(L * L), np.diag([1.0, -1.0]))


def dense_tm(U, L, m, csw, mu):
    """dense D_W(m) + clover(csw) + i mu gamma5 on the oracle's site-major, spin-minor ordering"""
    return _dense(U, L, m=m, csw=csw)[1] + 1j * mu * G5(L)


def sparse_tm(U, L, m, csw, mu):
    """the same operator as a scipy CSR matrix (the oracle's level-0 blocks, clover and twist added)"""
    import scipy.sparse as sp
    lv = O.Level()
    lv.compute_lvl0_matrix(U, O.Params(L=L, num_iters=1, block=2, m=m, nlevels=1))
    add_clover(lv, U, L, csw)
    add_twist(lv, mu)
    S = L * L
    site = np.arange(S)
    tgt = [site] + list(O.neighbours(L))
    rows, cols, vals = [], [], []
    for k in range(5):
        for i in range(2):
            for j in range(2):
                rows.append(2 * site + i)
                cols.append(2 * tgt[k] + j)
                vals.append(lv.D[:, k, i, j])
    return sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(2 * S, 2 * S))


def add_twist(lv, mu):
    """the oracle's level-0 operator (reference layout D[s][k][i][j]) -> D[s][0] += diag(i mu, -i mu)"""
    lv.D[:, 0, 0, 0] += 1j * mu
    lv.D[:, 0, 1, 1] -= 1j * mu


# ================================================================================================================
# CPU
# ================================================================================================================
@pytest.mark.parametrize("L", [8, 16])
@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_twisted_identities(L, csw):
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    m, mu = -0.08, 0.037
    M0, Mp, Mm = dense_tm(U, L, m, csw, 0.0), dense_tm(U, L, m, csw, mu), dense_tm(U, L, m, csw, -mu)
    G = G5(L)
    assert np.max(np.abs(G @ Mp @ G - Mm.conj().T)) < 1e-14
    assert np.max(np.abs(G @ Mp @ G - Mp.conj().T)) > 1.9 * mu              # no longer gamma5-hermitian
    N = Mp.conj().T @ Mp - (M0.conj().T @ M0 + mu ** 2 * np.eye(2 * L * L))
    assert np.max(np.abs(N)) < 1e-13


@pytest.mark.parametrize("L", [8, 16])
@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_free_field_smallest_singular_value(L, csw):
    """Free field, m = 0: D_W has an exact zero mode (momentum (pi, pi)), so the smallest singular value of D_tm is |mu|
    whatever the sign of mu (the clover field vanishes on the free field)."""
    U = np.ones((L * L, 2), dtype=complex)
    assert np.linalg.svd(dense_tm(U, L, 0.0, csw, 0.0), compute_uv=False).min() < 1e-12
    for mu in (0.05, -0.02):
        s = np.linalg.svd(dense_tm(U, L, 0.0, csw, mu), compute_uv=False)
        assert abs(s.min() - abs(mu)) < 1e-12, (mu, s.min())


@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_sparse_restatement_equals_dense(csw):
    L = 8
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    assert np.max(np.abs(sparse_tm(U, L, -0.03, csw, 0.02).toarray() - dense_tm(U, L, -0.03, csw, 0.02))) == 0.0


def test_params_checks():
    assert mg2d.make_params(32, -0.05).mu == 0.0
    p = mg2d.make_params(32, -0.05, mu=1e-3, csw=1.0)
    assert p.mu == 1e-3 and isinstance(p.mu, float)
    for bad in (float("nan"), float("inf"), -float("inf")):
        with pytest.raises(ValueError):
            mg2d.make_params(32, 0.0, mu=bad)
    with pytest.raises(ValueError):
        mg2d.make_params(32, 0.1, stencil="laplace", mu=1e-3)
    mg2d.make_params(32, 0.1, stencil="laplace", mu=0.0)
    with pytest.raises(ValueError):
        mg2d.make_params(32, -1.5, csw=1.0, mu=0.3)       # the clover bound 2 + m - |c_sw|/2 > 0 is kept as it is
    mg2d.make_params(32, -1.4, csw=1.0, mu=0.3)


def test_critical_mass_rejects_a_twisted_factory():
    from importlib import import_module
    critical = import_module("2d_multigrid_b200.critical")
    with pytest.raises(ValueError, match="mu == 0"):
        critical.estimate_critical_mass(None, lambda m: mg2d.make_params(16, m, mu=1e-3))


# ================================================================================================================
# GPU
# ================================================================================================================
def twist(mu, device):
    return 1j * mu * torch.tensor([1.0, -1.0], dtype=torch.complex128, device=device)


def half_tm(phi, lo, hi, U, U_lo, dg, r, colour, yoff):
    """one colour of the red-black sweep with the diagonal self block dg [Ly, Lx, 2]"""
    new = ((0 if r is None else r) - hop_ref(phi, lo, hi, U, U_lo)) / dg
    y = torch.arange(phi.shape[0], device=phi.device)[:, None]
    x = torch.arange(phi.shape[1], device=phi.device)[None, :]
    return torch.where(((x + y + yoff) % 2 == colour)[:, :, None], new, phi)


def rb2_tm(phi, lo2, hi2, U, U_lo2, U_hi, dgE, r, r_lo, r_hi, yoff):
    """colour 0 on rows -1 .. Ly from the old values two rows deep, then colour 1 on rows 0 .. Ly-1; dgE: rows -1 .. Ly"""
    Ly = phi.shape[0]
    E = torch.cat([lo2, phi, hi2], dim=0)
    UE = torch.cat([U_lo2, U, U_hi], dim=0)
    RE = None if r is None else torch.cat([r_lo, r, r_hi], dim=0)
    red = half_tm(E[1:Ly + 3], E[:1], E[Ly + 3:], UE[1:Ly + 3], UE[:1], dgE, RE, 0, yoff + 1)
    return half_tm(red[1:Ly + 1], red[:1], red[Ly + 1:], U, U_lo2, dgE[1:Ly + 1], r, 1, yoff)


def _capped(Lx, Ly):
    """the launchers' formulas (csrc/wilson.cu, csrc/wilson_rb2.cu): every CTA / warp loops, the last pass is partial"""
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
    S2 = Lx // 2 * Ly
    assert -(-S2 // 256) > sms() * 32, "wilson_rb_kernel is not in the capped regime"


def _tm_case(Lx, Ly, dtype, strip, yoff, seed, clover, mu=0.0173, capped=False):
    """apply (APPLY, RESID with fused dots), the two-colour sweep with and without r, both colours of the half sweep"""
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
    k = lambda t: t.to(CT[dtype]).contiguous()
    Uk, pk, rk = k(Ug).reshape(S, 2), k(pg).reshape(S, 2), k(rg).reshape(S, 2)
    lo2k, hi2k, Ulo2k, Uhik, rlok, rhik = k(lo2), k(hi2), k(U_lo2), k(U_hi), k(r_lo), k(r_hi)
    if clover:
        F = torch.empty(S, dtype=RT[dtype], device="cuda")
        call("mg2d_clover_field", P_(F), P_(Uk), P_(Ulo2k[1:]), P_(Uhik), csw, Lx, Ly, dtype, S_())
        if strip:
            F_lo, F_hi = (torch.randn((1, Lx), dtype=torch.float64, device="cuda", generator=g) * 0.3).to(RT[dtype]), \
                         (torch.randn((1, Lx), dtype=torch.float64, device="cuda", generator=g) * 0.3).to(RT[dtype])
        else:
            F_lo, F_hi = F.reshape(Ly, Lx)[-1:].clone(), F.reshape(Ly, Lx)[:1].clone()
        Fg, Flo, Fhi = F.reshape(Ly, Lx).double(), F_lo.double(), F_hi.double()
    else:
        F = F_lo = F_hi = None
        Fg, Flo, Fhi = (torch.zeros((n, Lx), dtype=torch.float64, device="cuda") for n in (Ly, 1, 1))
    tw = twist(mu, "cuda")
    dg = self_ref(Fg, m) + tw
    dgE = self_ref(torch.cat([Flo, Fg, Fhi], dim=0), m) + tw
    tol = TOL if dtype == C128 else TOL32
    if capped:
        _capped(Lx, Ly)
    what = (Lx, Ly, dtype, strip, clover)
    # apply; residual with the fused dots
    want = hop_ref(pg, lo2, hi2, Ug, U_lo2) + dg * pg
    out = torch.empty_like(pk)
    call("mg2d_wilson_tm_apply", P_(out), P_(pk), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(F), None, m, mu, Lx, Ly, 0,
         dtype, None, S_())
    assert rel(out, want) < tol, what + ("apply",)
    d = torch.zeros(4, dtype=torch.float64, device="cuda")
    call("mg2d_wilson_tm_apply", P_(out), P_(pk), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(F), P_(rk), m, mu, Lx, Ly, 1,
         dtype, P_(d), S_())
    res = rg - want
    assert rel(out, res) < tol, what + ("resid",)
    o64 = out.to(torch.complex128).reshape(-1)
    d = d.cpu().numpy()
    n2, ip, b2 = float((o64.abs() ** 2).sum()), complex(torch.vdot(o64, pg.reshape(-1))), float((rg.abs() ** 2).sum())
    assert abs(d[0] / n2 - 1) < TOL and abs(d[3] / b2 - 1) < TOL
    assert abs(complex(d[1], d[2]) - ip) < TOL * math.sqrt(n2 * float((pg.abs() ** 2).sum()))
    del out, o64, res, want
    # the one-pass two-colour sweep, with and without r
    for with_r in (True, False):
        o = torch.empty_like(pk)
        call("mg2d_wilson_tm_relax_rb2", P_(o), P_(pk), P_(lo2k), P_(hi2k), P_(Uk), P_(Ulo2k), P_(Uhik), P_(F), P_(F_lo), P_(F_hi),
             P_(rk if with_r else None), P_(rlok if with_r else None), P_(rhik if with_r else None), m, mu, Lx, Ly, yoff, dtype,
             None, S_())
        want = rb2_tm(pg, lo2, hi2, Ug, U_lo2, U_hi, dgE, rg if with_r else None, r_lo, r_hi, yoff)
        assert rel(o, want) < tol, what + ("rb2", with_r)
        del o, want
    # the half sweep (in place), both colours in turn
    ph = pk.clone()
    cur = pg
    for colour in (0, 1):
        call("mg2d_wilson_tm_relax_rb", P_(ph), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(F), P_(rk), m, mu, Lx, Ly,
             colour, yoff, dtype, S_())
        cur = half_tm(cur, lo2, hi2, Ug, U_lo2, dg, rg, colour, yoff)
        assert rel(ph, cur) < tol, what + ("rb", colour)


@pytest.mark.gpu
@pytest.mark.parametrize("clover", [False, True])
@pytest.mark.parametrize("Lx,Ly", [(6, 4), (34, 18), (130, 66), (256, 256)])
def test_tm_kernels_small(Lx, Ly, clover):
    for dtype in (C128, C64):
        _tm_case(Lx, Ly, dtype, False, 0, Lx * 7 + Ly, clover)


@pytest.mark.gpu
@pytest.mark.parametrize("clover", [False, True])
@pytest.mark.parametrize("dtype", [C128, C64])
def test_tm_kernels_4096(dtype, clover, gpu_mem):
    _tm_case(4096, 4096, dtype, False, 0, 21, clover)


@pytest.mark.gpu
@pytest.mark.parametrize("clover", [False, True])
def test_tm_kernels_capped_grid(clover, gpu_mem):
    """A ragged lattice large enough that the apply, the two-colour sweep and the half sweep all run on capped grids."""
    _tm_case(5000, 4128, C128, False, 0, 22, clover, capped=True)


@pytest.mark.gpu
@pytest.mark.parametrize("clover", [False, True])
@pytest.mark.parametrize("Ly,yoff,dtype", [(512, 1, C128), (512, 1, C64), (3, 1, C128)])
def test_tm_kernels_strips_explicit_halos(Ly, yoff, dtype, clover, gpu_mem):
    """Strips with explicit random halo rows of phi (two deep), links, r and the clover field."""
    _tm_case(4096 if Ly > 3 else 64, Ly, dtype, True, yoff, 23 + Ly, clover)


@pytest.mark.gpu
@pytest.mark.parametrize("clover", [False, True])
@pytest.mark.parametrize("L,Ly", [(4096, 512), (1024, 128), (256, 32)])
def test_tm_strips_equal_whole_lattice(L, Ly, clover, gpu_mem):
    """The 8-rank strips (an interior one and the last) with their real neighbour rows reproduce the whole lattice's rows
    of apply, residual, the two-colour sweep and each colour of the half sweep bit for bit."""
    m, mu, C = -0.05, 0.011, C128
    S = L * L
    g = gen(40 + L + clover)
    U = links(g, L, L).reshape(S, 2).contiguous()
    phi, r = crandn(g, S, 2), crandn(g, S, 2)
    row = lambda t, y: P_(t[(y % L) * L:])
    F = None
    if clover:
        F = torch.empty(S, dtype=torch.float64, device="cuda")
        call("mg2d_clover_field", P_(F), P_(U), row(U, -1), row(U, 0), 1.0, L, L, C, S_())
    fr = lambda y: None if F is None else row(F, y)
    ap, rs, sw = torch.empty_like(phi), torch.empty_like(phi), torch.empty_like(phi)
    call("mg2d_wilson_tm_apply", P_(ap), P_(phi), row(phi, -1), row(phi, 0), P_(U), row(U, -1), P_(F), None, m, mu, L, L, 0, C,
         None, S_())
    call("mg2d_wilson_tm_apply", P_(rs), P_(phi), row(phi, -1), row(phi, 0), P_(U), row(U, -1), P_(F), P_(r), m, mu, L, L, 1, C,
         None, S_())
    call("mg2d_wilson_tm_relax_rb2", P_(sw), P_(phi), row(phi, -2), row(phi, 0), P_(U), row(U, -2), row(U, 0), P_(F), fr(-1), fr(0),
         P_(r), row(r, -1), row(r, 0), m, mu, L, L, 0, C, None, S_())
    half = []
    for colour in (0, 1):
        h = phi.clone()
        call("mg2d_wilson_tm_relax_rb", P_(h), row(h, -1), row(h, 0), P_(U), row(U, -1), P_(F), P_(r), m, mu, L, L, colour, 0, C,
             S_())
        half.append(h)
    for y0 in (3 * Ly, L - Ly):
        rows = slice(y0 * L, (y0 + Ly) * L)
        y1 = y0 + Ly
        Fs = None if F is None else F[rows]
        fs = lambda y: None if F is None else row(F, y)
        o = torch.empty((Ly * L, 2), dtype=torch.complex128, device="cuda")
        call("mg2d_wilson_tm_apply", P_(o), P_(phi[rows]), row(phi, y0 - 1), row(phi, y1), P_(U[rows]), row(U, y0 - 1), P_(Fs), None,
             m, mu, L, Ly, 0, C, None, S_())
        assert torch.equal(o, ap[rows]), (y0, "apply")
        call("mg2d_wilson_tm_apply", P_(o), P_(phi[rows]), row(phi, y0 - 1), row(phi, y1), P_(U[rows]), row(U, y0 - 1), P_(Fs),
             P_(r[rows]), m, mu, L, Ly, 1, C, None, S_())
        assert torch.equal(o, rs[rows]), (y0, "resid")
        # (the two-row halos of the last strip are rows 0, 1: contiguous in the whole field)
        call("mg2d_wilson_tm_relax_rb2", P_(o), P_(phi[rows]), row(phi, y0 - 2), row(phi, y1), P_(U[rows]), row(U, y0 - 2), row(U, y1),
             P_(Fs), fs(y0 - 1), fs(y1), P_(r[rows]), row(r, y0 - 1), row(r, y1), m, mu, L, Ly, y0 & 1, C, None, S_())
        assert torch.equal(o, sw[rows]), (y0, "rb2")
        for colour in (0, 1):
            h = phi[rows].clone()
            call("mg2d_wilson_tm_relax_rb", P_(h), row(phi, y0 - 1), row(phi, y1), P_(U[rows]), row(U, y0 - 1), P_(Fs), P_(r[rows]),
                 m, mu, L, Ly, colour, y0 & 1, C, S_())
            assert torch.equal(h, half[colour][rows]), (y0, "rb", colour)
        del o


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("clover", [False, True])
def test_tm_entry_points_at_zero_mu_equal_wilson_and_sw(dtype, clover):
    """mu = 0 through the tm entry points gives the Wilson (F NULL) or SW entry points' results to rounding.  (A hierarchy
    with mu = 0 never calls the tm entry points.)"""
    Lx, Ly, m = 130, 66, 0.03
    S = Lx * Ly
    tol = 4e-16 * 4 if dtype == C128 else 6e-8 * 8
    g = gen(32)
    U = links(g, Ly, Lx, dtype).to(CT[dtype]).reshape(S, 2).contiguous()
    phi, r = crandn(g, S, 2).to(CT[dtype]), crandn(g, S, 2).to(CT[dtype])
    lo2, hi2, Ulo2, Uhi = phi[(Ly - 2) * Lx:], phi, U[(Ly - 2) * Lx:], U
    rlo, rhi = r[(Ly - 1) * Lx:], r
    F = Flo = Fhi = None
    if clover:
        F = torch.empty(S, dtype=RT[dtype], device="cuda")
        call("mg2d_clover_field", P_(F), P_(U), P_(Ulo2[Lx:]), P_(Uhi), 1.0, Lx, Ly, dtype, S_())
        Flo, Fhi = F[(Ly - 1) * Lx:], F
    sfx = "_sw" if clover else ""
    fa = (P_(F),) if clover else ()
    for mode, b in ((0, None), (1, r)):
        a, c = torch.empty_like(phi), torch.empty_like(phi)
        da, dc = torch.zeros(4, dtype=torch.float64, device="cuda"), torch.zeros(4, dtype=torch.float64, device="cuda")
        call(f"mg2d_wilson{sfx}_apply", P_(a), P_(phi), P_(lo2[Lx:]), P_(hi2), P_(U), P_(Ulo2[Lx:]), *fa, P_(b), m, Lx, Ly, mode,
             dtype, P_(da), S_())
        call("mg2d_wilson_tm_apply", P_(c), P_(phi), P_(lo2[Lx:]), P_(hi2), P_(U), P_(Ulo2[Lx:]), P_(F), P_(b), m, 0.0, Lx, Ly, mode,
             dtype, P_(dc), S_())
        assert rel(c, a) <= tol, mode
        assert float((dc - da).abs().max()) <= max(1e-13, 2 * tol) * float(da.abs().max()), mode
    fa2 = (P_(F), P_(Flo), P_(Fhi)) if clover else ()
    for rr in (r, None):
        a, c = torch.empty_like(phi), torch.empty_like(phi)
        rl, rh = (rlo, rhi) if rr is not None else (None, None)
        call(f"mg2d_wilson{sfx}_relax_rb2", P_(a), P_(phi), P_(lo2), P_(hi2), P_(U), P_(Ulo2), P_(Uhi), *fa2, P_(rr), P_(rl), P_(rh), m,
             Lx, Ly, 1, dtype, None, S_())
        call("mg2d_wilson_tm_relax_rb2", P_(c), P_(phi), P_(lo2), P_(hi2), P_(U), P_(Ulo2), P_(Uhi), P_(F), P_(Flo), P_(Fhi), P_(rr),
             P_(rl), P_(rh), m, 0.0, Lx, Ly, 1, dtype, None, S_())
        assert rel(c, a) <= 4 * tol                  # (the black stage reads the red stage's values)
        a, c = phi.clone(), phi.clone()
        for colour in (0, 1):
            call(f"mg2d_wilson{sfx}_relax_rb", P_(a), P_(a[(Ly - 1) * Lx:]), P_(a), P_(U), P_(Ulo2[Lx:]), *fa, P_(rr), m, Lx, Ly,
                 colour, 0, dtype, S_())
            call("mg2d_wilson_tm_relax_rb", P_(c), P_(c[(Ly - 1) * Lx:]), P_(c), P_(U), P_(Ulo2[Lx:]), P_(F), P_(rr), m, 0.0, Lx, Ly,
                 colour, 0, dtype, S_())
        assert rel(c, a) <= 4 * tol


# ---- the stored operator ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_twist_add_gives_the_restated_operator(csw):
    L, m, mu = 32, -0.04, 0.021
    U = O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))
    lvo = _dense(U, L, m=m, csw=csw)[0]
    add_twist(lvo, mu)
    for dt in ("complex128", "complex64"):
        p = mg2d.make_params(L, m, nlevels=1, csw=csw, mu=mu, matrix_free=False, dtype=dt)
        mg = mg2d.MG(p)
        mg.set_gauge(torch.as_tensor(U).cuda())
        D = mg2d.D_to_reference_layout(mg.LVL[0].D).to(torch.complex128).cpu().numpy()
        if dt == "complex128":
            # Wilson blocks and clover from their own kernels; the twist adds exactly i mu to the imaginary parts (zero before)
            assert np.array_equal(D.imag[:, 0, 0, 0], np.full(L * L, mu)) and np.array_equal(D.imag[:, 0, 1, 1], np.full(L * L, -mu))
            assert np.max(np.abs(D - lvo.D)) <= TOL * np.max(np.abs(lvo.D))
        else:
            assert np.max(np.abs(D - lvo.D)) <= TOL32 * np.max(np.abs(lvo.D))
        mg.close()
    # the entry point by itself, on a random stored operator: exactly +i mu / -i mu on the two self-block diagonals
    for dtype in (C128, C64):
        D = crandn(gen(9), L * L, 5, 2, 2).to(CT[dtype])
        D0 = D.clone()
        call("mg2d_twist_add", P_(D), mu, L * L, dtype, S_())
        want = D0.clone()
        want[:, 0, 0, 0] += 1j * torch.tensor(mu, dtype=RT[dtype])
        want[:, 0, 1, 1] -= 1j * torch.tensor(mu, dtype=RT[dtype])
        assert torch.equal(D, want), dtype


# ---- the norm identity -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("clover", [False, True])
def test_norm_identity_4096(clover, gpu_mem):
    """|D_tm x|^2 = |D x|^2 + mu^2 |x|^2 for random x (complex128), to 1e-12 relative: the cross term <D x, i mu g5 x> is
    purely imaginary because D is gamma5-hermitian."""
    L, m, mu = 4096, -0.06, 0.013
    S = L * L
    g = gen(50 + clover)
    U = links(g, L, L).reshape(S, 2).contiguous()
    x = crandn(g, S, 2)
    row = lambda t, y: P_(t[(y % L) * L:])
    F = None
    if clover:
        F = torch.empty(S, dtype=torch.float64, device="cuda")
        call("mg2d_clover_field", P_(F), P_(U), row(U, -1), row(U, 0), 1.0, L, L, C128, S_())
    a, b = torch.empty_like(x), torch.empty_like(x)
    call("mg2d_wilson_tm_apply", P_(a), P_(x), row(x, -1), row(x, 0), P_(U), row(U, -1), P_(F), None, m, mu, L, L, 0, C128, None,
         S_())
    call("mg2d_wilson_tm_apply", P_(b), P_(x), row(x, -1), row(x, 0), P_(U), row(U, -1), P_(F), None, m, 0.0, L, L, 0, C128, None,
         S_())
    na, nb, nx = (float(torch.linalg.vector_norm(t) ** 2) for t in (a, b, x))
    assert abs(na - (nb + mu * mu * nx)) <= 1e-12 * na, (na, nb, nx)


# ---- the Galerkin identity ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("quad", [1, 2, 3, 4])
def test_galerkin_carries_the_twist_to_every_level(quad):
    """Setups at mu and at 0 from the same supplied null vectors: on every coarse level self(mu) - self(0) = i mu Gamma5_c
    (Gamma5_c = diag(+1 x n/2, -1 x n/2)) to 1e-12 max|D|, the face blocks agree to rounding, and every projector is
    chirality-split (the identity rests on it)."""
    L, m, mu = 64, 0.02, 0.031
    U = torch.as_tensor(O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=30))).cuda()
    kw = dict(nlevels=3, block=[4, 2, 2], n_null=4, n_smooth=2, smoother="rbgs", null_iters=20, quad=quad, matrix_free=False)
    m0 = mg2d.setup(U, mg2d.make_params(L, m, **kw), init="device")
    nulls = [lv.phi_null.clone() for lv in m0.LVL[:3]]
    m0.close()
    a = mg2d.setup(U, mg2d.make_params(L, m, **kw), null_vectors=nulls)
    t = mg2d.setup(U, mg2d.make_params(L, m, mu=mu, **kw), null_vectors=nulls)
    for lvl in range(3):
        P = a.LVL[lvl].phi_null                                    # [S, nc, nf]
        h, hf = P.shape[1] // 2, P.shape[2] // 2
        assert float(P[:, :h, hf:].abs().max()) == 0.0 and float(P[:, h:, :hf].abs().max()) == 0.0, lvl
        assert torch.equal(P, t.LVL[lvl].phi_null), lvl
    for lvl in range(1, 4):
        Da, Dt = a.LVL[lvl].D, t.LVL[lvl].D                        # [S, 5, n, n]
        n = Da.shape[-1]
        g5 = torch.tensor([1.0] * (n // 2) + [-1.0] * (n // 2), dtype=torch.complex128, device="cuda")
        scale = float(Da.abs().max())
        assert float((Dt[:, 0] - Da[:, 0] - torch.diag(1j * mu * g5)).abs().max()) <= 1e-12 * scale, lvl
        assert float((Dt[:, 1:] - Da[:, 1:]).abs().max()) <= 1e-14 * scale, lvl
    a.close()
    t.close()


# ---- solves ------------------------------------------------------------------------------------------------------------
def _quenched(L, sweeps=30, seed=1234):
    return O.gauge_from_phases(O.gauge_quenched_phases(L, 6.0, sweeps=sweeps, seed=seed))


@pytest.mark.gpu
@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_reference_gs_flow_with_twist(csw):
    """The reference's flow (random start, GS smoother on the stored operator, stationary cycle) with the twist added to the
    oracle's level 0."""
    L, m, mu = 32, 0.02, 0.05
    U = _quenched(L)
    po = O.Params(L=L, num_iters=3, block=2, m=m, nlevels=2, null_iters=40, max_iters=300, res_threshold=1e-12)
    LVLo, NTLo = O.build_reference_problem(po, U)
    add_clover(LVLo[0], U, L, csw)
    add_twist(LVLo[0], mu)
    O.compute_near_null(LVLo, NTLo, po, po.quad)
    io = O.perform_MG(LVLo, NTLo, po)
    p = mg2d.make_params(L, m, nlevels=2, n_smooth=3, null_iters=40, max_iters=300, tol=1e-12, csw=csw, mu=mu)
    mg, ig = mg2d.run_reference_flow(p, torch.as_tensor(U).cuda())
    assert io["converged"] and ig["converged"] and ig["iters"] == io["iters"], (ig["iters"], io["iters"])
    x = mg.LVL[0].phi.cpu().numpy()
    assert np.max(np.abs(x - LVLo[0].phi)) < 1e-9 * np.max(np.abs(LVLo[0].phi))
    mg.close()


def _bench_like(L, m, mu, **kw):
    nlevels = max(1, int(round(math.log(L / 16, 4))))
    post = ([4, 2, 6] + [4] * nlevels)[:nlevels + 1]
    return mg2d.make_params(L, m, nlevels=nlevels, block=4, n_null=8, n_smooth=4, n_pre=0, n_post=post, smoother="rbgs",
                            null_iters=100, tol=1e-10, max_iters=500, mu=mu, **kw)


_MCRIT = {}


def _mcrit(L, U):
    if L not in _MCRIT:
        from importlib import import_module
        critical = import_module("2d_multigrid_b200.critical")
        _MCRIT[L], _ = critical.estimate_critical_mass(U, lambda m: _bench_like(L, m, 0.0), iters=4, refine=3)
    return _MCRIT[L]


@pytest.mark.gpu
@pytest.mark.parametrize("L,mu", [(64, 1e-2), (256, 1e-2), (256, 1e-3)])
def test_maximal_twist_solves(L, mu):
    """Quenched beta = 6 links at m = m_crit(mu = 0): FGCR(8) with the bench's cycle (its hierarchy for L: one coarse level
    at 64^2, two at 256^2) converges to a true residual <= 1e-10; the matrix-free and stored paths, and CUDA graphs on and
    off, take the same iterations; the complex64 preconditioner converges; the solution matches a sparse direct solve of the
    restated operator: within |b - D x| / |mu| (no singular value of D is below |mu|) and, at 64^2, to 1e-9.  (At 64^2 with mu = 1e-3 the one-coarse-level hierarchy, whose coarsest level is only
    relaxed, stalls above the tolerance in 500 iterations: the test takes that mu on the deeper 256^2 hierarchy.)"""
    import scipy.sparse.linalg as spla
    Un = _quenched(L, sweeps=200)
    U = torch.as_tensor(Un).cuda()
    mc = _mcrit(L, U)
    b = torch.zeros((L * L, 2), dtype=torch.complex128, device="cuda")
    b[L // 2 + (L // 2) * L, 0] = 1.0
    mgf = mg2d.setup(U, _bench_like(L, mc, mu), init="device")
    assert mgf.LVL[0].matrix_free
    nulls = [lv.phi_null.clone() for lv in mgf.LVL[:-1]]
    x, info = mg2d.solve(mgf, rhs=b, tol=1e-10, outer="gcr", restart=8)
    x = x.clone()
    assert info["converged"] and info["true_resnorm"] <= 1e-10, info
    _, ig = mg2d.solve(mgf, rhs=b, tol=1e-10, outer="gcr", restart=8, use_graph=True)
    assert ig["iters"] == info["iters"] and ig["true_resnorm"] <= 1e-10
    _, i32 = mg2d.solve(mgf, rhs=b, tol=1e-10, outer="gcr", restart=8, use_graph=True, precond_dtype="complex64")
    assert i32["converged"] and i32["true_resnorm"] <= 1e-10, i32
    mgs = mg2d.setup(U, _bench_like(L, mc, mu, matrix_free=False), null_vectors=nulls)
    assert not mgs.LVL[0].matrix_free
    _, i_s = mg2d.solve(mgs, rhs=b, tol=1e-10, outer="gcr", restart=8)
    assert i_s["iters"] == info["iters"], (i_s["iters"], info["iters"])
    xd = spla.spsolve(sparse_tm(Un, L, mc, 0.0, mu).tocsc(), b.cpu().numpy().reshape(-1))
    err = x.cpu().numpy().reshape(-1) - xd
    chk = torch.empty_like(x)
    mgf.LVL[0].apply_D(chk, x)
    assert np.linalg.norm(err) <= (1 + 1e-6) * float(torch.linalg.vector_norm(b - chk)) / mu
    if L == 64:
        assert np.max(np.abs(err)) < 1e-9 * np.max(np.abs(xd))
    mgf.close()
    mgs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("csw", [0.0, 1.0])
def test_strip_code_with_twist_equals_single_gpu(fused, csw):
    """The strip code with the rank as its own neighbour (fused or standalone smoother halos): the linked / standalone
    twisted two-colour sweep equals the single-GPU sweep, and the solve takes the same iterations to the same solution."""
    from importlib import import_module
    dmod = import_module("2d_multigrid_b200.dist")
    L, mu = 128, 3e-3
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=20, seed=1234, device=0)
    p = mg2d.make_params(L, 0.0, nlevels=2, block=4, n_null=8, n_smooth=3, n_pre=0, n_post=[4, 2, 8], smoother="rbgs",
                         null_iters=40, tol=1e-10, max_iters=100, csw=csw, mu=mu)
    rhs = torch.zeros((L * L, 2), dtype=torch.complex128, device="cuda")
    rhs[L // 2 + (L // 2) * L, 0] = 1.0
    ref = mg2d.setup(U, p, init="device")
    x_ref, i_ref = mg2d.solve(ref, rhs=rhs, tol=1e-10, outer="gcr")
    x_ref = x_ref.clone()
    comm = dmod.Comm.single(mg2d.Context(0), torch.device("cuda", 0))
    comm.fused = fused
    dmg = dmod.setup(U, p, comm, min_rows=16)
    lv0, rl0 = dmg.LVL[0], ref.LVL[0]
    assert lv0.distributed and lv0.matrix_free and rl0.matrix_free
    rows = slice(lv0.y0 * L, (lv0.y0 + lv0.Ly) * L)
    g = gen(61)
    ph, r = crandn(g, L * L, 2), crandn(g, L * L, 2)
    a, b = ph.clone(), ph[rows].clone()
    rl0.relax(3, smoother="rbgs", phi=a, r=r)
    lv0.relax(3, smoother="rbgs", phi=b, r=r[rows].clone())
    assert rel(b, a[rows]) < TOL          # (the linked sweep is another instantiation: equal to rounding, not bit for bit)
    x, info = mg2d.solve(dmg, rhs=rhs, tol=1e-10, outer="gcr")
    assert info["converged"] and info["iters"] == i_ref["iters"], (info["iters"], i_ref["iters"])
    dx = float((x - x_ref[rows]).abs().max() / x_ref.abs().max())
    assert dx < 1e-9 and info["true_resnorm"] < 1e-10, dx
    ref.close()
    dmg.close()
