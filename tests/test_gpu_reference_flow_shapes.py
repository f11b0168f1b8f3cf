"""The reference flow's own kernels at the baseline configurations' shapes against an fp64 reference.

The reference flow (mg2d.py, the BASELINE configurations, `smoother="gs" | "jacobi" | "mr"`, `ntl=True`) runs on kernels
the benchmark never calls: lexicographic Gauss-Seidel as anti-diagonal wavefronts in one cooperative launch
(mg2d_relax_gs), the Jacobi sweep and the MR smoother (mg2d_stencil_apply with per-vector fused dots + mg2d_mr_update),
the non-telescoping min-res weighting (mg2d_minres_solve, mg2d_scale_phi) and the scalar-Laplace multigrid of
csrc/scalar.cu.  At 16^2 a wavefront fits one CTA and a batched reduction one pass, so a lost barrier between CTAs or a
crossed reduction channel still converges there; these tests run the shapes where the fronts span several CTAs (several
rounds for batched vectors), the grids are capped and the Gram matrices are degenerate.

Each operation is restated from its definition as vectorised fp64 torch on whatever device the tensors are on; the CPU
tests anchor the restatements to the numpy oracle, the GPU tests hold the kernels to them on seeded synthetic operators
built on the device.  Tolerances, relative in the max-norm: complex128 1e-12; complex64 2e-5 against the fp64 reference
of the fp32-rounded inputs.  The scalar Gauss-Seidel claims the reference's summation order with exact a^2 = 4^level, so
it must equal the oracle bit for bit.  Every capped or multi-round case asserts so from the launcher's own formula.
"""
import importlib
import math

import numpy as np
import pytest
import torch

import mg2d
from oracle import mg_oracle as O
from oracle import scalar_s2 as S2
from test_gpu_bench_shapes import (C64, C128, CT, TOL, TOL32, P_, S_, _c, _diag_dominant, _maxrel, _periodic_halos, _t,
                                   assert_capped, call, crandn, gen, hop_dense, neighbours, rel, rounded, sms)

ST_THREADS = 256
GPB = {1: 256, 2: 64, 4: 16, 8: 8, 16: 8, 32: 8}      # sites per 256-thread CTA of the block stencil (GroupOf<N> lanes per site)
MAX_CTAS_PER_SM = 2048 // ST_THREADS                    # occupancy ceiling of a cooperative 256-thread launch


@pytest.fixture
def gpu_mem():
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    yield
    print(f"\npeak device memory {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ================================================================================================================
# fp64 reference.  Fields [nv, S, n] (site s = x + y*L); operator blocks in math layout Dm [S, 5, n, n]
# (the device stores them column-major: Dm = D_dev.transpose(-1, -2)); D0inv [S, n, n] in math layout.
# ================================================================================================================
def front(L, c, device):
    """sites of the anti-diagonal x + y = c and their four neighbours (slots 1..4: x+1, x-1, y+1, y-1, periodic)"""
    x = torch.arange(max(0, c - L + 1), min(c, L - 1) + 1, device=device)
    y = c - x
    return y * L + x, (y * L + (x + 1) % L, y * L + (x - 1) % L, ((y + 1) % L) * L + x, ((y - 1) % L) * L + x)


def gs_sweeps(phi, Dm, D0inv, r, L, num_iter):
    """f_relax with gs_flag = 1 (S6/level.h:113-123): x outer, y inner.  For the 5-point stencil with periodic wrap that
    order is the wavefront order c = x + y = 0 .. 2L-2: every site of front c reads fronts c-1 (new) and c+1 (old), and the
    wrap neighbours (x = 0 <- x = L-1 etc.) lie on fronts already updated or not, exactly as in the sequential loop.
    Returns the state after each sweep.  r None means r = 0."""
    out, states = phi.to(torch.complex128, copy=True), []
    fronts = [front(L, c, phi.device) for c in range(2 * L - 1)]
    for _ in range(num_iter):
        for s, nb in fronts:
            acc = sum(torch.einsum("sij,vsj->vsi", Dm[s, k + 1], out[:, nb[k]]) for k in range(4))
            if r is not None:
                acc = acc - r[:, s]
            out[:, s] = -torch.einsum("sij,vsj->vsi", D0inv[s], acc)
        states.append(out.clone())
    return states


def _grid(f, L):
    return f.reshape(f.shape[0], L, -1, f.shape[-1])


def hop(Dm, f, L, lo=None, hi=None):
    """sum_{k=1..4} D_k(s) f(s+d_k) on an L-wide strip; lo / hi: rows below / above ([nv, 1, L, n]), else periodic"""
    g = _grid(f, L)
    h = _periodic_halos(g) if lo is None else (lo, hi)
    return hop_dense(Dm.reshape(g.shape[1], L, 5, *Dm.shape[-2:]), neighbours(g, *h)).reshape(f.shape)


def apply_D(Dm, f, L):
    """f_apply_D (S6/level.h:251-265)"""
    return hop(Dm, f, L) + torch.einsum("sij,vsj->vsi", Dm[:, 0], f)


def jacobi(phi, Dm, D0inv, r, L):
    """f_relax with gs_flag = 0, one sweep"""
    acc = hop(Dm, phi, L)
    if r is not None:
        acc = acc - r
    return -torch.einsum("sij,vsj->vsi", D0inv, acc)


def mr(phi, Dm, r, L, num_iter, omega):
    """Level.relax_mr per vector: res = r - D phi; t = D res; alpha = omega <t,res>/<t,t>; phi += alpha res; res -= alpha t.
    The oracle stops at <t,t> = 0; alpha = 0 for that vector is the same thing."""
    phi = phi.to(torch.complex128, copy=True)
    res = r - apply_D(Dm, phi, L)
    for _ in range(num_iter):
        t = apply_D(Dm, res, L)
        tt = t.abs().square().sum((1, 2))
        tr = (t.conj() * res).sum((1, 2))
        alpha = torch.where(tt > 0, omega * tr / torch.where(tt > 0, tt, 1), 0)[:, None, None]
        phi += alpha * res
        res -= alpha * t
    return phi


def s2_residue(phi, b, L, scale, a):
    """S2:30-35: b - (1/a^2)(sum of the 4 neighbours - phi/scale) on the periodic L x L lattice (fp64)"""
    g = phi.reshape(L, L)
    nb = g.roll(-1, 1) + g.roll(1, 1) + g.roll(-1, 0) + g.roll(1, 0)
    return b - (1.0 / (a * a)) * (nb.reshape(-1) - phi / scale)


def s2_quad_sites(L, quad, device):
    """the four fine sites of every coarse site X (f_projection / f_interpolate, S2:74-143): x in {2x, 2x+sx}, y in
    {2y, 2y+sy} mod L, (sx, sy) = (+1, +1), (-1, +1), (-1, -1), (+1, -1) for quadrants 1..4, in the order (xa,ya), (xa,yb),
    (xb,ya), (xb,yb)"""
    Lc = L // 2
    X = torch.arange(Lc * Lc, device=device)
    xa, ya = 2 * (X % Lc), 2 * (X // Lc)
    sx, sy = (1 if quad in (1, 4) else -1), (1 if quad in (1, 2) else -1)
    xb, yb = (xa + sx) % L, (ya + sy) % L
    return xa + ya * L, xa + yb * L, xb + ya * L, xb + yb * L


def s2_project(b, phi, L, scale, a, quad):
    rt = s2_residue(phi, b, L, scale, a)
    s = s2_quad_sites(L, quad, b.device)
    return 0.25 * (rt[s[0]] + rt[s[1]] + rt[s[2]] + rt[s[3]])


def s2_interpolate(phi_f, phi_c, L, quad):
    out = phi_f.clone()
    for s in s2_quad_sites(L, quad, phi_f.device):
        out[s] += phi_c
    return out


# ================================================================================================================
# CPU: the reference against the numpy oracle
# ================================================================================================================
def _oracle_level(rng, L, n):
    lvo = O.Level()
    lvo.D = _c(rng, L * L, 5, n, n) * (0.15 / math.sqrt(n))
    lvo.D[:, 0] = _c(rng, L * L, n, n) * 0.2 + 3.0 * np.eye(n)
    lvo.phi, lvo.r = _c(rng, L * L, n), _c(rng, L * L, n)
    return lvo


@pytest.mark.parametrize("L,n", [(6, 1), (8, 2), (7, 4)])
def test_reference_smoothers_match_oracle(L, n):
    """the wavefront GS restatement == Level.relax(gs_flag=1) (the sequential x-outer loop's order), Jacobi ==
    Level.relax(gs_flag=0), r = 0 == the oracle with a zero r; two sweeps each"""
    rng = np.random.default_rng(10 * L + n)
    lvo = _oracle_level(rng, L, n)
    Dm, phi, r = _t(lvo.D), _t(lvo.phi)[None], _t(lvo.r)[None]
    D0inv = torch.linalg.inv(Dm[:, 0])
    for gs_flag in (1, 0):
        for with_r in (True, False):
            o = O.Level()
            o.D, o.phi, o.r = lvo.D, lvo.phi.copy(), lvo.r if with_r else np.zeros_like(lvo.r)
            o.relax(L, 2, gs_flag)
            if gs_flag:
                got = gs_sweeps(phi, Dm, D0inv, r if with_r else None, L, 2)[-1]
            else:
                got = jacobi(jacobi(phi, Dm, D0inv, r if with_r else None, L), Dm, D0inv, r if with_r else None, L)
            assert _maxrel(got[0], o.phi) < 1e-13, (gs_flag, with_r)
    # the order matters: Jacobi and GS differ at O(1)
    assert _maxrel(gs_sweeps(phi, Dm, D0inv, r, L, 1)[0], jacobi(phi, Dm, D0inv, r, L)) > 1e-2


@pytest.mark.parametrize("omega", [1.0, 0.7])
def test_reference_mr_matches_oracle(omega):
    """the batched MR restatement == Level.relax_mr vector by vector, including a zero vector (the oracle breaks on
    <t,t> = 0, the restatement keeps it unchanged) and vectors 1e6 apart in scale"""
    rng = np.random.default_rng(3)
    L, n, nv = 8, 2, 4
    lvo = _oracle_level(rng, L, n)
    scales = [1.0, 1e3, 0.0, 1e-3]
    phi = np.stack([s * _c(rng, L * L, n) for s in scales])
    r = np.stack([s * _c(rng, L * L, n) for s in scales])
    got = mr(_t(phi), _t(lvo.D), _t(r), L, 3, omega)
    for v in range(nv):
        o = O.Level()
        o.D, o.phi, o.r = lvo.D, phi[v].copy(), r[v]
        o.relax_mr(L, 3, omega)
        if scales[v] == 0:
            assert not got[v].abs().max() and not np.abs(o.phi).max()
        else:
            assert _maxrel(got[v], o.phi) < 1e-13, v


@pytest.mark.parametrize("L", [8, 12])
def test_reference_scalar_operators_match_oracle(L):
    """projection (all quadrants), interpolate, residue magnitude == oracle.scalar_s2 at levels 0 and 1"""
    rng = np.random.default_rng(L)
    p = S2.S2Params(2 * L, 0.1, 2)
    for lev in (0, 1):
        Ll = p.size[lev]
        phi, b = rng.normal(size=Ll * Ll), rng.normal(size=Ll * Ll)
        args = (Ll, p.scale[lev], p.a[lev])
        assert abs(float(s2_residue(_t(phi), _t(b), *args).abs().sum()) / S2.get_residue_mag(phi, b, lev, p) - 1) < 1e-14
        for quad in (1, 2, 3, 4):
            assert _maxrel(s2_project(_t(b), _t(phi), *args, quad), S2.projection(b, phi, lev, p, quad)) < 1e-14
        if lev == 0:
            continue
        for quad in (1, 2, 3, 4):
            pf, pc = rng.normal(size=(2 * Ll) ** 2), rng.normal(size=Ll * Ll)
            want, pc_o = pf.copy(), pc.copy()
            S2.interpolate(want, pc_o, lev, p, quad)
            assert np.array_equal(s2_interpolate(_t(pf), _t(pc), 2 * Ll, quad).numpy(), want) and not pc_o.any()


def _scaled_system(rng, n, spread):
    """B diag(s): a well-conditioned B with column norms spread over `spread` decades, the order shuffled so that the
    pivoting has to find it"""
    s = np.logspace(-spread / 2, spread / 2, n)[rng.permutation(n)] if n > 1 else np.ones(1)
    return (_c(rng, n, n) + 2 * np.eye(n)) * s[None, :], _c(rng, n), s


def _degenerate_grams(rng, n):
    """exactly rank-deficient n x n systems and their rank: two identical copies (rows and columns q0, q1 equal; the
    copies are 1e-2 of the others so the rounding left in the eliminated column stays far below eps*n*max|R_kk|), a copy
    that is zero (its row and column vanish), the all-zero matrix"""
    out = []
    if n >= 3:
        E = _c(rng, 64, n)
        E[:, 0] *= 1e-2
        E[:, 1] = E[:, 0]
        G = E.conj().T @ (_c(rng, 64, 64) * 0.1 + 3 * np.eye(64)) @ E
        G[1], G[:, 1] = G[0], G[:, 0]
        out.append(("duplicate", G, _c(rng, n), n - 1))
    if n >= 2:
        G = _c(rng, n, n) + 2 * np.eye(n)
        q = n // 2
        G[q], G[:, q] = 0, 0
        out.append(("zero copy", G, _c(rng, n), n - 1))
    out.append(("zero", np.zeros((n, n), dtype=complex), _c(rng, n), 0))
    return out


@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_reference_minres_oracle(n):
    """colpiv_householder_qr_solve == numpy.linalg.solve on well-conditioned and column-scaled systems; on the degenerate
    ones it decides the expected rank (zero unknowns), and f_scale_phi's definition"""
    rng = np.random.default_rng(n)
    A, b, _ = _scaled_system(rng, n, 0)
    assert _maxrel(O.colpiv_householder_qr_solve(A, b), np.linalg.solve(A, b)) < 1e-13
    A, b, s = _scaled_system(rng, n, 12)
    assert _maxrel(O.colpiv_householder_qr_solve(A, b) * s, np.linalg.solve(A, b) * s) < 1e-12
    for what, G, src, rank in _degenerate_grams(rng, n):
        x = O.colpiv_householder_qr_solve(G, src)
        assert int(np.sum(x == 0)) == n - rank, what
    phi, e, a = _c(rng, 50, 2), _c(rng, n, 50, 2), _c(rng, n)
    L1, NTL = O.Level(), [[O.Level() for _ in range(n)]]
    L1.phi = phi.copy()
    for q in range(n):
        NTL[0][q].phi = e[q].copy()
    O.scale_phi(L1, NTL, a, n, 0)
    assert _maxrel(_t(phi) + torch.einsum("q,qsi->si", _t(a), _t(e)), L1.phi) < 1e-15
    assert all(not NTL[0][q].phi.any() for q in range(n))


# ================================================================================================================
# GPU
# ================================================================================================================
def _operator(g, S, n, dtype):
    """seeded stored operator D [S, 5, n, n] (device layout) of the fp32-rounded values for complex64, and D0^-1 (device
    layout) from those values: both the kernel and the reference use this inverse"""
    D = rounded(crandn(g, S, 5, n, n) * (0.15 / math.sqrt(n)), dtype)
    D[:, 0] = rounded(_diag_dominant(g, S, n), dtype)
    Dm = D.transpose(-1, -2)
    D0inv = rounded(torch.linalg.inv(Dm[:, 0]), dtype)
    return Dm, D0inv, D.to(CT[dtype]), D0inv.transpose(-1, -2).contiguous().to(CT[dtype])


def _per_vector_rel(got, want):
    return max(rel(got[v], want[v]) for v in range(want.shape[0]))


# ---- 1. lexicographic Gauss-Seidel --------------------------------------------------------------------------------
def _gs_case(L, n, nvec, dtypes, r_modes, seed, multi_round=False):
    S = L * L
    for dtype in dtypes:
        g = gen(seed + dtype)
        Dm, D0inv, Dd, D0d = _operator(g, S, n, dtype)
        phi0 = rounded(crandn(g, nvec, S, n), dtype)
        r = rounded(crandn(g, nvec, S, n), dtype)
        tol = TOL if dtype == C128 else TOL32
        for with_r in r_modes:
            want = gs_sweeps(phi0, Dm, D0inv, r if with_r else None, L, 3)
            for num_iter in (1, 3):
                phi = phi0.to(CT[dtype], copy=True)
                rd = r.to(CT[dtype]) if with_r else None
                call("mg2d_relax_gs", P_(phi), P_(Dd), P_(D0d), P_(rd), n, L, num_iter, dtype, nvec, S * n, S_())
                err = _per_vector_rel(phi, want[num_iter - 1])
                assert err < tol, (L, n, nvec, dtype, with_r, num_iter, err)
            del want
        del Dm, D0inv, Dd, D0d, phi0, r


def _assert_fronts_span_ctas(L, n, nvec):
    """the longest front (L sites x nvec vectors) needs >= 2 CTAs, and at most one per SM, so the launcher's
    min(ceil(L*nvec/GPB), per_sm*num_SMs) launches them all whatever the occupancy: the fronts cross CTAs"""
    need = -(-L * nvec // GPB[n])
    assert 2 <= need <= sms(), (L, n, nvec, need)


@pytest.mark.gpu
@pytest.mark.parametrize("L,n", [(1024, 2), (256, 16), (64, 2)])
def test_gs_baseline_shapes(L, n, gpu_mem):
    """config 4 level 0 stored (1024^2, n = 2), config 4 level 1 (256^2, n = 16), config 2 (64^2, n = 2): num_iter 1 and 3,
    r given and NULL, complex128 and complex64.  The two larger ones spread each front over several CTAs; config 2's
    front fits one."""
    if L > 64:
        _assert_fronts_span_ctas(L, n, 1)
    _gs_case(L, n, 1, (C128, C64), (True, False), 100 + L + n)


@pytest.mark.gpu
@pytest.mark.parametrize("L,n", [(512, 1), (256, 4), (128, 8), (64, 32)])
def test_gs_block_sizes(L, n, gpu_mem):
    """n = 1, 4, 8, 32 at sizes where 2-16 CTAs share a front"""
    _assert_fronts_span_ctas(L, n, 1)
    _gs_case(L, n, 1, (C128, C64), (True, False), 200 + L + n)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_gs_batched_multi_round(dtype, gpu_mem):
    """near-null generation's call: nvec = 80 vectors S*n apart, r = NULL.  The longest fronts hold L*nvec = 81920 work
    items, more than the 8 CTAs/SM * num_SMs * GPB groups a cooperative launch of 256-thread CTAs can ever have: every
    group takes several rounds per front and the last round is partial"""
    L, n, nvec = 1024, 2, 80
    assert L * nvec > MAX_CTAS_PER_SM * sms() * GPB[n], (L * nvec, sms())
    _gs_case(L, n, nvec, (dtype,), (False,), 300)


@pytest.mark.gpu
def test_gs_batched_small(gpu_mem):
    """nvec = 4 with r given: the per-vector offsets of phi and r"""
    _assert_fronts_span_ctas(256, 16, 4)
    _gs_case(256, 16, 4, (C128,), (True,), 310)


@pytest.mark.gpu
def test_gs_strip_self_neighbour_1024(gpu_mem):
    """One sweep of mg2d_relax_gs_strip, through Level.relax on a single rank that is its own strip neighbour (global
    fronts, the upper neighbour of the last row delivered through the halo buffer and its progress flag), equals
    mg2d_relax_gs bit for bit at config 4's levels 0 (1024^2, n = 2) and 1 (256^2, n = 16)."""
    dmod = importlib.import_module("2d_multigrid_b200.dist")
    p = mg2d.make_params(1024, 0.02, nlevels=1, block=4, n_null=8, smoother="gs", matrix_free=False)
    comm = dmod.Comm.single(mg2d.Context(0), torch.device("cuda", 0))
    dmg = dmod.DistMG(p, comm, min_rows=8)
    assert [d for d, _ in dmg.plan] == [True, True]
    g = gen(320)
    for lv, n in zip(dmg.LVL, (2, 16)):
        assert lv.distributed and lv.n == n and lv.Ly == lv.L
        Dm, _, Dd, _ = _operator(g, lv.S, n, C128)
        lv.D, lv.D0inv = Dd, None
        v, rr = crandn(g, lv.S, n), crandn(g, lv.S, n)
        strip = v.clone()
        lv.relax(1, phi=strip, r=rr, smoother="gs")
        whole = v.clone()
        call("mg2d_relax_gs", P_(whole), P_(Dd), P_(lv.D0inv), P_(rr), n, lv.L, 1, C128, 1, lv.S * n, S_())
        assert torch.equal(strip, whole), n
        assert not torch.equal(whole, v)
        del Dm, Dd
    assert comm.p2p_errors() == 0
    dmg.close()


# ---- 2. Jacobi and MR ------------------------------------------------------------------------------------------------
def _assert_stencil_capped(S, n):
    """launch_stencil: min(ceil(S/GPB), 4096) CTAs in x, each looping over >= 2 steps of GPB sites"""
    steps = -(-S // GPB[n])
    assert steps >= 2 * 4096, f"stencil_kernel {S} sites n = {n}: {steps} steps on {min(steps, 4096)} CTAs"


@pytest.mark.gpu
@pytest.mark.parametrize("L,n", [(1024, 2), (256, 16)])
@pytest.mark.parametrize("dtype", [C128, C64])
def test_jacobi(L, n, dtype, gpu_mem):
    """mg2d_relax_jacobi on the whole lattice (periodic halos, hstride = vstride = S*n), nvec 1 and 4, r given and NULL"""
    S = L * L
    _assert_stencil_capped(S, n)
    g = gen(400 + L + dtype)
    Dm, D0inv, Dd, D0d = _operator(g, S, n, dtype)
    tol = TOL if dtype == C128 else TOL32
    for nvec in (1, 4):
        phi = rounded(crandn(g, nvec, S, n), dtype)
        r = rounded(crandn(g, nvec, S, n), dtype)
        for with_r in (True, False):
            want = jacobi(phi, Dm, D0inv, r if with_r else None, L)
            inp, out = phi.to(CT[dtype]), torch.full((nvec, S, n), math.nan, dtype=CT[dtype], device="cuda")
            lo = P_(inp) + (L - 1) * L * n * inp.element_size()
            rd = r.to(CT[dtype]) if with_r else None
            call("mg2d_relax_jacobi", P_(out), P_(inp), lo, P_(inp), P_(Dd), P_(D0d), P_(rd),
                 n, L, L, dtype, nvec, S * n, S * n, S_())
            assert _per_vector_rel(out, want) < tol, (nvec, with_r)


@pytest.mark.gpu
def test_jacobi_strip_1024x128(gpu_mem):
    """Level.relax on a strip: 1024 x 128 rows [384, 512) of a 1024^2 lattice, n = 2, nvec = 4, halo rows as separate
    buffers hstride = L*n apart; equals the whole-lattice reference on those rows"""
    L, Ly, y0, n, nvec = 1024, 128, 384, 2, 4
    g = gen(410)
    Dm, D0inv, Dd, D0d = _operator(g, L * L, n, C128)
    phi, r = crandn(g, nvec, L * L, n), crandn(g, nvec, L * L, n)
    want = jacobi(phi, Dm, D0inv, r, L)
    rows = slice(y0 * L, (y0 + Ly) * L)
    Sl = Ly * L
    inp, rs = phi[:, rows].contiguous(), r[:, rows].contiguous()
    lo = phi[:, (y0 - 1) * L:y0 * L].contiguous()
    hi = phi[:, (y0 + Ly) * L:(y0 + Ly + 1) * L].contiguous()
    out = torch.full_like(inp, math.nan)
    call("mg2d_relax_jacobi", P_(out), P_(inp), P_(lo), P_(hi), P_(Dd[rows].contiguous()), P_(D0d[rows].contiguous()), P_(rs),
         n, L, Ly, C128, nvec, Sl * n, L * n, S_())
    assert _per_vector_rel(out, want[:, rows]) < TOL


_MR_SCALES = [1.0, 1e3, 0.0, 1e-3, 1e6, 1e-6, 10.0, 0.1]


@pytest.mark.gpu
@pytest.mark.parametrize("L,n", [(1024, 2), (256, 16)])
@pytest.mark.parametrize("dtype", [C128, C64])
def test_mr_smoother(L, n, dtype, gpu_mem):
    """Level.relax(3, smoother="mr") on a stored operator, nvec 1, 4, 8, omega 1.0 and 0.7.  In a batch vector 2 is zero
    (phi = r = 0: <t,t> = 0, it must stay exactly zero while the others move) and the others are 1e-6..1e6 apart in scale,
    so a dot read from another vector's reduction channel is an O(1) error in that vector's alpha."""
    S = L * L
    _assert_stencil_capped(S, n)
    p = mg2d.make_params(L, 0.1, nlevels=0, matrix_free=False, dtype="complex128" if dtype == C128 else "complex64")
    mg = mg2d.MG(p)
    lv = mg.LVL[0]
    g = gen(500 + L + dtype)
    Dm, _, Dd, _ = _operator(g, S, n, dtype)
    lv.n, lv.L, lv.Ly, lv.S = n, L, L, S
    lv.D, lv.D0inv, lv.M = Dd, None, None
    tol = TOL if dtype == C128 else TOL32
    for nvec in (1, 4, 8):
        sc = torch.tensor(_MR_SCALES[:nvec] if nvec > 1 else [1.0], dtype=torch.float64, device="cuda")[:, None, None]
        phi0 = rounded(crandn(g, nvec, S, n) * sc, dtype)
        r = rounded(crandn(g, nvec, S, n) * sc, dtype)
        for omega in (1.0, 0.7):
            mg.p.mr_omega = omega
            want = mr(phi0, Dm, r, L, 3, omega)
            phi = phi0.to(CT[dtype], copy=True)
            lv.relax(3, phi=phi if nvec > 1 else phi[0], r=r.to(CT[dtype]) if nvec > 1 else r[0].to(CT[dtype]), smoother="mr")
            for v in range(nvec):
                if float(sc[v]) == 0:
                    assert not phi[v].abs().max(), (nvec, omega)
                else:
                    assert rel(phi[v], want[v]) < tol, (nvec, omega, v, rel(phi[v], want[v]))
                    assert rel(phi[v], phi0[v]) > 1e-3
            del want
    mg.close()


# ---- 3. NTL min-res weighting ----------------------------------------------------------------------------------------
def _minres(A, b):
    n = A.shape[0]
    gram = torch.tensor(np.stack([A.real, A.imag], -1).reshape(-1), dtype=torch.float64, device="cuda")
    src = torch.tensor(np.stack([b.real, b.imag], -1).reshape(-1), dtype=torch.float64, device="cuda")
    a = torch.full((8,), math.nan, dtype=torch.float64, device="cuda")
    call("mg2d_minres_solve", P_(gram), P_(src), n, P_(a), S_())
    av = a.cpu().numpy()
    return av[0:2 * n:2] + 1j * av[1:2 * n:2]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3, 4])
def test_minres_solve(n):
    """mg2d_minres_solve against colpiv_householder_qr_solve: well conditioned (and numpy.linalg.solve), columns scaled
    over 12 decades (the pivot order matters: a rank threshold far above eps*n would drop the small columns), and exactly
    rank-deficient systems, where kernel and oracle must put the same unknowns to zero"""
    rng = np.random.default_rng(600 + n)
    for _ in range(4):
        A, b, _ = _scaled_system(rng, n, 0)
        x = _minres(A, b)
        assert _maxrel(x, O.colpiv_householder_qr_solve(A, b)) < TOL
        assert _maxrel(x, np.linalg.solve(A, b)) < TOL
        A, b, s = _scaled_system(rng, n, 12)
        x, xo = _minres(A, b), O.colpiv_householder_qr_solve(A, b)
        assert _maxrel(x * s, xo * s) < 1e-11, (x, xo)
        assert np.all(x != 0)
    for what, G, src, rank in _degenerate_grams(rng, n):
        x, xo = _minres(G, src), O.colpiv_householder_qr_solve(G, src)
        assert np.array_equal(x == 0, xo == 0) and int(np.sum(x == 0)) == n - rank, (what, x, xo)
        if rank:
            assert _maxrel(x, xo) < 1e-10, (what, x, xo)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_scale_phi_1024(dtype, gpu_mem):
    """mg2d_scale_phi at 1024^2, n = 2 (2^21 elements on a capped grid), ncopies 1..4, estride = S*n: phi += sum a_q e_q,
    every e_q zeroed, copies beyond ncopies untouched"""
    S, n = 1024 * 1024, 2
    N = S * n
    nb = -(-N // 256)
    assert_capped(N, min(nb, sms() * 8, 4096) * 256, "scale_phi_kernel")
    g = gen(700 + dtype)
    tol = TOL if dtype == C128 else TOL32
    for nc in (1, 2, 3, 4):
        phi0 = rounded(crandn(g, S, n), dtype)
        E0 = rounded(crandn(g, 4, S, n), dtype)
        a = torch.randn(2 * nc, dtype=torch.float64, device="cuda", generator=g)
        ac = torch.complex(a[0::2], a[1::2])
        want = phi0 + torch.einsum("q,qsi->si", rounded(ac, dtype) if dtype == C64 else ac, E0[:nc])
        phi, E = phi0.to(CT[dtype], copy=True), E0.to(CT[dtype], copy=True)
        call("mg2d_scale_phi", P_(phi), P_(E), N, P_(a), nc, N, dtype, S_())
        assert rel(phi, want) < tol, nc
        assert not E[:nc].abs().max() and torch.equal(E[nc:], E0[nc:].to(CT[dtype])), nc


@pytest.mark.gpu
def test_ntl_min_res_and_scale_phi_config3(gpu_mem):
    """min_res(mg, 4, 0) and scale_phi of mg.py at level 0 of a config-3-shaped hierarchy (Wilson 256^2, near-critical,
    ntl, 4 copies) against O.min_res / O.scale_phi on the same operator, residual and copy fields.  The oracle's
    scale_phi gets the kernel's weights, so the phi check holds mg2d_scale_phi alone to 1e-12."""
    L, nc = 256, 4
    U = mg2d.gauge.quenched_links_device(L, 6.0, sweeps=20, seed=1234, device=0)
    p = mg2d.make_params(L, -0.03, nlevels=3, block=4, n_null=8, ntl=True, n_copies=nc, matrix_free=False)
    mg = mg2d.MG(p)
    mg.init_fields()
    mg.set_gauge(U)
    lv = mg.LVL[0]
    g = gen(800)
    E = mg._ntl_fields(0)
    E.copy_(crandn(g, 4, lv.S, lv.n))
    lv.r.copy_(crandn(g, lv.S, lv.n))
    lv.phi.copy_(crandn(g, lv.S, lv.n))
    po = O.Params(L=L, num_iters=2, block=4, m=-0.03, nlevels=3)
    LV, NT = O.Level(), [[O.Level() for _ in range(nc)]]
    LV.D = mg2d.D_to_reference_layout(lv.D).cpu().numpy()
    LV.r, LV.phi = lv.r.cpu().numpy(), lv.phi.cpu().numpy()
    for q in range(nc):
        NT[0][q].phi = E[q].cpu().numpy()
    a = mg2d.mg.min_res(mg, nc, 0)
    av = a[:2 * nc].cpu().numpy()
    w = av[0::2] + 1j * av[1::2]
    wo = O.min_res([LV], NT, nc, 0, po)
    assert np.max(np.abs(w - wo)) < 1e-10 * np.max(np.abs(wo)), (w, wo)
    mg2d.mg.scale_phi(mg, lv, a, nc, 0)
    O.scale_phi(LV, NT, w, nc, 0)
    assert _maxrel(lv.phi.cpu(), LV.phi) < TOL
    assert not E.abs().max()
    mg.close()


# ---- 4. scalar-Laplace kernels ---------------------------------------------------------------------------------------
def _s2_relax_grid(L):
    """mg2d_s2_relax launches min(ceil(L/256), per_sm*num_SMs) CTAs; with ceil(L/256) <= num_SMs that is all of them"""
    need = -(-L // 256)
    assert need <= sms()
    return need


@pytest.mark.gpu
@pytest.mark.parametrize("L,lev", [(64, 0), (300, 0), (300, 1), (512, 0), (4096, 0)])
def test_s2_relax_bit_exact(L, lev, gpu_mem):
    """mg2d_s2_relax through mg2d.scalar == the oracle's front loop bit for bit (same summation order; b a^2 with
    a = 2^level is exact).  L = 64: one CTA (__syncthreads branch); 300: a ragged second CTA; 512: two full CTAs;
    4096: 16 CTAs; the last three take the grid.sync() branch."""
    grid = _s2_relax_grid(L)
    assert (grid == 1) == (L == 64)
    smg = mg2d.scalar.ScalarMG(L << lev, 0.1, lev)
    p = S2.S2Params(L << lev, 0.1, lev)
    assert smg.size[lev] == p.size[lev] == L and smg.a[lev] == p.a[lev] == 2.0 ** lev and smg.scale[lev] == p.scale[lev]
    rng = np.random.default_rng(L + lev)
    phi0, b = rng.normal(size=L * L), rng.normal(size=L * L)
    for num_iter in (1, 3):
        want = phi0.copy()
        S2.relax(want, b, lev, num_iter, p)
        phi, bd = torch.tensor(phi0, device="cuda"), torch.tensor(b, device="cuda")
        smg.relax(phi, bd, lev, num_iter)
        got = phi.cpu().numpy()
        assert np.array_equal(got, want), (num_iter, int(np.sum(got != want)), float(np.max(np.abs(got - want))))


def _sgrid_threads(n):
    return min(-(-n // 256), sms() * 8, 4096) * 256


@pytest.mark.gpu
@pytest.mark.parametrize("L", [64, 4096])
def test_s2_project_interpolate(L, gpu_mem):
    """mg2d_s2_project and mg2d_s2_interpolate for quadrants 1..4 (2..4 wrap 2x-1 -> L-1) at levels 0 and 1 scales; at
    4096 the Lc^2 = 4M coarse sites are more than a capped grid covers.  Interpolate zeroes phi_c."""
    Lc = L // 2
    if L == 4096:
        assert_capped(Lc * Lc, _sgrid_threads(Lc * Lc), "s2 project / interpolate")
    smg = mg2d.scalar.ScalarMG(L, 0.1, 1)
    g = torch.Generator(device="cuda")
    g.manual_seed(900 + L)
    phi = torch.randn(L * L, dtype=torch.float64, device="cuda", generator=g)
    b = torch.randn(L * L, dtype=torch.float64, device="cuda", generator=g)
    for quad in (1, 2, 3, 4):
        rc = torch.full((Lc * Lc,), math.nan, dtype=torch.float64, device="cuda")
        smg.projection(rc, b, phi, 0, quad)
        want = s2_project(b, phi, L, smg.scale[0], smg.a[0], quad)
        assert rel(rc, want) < TOL, quad
        pc = torch.randn(Lc * Lc, dtype=torch.float64, device="cuda", generator=g)
        want = s2_interpolate(phi, pc, L, quad)
        pf = phi.clone()
        smg.interpolate(pf, pc, 1, quad)
        assert torch.equal(pf, want) and not pc.abs().max(), quad


@pytest.mark.gpu
def test_s2_residue_mag_and_scale(gpu_mem):
    """mg2d_s2_residue_mag at 4096^2 (capped grid) against the fp64 sum of |r|; mg2d_s2_scale on a length that is not a
    multiple of 256"""
    L = 4096
    assert_capped(L * L, _sgrid_threads(L * L), "s2_residue_mag_kernel")
    smg = mg2d.scalar.ScalarMG(L, 0.1, 1)
    g = torch.Generator(device="cuda")
    g.manual_seed(950)
    smg.phi[0].copy_(torch.randn(L * L, dtype=torch.float64, device="cuda", generator=g))
    smg.r[0].copy_(torch.randn(L * L, dtype=torch.float64, device="cuda", generator=g))
    want = float(s2_residue(smg.phi[0], smg.r[0], L, smg.scale[0], smg.a[0]).abs().sum())
    assert abs(smg.get_residue_mag(0) / want - 1) < TOL
    for n in (1000003, 255):
        x0 = torch.randn(n, dtype=torch.float64, device="cuda", generator=g)
        x = x0.clone()
        smg.ctx.call("mg2d_s2_scale", x.data_ptr(), 0.37, n, S_())
        assert torch.equal(x, x0 * 0.37), n
