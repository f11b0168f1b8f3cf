"""The multigrid setup kernels at the benchmark's shapes, precisions and strip geometries against an fp64 reference.

The setup builds the hierarchy every solve runs on: near-null vectors packed into the projector P (mg2d_pack_null, after
the chunk renormalisation mg2d_norm2 + mg2d_scale_inv_norm), orthonormalised per aggregate (mg2d_norm_nn, mg2d_ortho x2,
mg2d_check_ortho), and the Galerkin operator D_c = P D_f P^dagger (mg2d_coarse_matrix; on the first coarse level also its
rank-`block` hopping factors, mg2d_hop_factors) from the stored level-0 operator (mg2d_lvl0_matrix + mg2d_clover_add).  At
4096^2 with 4x4 aggregates the launchers cap the grid, so every CTA / warp / thread loops over many aggregates or
elements; on 2/4/8 GPUs the fine levels are strips whose projector and link halo rows belong to the neighbouring rank.
A wrong setup does not stop FGCR from converging -- it only costs iterations -- so these kernels get their own checks.

Each operation is restated from its definition (layouts: include/mg2d.h) as vectorised fp64 torch over gathered
aggregates; the CPU tests anchor that restatement to the numpy oracle, the GPU tests hold the kernels to it on seeded
synthetic inputs generated on the device.  Tolerances as in test_gpu_bench_shapes: relative max-norm 1e-12 for complex128,
2e-5 for complex64 against the fp64 reference of the fp32-rounded inputs; Gram-Schmidt on ill-conditioned rows scales them
by each aggregate's condition number.  Every capped case asserts >= 2 passes with a partial last one.
"""
import math

import numpy as np
import pytest
import torch

import mg2d
from oracle import mg_oracle as O
from test_gpu_bench_shapes import (C64, C128, CT, TOL, TOL32, P_, S_, _c, _maxrel, _t, assert_capped, call, crandn, gen,
                                   gpu_mem, owner, rel, sms, wilson_proj)  # noqa: F401 (gpu_mem: fixture)


# ================================================================================================================
# fp64 reference.  P [S, nc, nf] (row ic of site s); an aggregate's rows gathered as R [nX, nc, block^2 * nf] with the
# fine sites in the kernels' order b = x1*block + y1.  Operator blocks in math layout (Dm = D_dev.transpose(-1, -2)).
# ================================================================================================================
def agg_sites(Lxf, Lyf, block, quad, device, X0=0, X1=None):
    """[X1-X0, block^2] fine sites of aggregates X0..X1-1 (X = xc + yc*Lxc), based at (block*xc - dx, block*yc - dy)."""
    dx, dy = int(quad in (2, 3)), int(quad in (3, 4))
    Lxc = Lxf // block
    X = torch.arange(X0, (Lxc * (Lyf // block)) if X1 is None else X1, device=device)
    b = torch.arange(block * block, device=device)
    xf = (block * (X % Lxc)[:, None] - dx + (b // block)[None]) % Lxf
    yf = (block * (X // Lxc)[:, None] - dy + (b % block)[None]) % Lyf
    return yf * Lxf + xf


def rows_of(P, sites):
    """R [nX, nc, bb*nf] of the aggregates whose sites are `sites` [nX, bb], in fp64."""
    Pa = P[sites].to(torch.complex128)                            # [nX, bb, nc, nf]
    return Pa.permute(0, 2, 1, 3).reshape(Pa.shape[0], Pa.shape[2], -1)


def scatter_rows(P, sites, R):
    nX, bb = sites.shape
    P[sites] = R.reshape(nX, R.shape[1], bb, -1).permute(0, 2, 1, 3).to(P.dtype)


def block_norm(R):
    """f_block_norm of every row (f_norm_nn)"""
    return R / R.abs().square().sum(-1, keepdim=True).sqrt()


def ortho(R):
    """f_ortho: modified Gram-Schmidt per aggregate with t -= (<u,t>/|u|) u (S6/near_null.h:165), then block-normalise."""
    R = R.clone()
    for d1 in range(R.shape[1]):
        t = R[:, d1]
        for d2 in range(d1):
            u = R[:, d2]
            nrm = u.abs().square().sum(-1).sqrt()
            dot = (u.conj() * t).sum(-1)
            t -= (dot / nrm)[:, None] * u
        t /= t.abs().square().sum(-1, keepdim=True).sqrt()
    return R


def check_ortho(R):
    """f_check_ortho: max over aggregates and d2 < d1 of |<row d1, row d2>|"""
    G = (R.conj() @ R.transpose(-1, -2)).abs()
    return float(torch.tril(G, diagonal=-1).max())


def condition(R):
    """per-aggregate condition number of the rows (block-normalised), from the eigenvalues of R R^dagger.  LAPACK on the
    host: torch's batched CUDA Hermitian eigensolver (cusolverDnXsyevBatched) rejects these batches."""
    ev = torch.linalg.eigvalsh((R @ R.conj().transpose(-1, -2)).cpu())
    return (ev[:, -1] / ev[:, 0]).sqrt().to(R.device)


def pack_null(Pprev, V, nvec, wilson):
    """tail of f_near_null (S6/level.h:217-246) on sites [a, b): V [nvec, b-a, nf] -> rows of P; rows a vector does not
    reach keep their previous contents."""
    out = Pprev.clone()
    nc, nf = out.shape[1], out.shape[2]
    Vc = V.conj().transpose(0, 1)                                 # [S, nvec, nf]
    if not wilson:
        out[:, :nvec] = Vc
    else:
        h, H = nf // 2, nc // 2
        out[:, :nvec, :h], out[:, :nvec, h:] = Vc[..., :h], 0
        out[:, H:H + nvec, h:], out[:, H:H + nvec, :h] = Vc[..., h:], 0
    return out


def _rows_at(P, P_lo, P_hi, y, x, Lx, Ly):
    """P at (x, y) of a strip with y in -1..Ly: row -1 = P_lo [Lx, ...], row Ly = P_hi [Lx, ...]"""
    main = P[y.clamp(0, Ly - 1) * Lx + x]
    y = y.reshape(y.shape + (1,) * (main.dim() - y.dim()))
    return torch.where(y < 0, P_lo[x], torch.where(y >= Ly, P_hi[x], main))


def coarse_matrix(Dm, P, P_lo, P_hi, Lx, Ly, block, quad, X0=0, X1=None):
    """D_c(X) = sum_{s in X} sum_k P(s) D_k(s) P(s+d_k)^dagger for aggregates X0..X1-1 of an Lx x Ly strip, term k routed
    to slot 0 when s+d_k lies in the same aggregate, else to face slot k (S6/modules_main.h:130-155).  Dm [S, 5, nf, nf]
    math layout; P_lo / P_hi: the projector rows below / above the strip.  Returns [nX, 5, nc, nc] (math layout)."""
    sites = agg_sites(Lx, Ly, block, quad, P.device, X0, X1)
    y, x = sites // Lx, sites % Lx
    b = torch.arange(block * block, device=P.device)
    x1, y1 = b // block, b % block
    Ps = P[sites].to(torch.complex128)
    nX, nc = sites.shape[0], P.shape[1]
    out = torch.zeros((nX, 5, nc, nc), dtype=torch.complex128, device=P.device)
    nbr = [(y, x), (y, (x + 1) % Lx), (y, (x - 1) % Lx), (y + 1, x), (y - 1, x)]
    face = [None, x1 == block - 1, x1 == 0, y1 == block - 1, y1 == 0]
    for k in range(5):
        Pn = _rows_at(P, P_lo, P_hi, nbr[k][0], nbr[k][1], Lx, Ly).to(torch.complex128)
        t = torch.einsum("xbij,xbjl,xbml->xbim", Ps, Dm[sites, k].to(torch.complex128), Pn.conj())
        if k == 0:
            out[:, 0] += t.sum(1)
        else:
            f = face[k][None, :, None, None]
            out[:, 0] += torch.where(f, 0, t).sum(1)
            out[:, k] += torch.where(f, t, 0).sum(1)
    return out


def _chunks(n, size):
    for a in range(0, n, size):
        yield a, min(n, a + size)


# ================================================================================================================
# CPU: the reference against the numpy oracle
# ================================================================================================================
_ORACLE_CASES = [(8, 2, 4), (16, 2, 8), (8, 4, 16), (16, 4, 16)]


def _oracle_params(L, block, nc, **kw):
    return O.Params(L=L, num_iters=1, block=block, m=0.0, nlevels=1, n_dof_scale=nc, **kw)


@pytest.mark.parametrize("L,block", [(8, 2), (8, 4), (16, 4)])
def test_reference_aggregates_match_oracle(L, block):
    for quad in (1, 2, 3, 4):
        sites = agg_sites(L, L, block, quad, "cpu")
        assert np.array_equal(sites.numpy(), O.aggregates(L, L // block, block, quad))
        own = owner(L, L, block, quad, "cpu")
        assert torch.equal(own[sites], torch.arange(sites.shape[0])[:, None].expand_as(sites))


@pytest.mark.parametrize("L,block,nc", _ORACLE_CASES)
def test_reference_orthonormalisation_matches_oracle(L, block, nc):
    """norm_nn, ortho (twice) and check_ortho per aggregate == Level.norm_nn / ortho / check_ortho, all quadrants."""
    rng = np.random.default_rng(L * block + nc)
    p = _oracle_params(L, block, nc)
    for quad in (1, 2, 3, 4):
        lvo = O.Level()
        lvo.phi_null = _c(rng, L * L, nc, 2)
        sites = agg_sites(L, L, block, quad, "cpu")
        R = rows_of(_t(lvo.phi_null), sites)
        got = _t(lvo.phi_null).clone()
        R = block_norm(R)
        scatter_rows(got, sites, R)
        lvo.norm_nn(0, quad, p)
        assert _maxrel(got, lvo.phi_null) < 1e-13
        # from the oracle's unorthogonalised rows, each check_ortho non-trivial
        assert abs(check_ortho(R) / lvo.check_ortho(0, quad, p) - 1) < 1e-13
        for _ in range(2):
            R = ortho(R)
            scatter_rows(got, sites, R)
            lvo.ortho(0, quad, p)
            assert _maxrel(got, lvo.phi_null) < 1e-13
        assert abs(check_ortho(R) - lvo.check_ortho(0, quad, p)) < 1e-15 and check_ortho(R) < 1e-13


@pytest.mark.parametrize("L,block,nc", _ORACLE_CASES)
def test_reference_coarse_matrix_matches_oracle(L, block, nc):
    rng = np.random.default_rng(3 * L + block + nc)
    p = _oracle_params(L, block, nc)
    Df = _c(rng, L * L, 5, 2, 2)
    P = _c(rng, L * L, nc, 2)
    Pt = _t(P)
    for quad in (1, 2, 3, 4):
        got = coarse_matrix(_t(Df), Pt, Pt[-L:], Pt[:L], L, L, block, quad)
        assert _maxrel(got, O.compute_coarse_matrix(Df, P, 0, quad, p)) < 1e-13


@pytest.mark.parametrize("L,block,nc", _ORACLE_CASES)
def test_reference_pack_null_matches_oracle(L, block, nc):
    """The tail of Level.near_null (conjugate + chirality split) on the vectors its relaxation produced.  A Jacobi sweep of
    D = 1 + (hop to x+1 only) with r = 0 maps phi to -phi(s+x), then the chunk renormalisation divides by |phi|."""
    rng = np.random.default_rng(L + nc)
    p = _oracle_params(L, block, nc, gs_flag=0, null_iters=1, null_chunk=1)
    S = L * L
    lvo = O.Level()
    lvo.D = np.zeros((S, 5, 2, 2), dtype=complex)
    lvo.D[:, 0] = lvo.D[:, 1] = np.eye(2)
    lvo.phi_null = _c(rng, S, nc, 2)
    xp = O.neighbours(L)[0]
    V = np.stack([-lvo.phi_null[xp, v] / np.linalg.norm(lvo.phi_null[:, v]) for v in range(nc // 2)])
    prev = _t(lvo.phi_null)
    lvo.near_null(0, p)
    assert _maxrel(pack_null(prev, _t(V), nc // 2, True), lvo.phi_null) < 1e-14
    # laplace rows: every row from a vector
    Vl = _c(rng, nc, S, 1)
    assert torch.equal(pack_null(_t(_c(rng, S, nc, 1)), _t(Vl), nc, False), _t(Vl).conj().transpose(0, 1))


def test_reference_strips_equal_whole_lattice_setup():
    """coarse_matrix on a strip of rows [y0, y0+Ly) with the neighbouring projector rows as explicit P_lo / P_hi equals the
    whole-lattice result on those coarse rows."""
    rng = np.random.default_rng(12)
    L, block, nc = 16, 4, 8
    Df, P = _t(_c(rng, L * L, 5, 2, 2)), _t(_c(rng, L * L, nc, 2))
    whole = coarse_matrix(Df, P, P[-L:], P[:L], L, L, block, 1)
    Lc = L // block
    for y0, Ly in ((4, 8), (12, 4), (0, 4)):
        rows = slice(y0 * L, (y0 + Ly) * L)
        lo, hi = P[((y0 - 1) % L) * L:][:L], P[((y0 + Ly) % L) * L:][:L]
        got = coarse_matrix(Df[rows], P[rows], lo, hi, L, Ly, block, 1)
        assert _maxrel(got, whole[(y0 // block) * Lc:((y0 + Ly) // block) * Lc]) < 1e-15
        # the strip's own wrap rows in place of the neighbour's are not the same operator
        wrong = coarse_matrix(Df[rows], P[rows], P[rows][-L:], P[rows][:L], L, Ly, block, 1)
        assert _maxrel(wrong, whole[(y0 // block) * Lc:((y0 + Ly) // block) * Lc]) > 1e-3


# ================================================================================================================
# GPU
# ================================================================================================================
def _links(g, S):
    th = torch.rand((S, 2), dtype=torch.float64, device="cuda", generator=g) * (2 * math.pi)
    return torch.polar(torch.ones_like(th), th)


def _row(t, y, L):
    """row y (mod the lattice) of a site-major field of width L, as its own buffer"""
    n = t.shape[0] // L
    return t[(y % n) * L:(y % n + 1) * L].clone()


def _status():
    return torch.zeros(1, dtype=torch.int32, device="cuda")


def _grid_stream(n):
    return min(-(-n // 256), sms() * 8, 4096) * 256                # threads of stream_grid (blas.cu)


# ---- 1. near-null renormalisation and projector packing ------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_chunk_renormalisation_4096(dtype, gpu_mem):
    """mg2d_norm2 + mg2d_scale_inv_norm on the 8 near-null vectors of level 0 (2 * 4096^2 elements each): v / |v|."""
    N, nv = 2 * 4096 * 4096, 8
    assert_capped(N, _grid_stream(N), "scale_inv_norm_kernel")
    g = gen(31 + dtype)
    V0 = crandn(g, nv, N, dtype=CT[dtype])
    V0 *= torch.logspace(-3, 4, nv, dtype=torch.float64, device="cuda").to(CT[dtype])[:, None]   # one scale per vector
    V = V0.clone()
    nrm = torch.zeros(nv, dtype=torch.float64, device="cuda")
    for v in range(nv):
        call("mg2d_norm2", P_(V[v]), N, dtype, P_(nrm[v:]), S_())
    for v in range(nv):
        call("mg2d_scale_inv_norm", P_(V[v]), P_(nrm[v:]), N, dtype, S_())
    tol = TOL if dtype == C128 else TOL32
    for v in range(nv):
        v64 = V0[v].to(torch.complex128)
        n2 = float(v64.abs().square().sum())
        assert abs(float(nrm[v]) / n2 - 1) < TOL, v
        assert rel(V[v], v64 / math.sqrt(n2)) < tol, v


def _pack_case(L, nf, nc, wilson, dtype, nvecs, seed):
    S = L * L
    g = gen(seed)
    Pprev = crandn(g, S, nc, nf, dtype=CT[dtype])
    nmax = nc // 2 if wilson else nc
    V = crandn(g, nmax, S, nf, dtype=CT[dtype])
    total = S * nc * nf
    assert_capped(total, min(-(-total // 256), sms() * 16) * 256, "pack_null_kernel")
    P = torch.empty_like(Pprev)
    for nvec in nvecs:
        P.copy_(Pprev)
        call("mg2d_pack_null", P_(P), P_(V), nvec, S * nf, nf, nc, S, int(wilson), dtype, S_())
        for a, b in _chunks(S, 1 << 21):
            assert torch.equal(P[a:b], pack_null(Pprev[a:b], V[:nvec, a:b], nvec, wilson)), (nvec, a)


@pytest.mark.gpu
def test_pack_null_wilson_4096(gpu_mem):
    """Wilson branch at level 0 (5.4e8 elements): nvec = nc/2 as the setup calls it, and nvec < nc/2 (the other rows keep
    their contents).  A copy with conjugation: bit-exact."""
    _pack_case(4096, 2, 16, True, C128, (8, 3), 32)


@pytest.mark.gpu
def test_pack_null_laplace_1024(gpu_mem):
    _pack_case(1024, 1, 16, False, C64, (16, 5), 33)


# ---- 2. per-aggregate orthonormalisation -----------------------------------------------------------------------------
def _input_rows(g, S, nc, nf, dtype, near_null):
    """independent random rows, or near-null-like ones: one shared component per site plus 1e-3 x random"""
    P0 = crandn(g, S, nc, nf, dtype=CT[dtype])
    if near_null:
        P0.mul_(1e-3).add_(crandn(g, S, 1, nf, dtype=CT[dtype]))
    return P0


def _orthonormalise_case(L, blk, nf, nc, dtype, quad, near_null, seed):
    S, nagg = L * L, (L // blk) ** 2
    assert_capped(nagg, min(-(-nagg // 4), sms() * 32) * 4, f"aggregate_rows_kernel {L}^2 block {blk}")
    P0 = _input_rows(gen(seed), S, nc, nf, dtype, near_null)
    P = P0.clone()
    status = _status()
    args = (nf, nc, L, L, blk, quad, dtype)
    call("mg2d_norm_nn", P_(P), *args, P_(status), S_())
    tol = TOL if dtype == C128 else TOL32
    chunk = max(1, (1 << 31) // (nc * blk * blk * nf * 16))
    errs = []
    for a, b in _chunks(nagg, chunk):
        sites = agg_sites(L, L, blk, quad, "cuda", a, b)
        errs.append(rel(rows_of(P, sites), block_norm(rows_of(P0, sites))))
    assert all(e < tol for e in errs), ("norm_nn", max(errs))
    call("mg2d_ortho", P_(P), *args, P_(status), S_())
    call("mg2d_ortho", P_(P), *args, P_(status), S_())
    out = torch.full((1,), -1.0, dtype=torch.float64, device="cuda")
    call("mg2d_check_ortho", P_(P), *args, P_(out), S_())
    assert int(status.item()) == 0
    assert 0.0 <= float(out.item()) < (1e-12 if dtype == C128 else TOL32)
    worst, kmax = [], 0.0
    for a, b in _chunks(nagg, chunk):
        sites = agg_sites(L, L, blk, quad, "cuda", a, b)
        R0 = block_norm(rows_of(P0, sites))
        want, got = ortho(ortho(R0)), rows_of(P, sites)
        err = (got - want).abs().amax(-1).amax(-1) / want.abs().amax(-1).amax(-1)
        if near_null:       # Gram-Schmidt amplifies rounding by the condition number of the rows it starts from
            kappa = condition(R0)
            kmax = max(kmax, float(kappa.max()))
            err = err / kappa
        worst.append(float(torch.nan_to_num(err, nan=math.inf).max()))
        del R0, want, got
    assert all(w < tol for w in worst), ("ortho", max(worst), kmax)
    if near_null:
        assert kmax > 100, kmax          # the input really is ill-conditioned


@pytest.mark.gpu
@pytest.mark.parametrize("near_null", [False, True])
def test_orthonormalise_level0_4096(near_null, gpu_mem):
    """norm_nn, ortho x2, check_ortho (the compute_near_null sequence) at level 0: nf 2, nc 16, 4x4 aggregates, 2^20 of
    them (one 32-element warp-row per aggregate row)."""
    _orthonormalise_case(4096, 4, 2, 16, C128, 1, near_null, 40 + near_null)


@pytest.mark.gpu
@pytest.mark.parametrize("near_null", [False, True])
@pytest.mark.parametrize("dtype", [C128, C64])
def test_orthonormalise_level1_1024(dtype, near_null, gpu_mem):
    _orthonormalise_case(1024, 4, 16, 16, dtype, 1, near_null, 42 + 2 * dtype + near_null)


@pytest.mark.gpu
@pytest.mark.parametrize("quad", [2, 3, 4])
def test_orthonormalise_quadrants_512(quad, gpu_mem):
    """Quadrants 2-4 (aggregates wrap around the lattice edge) at a capped block-2 shape: 512^2, nf = nc = 8."""
    for near_null in (False, True):
        _orthonormalise_case(512, 2, 8, 8, C128, quad, near_null, 50 + quad + 4 * near_null)


# ---- 3. edges of the grid-stride loops -----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("L,blk,nf,nc", [(512, 2, 8, 8), (4096, 4, 2, 16)])
def test_aggregate_rows_edges(L, blk, nf, nc, gpu_mem):
    """check_ortho finds an overlap planted in the last aggregate (the partial last pass) and, on the same output
    buffer, the smaller one of aggregate 0 once the first is gone (the launcher resets the maximum); ortho and norm_nn
    leave exactly orthonormal rows unchanged with status 0 and flag a zero / tiny row in the last aggregate."""
    nagg = (L // blk) ** 2
    assert_capped(nagg, min(-(-nagg // 4), sms() * 32) * 4, "aggregate_rows_kernel")
    for quad in ((1, 2, 3, 4) if L == 512 else (1,)):
        sites = agg_sites(L, L, blk, quad, "cuda")
        base = torch.zeros((L * L, nc, nf), dtype=torch.complex128, device="cuda")
        for d in range(nc):         # row d of every aggregate: the unit vector at (b, j) = divmod(d, nf), exactly orthonormal
            base[sites[:, d // nf], d, d % nf] = 1.0
        last, first = sites[-1], sites[0]
        P = base.clone()
        P[last[0], nc - 1, 0] = 0.3 + 0.4j            # |<row nc-1, row 0>| = 0.5 in the last aggregate
        P[first[0], 2, 0] = 0.25j                      # |<row 2, row 0>| = 0.25 in aggregate 0
        args = (nf, nc, L, L, blk, quad, C128)
        out = torch.zeros(1, dtype=torch.float64, device="cuda")
        for planted_last in (True, False):
            if not planted_last:
                P[last[0], nc - 1, 0] = 0
            want = max(check_ortho(rows_of(P, sites[a:b])) for a, b in _chunks(nagg, 1 << 16))
            call("mg2d_check_ortho", P_(P), *args, P_(out), S_())
            assert abs(float(out.item()) - want) <= 1e-15 * want, (quad, planted_last, float(out.item()), want)
            assert abs(want - (0.5 if planted_last else 0.25)) < 1e-15
        for fn in ("mg2d_norm_nn", "mg2d_ortho"):
            P = base.clone()
            status = _status()
            call(fn, P_(P), *args, P_(status), S_())
            assert int(status.item()) == 0 and torch.equal(P, base), (fn, quad)
        P = base.clone()
        P[last[0], 0, 0] = 0                           # a zero row: ortho divides by its norm for every later row
        status = _status()
        call("mg2d_ortho", P_(P), *args, P_(status), S_())
        assert int(status.item()) & 2, quad
        P = base.clone()
        P[last[(nc - 1) // nf], nc - 1, (nc - 1) % nf] = 1e-45      # a block norm below the reference's 1e-40
        status = _status()
        call("mg2d_norm_nn", P_(P), *args, P_(status), S_())
        assert int(status.item()) & 1, quad
        del base, P


def _small_hierarchy(L=16):
    p = mg2d.make_params(L, 0.05, nlevels=1, block=4, n_null=8, n_smooth=2, null_iters=8, matrix_free=False)
    mg = mg2d.MG(p)
    mg.init_reference_fields()
    mg.set_gauge(torch.as_tensor(O.gauge_gaussian(L, width=0.4, seed=9)).cuda())
    return mg


@pytest.mark.gpu
@pytest.mark.parametrize("row_norm", [None, 0.0, 1e-45])
def test_compute_near_null_rejects_degenerate_rows(row_norm):
    """compute_near_null(gen_null=0) on supplied vectors: healthy rows pass (check_ortho < 1e-12); one aggregate row of
    norm 0 or ~1e-45 raises FloatingPointError (the reference exits on a block norm below 1e-40)."""
    mg = _small_hierarchy()
    lv = mg.LVL[0]
    if row_norm is not None:
        sites = agg_sites(lv.L, lv.L, lv.block, 1, "cuda")[5]
        v = torch.zeros_like(lv.phi_null[sites, 3, :])
        v[0, 0] = row_norm
        lv.phi_null[sites, 3, :] = v
        with pytest.raises(FloatingPointError):
            mg2d.compute_near_null(mg, gen_null=0)
    else:
        mg2d.compute_near_null(mg, gen_null=0)
        assert max(mg.info["ortho_worst"]) < 1e-12
    mg.close()


# ---- 4 + 5. Galerkin operator, hop factors, strips with real neighbour rows -------------------------------------------
def _coarse_call(Dc, Df, P, P_lo, P_hi, nf, nc, Lx, Ly, blk, quad, dtype):
    call("mg2d_coarse_matrix", P_(Dc), P_(Df), P_(P), P_(P_lo), P_(P_hi), nf, nc, Lx, Ly, blk, quad, dtype, S_())


def _check_coarse(Dc, Df, P, P_lo, P_hi, nf, nc, Lx, Ly, blk, quad, dtype):
    """Dc (device layout) against the reference, in chunks of aggregates with an explicit fine halo row."""
    Dm = Df.view(-1, 5, nf, nf).transpose(-1, -2)
    nagg = (Lx // blk) * (Ly // blk)
    chunk = max(Lx // blk, (1 << 28) // (blk * blk * nc * nc * 16))
    errs = []
    for a, b in _chunks(nagg, chunk):
        want = coarse_matrix(Dm, P, P_lo, P_hi, Lx, Ly, blk, quad, a, b)
        errs.append(rel(Dc[a:b].transpose(-1, -2), want))
        del want
    tol = TOL if dtype == C128 else TOL32
    assert all(e < tol for e in errs), (Lx, Ly, quad, dtype, max(errs))


def _nan_like(shape, dtype):
    return torch.full(shape, complex(math.nan, math.nan), dtype=CT[dtype], device="cuda")


@pytest.mark.gpu
def test_galerkin_level0_4096(gpu_mem):
    """Level 0 -> 1 of the benchmark: fine operator from mg2d_lvl0_matrix on random links + mg2d_clover_add (csw = 1),
    random dense P; mg2d_coarse_matrix against the reference, mg2d_hop_factors against its face slots, and the level-0
    strips of the 8-rank plan (4096 x 512: an interior one and the last, whose upper neighbour is global row 0) with their
    true neighbour rows: the same rows of the whole-lattice results bit for bit."""
    L, blk, nf, nc, m = 4096, 4, 2, 16, -0.05
    S, Lc = L * L, L // blk
    nagg = Lc * Lc
    assert_capped(nagg, min(nagg, sms() * 8), "coarse_matrix_kernel (level 0)")
    assert_capped(nagg, min(-(-nagg // 8), sms() * 16) * 8, "hop_factors_kernel")
    g = gen(60)
    U = _links(g, S)
    F = torch.empty(S, dtype=torch.float64, device="cuda")
    call("mg2d_clover_field", P_(F), P_(U), P_(_row(U, -1, L)), P_(_row(U, 0, L)), 1.0, L, L, C128, S_())
    Df = torch.empty((S, 5, nf, nf), dtype=torch.complex128, device="cuda")
    call("mg2d_lvl0_matrix", P_(Df), P_(U), P_(_row(U, -1, L)), m, 0, L, L, C128, S_())
    call("mg2d_clover_add", P_(Df), P_(F), S, C128, S_())
    # the stored operator itself: (2+m) 1 + F s3 and U-weighted spin projectors (S6/level.h:155-172)
    proj = wilson_proj("cuda")
    Dm = Df.view(L, L, 5, nf, nf).transpose(-1, -2)
    Ug = U.view(L, L, 2)
    for y0 in range(0, L, 512):
        ys = slice(y0, y0 + 512)
        Fs = F.view(L, L)[ys]
        Uym = Ug[(torch.arange(y0, y0 + 512, device="cuda") - 1) % L, :, 1]
        coef = (Ug[ys, :, 0], Ug[ys, :, 0].roll(1, dims=1).conj(), Ug[ys, :, 1], Uym.conj())
        assert rel(Dm[ys, :, 0, 0, 0], (2 + m) + Fs) < 1e-15 and rel(Dm[ys, :, 0, 1, 1], (2 + m) - Fs) < 1e-15
        assert float(Dm[ys, :, 0, 0, 1].abs().max()) == 0.0 and float(Dm[ys, :, 0, 1, 0].abs().max()) == 0.0
        for k in range(4):
            assert rel(Dm[ys, :, k + 1], coef[k][..., None, None] * proj[k]) < 1e-15, (y0, k)
    del Dm, Ug, coef, Uym, Fs
    P = crandn(g, S, nc, nf)
    P_lo, P_hi = _row(P, -1, L), _row(P, 0, L)
    Dc = _nan_like((nagg, 5, nc, nc), C128)
    _coarse_call(Dc, Df, P, P_lo, P_hi, nf, nc, L, L, blk, 1, C128)
    _check_coarse(Dc, Df, P, P_lo, P_hi, nf, nc, L, L, blk, 1, C128)
    A = _nan_like((nagg, 4 * blk, nc), C128)
    B = _nan_like((nagg, 4 * blk, nc), C128)
    status = _status()
    call("mg2d_hop_factors", P_(A), P_(B), P_(Df), P_(P), P_(P_lo), P_(P_hi), nf, nc, L, L, blk, C128, P_(status), S_())
    assert int(status.item()) == 0
    errs = []
    for a, b in _chunks(nagg, 1 << 16):
        rec = torch.einsum("xkbi,xkbj->xkij", A[a:b].view(-1, 4, blk, nc), B[a:b].view(-1, 4, blk, nc).conj())
        errs.append(rel(rec, Dc[a:b, 1:].transpose(-1, -2)))
    assert all(e < TOL for e in errs), max(errs)
    for y0 in (3 * 512, L - 512):
        Ly = 512
        rows, crows = slice(y0 * L, (y0 + Ly) * L), slice((y0 // blk) * Lc, ((y0 + Ly) // blk) * Lc)
        Us, U_lo, U_hi = U[rows].clone(), _row(U, y0 - 1, L), _row(U, y0 + Ly, L)
        Fs = torch.empty(Ly * L, dtype=torch.float64, device="cuda")
        call("mg2d_clover_field", P_(Fs), P_(Us), P_(U_lo), P_(U_hi), 1.0, L, Ly, C128, S_())
        assert torch.equal(Fs, F[rows]), y0
        Ds = torch.empty((Ly * L, 5, nf, nf), dtype=torch.complex128, device="cuda")
        call("mg2d_lvl0_matrix", P_(Ds), P_(Us), P_(U_lo), m, 0, L, Ly, C128, S_())
        call("mg2d_clover_add", P_(Ds), P_(Fs), Ly * L, C128, S_())
        assert torch.equal(Ds, Df[rows]), y0
        Ps, Ps_lo, Ps_hi = P[rows].clone(), _row(P, y0 - 1, L), _row(P, y0 + Ly, L)
        Dcs = _nan_like((Ly // blk * Lc, 5, nc, nc), C128)
        _coarse_call(Dcs, Ds, Ps, Ps_lo, Ps_hi, nf, nc, L, Ly, blk, 1, C128)
        assert torch.equal(Dcs, Dc[crows]), y0
        As, Bs = _nan_like((Ly // blk * Lc, 4 * blk, nc), C128), _nan_like((Ly // blk * Lc, 4 * blk, nc), C128)
        status = _status()
        call("mg2d_hop_factors", P_(As), P_(Bs), P_(Ds), P_(Ps), P_(Ps_lo), P_(Ps_hi), nf, nc, L, Ly, blk, C128, P_(status), S_())
        assert int(status.item()) == 0
        assert torch.equal(As, A[crows]) and torch.equal(Bs, B[crows]), y0
        del Us, Fs, Ds, Ps, Dcs, As, Bs


@pytest.mark.gpu
@pytest.mark.parametrize("L,dtype", [(1024, C128), (1024, C64), (256, C128)])
def test_galerkin_coarse_levels(L, dtype, gpu_mem):
    """Levels 1 -> 2 (1024^2) and 2 -> 3 (256^2, the first replicated level of the 8-rank plan): random 16 x 16 blocks,
    random P; then the 8-rank strips (L x L/8: an interior one and the last) with true neighbour rows, bit for bit."""
    blk, nf, nc = 4, 16, 16
    S, Lc = L * L, L // blk
    nagg = Lc * Lc
    assert_capped(nagg, min(nagg, sms() * 8), f"coarse_matrix_kernel {L}^2")
    g = gen(70 + L + dtype)
    Df = crandn(g, S, 5, nf, nf, dtype=CT[dtype])
    P = crandn(g, S, nc, nf, dtype=CT[dtype])
    P_lo, P_hi = _row(P, -1, L), _row(P, 0, L)
    Dc = _nan_like((nagg, 5, nc, nc), dtype)
    _coarse_call(Dc, Df, P, P_lo, P_hi, nf, nc, L, L, blk, 1, dtype)
    _check_coarse(Dc, Df, P, P_lo, P_hi, nf, nc, L, L, blk, 1, dtype)
    Ly = L // 8
    for y0 in (3 * Ly, L - Ly):
        rows, crows = slice(y0 * L, (y0 + Ly) * L), slice((y0 // blk) * Lc, ((y0 + Ly) // blk) * Lc)
        Dcs = _nan_like((Ly // blk * Lc, 5, nc, nc), dtype)
        _coarse_call(Dcs, Df[rows].clone(), P[rows].clone(), _row(P, y0 - 1, L), _row(P, y0 + Ly, L), nf, nc, L, Ly, blk, 1, dtype)
        assert torch.equal(Dcs, Dc[crows]), y0
        del Dcs


@pytest.mark.gpu
def test_galerkin_quadrants_512(gpu_mem):
    """Quadrants 1-4 at the capped block-2 shape (512^2, nf = nc = 8): aggregates and their faces wrap the lattice edge."""
    L, blk, nf, nc = 512, 2, 8, 8
    nagg = (L // blk) ** 2
    assert_capped(nagg, min(nagg, sms() * 8), "coarse_matrix_kernel 512^2 block 2")
    g = gen(80)
    Df = crandn(g, L * L, 5, nf, nf)
    P = crandn(g, L * L, nc, nf)
    P_lo, P_hi = _row(P, -1, L), _row(P, 0, L)
    for quad in (1, 2, 3, 4):
        Dc = _nan_like((nagg, 5, nc, nc), C128)
        _coarse_call(Dc, Df, P, P_lo, P_hi, nf, nc, L, L, blk, quad, C128)
        _check_coarse(Dc, Df, P, P_lo, P_hi, nf, nc, L, L, blk, quad, C128)
