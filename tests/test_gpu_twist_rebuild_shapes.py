"""The self-block rebuild behind MG.set_twist against an fp64 reference: mg2d_twist_set, mg2d_block_inverse (with partial
pivoting) at every n, mg2d_premultiply, mg2d_lowrank_pack_a and the whole set_twist chain, with clover and a stored level 0.

set_twist changes the twisted mass of a built hierarchy in place: mg2d_twist_set sets the imaginary self-block diagonal to
base + delta Gamma5_c, and mg2d_block_inverse, mg2d_premultiply, mg2d_lowrank_pack_a and mg2d_to_half rebuild every buffer
that depends on the self blocks.  The multigrid is only a preconditioner inside FGCR: a subtly wrong D0^-1, M or F costs
iterations and never gives a wrong answer, so these kernels get their own checks.  The self blocks of a twisted coarse level
near the critical mass are not diagonally dominant, so the row swaps of the pivoting inverse run here against a reference
(the other shape tests invert diagonally dominant blocks only, which never pivot).

Each operation is restated from its definition (layouts: include/mg2d.h; the low-rank lane order: stencil.cu, LowRank) as
vectorised fp64 torch; the CPU tests anchor the restatements to the numpy oracle, to scipy's LU and to the sweep that reads
the lane order, the GPU tests hold the kernels to them on seeded synthetic inputs generated on the device and on hierarchies
built at 1024^2 with the benchmark's cycle.  Tolerances as in test_gpu_bench_shapes: relative max-norm 1e-12 for complex128,
2e-5 for complex64 against the fp64 reference of the rounded inputs; inverses of blocks that are not well conditioned get
that tolerance times each block's condition number (infinity norm, from the fp64 inverse).  Every capped case asserts >= 2
passes with a partial last one.
"""
import math

import numpy as np
import pytest
import torch

import mg2d
from mg2d import _lib
from oracle import mg_oracle as O
from test_gpu_bench_shapes import (C64, C128, CT, TOL, TOL32, P_, S_, _c, _periodic_halos, _t, assert_capped, call, crandn,
                                   gen, gpu_mem, hop_lowrank, neighbours, rb_half, rel, rounded, sms)  # noqa: F401 (gpu_mem)
from test_gpu_setup_shapes import agg_sites, block_norm, coarse_matrix, ortho, pack_null, rows_of, scatter_rows
from test_twisted_mass import G5, add_twist, dense_tm

RT = {C128: torch.float64, C64: torch.float32}


# ================================================================================================================
# fp64 reference.  Operator blocks: device layout D[s][k][j][i] (column-major), math layout = D.transpose(-1, -2).
# ================================================================================================================
def gamma5_c(n, device="cpu"):
    """diag of Gamma5_c = diag(+1 x n/2, -1 x n/2): gamma5 = sigma3 on level 0 (n = 2), its Galerkin image on a
    chirality-split projector on the coarse levels"""
    return torch.cat([torch.ones(n // 2), -torch.ones(n - n // 2)]).to(torch.float64).to(device)


def twist_set_ref(D, base, delta):
    """mg2d_twist_set: D [S, 5, n, n] with Im D[s][0](i,i) = base[s][i] + delta Gamma5_c(i,i), summed in fp64 and rounded
    once to D's precision; every other number untouched"""
    n = D.shape[-1]
    out = D.clone()
    idx = torch.arange(n, device=D.device)
    im = (base + delta * gamma5_c(n, D.device)).to(out.real.dtype)
    out[:, 0, idx, idx] = torch.complex(out[:, 0, idx, idx].real, im)
    return out


def bits(t):
    r = torch.view_as_real(t) if t.is_complex() else t
    return r.contiguous().view({8: torch.int64, 4: torch.int32, 2: torch.int16}[r.element_size()])


def bits_equal(a, b):
    return tuple(a.shape) == tuple(b.shape) and torch.equal(bits(a), bits(b))


def pivot_trace(A):
    """Rows chosen by Gauss-Jordan with partial pivoting on A [S, n, n] (math layout), in fp64: step c takes the largest
    |a|^2 at or below the diagonal of column c, ties to the smallest row (block_inverse_kernel), and swaps it with row c.
    Gauss-Jordan eliminates the rows below the pivot as LU does, so the choices are LU's.  Returns [S, n]."""
    A = A.to(torch.complex128).clone()
    S, n, _ = A.shape
    piv = torch.empty((S, n), dtype=torch.long, device=A.device)
    ar = torch.arange(S, device=A.device)
    for c in range(n):
        col = A[:, c:, c]
        r = c + torch.argmax(col.real ** 2 + col.imag ** 2, dim=1)      # argmax: the first maximal index
        piv[:, c] = r
        rc = A[ar, c].clone()
        A[ar, c] = A[ar, r]
        A[ar, r] = rc
        A[:, c + 1:] -= (A[:, c + 1:, c] / A[:, c, c][:, None])[..., None] * A[:, c, None]
    return piv


def pivots(piv):
    """[S] bool: the site swaps rows at some step"""
    return (piv != torch.arange(piv.shape[1], device=piv.device)).any(1)


def cond_inf(A, Ainv):
    """per-block condition number in the infinity norm"""
    return A.abs().sum(-1).amax(-1) * Ainv.abs().sum(-1).amax(-1)


def block_err(got, want):
    """per block max |got - want| / max |want|; NaN / inf in `got` -> inf"""
    e = (got.to(torch.complex128) - want).abs().amax((-2, -1)) / want.abs().amax((-2, -1))
    return torch.nan_to_num(e, nan=math.inf)


def self_blocks(kind, Z):
    """Self blocks A [S, n, n] (math layout, fp64) from the Gaussian draws Z [S, n, n]:
    permuted   well conditioned (3 I + 0.5 Z / sqrt(n): every eigenvalue within about 1 of 3), rows cycled up by one: the
               dominant entry of column c sits in row c-1 (column 0: row n-1), so every column but the last pivots
    gaussian   Z (condition numbers up to ~1e4)
    zero_diag  Z with a zero diagonal: without pivoting the first step divides by zero
    ties       0.3 Z, column 0 small except two entries of modulus exactly 4 (phases 1, i, -1, -i, exact in fp32) in rows
               1 and n-1 (n >= 3: the pivot takes row 1) or rows 0 and 1 (n = 2: row 0 stays)"""
    S, n, _ = Z.shape
    if kind == "permuted":
        A = 3.0 * torch.eye(n, dtype=Z.dtype, device=Z.device) + (0.5 / math.sqrt(n)) * Z
        return A.roll(-1, dims=-2)
    if kind == "gaussian":
        return Z.clone()
    if kind == "zero_diag":
        A = Z.clone()
        A.diagonal(dim1=-2, dim2=-1).zero_()
        return A
    assert kind == "ties" and n >= 2
    A = 0.3 * Z
    A[:, :, 0] *= 0.1
    r0, r1 = (1, n - 1) if n >= 3 else (0, 1)
    ph = torch.tensor([1, 1j, -1, -1j], dtype=Z.dtype, device=Z.device)
    quad = lambda z: (torch.floor((torch.angle(z) + math.pi) / (math.pi / 2)).long() % 4)     # noqa: E731
    A[:, r0, 0] = 4 * ph[quad(Z[:, r0, 1])]
    A[:, r1, 0] = 4 * ph[quad(Z[:, r1, 1])]
    return A


def lr_index(n, R):
    """Lane order of the low-rank factors F[s][2][IT][32] (stencil.cu, LowRank): Bc[t][g] = conj(b_q)_j with q = g / LP,
    j = (g % LP) IT + t, and MA[t][g] = ma_{q,i} with i = g % n, q = t H + g / n (Q = 4R, IT = nR/8, LP = 32/Q, H = 32/n).
    Returns ((qb, jb), (qa, ia)), each [IT, 32]."""
    Q, IT = 4 * R, n * R // 8
    LP, H = 32 // Q, 32 // n
    t, g = torch.arange(IT)[:, None], torch.arange(32)[None, :]
    return ((g // LP).expand(IT, 32), (g % LP) * IT + t), (t * H + g // n, (g % n).expand(IT, 32))


def lr_ma_ref(A, inv, n, R):
    """the -D0inv A half of F [S, IT, 32] in fp64 (A [S, 4R, n]; inv [S, n, n] math layout) in lane order"""
    _, (qa, ia) = lr_index(n, R)
    MA = -torch.einsum("sil,sql->sqi", inv.to(torch.complex128), A.to(torch.complex128))
    return MA[:, qa.to(A.device), ia.to(A.device)]


def lr_pack_ref(A, B, inv, n, R):
    """F [S, 2, IT, 32] in fp64: conj(B) and -D0inv A (B [S, 4R, n]) in lane order"""
    (qb, jb), _ = lr_index(n, R)
    Bc = B.to(torch.complex128).conj()
    return torch.stack([Bc[:, qb.to(A.device), jb.to(A.device)], lr_ma_ref(A, inv, n, R)], 1)


def lr_sweep_update(F, nb, n, R):
    """What stencil_rb_lr_kernel computes from F at one site: lane g dots its IT entries of Bc with the neighbour of face
    k = 1 + q/R, q = g / LP (stage 1: t_q summed over the LP lanes of q), then multiplies its IT entries of MA with
    t_{t H + g / n} and the lanes of equal g % n are summed (stage 2).  nb [4, S, n]: the neighbours in slots 1..4."""
    Q, IT = 4 * R, n * R // 8
    LP = 32 // Q
    (qb, jb), (qa, _) = lr_index(n, R)
    k = (qb[0] // R).to(F.device)                                      # face of each lane (slot k + 1)
    S = F.shape[0]
    nbg = nb[k[None, :].expand(IT, 32), :, jb.to(F.device)]            # [IT, 32, S]
    part = (F[:, 0] * nbg.permute(2, 0, 1)).sum(1)                     # [S, 32]
    tq = part.reshape(S, Q, LP).sum(-1)                                # [S, Q]
    acc = (F[:, 1] * tq[:, qa.to(F.device)]).sum(1)                    # [S, 32]
    return acc.reshape(S, 32 // n, n).sum(1)


# ================================================================================================================
# CPU: the reference against the oracle, scipy and the sweep
# ================================================================================================================
@pytest.mark.parametrize("L,block,nc", [(8, 2, 4), (8, 2, 8), (16, 4, 16), (8, 4, 32)])
def test_reference_gamma5_c_is_the_galerkin_image_of_sigma3(L, block, nc):
    """On chirality-split projector rows orthonormal per aggregate (pack_null + ortho, as the setup builds them), the Galerkin
    product of the level-0 twist i mu sigma3 is i mu Gamma5_c on the self blocks and nothing on the faces; n = 2 is sigma3
    itself (the oracle's gamma5)."""
    rng = np.random.default_rng(nc + L)
    S, mu = L * L, 0.37
    P = pack_null(_t(_c(rng, S, nc, 2)), _t(_c(rng, nc // 2, S, 2)), nc // 2, True)
    sites = agg_sites(L, L, block, 1, "cpu")
    R = block_norm(rows_of(P, sites))
    R = ortho(ortho(R))
    scatter_rows(P, sites, R)
    Dm = torch.zeros((S, 5, 2, 2), dtype=torch.complex128)
    Dm[:, 0] = 1j * mu * torch.diag(gamma5_c(2)).to(torch.complex128)
    Dc = coarse_matrix(Dm, P, P[-L:], P[:L], L, L, block, 1)
    want = 1j * mu * torch.diag(gamma5_c(nc)).to(torch.complex128)
    assert float((Dc[:, 0] - want).abs().max()) < 1e-13
    assert float(Dc[:, 1:].abs().max()) == 0.0
    assert torch.equal(gamma5_c(2), torch.as_tensor(np.diag(G5(1)).copy()))


def test_reference_twist_set_is_the_oracles_twist():
    """twist_set_ref on the oracle's level-0 operator at twist 0 with delta = mu equals the oracle's i mu gamma5 added to it,
    bit for bit (one fp64 sum), and delta = 0 returns the input."""
    L, mu = 8, 0.0173
    lvo = O.Level()
    lvo.compute_lvl0_matrix(O.gauge_gaussian(L, width=0.4, seed=9), O.Params(L=L, num_iters=1, block=2, m=-0.05, nlevels=1))
    D = _t(lvo.D).transpose(-1, -2).contiguous()                       # device layout
    base = D[:, 0].diagonal(dim1=-2, dim2=-1).imag.contiguous()
    got = twist_set_ref(D, base, mu)
    add_twist(lvo, mu)
    assert bits_equal(got, _t(lvo.D).transpose(-1, -2).contiguous())
    assert bits_equal(twist_set_ref(D, base, 0.0), D)


@pytest.mark.parametrize("n", [2, 4, 8, 16, 32])
def test_reference_pivot_trace_matches_lu_and_the_inputs(n):
    """pivot_trace == scipy's partial-pivoting LU on real blocks (|a| orders as |a|^2 there); the synthetic inputs pivot as
    they claim: every column but the last of `permuted`, column 0 of every `zero_diag` block, row 1 (n >= 3) or row 0 (n = 2)
    among the exact ties."""
    import scipy.linalg as sl
    rng = np.random.default_rng(n)
    Ar = rng.normal(size=(64, n, n))
    got = pivot_trace(_t(Ar).to(torch.complex128))
    for s in range(64):
        assert np.array_equal(got[s].numpy(), sl.lu_factor(Ar[s])[1]), s
    Z = _t(_c(rng, 256, n, n))
    ar = torch.arange(n)
    piv = pivot_trace(self_blocks("permuted", Z))
    assert bool((piv[:, :n - 1] != ar[:n - 1]).all())
    assert bool((pivot_trace(self_blocks("zero_diag", Z))[:, 0] != 0).all())
    T = self_blocks("ties", Z)
    r0, r1 = (1, n - 1) if n >= 3 else (0, 1)
    assert torch.equal(T[:, r0, 0].abs(), torch.full((256,), 4.0, dtype=torch.float64))
    assert torch.equal(T[:, r1, 0].abs(), T[:, r0, 0].abs())
    assert bool((pivot_trace(T)[:, 0] == r0).all())
    for kind in ("permuted", "gaussian", "zero_diag", "ties"):
        A = self_blocks(kind, Z)
        assert float((A @ torch.linalg.inv(A) - torch.eye(n, dtype=A.dtype)).abs().max()) < 1e-9, kind


@pytest.mark.parametrize("n,R", [(16, 4), (8, 2)])
def test_reference_lane_order_is_the_lowrank_sweep(n, R):
    """Every (q, j) of conj(B) and every (q, i) of -D0inv A has exactly one lane, and the sweep read from lr_pack_ref in the
    kernel's lane order gives -D0inv sum_q A_q (B_q^dagger phi(s + d_k(q))), the low-rank update of the dense reference."""
    Q, IT = 4 * R, n * R // 8
    (qb, jb), (qa, ia) = lr_index(n, R)
    assert sorted((qb * n + jb).reshape(-1).tolist()) == list(range(Q * n))
    assert sorted((qa * n + ia).reshape(-1).tolist()) == list(range(Q * n))
    rng = np.random.default_rng(n + R)
    S = 64
    A, B, inv, nb = (_t(_c(rng, S, Q, n)), _t(_c(rng, S, Q, n)), _t(_c(rng, S, n, n)), _t(_c(rng, 4, S, n)))
    F = lr_pack_ref(A, B, inv, n, R)
    assert F.shape == (S, 2, IT, 32)
    hop = sum(torch.einsum("sqi,sq->si", A[:, k * R:(k + 1) * R],
                           torch.einsum("sqj,sj->sq", B[:, k * R:(k + 1) * R].conj(), nb[k])) for k in range(4))
    want = -torch.einsum("sij,sj->si", inv, hop)
    assert _maxrel(lr_sweep_update(F, nb, n, R), want) < 1e-13


def _maxrel(a, b):
    return float((a - b).abs().max() / b.abs().max())


# ================================================================================================================
# GPU
# ================================================================================================================
def _capped_sites(per_pass):
    """a site count with 2.5 passes of a grid-stride loop that covers `per_pass` sites per pass (odd, so never a multiple of
    the block size)"""
    return (5 * per_pass) // 2 | 1


def _inverse_warps(n, dtype):
    """warps per CTA of launch_inverse (stencil.cu): as many 2 n^2 workspaces as fit 48 KB, at most 8"""
    per_warp = 2 * n * n * (16 if dtype == C128 else 8)
    return max(1, min(48 * 1024 // per_warp, 8))


def _block_inverse(A, dtype):
    """mg2d_block_inverse on self blocks A [S, n, n] (math layout, fp64 values representable in dtype), slot 0 of a 5-slot
    operator whose other slots hold NaN (the kernel must not read them); returns D0inv in math layout"""
    S, n, _ = A.shape
    D = torch.full((S, 5, n, n), complex(math.nan, math.nan), dtype=CT[dtype], device="cuda")
    D[:, 0] = A.transpose(-1, -2).to(CT[dtype])
    inv = torch.full((S, n, n), complex(math.nan, math.nan), dtype=CT[dtype], device="cuda")
    call("mg2d_block_inverse", P_(inv), P_(D), n, S, dtype, S_())
    return inv.transpose(-1, -2)


def _check_inverse(got, A, tol, scaled, what):
    """got vs the fp64 inverse of A, per block: err < tol (scaled: tol times the block's condition number)"""
    want = torch.linalg.inv(A)
    err = block_err(got, want)
    kappa = cond_inf(A, want)
    worst = float((err / kappa).max() if scaled else err.max())
    assert worst < tol, (what, worst, float(kappa.max()))
    return float(kappa.max())


# ---- 1. mg2d_twist_set --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("n", [2, 4, 8, 16, 32])
def test_twist_set(n, dtype, gpu_mem):
    """Im D[s][0](i,i) = (base + delta Gamma5_c).to(T) bit for bit on a capped grid with S n not a multiple of 256; the real
    parts, the off-diagonal entries and slots 1-4 bit-identical to the input; delta = 0 writes base.to(T).  In complex64
    the sum rounded twice, (T)base + (T)delta, differs on a sizeable fraction of the elements: the check sees it."""
    S = _capped_sites(sms() * 8 * 256) // n | 1
    nel = S * n
    assert nel % 256
    assert_capped(nel, min(-(-nel // 256), sms() * 8) * 256, f"twist_set_kernel n {n}")
    g = gen(300 + 2 * n + dtype)
    D0 = crandn(g, S, 5, n, n, dtype=CT[dtype])
    base = torch.randn((S, n), dtype=torch.float64, device="cuda", generator=g) * 3.0
    base[::7] = base[::7].to(torch.float32).to(torch.float64)         # some exactly representable in fp32
    g5 = gamma5_c(n, "cuda")
    for delta in (0.0173 + 2.0 ** -33, -0.31, 0.0):
        D = D0.clone()
        call("mg2d_twist_set", P_(D), P_(base), delta, n, S, dtype, S_())
        assert bits_equal(D, twist_set_ref(D0, base, delta)), delta
        im = D[:, 0].diagonal(dim1=-2, dim2=-1).imag
        if delta == 0.0:
            assert bits_equal(im, base.to(RT[dtype]))
        elif dtype == C64:
            twice = base.to(torch.float32) + (delta * g5).to(torch.float32)
            differ = float((bits(twice) != bits(im)).double().mean())
            assert differ > 0.05, differ
        del D, im


@pytest.mark.gpu
def test_twist_set_refusals():
    """n outside {2, 4, 8, 16, 32} -> MG2D_EUNSUPPORTED, a non-finite delta -> MG2D_EINVAL; nothing is written"""
    for n in (1, 3, 64):
        D = torch.zeros((4, 5, n, n), dtype=torch.complex128, device="cuda")
        base = torch.ones((4, n), dtype=torch.float64, device="cuda")
        with pytest.raises(mg2d.MG2DError, match=r"mg2d_twist_set failed \(-3\)"):
            call("mg2d_twist_set", P_(D), P_(base), 0.1, n, 4, C128, S_())
    D = torch.zeros((4, 5, 2, 2), dtype=torch.complex128, device="cuda")
    base = torch.ones((4, 2), dtype=torch.float64, device="cuda")
    for bad in (math.nan, math.inf, -math.inf):
        with pytest.raises(mg2d.MG2DError, match=r"mg2d_twist_set failed \(-1\)"):
            call("mg2d_twist_set", P_(D), P_(base), bad, 2, 4, C128, S_())
    torch.cuda.synchronize()
    assert float(D.abs().max()) == 0.0


# ---- 2. mg2d_block_inverse with pivoting ---------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("n", [1, 2, 4, 8, 16, 32])
def test_block_inverse_pivoting(n, dtype, gpu_mem):
    """Permuted diagonally dominant blocks (plain tolerance; every column but the last pivots), dense Gaussian blocks, zero
    diagonals and exact ties (tolerance times the condition number), on a capped grid; every result bit-reproducible."""
    warps = _inverse_warps(n, dtype)
    S = _capped_sites(sms() * 16 * warps)
    assert_capped(S, min(-(-S // warps), sms() * 16) * warps, f"block_inverse_kernel n {n}")
    tol = TOL if dtype == C128 else TOL32
    Z = crandn(gen(400 + 2 * n + dtype), S, n, n)
    ar = torch.arange(n, device="cuda")
    for kind in (("gaussian",) if n == 1 else ("permuted", "gaussian", "zero_diag", "ties")):
        A = rounded(self_blocks(kind, Z), dtype)
        piv = pivot_trace(A)
        if kind == "permuted":
            assert bool((piv[:, :n - 1] != ar[:n - 1]).all())
        elif kind == "gaussian" and n > 1:
            assert float(pivots(piv).double().mean()) > 0.4
        elif kind == "zero_diag":
            assert bool((piv[:, 0] != 0).all())
        elif kind == "ties":
            r0, r1 = (1, n - 1) if n >= 3 else (0, 1)
            assert torch.equal(A[:, r0, 0].abs(), A[:, r1, 0].abs()) and bool((piv[:, 0] == r0).all())
        got = _block_inverse(A, dtype)
        _check_inverse(got, A, tol, kind != "permuted", (kind, n, dtype))
        assert bits_equal(_block_inverse(A, dtype), got), kind
        del A, got, piv


# ---- 3. mg2d_premultiply ------------------------------------------------------------------------------------------------
def premultiply_err(M, Dd, inv):
    """M [S, 4, n, n] against -inv D_k in fp64, per block relative to max (|inv| |D_k|) (the dot products' own scale);
    M, Dd [S, 5, n, n] and inv [S, n, n] in device layout"""
    Im = inv.transpose(-1, -2).to(torch.complex128)
    Dk = Dd[:, 1:].transpose(-1, -2).to(torch.complex128)
    want = -torch.einsum("sij,skjl->skil", Im, Dk)
    scale = torch.einsum("sij,skjl->skil", Im.abs(), Dk.abs()).amax((-2, -1))
    err = torch.nan_to_num((M.transpose(-1, -2).to(torch.complex128) - want).abs().amax((-2, -1)) / scale, nan=math.inf)
    return float(err.max())


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("n", [1, 2, 4, 8, 16])
def test_premultiply(n, dtype, gpu_mem):
    """M = -D0^-1 D_k on a capped grid with non-dominant self blocks (zero diagonal, Gaussian) and twisted ones
    (D0 + i mu Gamma5_c), D0^-1 from mg2d_block_inverse as the rebuild makes it."""
    S = _capped_sites(sms() * 16)
    assert_capped(S, min(S, sms() * 16), f"premultiply_kernel n {n}")
    g = gen(500 + 2 * n + dtype)
    D = crandn(g, S, 5, n, n)
    tol = TOL if dtype == C128 else TOL32
    kinds = ("gaussian",) if n == 1 else ("zero_diag", "gaussian", "twisted")
    Z = D[:, 0].transpose(-1, -2).clone()
    M = torch.empty((S, 4, n, n), dtype=CT[dtype], device="cuda")
    for kind in kinds:
        A = self_blocks("gaussian" if kind == "twisted" else kind, Z)
        if kind == "twisted":
            A = A + 0.05j * torch.diag(gamma5_c(n, "cuda")).to(torch.complex128)
        D[:, 0] = A.transpose(-1, -2)
        Dd = D.to(CT[dtype])
        inv = _block_inverse(rounded(A, dtype), dtype).transpose(-1, -2).contiguous()
        M.fill_(complex(math.nan, math.nan))
        call("mg2d_premultiply", P_(M), P_(Dd), P_(inv), n, S, dtype, S_())
        err = premultiply_err(M, Dd, inv)
        assert err < tol, (kind, n, dtype, err)
        del Dd, inv


# ---- 4. mg2d_lowrank_pack_a and the (8, 2) factors ---------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("n,R", [(16, 4), (8, 2)])
def test_lowrank_pack_a(n, R, dtype, gpu_mem):
    """lowrank_pack with D0inv, then lowrank_pack_a with a new D0inv': F equals lowrank_pack with D0inv' bit for bit and its
    conj(B) half is untouched; both halves against the fp64 restatement of the lane order (conj(B) exactly)."""
    S = _capped_sites(sms() * 16 * 8)
    assert_capped(S, min(-(-S // 8), sms() * 16) * 8, f"lowrank_pack_kernel ({n}, {R})")
    Q, IT = 4 * R, n * R // 8
    g = gen(600 + n + dtype)
    A, B = crandn(g, S, Q, n, dtype=CT[dtype]), crandn(g, S, Q, n, dtype=CT[dtype])
    inv1, inv2 = crandn(g, S, n, n, dtype=CT[dtype]), crandn(g, S, n, n, dtype=CT[dtype])     # device layout
    tol = TOL if dtype == C128 else TOL32

    def pack(inv):
        F = torch.full((S, 2, IT, 32), complex(math.nan, math.nan), dtype=CT[dtype], device="cuda")
        call("mg2d_lowrank_pack", P_(F), P_(A), P_(B), P_(inv), n, R, S, dtype, S_())
        return F

    F = pack(inv1)
    want = lr_pack_ref(A, B, inv1.transpose(-1, -2), n, R)
    assert bits_equal(F[:, 0], want[:, 0].to(CT[dtype]))
    assert rel(F[:, 1], want[:, 1]) < tol
    F_b = F[:, 0].clone()
    call("mg2d_lowrank_pack_a", P_(F), P_(A), P_(inv2), n, R, S, dtype, S_())
    assert bits_equal(F, pack(inv2))
    assert bits_equal(F[:, 0], F_b)
    assert rel(F[:, 1], lr_pack_ref(A, B, inv2.transpose(-1, -2), n, R)[:, 1]) < tol


def _lr82_case(Lx, Ly, dtype, strip, yoff, nvs, cmodes, seed):
    """mg2d_lowrank_pack + mg2d_relax_rb_lr at (n, rank) = (8, 2) against the dense-reference half sweeps (the (16, 4) case is
    test_gpu_bench_shapes._lr_case)"""
    n, R = 8, 2
    S, Q = Lx * Ly, 4 * R
    g = gen(seed)
    D0 = rounded(crandn(g, S, n, n) * (0.5 / math.sqrt(n)) + 3.0 * torch.eye(n, dtype=torch.complex128, device="cuda"), dtype)
    D0inv = rounded(torch.linalg.inv(D0), dtype)
    del D0
    A, B = rounded(crandn(g, S, Q, n) * 0.3, dtype), rounded(crandn(g, S, Q, n) * 0.3, dtype)
    Dk = D0inv.transpose(-1, -2).to(CT[dtype]).contiguous()
    Ad, Bd = A.to(CT[dtype]), B.to(CT[dtype])                      # (named: a temporary's memory is reused at once)
    F = torch.empty((S, 2, n * R // 8, 32), dtype=CT[dtype], device="cuda")
    call("mg2d_lowrank_pack", P_(F), P_(Ad), P_(Bd), P_(Dk), n, R, S, dtype, S_())
    del Ad, Bd
    Ag, Bg, D0i = A.reshape(Ly, Lx, Q, n), B.reshape(Ly, Lx, Q, n), D0inv.reshape(Ly, Lx, n, n)
    if not strip:
        nsteps = -(-(Lx // 2) * Ly // 8)
        assert_capped(nsteps, min(nsteps, sms() * 32), f"stencil_rb_lr_kernel (8, 2) {Lx}x{Ly}")
    tol = TOL if dtype == C128 else TOL32
    for nv in nvs:
        for cmode in cmodes:
            phi0 = rounded(crandn(g, nv, S, n), dtype)
            r = rounded(crandn(g, nv, S, n), dtype) if cmode else None
            c_ref = None if r is None else torch.einsum("yxij,vyxj->vyxi", D0i, r.reshape(nv, Ly, Lx, n)).reshape(nv, S, n)
            if strip:
                lo, hi = rounded(crandn(g, nv, Lx, n), dtype), rounded(crandn(g, nv, Lx, n), dtype)
            outs = []
            for rep in range(2):
                phi = phi0.to(CT[dtype], copy=True)
                cbuf = torch.zeros_like(phi) if cmode != 2 else c_ref.to(CT[dtype]).contiguous()
                if strip:
                    lod, hid = lo.to(CT[dtype]), hi.to(CT[dtype])
                    lop, hip, hs = P_(lod), P_(hid), Lx * n
                else:
                    lop, hip, hs = P_(phi) + (Ly - 1) * Lx * n * phi.element_size(), P_(phi), S * n
                rk = r.to(CT[dtype]) if r is not None else None
                for colour in (0, 1):
                    call("mg2d_relax_rb_lr", P_(phi), lop, hip, P_(F), P_(Dk), P_(rk), P_(cbuf), cmode, n, R, Lx, Ly, colour, yoff,
                         dtype, nv, S * n, hs, None, S_())
                outs.append((phi, cbuf))
            assert bits_equal(outs[0][0], outs[1][0]), (nv, cmode)
            want = phi0.reshape(nv, Ly, Lx, n)
            rr = None if r is None else r.reshape(nv, Ly, Lx, n)
            for colour in (0, 1):
                h = (lo.reshape(nv, 1, Lx, n), hi.reshape(nv, 1, Lx, n)) if strip else _periodic_halos(want)
                want = rb_half(want, hop_lowrank(Ag, Bg, neighbours(want, *h)), D0i, rr, colour, yoff)
            assert rel(outs[0][0], want) < tol, (Lx, Ly, dtype, nv, cmode)
            if cmode == 1:
                assert rel(outs[0][1], c_ref) < tol
            del outs


@pytest.mark.gpu
def test_lowrank_sweep_8_2_level1_512(gpu_mem):
    """(8, 2): level 1 of a 1024^2 problem on 2x2 aggregates with 4 null vectors, periodic, capped grid: NV 1 and 4,
    cmode 0/1/2; then the 512 x 64 strip with explicit halo rows, yoff 1, in complex64."""
    _lr82_case(512, 512, C128, False, 0, (1, 4), (0, 1, 2), 700)
    _lr82_case(512, 64, C64, True, 1, (4, 1), (1, 2), 701)


# ---- 5. the whole set_twist chain at 1024^2 ----------------------------------------------------------------------------
L_CHAIN = 1024
_STATE = {}


def _links():
    if "U" not in _STATE:
        _STATE["U"] = mg2d.gauge.quenched_links_device(L_CHAIN, 6.0, sweeps=30, seed=1234)
    return _STATE["U"]


def _chain_params(mass, block=4, n_null=8, **kw):
    nlevels = 3 if block == 4 else 4                                   # coarsest level 16^2 / 64^2
    post = ([4, 2, 6] + [4] * nlevels)[:nlevels + 1]                   # the benchmark's cycle (bench.post_sweeps)
    return mg2d.make_params(L_CHAIN, mass, nlevels=nlevels, block=block, n_null=n_null, n_smooth=4, n_pre=0, n_post=post,
                            smoother="rbgs", null_iters=60, tol=1e-10, max_iters=500, **kw)


def _mcrit(csw):
    """m_crit of the 1024^2 links with clover coefficient csw (multigrid inverse iteration, as the benchmark locates it)"""
    if ("mcrit", csw) not in _STATE:
        from importlib import import_module
        critical = import_module("2d_multigrid_b200.critical")
        _STATE[("mcrit", csw)], _ = critical.estimate_critical_mass(_links(), lambda m: _chain_params(m, csw=csw), iters=3, refine=2)
    return _STATE[("mcrit", csw)]


def _tm_resid(mg, x, b, mu):
    """|b - D_tm(mu) x| / |b| through mg2d_wilson_tm_apply with the level's clover field, independent of the hierarchy's p.mu"""
    lv = mg.LVL[0]
    out = torch.empty_like(x)
    lo, hi = lv._halo(x)
    mg.ctx.call("mg2d_wilson_tm_apply", P_(out), P_(x), lo, hi, P_(lv.U), lv.U_lo_ptr, P_(lv.clover), P_(b), float(mg.p.mass),
                float(mu), lv.L, lv.Ly, _lib.MODE_RESID, _lib.C128, None, S_())
    return float(torch.linalg.vector_norm(out) / torch.linalg.vector_norm(b))


_BUFS = ("D", "D0inv", "M", "F", "Dh", "D0inv_h")


def _snap(mg):
    return {(lv.lvl, k): getattr(lv, k).clone() for lv in mg.LVL for k in _BUFS if getattr(lv, k) is not None}


def _half_bits_equal(h, t32):
    """a __half2 copy (stored as float32 words) holds each fp32 component rounded to nearest fp16"""
    return torch.equal(h.view(torch.float16).reshape(-1).view(torch.int16),
                       torch.view_as_real(t32).to(torch.float16).reshape(-1).view(torch.int16))


def _check_level(lv, snap, base, delta, A, tol, report):
    """One level after set_twist: D changed only on the imaginary self-block diagonal (bit for bit), D0^-1 against the fp64
    inverse of the new self blocks (tolerance times the condition number), M = -D0^-1 D_k and the -D0^-1 A half of F against
    fp64 from the kernel's D0^-1, F's conj(B) half untouched, the half copies the rounding of the new buffers."""
    l = lv.lvl
    what = (l, lv.mg.p.dtype)
    assert bits_equal(lv.D, twist_set_ref(snap[(l, "D")], base, delta)), what
    A0 = lv.D[:, 0].transpose(-1, -2).to(torch.complex128)
    if lv.D0inv is not None:
        kappa = _check_inverse(lv.D0inv.transpose(-1, -2), A0, tol, True, what)
        if report is not None and lv.n > 2:
            frac = float(pivots(pivot_trace(A0)).double().mean())
            report.append(f"level {l} ({lv.mg.p.dtype}, n {lv.n}, {lv.S} sites): max condition {kappa:.3g}, "
                          f"{100 * frac:.1f}% of the twisted self blocks pivot")
    if lv.M is not None:
        err = premultiply_err(lv.M, lv.D, lv.D0inv)
        assert err < tol, (what, err)
    if lv.F is not None:
        assert bits_equal(lv.F[:, 0], snap[(l, "F")][:, 0]), what
        if A is not None:
            assert rel(lv.F[:, 1], lr_ma_ref(A, lv.D0inv.transpose(-1, -2), lv.n, lv.lr_rank)) < tol, what
    if lv.Dh is not None:
        assert _half_bits_equal(lv.Dh, lv.D) and _half_bits_equal(lv.D0inv_h, lv.D0inv), what


_VARIANTS = {"wilson": {}, "clover": {"csw": 1.0}, "stored_level0": {"matrix_free": False},
             "block2_rank2": {"block": 2, "n_null": 4}, "built_twisted": {"mu": 0.011}}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(_VARIANTS))
def test_set_twist_chain_1024(variant, gpu_mem):
    """Hierarchies with the benchmark's cycle at 1024^2 near the critical mass (low-rank first coarse level, pre-multiplied
    deeper levels, complex64+half shadow): after set_twist(mu) every level and the shadow hold what the fp64 reference gives
    from the kept state, a twisted solve reaches a true residual <= 1e-10 of D_tm(mu), and set_twist(mu_b) restores every
    buffer bit for bit."""
    kw = dict(_VARIANTS[variant])
    U = _links()
    mass = _mcrit(kw.get("csw", 0.0)) + 1e-3
    mg = mg2d.setup(U, _chain_params(mass, **kw), init="device")
    mu_b = mg.p.mu
    b = torch.randn((L_CHAIN * L_CHAIN, 2), dtype=torch.complex128, device="cuda", generator=gen(800))
    for pd in (None, "complex64+half"):         # a few cycles build D0^-1, M, F of both hierarchies and the half copies
        mg2d.solve(mg, rhs=b, tol=1e-10, max_iters=3, outer="gcr", restart=8, precond_dtype=pd)
    sh = mg.info["single"]
    rank = 2 if variant == "block2_rank2" else 4
    assert mg.LVL[1].F is not None and mg.LVL[1].lr_rank == rank and sh.LVL[1].F is not None
    assert all(lv.M is not None for lv in mg.LVL[2:])
    assert mg.LVL[0].matrix_free == (variant != "stored_level0")
    assert any(l32.Dh is not None for l32 in sh.LVL)
    snap, snap32 = _snap(mg), _snap(sh)
    mu = 0.0173 if mu_b == 0.0 else -0.02
    mg.set_twist(mu)
    st = mg.info["twist"]
    assert st["mu_b"] == mu_b
    delta = mu - mu_b
    report = []
    for lv, l32 in zip(mg.LVL, sh.LVL):
        if lv.D is None:
            assert lv.lvl == 0 and lv.matrix_free and l32.D is None
            continue
        _check_level(lv, snap, st["base"][lv.lvl], delta, st["A"][lv.lvl], TOL, report)
        _check_level(l32, snap32, st["base"][lv.lvl], delta, None, TOL32, None)
        if l32.F is not None:
            assert bits_equal(l32.F, lv.F.to(torch.complex64))
    print(f"\n{variant}: m = m_crit {mass - 1e-3:+.5f} + 1e-3, mu {mu}\n  " + "\n  ".join(report))
    x, info = mg2d.solve(mg, rhs=b, tol=1e-10, outer="gcr", restart=8, precond_dtype="complex64+half")
    assert info["converged"], info["resnorms"][-3:]
    assert _tm_resid(mg, x, b, mu) <= 1e-10
    mg.set_twist(mu_b)
    for now, then in ((_snap(mg), snap), (_snap(sh), snap32)):
        assert set(now) == set(then)
        for k, v in now.items():
            assert bits_equal(v, then[k]), k
    mg.close()


@pytest.mark.gpu
def test_normal_solve_clover_against_dense_32():
    """normal_solve on a Wilson-clover hierarchy (csw = 1) against the dense normal equations, as
    test_rhmc_mg.test_normal_solve_against_dense_32 does for Wilson"""
    from test_rhmc_mg import _links as links, _p, _rhs
    L, m, tol = 32, 0.1, 1e-10
    U, th = links(L, beta=2.0)
    mg = mg2d.setup(U, _p(L, 4, 1, m=m, csw=1.0), init="device")
    assert mg.LVL[0].clover is not None
    b = _rhs(L)
    shifts = [1e-3, 0.0, 1e-5, 0.1]
    X, info = mg2d.normal_solve(mg, b, shifts, tol, use_graph=True)
    assert mg.p.mu == 0.0 and info["converged"] and max(info["true_residuals"]) <= tol, info["true_residuals"]
    D = dense_tm(np.exp(1j * th.cpu().numpy()), L, m, 1.0, 0.0)
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


# ---- 6. mg2d_gamma5 in place ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("S", [4096 * 4096, 1_000_003, 255])
def test_gamma5_in_place_and_out_of_place(S, gpu_mem):
    """out = in * [1, -1] bit for bit, out of place (in untouched) and in place (out == in, as normal_solve calls it)"""
    if S > sms() * 8 * 256:
        assert_capped(S, min(-(-S // 256), sms() * 8) * 256, f"gamma5_kernel {S}")
    x = crandn(gen(900 + S % 97), S, 2)
    want = torch.stack([x[:, 0], -x[:, 1]], 1)
    x0 = x.clone()
    out = torch.full_like(x, complex(math.nan, math.nan))
    call("mg2d_gamma5", P_(out), P_(x), S, S_())
    assert bits_equal(out, want) and bits_equal(x, x0)
    call("mg2d_gamma5", P_(x), P_(x), S, S_())
    assert bits_equal(x, want)
