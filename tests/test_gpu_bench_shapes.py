"""The solver's hot-path kernels at the benchmark's shapes, precisions and strip geometries against an fp64 reference.

The headline solve (4096^2 Wilson, 16 dof on the coarse levels, 4x4 aggregates, FGCR(8)) runs its kernels on grids so
large that the launchers cap the grid: every CTA / warp then loops over several work items, a regime the small parity
tests never reach.  On 2/4/8 GPUs the levels are strips (Ly < Lx) whose halo rows are not the periodic wrap, and the
preconditioner runs in complex64 and half precision.  Here each operation is restated from its definition (layouts:
include/mg2d.h) as vectorised torch in fp64 on whatever device the tensors live on -- no kernel index tricks.  The CPU
tests anchor that reference to the numpy oracle; the GPU tests hold the kernels to it on seeded synthetic operators
generated on the device (a set-up 4096^2 hierarchy would not fit beside its reference).

Tolerances, relative in the max-norm: complex128 1e-12; complex64 2e-5 against the fp64 reference of the fp32-rounded
inputs; the half-precision sweep 2e-5 against the fp64 reference of the half-rounded blocks.  Every capped-grid case
asserts, from the SM count and the launcher's formula, at least two passes per CTA / warp with a partial last one.
"""
import math

import numpy as np
import pytest
import torch

import mg2d
from oracle import mg_oracle as O

TOL = 1e-12
TOL32 = 2e-5
C128, C64 = 0, 1
CT = {C128: torch.complex128, C64: torch.complex64}


# ================================================================================================================
# fp64 reference.  Fields are grids [..., Ly, Lx, n] (site s = x + y*Lx); blocks are in math layout [..., i, j]
# (the device stores them column-major: D_dev[s][k][j][i], so Dm = D_dev.transpose(-1, -2)).
# ================================================================================================================
def neighbours(f, lo, hi):
    """f(s+x), f(s-x), f(s+y), f(s-y) (stencil slots 1..4) of a strip f [..., Ly, Lx, n]: x periodic, row -1 = the last
    row of `lo` [..., d, Lx, n], row Ly = the first row of `hi`."""
    e = torch.cat([lo[..., -1:, :, :], f, hi[..., :1, :, :]], dim=-3)
    return f.roll(-1, dims=-2), f.roll(1, dims=-2), e[..., 2:, :, :], e[..., :-2, :, :]


def hop_dense(Dm, nb):
    """sum_{k=1..4} D_k(s) f(s+d_k); Dm [Ly, Lx, 5, n, n]."""
    return sum(torch.einsum("yxij,...yxj->...yxi", Dm[:, :, k + 1], nb[k]) for k in range(4))


def hop_lowrank(A, B, nb):
    """The same with D_k = sum_b A_q B_q^dagger, q = (k-1)*R + b; A, B [Ly, Lx, 4R, n]."""
    R = A.shape[-2] // 4
    out = 0
    for k in range(4):
        t = torch.einsum("yxqj,...yxj->...yxq", B[:, :, k * R:(k + 1) * R].conj(), nb[k])
        out = out + torch.einsum("yxqi,...yxq->...yxi", A[:, :, k * R:(k + 1) * R], t)
    return out


def colour_mask(Lx, Ly, colour, yoff, device):
    y = torch.arange(Ly, device=device)[:, None]
    x = torch.arange(Lx, device=device)[None, :]
    return ((x + y + yoff) % 2 == colour)[:, :, None]


def rb_half(phi, hop, D0inv, r, colour, yoff):
    """Red-black half sweep (f_relax's update rule): sites with (x+y+yoff)%2 == colour get -D0^-1 (hop - r)."""
    rhs = hop if r is None else hop - r
    new = -torch.einsum("yxij,...yxj->...yxi", D0inv, rhs)
    return torch.where(colour_mask(phi.shape[-2], phi.shape[-3], colour, yoff, phi.device), new, phi)


def wilson_proj(device):
    """(1 - sigma_1)/2, (1 + sigma_1)/2, (1 - sigma_2)/2, (1 + sigma_2)/2: the spin structure of slots 1..4 (S6/level.h:155-172)."""
    I = torch.eye(2, dtype=torch.complex128, device=device)
    g1 = torch.tensor([[0, 1], [1, 0]], dtype=torch.complex128, device=device)
    g2 = torch.tensor([[0, -1j], [1j, 0]], dtype=torch.complex128, device=device)
    return [0.5 * (I - g1), 0.5 * (I + g1), 0.5 * (I - g2), 0.5 * (I + g2)]


def wilson_hop(f, lo, hi, U, U_lo):
    """Level-0 Wilson hop matrix-free from the links U [Ly, Lx, 2] = (U_x, U_y); U_lo: link rows below (last = row -1)."""
    nb = neighbours(f, lo, hi)
    Uy_m = torch.cat([U_lo[-1:, :, 1], U[:-1, :, 1]], dim=0)
    coef = (U[..., 0], U[..., 0].roll(1, dims=1).conj(), U[..., 1], Uy_m.conj())
    P = wilson_proj(f.device)
    return sum(coef[k][..., None] * torch.einsum("ij,...j->...i", P[k], nb[k]) for k in range(4))


def wilson_half(phi, lo, hi, U, U_lo, r, mass, colour, yoff):
    hop = wilson_hop(phi, lo, hi, U, U_lo)
    new = ((0 if r is None else r) - hop) / (2.0 + mass)
    return torch.where(colour_mask(phi.shape[-2], phi.shape[-3], colour, yoff, phi.device), new, phi)


def wilson_rb2(phi, lo2, hi2, U, U_lo2, U_hi, r, r_lo, r_hi, mass, yoff):
    """Both colours, out of place: colour 0 on the rows -1..Ly (from old values two rows deep), then colour 1 on the
    rows 0..Ly-1 from those new values.  Halos: phi rows -2,-1 / Ly,Ly+1; links rows -2,-1 / Ly; r rows -1 / Ly."""
    Ly = phi.shape[-3]
    E = torch.cat([lo2, phi, hi2], dim=0)                       # rows -2 .. Ly+1
    UE = torch.cat([U_lo2, U, U_hi], dim=0)                     # rows -2 .. Ly
    RE = None if r is None else torch.cat([r_lo, r, r_hi], dim=0)   # rows -1 .. Ly
    red = wilson_half(E[1:Ly + 3], E[:1], E[Ly + 3:], UE[1:Ly + 3], UE[:1], RE, mass, 0, yoff + 1)   # rows -1 .. Ly
    return wilson_half(red[1:Ly + 1], red[:1], red[Ly + 1:], U, U_lo2, r, mass, 1, yoff)


def owner(Lxf, Lyf, block, quad, device):
    """owner[s] = coarse site of fine site s: aggregates based at (block*xc - dx, block*yc - dy) (f_get_base_site)."""
    dx, dy = int(quad in (2, 3)), int(quad in (3, 4))
    y = torch.arange(Lyf, device=device)[:, None]
    x = torch.arange(Lxf, device=device)[None, :]
    return (((x + dx) % Lxf) // block + (((y + dy) % Lyf) // block) * (Lxf // block)).reshape(-1)


def _sum_aggregates(Pv, own, block):
    nagg = Pv.shape[0] // (block * block)
    return Pv[torch.argsort(own, stable=True)].reshape(nagg, block * block, -1).sum(1)


def restrict(vf, P, own, block):
    """vc(X) = sum_{s in X} P(s) vf(s); P [S, nc, nf]."""
    return _sum_aggregates(torch.einsum("sij,sj->si", P, vf), own, block)


def prolong(vf, vc, P, own, accumulate=True):
    """vf(s) (+)= P(s)^dagger vc(X(s))."""
    add = torch.einsum("sij,si->sj", P.conj(), vc[own])
    return vf + add if accumulate else add


def restrict_chiral(vf, Pc, own, block):
    """Pc [S, nc, nf/2]: row i < nc/2 acts on the upper half of the spinor, row i >= nc/2 on the lower half."""
    h, hf = Pc.shape[1] // 2, Pc.shape[2]
    Pv = torch.cat([torch.einsum("sij,sj->si", Pc[:, :h], vf[:, :hf]), torch.einsum("sij,sj->si", Pc[:, h:], vf[:, hf:])], 1)
    return _sum_aggregates(Pv, own, block)


def prolong_chiral(vf, vc, Pc, own, accumulate=True):
    h = Pc.shape[1] // 2
    w = vc[own]
    add = torch.cat([torch.einsum("sij,si->sj", Pc[:, :h].conj(), w[:, :h]), torch.einsum("sij,si->sj", Pc[:, h:].conj(), w[:, h:])], 1)
    return vf + add if accumulate else add


def chiral_dense(Pc):
    """The dense projector a chirality-compacted one stands for (zeros in the other chirality's columns)."""
    S, nc, hf = Pc.shape
    P = torch.zeros((S, nc, 2 * hf), dtype=Pc.dtype, device=Pc.device)
    P[:, :nc // 2, :hf] = Pc[:, :nc // 2]
    P[:, nc // 2:, hf:] = Pc[:, nc // 2:]
    return P


def lazy_coefficients(bs, as_):
    """FGCR lazy update (comment above gcr_step_lazy_kernel): zh_j = z_j - sum_{i<j} b_ij zh_i = sum_{i<=j} c_ij z_i,
    g_i = sum_j a_j c_ij.  bs[j] = (b_0j .. b_{j-1}j), as_[j] = a_j.  Returns C [8, 8] (C[i, j] = c_ij) and g [8]."""
    C = np.zeros((8, 8), dtype=complex)
    g = np.zeros(8, dtype=complex)
    for j, (b, a) in enumerate(zip(bs, as_)):
        C[j, j] = 1.0
        for i in range(j):
            C[:, j] -= b[i] * C[:, i]
        g += a * C[:, j]
    return C, g


# ================================================================================================================
# CPU: the reference against the numpy oracle
# ================================================================================================================
def _c(rng, *s):
    return rng.normal(size=s) + 1j * rng.normal(size=s)


def _t(a):
    return torch.as_tensor(np.ascontiguousarray(a))


def _periodic_halos(f, depth=1):
    return f[..., -depth:, :, :], f[..., :depth, :, :]


def _maxrel(a, b):
    a = a.numpy() if torch.is_tensor(a) else a
    b = b.numpy() if torch.is_tensor(b) else b
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.mark.parametrize("L,n", [(8, 2), (10, 4), (16, 16)])
def test_reference_block_stencil_matches_oracle(L, n):
    rng = np.random.default_rng(L + n)
    D = _c(rng, L * L, 5, n, n) * 0.2
    D[:, 0] += 3.0 * np.eye(n)
    lvo = O.Level()
    lvo.D, lvo.phi, lvo.r = D, _c(rng, L * L, n), _c(rng, L * L, n)
    Dm = _t(D).reshape(L, L, 5, n, n)
    phi, r = _t(lvo.phi).reshape(L, L, n), _t(lvo.r).reshape(L, L, n)
    D0inv = torch.linalg.inv(Dm[:, :, 0])
    app = hop_dense(Dm, neighbours(phi, *_periodic_halos(phi))) + torch.einsum("yxij,yxj->yxi", Dm[:, :, 0], phi)
    assert _maxrel(app.reshape(-1, n), lvo.apply_D(lvo.phi, L)) < 1e-13
    assert _maxrel((r - app).reshape(-1, n), lvo.residue(L)) < 1e-13
    for _ in range(2):
        for colour in (0, 1):
            phi = rb_half(phi, hop_dense(Dm, neighbours(phi, *_periodic_halos(phi))), D0inv, r, colour, 0)
    lvo.relax_rb(L, 2)
    assert _maxrel(phi.reshape(-1, n), lvo.phi) < 1e-13


@pytest.mark.parametrize("L,n,R", [(8, 16, 4), (16, 8, 2)])
def test_reference_lowrank_sweep_matches_oracle(L, n, R):
    """The low-rank hop sum_b A_q B_q^dagger against the oracle's sweep on the dense blocks it stands for."""
    rng = np.random.default_rng(3 * L + R)
    A, B = _c(rng, L * L, 4 * R, n) * 0.3, _c(rng, L * L, 4 * R, n) * 0.3
    D = np.zeros((L * L, 5, n, n), dtype=complex)
    D[:, 0] = _c(rng, L * L, n, n) * 0.2 + 3.0 * np.eye(n)
    for k in range(4):
        D[:, k + 1] = np.einsum("sbi,sbj->sij", A[:, k * R:(k + 1) * R], np.conj(B[:, k * R:(k + 1) * R]))
    lvo = O.Level()
    lvo.D, lvo.phi, lvo.r = D, _c(rng, L * L, n), _c(rng, L * L, n)
    At, Bt = _t(A).reshape(L, L, 4 * R, n), _t(B).reshape(L, L, 4 * R, n)
    phi, r = _t(lvo.phi).reshape(L, L, n), _t(lvo.r).reshape(L, L, n)
    D0inv = torch.linalg.inv(_t(D[:, 0]).reshape(L, L, n, n))
    for colour in (0, 1):
        phi = rb_half(phi, hop_lowrank(At, Bt, neighbours(phi, *_periodic_halos(phi))), D0inv, r, colour, 0)
    lvo.relax_rb(L, 1)
    assert _maxrel(phi.reshape(-1, n), lvo.phi) < 1e-13


def test_reference_strips_equal_whole_lattice():
    """A half sweep on a strip of rows [y0, y0+Ly) with the neighbouring rows as explicit halos and yoff = y0 % 2 equals
    the whole-lattice sweep there (block stencil and both Wilson sweeps): the strip arguments of the reference are right."""
    rng = np.random.default_rng(5)
    L, n, m = 12, 4, -0.07
    D = _t(_c(rng, L, L, 5, n, n) * 0.2)
    D[:, :, 0] += 3.0 * torch.eye(n, dtype=torch.complex128)
    D0inv = torch.linalg.inv(D[:, :, 0])
    phi, r = _t(_c(rng, L, L, n)), _t(_c(rng, L, L, n))
    whole = rb_half(phi, hop_dense(D, neighbours(phi, *_periodic_halos(phi))), D0inv, r, 1, 0)
    U = _t(np.exp(1j * rng.uniform(-np.pi, np.pi, size=(L, L, 2))))
    psi, rw = _t(_c(rng, L, L, 2)), _t(_c(rng, L, L, 2))
    w_whole = wilson_rb2(psi, psi[-2:], psi[:2], U, U[-2:], U[:1], rw, rw[-1:], rw[:1], m, 0)
    for y0, Ly in ((3, 5), (8, 4), (0, 3)):
        rows = [(y0 + d) % L for d in range(-2, Ly + 2)]
        f, rr, Dm = phi[rows[2:-2]], r[rows[2:-2]], D[rows[2:-2]]
        got = rb_half(f, hop_dense(Dm, neighbours(f, phi[rows[1:2]], phi[rows[-2:-1]])), D0inv[rows[2:-2]], rr, 1, y0 % 2)
        assert _maxrel(got, whole[rows[2:-2]]) < 1e-15
        got = wilson_rb2(psi[rows[2:-2]], psi[rows[:2]], psi[rows[-2:]], U[rows[2:-2]], U[rows[:2]], U[rows[-2:-1]],
                         rw[rows[2:-2]], rw[rows[1:2]], rw[rows[-2:-1]], m, y0 % 2)
        assert _maxrel(got, w_whole[rows[2:-2]]) < 1e-15


@pytest.mark.parametrize("L", [8, 16])
def test_reference_wilson_matches_oracle(L):
    """Matrix-free hop from the links == the oracle's stored level-0 operator; both red-black forms == relax_rb."""
    rng = np.random.default_rng(L)
    m = -0.05
    po = O.Params(L=L, num_iters=2, block=2, m=m, nlevels=1)
    Uf = O.gauge_gaussian(L, width=0.4, seed=9)
    lvo = O.Level()
    lvo.compute_lvl0_matrix(Uf, po)
    lvo.phi, lvo.r = _c(rng, L * L, 2), _c(rng, L * L, 2)
    U = _t(Uf).reshape(L, L, 2)
    phi, r = _t(lvo.phi).reshape(L, L, 2), _t(lvo.r).reshape(L, L, 2)
    app = wilson_hop(phi, *_periodic_halos(phi), U, U[-1:]) + (2.0 + m) * phi
    assert _maxrel(app.reshape(-1, 2), lvo.apply_D(lvo.phi, L)) < 1e-13
    half = phi
    for colour in (0, 1):
        half = wilson_half(half, *_periodic_halos(half), U, U[-1:], r, m, colour, 0)
    two = wilson_rb2(phi, phi[-2:], phi[:2], U, U[-2:], U[:1], r, r[-1:], r[:1], m, 0)
    lvo.relax_rb(L, 1)
    assert _maxrel(half.reshape(-1, 2), lvo.phi) < 1e-13
    assert _maxrel(two.reshape(-1, 2), lvo.phi) < 1e-13


@pytest.mark.parametrize("L,block,nf,nc", [(8, 2, 2, 4), (16, 4, 2, 16), (12, 2, 4, 8)])
def test_reference_transfer_matches_oracle(L, block, nf, nc):
    rng = np.random.default_rng(L * block)
    Lc = L // block
    po = O.Params(L=L, num_iters=2, block=block, m=0.1, nlevels=1)
    Pc = _c(rng, L * L, nc, nf // 2)
    P = chiral_dense(_t(Pc)).numpy()
    lvo = O.Level()
    lvo.phi_null = P
    vf, vc = _c(rng, L * L, nf), _c(rng, Lc * Lc, nc)
    for quad in (1, 2, 3, 4):
        own = owner(L, L, block, quad, "cpu")
        want = lvo.restriction(vf, 0, po, quad)
        assert _maxrel(restrict(_t(vf), _t(P), own, block), want) < 1e-13
        assert _maxrel(restrict_chiral(_t(vf), _t(Pc), own, block), want) < 1e-13
        fo = vf.copy()
        lvo.prolongation(fo, vc, 1, po, quad)
        assert _maxrel(prolong(_t(vf), _t(vc), _t(P), own), fo) < 1e-13
        assert _maxrel(prolong_chiral(_t(vf), _t(vc), _t(Pc), own), fo) < 1e-13
        assert _maxrel(prolong_chiral(_t(vf), _t(vc), _t(Pc), own, accumulate=False), fo - vf) < 1e-13


def test_reference_lazy_gcr_equals_explicit_orthogonalisation():
    """x + sum_i g_i z_i of the lazy recursion == x + sum_j a_j zh_j with the directions orthogonalised explicitly."""
    rng = np.random.default_rng(11)
    z = _c(rng, 8, 50)
    bs = [_c(rng, j) for j in range(8)]
    as_ = list(_c(rng, 8))
    zh = []
    for j in range(8):
        zh.append(z[j] - sum(bs[j][i] * zh[i] for i in range(j)))
    _, g = lazy_coefficients(bs, as_)
    assert _maxrel(g @ z, sum(a * v for a, v in zip(as_, zh))) < 1e-13


# ================================================================================================================
# GPU
# ================================================================================================================
_CTX = None


def ctx():
    global _CTX
    if _CTX is None:
        _CTX = mg2d._lib.Context(0)
    return _CTX


def call(name, *args):
    ctx().call(name, *args)


def P_(t):
    return None if t is None else t.data_ptr()


def S_():
    return torch.cuda.current_stream().cuda_stream


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def assert_capped(work, grid, what):
    """A grid-stride loop over `work` items on `grid` CTAs / warps: >= 2 passes and a partial last pass."""
    passes = -(-work // grid)
    assert passes >= 2 and work % grid != 0, f"{what}: {work} items on {grid} -> {passes} passes (the capped regime is gone)"


def rel(got, want):
    """max |got - want| / max |want| in fp64, in chunks (no full-size temporaries); NaN when either side holds a NaN
    (Python's max() would silently drop it)."""
    g, w = got.reshape(-1), want.reshape(-1)
    num = den = 0.0
    for i in range(0, w.numel(), 1 << 24):
        wi = w[i:i + (1 << 24)].to(torch.complex128)
        d = float((g[i:i + (1 << 24)].to(torch.complex128) - wi).abs().max())
        if math.isnan(d):
            return math.nan
        num = max(num, d)
        den = max(den, float(wi.abs().max()))
    return num / max(den, 1e-300)


def crandn(gen, *shape, dtype=torch.complex128):
    return torch.randn(shape, dtype=dtype, device="cuda", generator=gen)


def gen(seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return g


def rounded(t, dtype):
    """the inputs a kernel of `dtype` sees, as fp64 (the reference's inputs)"""
    return t.to(CT[dtype]).to(torch.complex128)


@pytest.fixture(autouse=False)
def gpu_mem():
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    yield
    print(f"\npeak device memory {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _diag_dominant(g, S, n, dtype=torch.complex128):
    D0 = crandn(g, S, n, n, dtype=dtype) * 0.2
    D0 += 3.0 * torch.eye(n, dtype=dtype, device="cuda")
    return D0


# ---- level 1: low-rank sweep ----------------------------------------------------------------------------------
def _lr_case(Lx, Ly, dtype, strip, yoff, nvs, cmodes, seed):
    n, R = 16, 4
    S, Q = Lx * Ly, 16
    g = gen(seed)
    D0 = rounded(_diag_dominant(g, S, n), dtype)
    D0inv = torch.linalg.inv(D0)                                    # the reference's inverse; the kernel gets it too
    del D0
    A, B = rounded(crandn(g, S, Q, n) * 0.25, dtype), rounded(crandn(g, S, Q, n) * 0.25, dtype)
    # packed in complex128 as the setup does; the complex64 preconditioner receives a converted copy
    F = torch.empty((S, 2, n * R // 8, 32), dtype=torch.complex128, device="cuda")
    Dk = D0inv.transpose(-1, -2).contiguous()                       # device layout (column-major blocks)
    call("mg2d_lowrank_pack", P_(F), P_(A), P_(B), P_(Dk), n, R, S, C128, S_())
    F, Dk = F.to(CT[dtype]), Dk.to(CT[dtype])
    assert_capped(S, min(-(-S // 8), sms() * 16) * 8, "lowrank_pack_kernel")
    Ag, Bg, D0i = A.reshape(Ly, Lx, Q, n), B.reshape(Ly, Lx, Q, n), D0inv.reshape(Ly, Lx, n, n)
    nsteps = -(-(Lx // 2) * Ly // 8)
    assert_capped(nsteps, min(nsteps, sms() * 32), f"stencil_rb_lr_kernel {Lx}x{Ly}")
    tol = TOL if dtype == C128 else TOL32
    for nv in nvs:
        for cmode in cmodes:
            phi0 = rounded(crandn(g, nv, S, n), dtype)
            r = rounded(crandn(g, nv, S, n), dtype) if cmode else None
            c_ref = None if r is None else torch.einsum("yxij,vyxj->vyxi", D0i, r.reshape(nv, Ly, Lx, n)).reshape(nv, S, n).contiguous()
            if strip:
                lo, hi = rounded(crandn(g, nv, Lx, n), dtype), rounded(crandn(g, nv, Lx, n), dtype)
                hs = Lx * n
            outs = []
            for rep in range(2):
                phi = phi0.to(CT[dtype], copy=True)
                cbuf = torch.zeros_like(phi) if cmode != 2 else c_ref.to(CT[dtype], copy=True)
                if strip:
                    lod, hid = lo.to(CT[dtype]), hi.to(CT[dtype])
                    lop, hip = P_(lod), P_(hid)
                else:
                    lop, hip, hs = P_(phi) + (Ly - 1) * Lx * n * phi.element_size(), P_(phi), S * n
                rk = r.to(CT[dtype]) if r is not None else None
                for colour in (0, 1):
                    call("mg2d_relax_rb_lr", P_(phi), lop, hip, P_(F), P_(Dk), P_(rk), P_(cbuf), cmode, n, R, Lx, Ly, colour, yoff,
                         dtype, nv, S * n, hs, None, S_())
                outs.append((phi, cbuf))
            assert torch.equal(outs[0][0], outs[1][0]), (nv, cmode)
            want = phi0.reshape(nv, Ly, Lx, n)
            rr = None if r is None else r.reshape(nv, Ly, Lx, n)
            for colour in (0, 1):
                h = (lo.reshape(nv, 1, Lx, n), hi.reshape(nv, 1, Lx, n)) if strip else _periodic_halos(want)
                hop = hop_lowrank(Ag, Bg, neighbours(want, *h))
                want = rb_half(want, hop, D0i, rr, colour, yoff)
            assert rel(outs[0][0], want) < tol, (Lx, Ly, dtype, nv, cmode)
            if cmode == 1:
                assert rel(outs[0][1], c_ref) < tol
            del outs, phi, cbuf


@pytest.mark.gpu
def test_lowrank_sweep_level1_1024(gpu_mem):
    """mg2d_lowrank_pack + mg2d_relax_rb_lr on the benchmark's level 1 (1024^2, 16 dof, rank 4): cmode 0/1/2, NV 1 and 4."""
    _lr_case(1024, 1024, C128, False, 0, (1, 4), (0, 1, 2), 1)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_lowrank_sweep_level1_strip(dtype, gpu_mem):
    """Level 1 of the 8-rank plan (1024 x 128), explicit halo rows, NV = 4 with hstride = L*n, yoff = 1."""
    _lr_case(1024, 128, dtype, True, 1, (4, 1) if dtype == C128 else (1,), (0, 1, 2) if dtype == C128 else (1, 2), 2)


@pytest.mark.gpu
def test_block_inverse_1024(gpu_mem):
    """mg2d_block_inverse on the 1024^2 level (capped grid); complex64 keeps the 5-slot operator at 10 GB."""
    S, n = 1024 * 1024, 16
    g = gen(3)
    D = torch.empty((S, 5, n, n), dtype=torch.complex64, device="cuda")
    D[:, 0] = _diag_dominant(g, S, n, torch.complex64)
    inv = torch.empty((S, n, n), dtype=torch.complex64, device="cuda")
    call("mg2d_block_inverse", P_(inv), P_(D), n, S, C64, S_())
    warps = min(48 * 1024 // (2 * n * n * 16), 8)
    assert_capped(S, min(-(-S // warps), sms() * 16) * warps, "block_inverse_kernel")
    want = torch.linalg.inv(D[:, 0].transpose(-1, -2).to(torch.complex128))
    assert rel(inv.transpose(-1, -2), want) < TOL32


# ---- hop factors 4096^2 -> 1024^2 -------------------------------------------------------------------------------
@pytest.mark.gpu
def test_hop_factors_4096(gpu_mem):
    """mg2d_hop_factors on the benchmark's level 0 -> 1 (Wilson fine operator from random links, random dense projector):
    sum_b A_q B_q^dagger equals the Galerkin hop block sum over the face links P(s) D_k(s) P(s+d_k)^dagger."""
    L, blk, nc, nf = 4096, 4, 16, 2
    Lc = L // blk
    g = gen(4)
    th = torch.rand((L * L, 2), dtype=torch.float64, device="cuda", generator=g) * (2 * math.pi)
    U = torch.polar(torch.ones_like(th), th)
    del th
    Df = torch.empty((L * L, 5, 2, 2), dtype=torch.complex128, device="cuda")
    call("mg2d_lvl0_matrix", P_(Df), P_(U), P_(U) + (L - 1) * L * 2 * 16, -0.05, 0, L, L, C128, S_())
    del U
    P = crandn(g, L * L, nc, nf)
    A = torch.empty((Lc * Lc, 4 * blk, nc), dtype=torch.complex128, device="cuda")
    B = torch.empty_like(A)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    rowb = L * nc * nf * 16
    call("mg2d_hop_factors", P_(A), P_(B), P_(Df), P_(P), P_(P) + (L - 1) * rowb, P_(P), nf, nc, L, L, blk, C128, P_(status), S_())
    nagg = Lc * Lc
    assert_capped(nagg, min(-(-nagg // 8), sms() * 16) * 8, "hop_factors_kernel")
    assert int(status.item()) == 0
    Dm = Df.reshape(L, L, 5, 2, 2).transpose(-1, -2)
    Pg = P.reshape(L, L, nc, nf)
    A4, B4 = A.reshape(Lc, Lc, 4, blk, nc), B.reshape(Lc, Lc, 4, blk, nc)
    worst = 0.0
    for yc0 in range(0, Lc, 64):
        ys = slice(blk * yc0, blk * (yc0 + 64))
        rows = torch.arange(blk * yc0 - 1, blk * (yc0 + 64) + 1, device="cuda") % L     # one fine row either side
        Pe, De = Pg[rows], Dm[rows]
        rec = torch.einsum("yxkbi,yxkbj->yxkij", A4[yc0:yc0 + 64], B4[yc0:yc0 + 64].conj())
        want = []
        for k in range(4):
            if k < 2:                       # x faces: column blk-1 (k=1) / 0 (k=2) of every aggregate, all its rows
                x1, sh = (blk - 1, -1) if k == 0 else (0, 1)
                Ps = Pe[1:-1, x1::blk]
                Pn = Pe[1:-1].roll(sh, dims=1)[:, x1::blk]
                t = torch.einsum("yxij,yxjl,yxml->yxim", Ps, De[1:-1, x1::blk, k + 1], Pn.conj())
                want.append(t.reshape(64, blk, Lc, nc, nc).sum(1))
            else:                           # y faces: row blk-1 (k=3) / 0 (k=4), all its columns
                y1, dy = (blk - 1, 1) if k == 2 else (0, -1)
                Ps = Pe[1 + y1::blk][:64]
                Pn = Pe[1 + y1 + dy::blk][:64]
                t = torch.einsum("yxij,yxjl,yxml->yxim", Ps, De[1 + y1::blk][:64, :, k + 1], Pn.conj())
                want.append(t.reshape(64, Lc, blk, nc, nc).sum(2))
        want = torch.stack(want, 2)
        worst = max(worst, rel(rec, want))
        del rec, want, t, Pe, De
    assert worst < TOL


# ---- level 2 (256^2): pre-multiplied and half-precision sweeps ----------------------------------------------------
def _stencil_operator(g, S, n, dtype):
    """D [S, 5, n, n] device layout with diagonally dominant self blocks, rounded to `dtype`, and its math-layout copy."""
    D = crandn(g, S, 5, n, n) * 0.2
    D[:, 0] += 3.0 * torch.eye(n, dtype=torch.complex128, device="cuda")
    D = rounded(D, dtype)
    return D.to(CT[dtype]), D.transpose(-1, -2)


def _pm_case(Lx, Ly, dtype, strip, yoff, nvs, cmodes, seed):
    n, S = 16, Lx * Ly
    g = gen(seed)
    Dd, Dm = _stencil_operator(g, S, n, dtype)
    D0inv = torch.linalg.inv(Dm[:, 0])
    inv = torch.empty((S, n, n), dtype=CT[dtype], device="cuda")
    call("mg2d_block_inverse", P_(inv), P_(Dd), n, S, dtype, S_())
    tol = TOL if dtype == C128 else TOL32
    assert rel(inv.transpose(-1, -2), D0inv) < tol
    M = torch.empty((S, 4, n, n), dtype=CT[dtype], device="cuda")
    call("mg2d_premultiply", P_(M), P_(Dd), P_(inv), n, S, dtype, S_())
    assert rel(M.transpose(-1, -2), -torch.einsum("sij,skjl->skil", D0inv, Dm[:, 1:])) < tol
    if S > sms() * 16:
        assert_capped(S, sms() * 16, "premultiply_kernel")
    Dg, D0i = Dm.reshape(Ly, Lx, 5, n, n), D0inv.reshape(Ly, Lx, n, n)
    for nv in nvs:
        for cmode in cmodes:
            phi0 = rounded(crandn(g, nv, S, n), dtype)
            r = rounded(crandn(g, nv, S, n), dtype) if cmode else None
            c_ref = None if r is None else torch.einsum("sij,vsj->vsi", D0inv, r).contiguous()
            if strip:
                lo, hi = rounded(crandn(g, nv, Lx, n), dtype), rounded(crandn(g, nv, Lx, n), dtype)
            outs = []
            for rep in range(2):
                phi = phi0.to(CT[dtype], copy=True)
                cbuf = torch.zeros_like(phi) if cmode != 2 else c_ref.to(CT[dtype], copy=True)
                if strip:
                    lod, hid = lo.to(CT[dtype]), hi.to(CT[dtype])
                    lop, hip, hs = P_(lod), P_(hid), Lx * n
                else:
                    lop, hip, hs = P_(phi) + (Ly - 1) * Lx * n * phi.element_size(), P_(phi), S * n
                rk = r.to(CT[dtype]) if r is not None else None
                for colour in (0, 1):
                    call("mg2d_relax_rb_pm", P_(phi), lop, hip, P_(M), P_(inv), P_(rk), P_(cbuf), cmode, n, Lx, Ly, colour, yoff,
                         dtype, nv, S * n, hs, None, S_())
                outs.append((phi, cbuf))
            assert torch.equal(outs[0][0], outs[1][0]), (nv, cmode)
            want = phi0.reshape(nv, Ly, Lx, n)
            rr = None if r is None else r.reshape(nv, Ly, Lx, n)
            for colour in (0, 1):
                h = (lo.reshape(nv, 1, Lx, n), hi.reshape(nv, 1, Lx, n)) if strip else _periodic_halos(want)
                want = rb_half(want, hop_dense(Dg, neighbours(want, *h)), D0i, rr, colour, yoff)
            assert rel(outs[0][0], want) < tol, (Lx, Ly, dtype, nv, cmode)
            if cmode == 1:
                assert rel(outs[0][1], c_ref) < tol


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_premultiplied_sweep_level2_256(dtype, gpu_mem):
    """mg2d_block_inverse, mg2d_premultiply (capped grid) and mg2d_relax_rb_pm at 256^2, 16 dof: NV 1 and 4, cmode 0/1/2."""
    _pm_case(256, 256, dtype, False, 0, (1, 4), (0, 1, 2), 5)


@pytest.mark.gpu
@pytest.mark.parametrize("Lx,Ly,yoff", [(256, 32, 1), (64, 32, 0)])
@pytest.mark.parametrize("dtype", [C128, C64])
def test_premultiplied_sweep_strips(Lx, Ly, yoff, dtype, gpu_mem):
    """Levels 2 and 3 of the 8-rank plan: explicit halo rows, NV = 4 with hstride = L*n (and NV = 1)."""
    _pm_case(Lx, Ly, dtype, True, yoff, (4, 1), (0, 1, 2), 6)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [64, 16])
@pytest.mark.parametrize("dtype", [C128, C64])
def test_persistent_sweeps_small_levels(L, dtype, gpu_mem):
    """mg2d_relax_rb_pm_sweeps (all sweeps of a relax call in one cooperative launch) at the bench's levels 3 and 4."""
    n, S, nsw = 16, L * L, 3
    g = gen(7 + L)
    Dd, Dm = _stencil_operator(g, S, n, dtype)
    D0inv = torch.linalg.inv(Dm[:, 0])
    inv = D0inv.transpose(-1, -2).to(CT[dtype]).contiguous()
    M = torch.empty((S, 4, n, n), dtype=CT[dtype], device="cuda")
    call("mg2d_premultiply", P_(M), P_(Dd), P_(inv), n, S, dtype, S_())
    tol = TOL if dtype == C128 else TOL32
    Dg, D0i = Dm.reshape(L, L, 5, n, n), D0inv.reshape(L, L, n, n)
    for with_r in (True, False):
        phi0 = rounded(crandn(g, S, n), dtype)
        r = rounded(crandn(g, S, n), dtype) if with_r else None
        outs = []
        for rep in range(2):
            phi = phi0.to(CT[dtype], copy=True)
            cbuf = torch.zeros_like(phi)
            call("mg2d_relax_rb_pm_sweeps", P_(phi), P_(M), P_(inv), P_(None if r is None else r.to(CT[dtype])), P_(cbuf), n, L,
                 nsw, dtype, S_())
            outs.append(phi)
        assert torch.equal(outs[0], outs[1])
        want = phi0.reshape(L, L, n)
        rr = None if r is None else r.reshape(L, L, n)
        for _ in range(nsw):
            for colour in (0, 1):
                want = rb_half(want, hop_dense(Dg, neighbours(want, *_periodic_halos(want))), D0i, rr, colour, 0)
        assert rel(outs[0], want) < tol, (L, dtype, with_r)


def _half_rounded(t32):
    """what mg2d_to_half stores: each fp32 component rounded to nearest fp16"""
    return torch.view_as_complex(torch.view_as_real(t32).to(torch.float16).to(torch.float64).contiguous())


@pytest.mark.gpu
@pytest.mark.parametrize("Lx,Ly,strip", [(256, 256, False), (64, 64, False), (16, 16, False), (256, 32, True)])
def test_half_precision_sweep(Lx, Ly, strip, gpu_mem):
    """mg2d_to_half + mg2d_relax_rb_half (16 dof) against the fp64 sweep with the half-rounded blocks."""
    n, S = 16, Lx * Ly
    g = gen(8 + Lx + Ly)
    D32, Dm = _stencil_operator(g, S, n, C64)
    inv32 = torch.linalg.inv(Dm[:, 0]).transpose(-1, -2).to(torch.complex64).contiguous()
    Dh = torch.empty(D32.shape, dtype=torch.float32, device="cuda")
    invh = torch.empty(inv32.shape, dtype=torch.float32, device="cuda")
    call("mg2d_to_half", P_(Dh), P_(D32), D32.numel(), S_())
    call("mg2d_to_half", P_(invh), P_(inv32), inv32.numel(), S_())
    assert torch.equal(Dh.view(torch.float16).reshape(-1), torch.view_as_real(D32).to(torch.float16).reshape(-1))
    Dg = _half_rounded(D32).transpose(-1, -2).reshape(Ly, Lx, 5, n, n)
    Ig = _half_rounded(inv32).transpose(-1, -2).reshape(Ly, Lx, n, n)
    for with_r in (True, False):
        for yoff in ((0, 1) if strip else (0,)):
            phi0 = rounded(crandn(g, S, n), C64)
            r = rounded(crandn(g, S, n), C64) if with_r else None
            if strip:
                lo, hi = rounded(crandn(g, Lx, n), C64), rounded(crandn(g, Lx, n), C64)
            outs = []
            for rep in range(2):
                phi = phi0.to(torch.complex64, copy=True)
                if strip:
                    lod, hid = lo.to(torch.complex64), hi.to(torch.complex64)
                    lop, hip = P_(lod), P_(hid)
                else:
                    lop, hip = P_(phi) + (Ly - 1) * Lx * n * 8, P_(phi)
                for colour in (0, 1):
                    call("mg2d_relax_rb_half", P_(phi), lop, hip, P_(Dh), P_(invh), P_(None if r is None else r.to(torch.complex64)),
                         n, Lx, Ly, colour, yoff, S_())
                outs.append(phi)
            assert torch.equal(outs[0], outs[1])
            want = phi0.reshape(Ly, Lx, n)
            rr = None if r is None else r.reshape(Ly, Lx, n)
            for colour in (0, 1):
                h = (lo.reshape(1, Lx, n), hi.reshape(1, Lx, n)) if strip else _periodic_halos(want)
                want = rb_half(want, hop_dense(Dg, neighbours(want, *h)), Ig, rr, colour, yoff)
            assert rel(outs[0], want) < TOL32, (Lx, Ly, with_r, yoff)


# ---- restriction / prolongation ----------------------------------------------------------------------------------
def _transfer_case(Lf, blk, nf, nc, dtype, chiral, quads, seed):
    Lc = Lf // blk
    Sf, Sc = Lf * Lf, Lc * Lc
    g = gen(seed)
    Pw = rounded(crandn(g, Sf, nc, nf // 2 if chiral else nf), dtype)
    Pk = Pw.to(CT[dtype])
    vf0 = rounded(crandn(g, Sf, nf), dtype)
    vc0 = rounded(crandn(g, Sc, nc), dtype)
    tol = TOL if dtype == C128 else TOL32
    R, Pr = (restrict_chiral, prolong_chiral) if chiral else (restrict, prolong)
    for quad in quads:
        own = owner(Lf, Lf, blk, quad, "cuda")
        outs = []
        for rep in range(2):
            vc = torch.empty((Sc, nc), dtype=CT[dtype], device="cuda")
            call("mg2d_restrict_chiral" if chiral else "mg2d_restrict", P_(vc), P_(vf0.to(CT[dtype])), P_(Pk), nf, nc, Lf, Lf, blk,
                 quad, dtype, S_())
            outs.append(vc)
        assert torch.equal(outs[0], outs[1])
        assert rel(outs[0], R(vf0, Pw, own, blk)) < tol, ("restrict", Lf, nf, nc, quad)
        del outs
        for accumulate in ((1, 0) if chiral else (1,)):
            for zero_vc in (0, 1):
                vf = vf0.to(CT[dtype], copy=True)
                vc = vc0.to(CT[dtype], copy=True)
                if chiral:
                    call("mg2d_prolong_chiral", P_(vf), P_(vc), P_(Pk), nf, nc, Lf, Lf, blk, quad, zero_vc, accumulate, dtype, S_())
                else:
                    call("mg2d_prolong_add", P_(vf), P_(vc), P_(Pk), nf, nc, Lf, Lf, blk, quad, zero_vc, dtype, S_())
                assert rel(vf, Pr(vf0, vc0, Pw, own, accumulate=bool(accumulate))) < tol, ("prolong", Lf, quad, accumulate)
                if zero_vc:
                    assert float(vc.abs().max()) == 0.0
                else:
                    assert torch.equal(vc, vc0.to(CT[dtype]))
                del vf, vc


@pytest.mark.gpu
def test_transfer_level0_4096(gpu_mem):
    """restrict_chiral_nf2_nc16_blk4 / prolong_chiral_nf2_blk4<16> at 4096^2 -> 1024^2: quads 1..4, accumulate, zero_vc."""
    nagg = 1024 * 1024
    assert_capped(-(-nagg // 16), sms() * 32, "restrict_chiral_nf2_nc16_blk4_kernel")
    assert_capped(-(-nagg // 8), sms() * 32, "prolong_chiral_nf2_blk4_kernel (blocks)")
    _transfer_case(4096, 4, 2, 16, C128, True, (1, 2, 3, 4), 9)


@pytest.mark.gpu
def test_transfer_level0_4096_complex64(gpu_mem):
    _transfer_case(4096, 4, 2, 16, C64, True, (1, 3), 10)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_transfer_level1_1024(dtype, gpu_mem):
    """restrict/prolong_chiral<16,16> (and the dense mg2d_restrict / mg2d_prolong_add) at 1024^2 -> 256^2."""
    nsteps = -(-(256 * 256) // 8)
    assert_capped(nsteps, min(nsteps, sms() * 32), "restrict/prolong_chiral_kernel<16,16>")
    _transfer_case(1024, 4, 16, 16, dtype, True, (1, 2, 3, 4) if dtype == C128 else (2,), 11)
    _transfer_case(1024, 4, 16, 16, dtype, False, (1, 4), 12)


# ---- level 0 Wilson operator -----------------------------------------------------------------------------------------
def _links(g, Ly, Lx, dtype=C128):
    th = torch.rand((Ly, Lx, 2), dtype=torch.float64, device="cuda", generator=g) * (2 * math.pi)
    return rounded(torch.polar(torch.ones_like(th), th), dtype)


def _wilson_case(Lx, Ly, dtype, strip, yoff, seed):
    m = -0.05
    S = Lx * Ly
    g = gen(seed)
    U = _links(g, Ly, Lx, dtype).reshape(S, 2)
    phi, r = rounded(crandn(g, S, 2), dtype), rounded(crandn(g, S, 2), dtype)
    Ug, pg, rg = U.reshape(Ly, Lx, 2), phi.reshape(Ly, Lx, 2), r.reshape(Ly, Lx, 2)
    if strip:
        lo2, hi2 = rounded(crandn(g, 2, Lx, 2), dtype), rounded(crandn(g, 2, Lx, 2), dtype)
        U_lo2, U_hi = _links(g, 2, Lx, dtype), _links(g, 1, Lx, dtype)
        r_lo, r_hi = rounded(crandn(g, 1, Lx, 2), dtype), rounded(crandn(g, 1, Lx, 2), dtype)
    else:
        lo2, hi2, U_lo2, U_hi, r_lo, r_hi = pg[-2:], pg[:2], Ug[-2:], Ug[:1], rg[-1:], rg[:1]
    k = lambda t: t.to(CT[dtype]).contiguous()
    Uk, pk, rk = k(U), k(phi), k(r)
    lo2k, hi2k, Ulo2k, Uhik, rlok, rhik = k(lo2), k(hi2), k(U_lo2), k(U_hi), k(r_lo), k(r_hi)
    tol = TOL if dtype == C128 else TOL32
    # apply, and residual with the fused dots
    want = wilson_hop(pg, lo2, hi2, Ug, U_lo2) + (2.0 + m) * pg
    out = torch.empty_like(pk)
    call("mg2d_wilson_apply", P_(out), P_(pk), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), None, m, Lx, Ly, 0, dtype, None, S_())
    assert rel(out, want) < tol
    res = rg - want
    dd = []
    for rep in range(2):
        d = torch.zeros(4, dtype=torch.float64, device="cuda")
        call("mg2d_wilson_apply", P_(out), P_(pk), P_(lo2k[1:]), P_(hi2k), P_(Uk), P_(Ulo2k[1:]), P_(rk), m, Lx, Ly, 1, dtype, P_(d), S_())
        dd.append(d)
    assert torch.equal(dd[0], dd[1])
    assert rel(out, res) < tol
    out64 = out.to(torch.complex128)
    d = dd[0].cpu().numpy()
    dref = (float((out64.abs() ** 2).sum()), complex(torch.vdot(out64.reshape(-1), phi.reshape(-1))), float((r.abs() ** 2).sum()))
    assert abs(d[0] / dref[0] - 1) < TOL and abs(d[3] / dref[2] - 1) < TOL
    assert abs(complex(d[1], d[2]) - dref[1]) < TOL * math.sqrt(dref[0] * float((phi.abs() ** 2).sum()))
    del out, out64, res, want
    # the one-pass two-colour sweep, with and without r
    for with_r in (True, False):
        outs = []
        for rep in range(2):
            o = torch.empty_like(pk)
            call("mg2d_wilson_relax_rb2", P_(o), P_(pk), P_(lo2k), P_(hi2k), P_(Uk), P_(Ulo2k), P_(Uhik),
                 P_(rk if with_r else None), P_(rlok if with_r else None), P_(rhik if with_r else None), m, Lx, Ly, yoff, dtype, None, S_())
            outs.append(o)
        assert torch.equal(outs[0], outs[1])
        want = wilson_rb2(pg, lo2, hi2, Ug, U_lo2, U_hi, rg if with_r else None, r_lo, r_hi, m, yoff)
        assert rel(outs[0], want) < tol, (Lx, Ly, dtype, with_r)
        del outs, want


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_wilson_level0_4096(dtype, gpu_mem):
    """mg2d_wilson_apply (apply; residual + dots) and mg2d_wilson_relax_rb2 (row chunks of 128) on the 4096^2 lattice."""
    _wilson_case(4096, 4096, dtype, False, 0, 13)


@pytest.mark.gpu
@pytest.mark.parametrize("Ly,yoff", [(512, 1), (2048, 0)])
def test_wilson_level0_strips(Ly, yoff, gpu_mem):
    """Level-0 strips of the 8- and 2-rank plans with explicit two-row halos of phi and links and one-row halos of r."""
    _wilson_case(4096, Ly, C128, True, yoff, 14 + Ly)
    if Ly == 512:
        _wilson_case(4096, Ly, C64, True, yoff, 15)


# ---- outer FGCR vector kernels ------------------------------------------------------------------------------------------
def _grid_blas(n, U):
    nb = -(-n // (256 * U))
    return min(nb, sms() * 8, 4096) * 256 * U          # elements per outer pass (stream_grid in blas.cu)


_DOTS_U = {1: 4, 2: 4, 3: 2, 4: 2, 5: 2, 6: 1, 7: 1, 8: 1}
_ORTHO_W_U = {0: 4, 1: 4, 2: 2, 3: 2, 4: 2, 5: 1, 6: 1, 7: 1, 8: 1}


def _cplx(d, k):
    return complex(d[2 * k], d[2 * k + 1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
def test_gcr_kernels_4096(dtype, gpu_mem):
    """mg2d_gcr_dots / gcr_ortho (with and without z) / gcr_step / gcr_step_lazy / gcr_xupdate / norm2 / cdot_batch on the
    level-0 vectors of the benchmark (2 * 4096^2 elements), every nj, one stored direction with |W_j|^2 = 0."""
    N = 2 * 4096 * 4096
    for U in sorted(set(_DOTS_U.values()) | set(_ORTHO_W_U.values())):
        assert_capped(N, _grid_blas(N, U), f"FGCR kernels, {U} elements per thread and pass")
    g = gen(16)
    ct = CT[dtype]
    tol = TOL if dtype == C128 else TOL32
    W64 = rounded(crandn(g, 8, N), dtype)
    Z64 = rounded(crandn(g, 8, N), dtype)
    W, Z = W64.to(ct), Z64.to(ct)
    w64, r64 = rounded(crandn(g, N), dtype), rounded(crandn(g, N), dtype)
    wk, rk = w64.to(ct), r64.to(ct)
    wn2_h = np.abs(np.random.default_rng(1).normal(size=8)) * N + 1.0
    wn2_h[3] = 0.0                                                    # the d > 0 guards
    wn2 = torch.tensor(wn2_h, dtype=torch.float64, device="cuda")

    def dev(x):
        return torch.tensor(np.asarray(x, dtype=np.float64), device="cuda")

    # norm2, cdot_batch (1 and 64 pairs): inputs exact in both precisions, sums in fp64
    outs = []
    for rep in range(2):
        o = torch.zeros(2 + 2 * 64, dtype=torch.float64, device="cuda")
        call("mg2d_norm2", P_(wk), N, dtype, P_(o), S_())
        call("mg2d_cdot_batch", P_(W), N, 8, P_(Z), N, 8, N, dtype, P_(o[2:]), S_())
        outs.append(o)
    assert torch.equal(outs[0], outs[1])
    o = outs[0].cpu().numpy()
    assert abs(o[0] / float((w64.abs() ** 2).sum()) - 1) < TOL
    gram = (W64.conj() @ Z64.T).cpu().numpy()
    got = (o[2:2 + 128:2] + 1j * o[3:2 + 128:2])[:64].reshape(8, 8)
    assert np.max(np.abs(got - gram)) < TOL * np.max(np.abs(gram))
    o1 = torch.zeros(2, dtype=torch.float64, device="cuda")
    call("mg2d_cdot_batch", P_(wk), N, 1, P_(rk), N, 1, N, dtype, P_(o1), S_())
    want = complex(torch.vdot(w64, r64))
    assert abs(_cplx(o1.cpu().numpy(), 0) - want) < TOL * abs(want)
    # projections <W_j, w>
    proj = (W64.conj() @ w64).cpu().numpy()
    for nj in range(1, 9):
        outs = []
        for rep in range(2):
            o = torch.zeros(16, dtype=torch.float64, device="cuda")
            call("mg2d_gcr_dots", P_(W), N, nj, P_(wk), N, dtype, P_(o), S_())
            outs.append(o)
        assert torch.equal(outs[0], outs[1]), nj
        got = np.array([_cplx(outs[0].cpu().numpy(), j) for j in range(nj)])
        assert np.max(np.abs(got - proj[:nj])) < TOL * np.max(np.abs(proj)), nj
    # orthogonalisation: dots_j random (the kernel takes them as given), beta_j = -dots_j / |W_j|^2
    rng = np.random.default_rng(2)
    dots_h = (rng.normal(size=8) + 1j * rng.normal(size=8)) * N
    dots = dev(np.stack([dots_h.real, dots_h.imag], -1).reshape(-1))
    beta = np.where(wn2_h > 0, -dots_h / np.where(wn2_h > 0, wn2_h, 1.0), 0.0)
    z64 = rounded(crandn(g, N), dtype)
    for with_z in (True, False):
        for nj in range(0, 9):
            bt = torch.tensor(beta[:nj], dtype=torch.complex128, device="cuda")
            w_ref = w64 + (bt @ W64[:nj] if nj else 0)
            z_ref = z64 + (bt @ Z64[:nj] if nj else 0)
            red_ref = (float((w_ref.abs() ** 2).sum()), complex(torch.vdot(w_ref, r64)))
            res = []
            for rep in range(2):
                w, z = wk.clone(), z64.to(ct, copy=True)
                o = torch.zeros(4, dtype=torch.float64, device="cuda")
                call("mg2d_gcr_ortho", P_(w), P_(z) if with_z else None, P_(rk), P_(W), P_(Z) if with_z else None, N, nj, P_(dots),
                     P_(wn2), N, dtype, P_(o), S_())
                res.append((w, z, o))
            assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][2], res[1][2]), (with_z, nj)
            w, z, o = res[0]
            assert rel(w, w_ref) < tol, (with_z, nj)
            if with_z:
                assert rel(z, z_ref) < tol, nj
            else:
                assert torch.equal(z, z64.to(ct))
            o = o.cpu().numpy()
            assert abs(o[0] / red_ref[0] - 1) < tol, (with_z, nj)
            assert abs(complex(o[1], o[2]) - red_ref[1]) < tol * math.sqrt(red_ref[0] * float((r64.abs() ** 2).sum()))
            del res, w, z, w_ref, z_ref
    # step: x += a z, r -= a w, |r|^2, |w|^2 -> slot
    x64 = rounded(crandn(g, N), dtype)
    wr_h = np.array([float(N), 0.3 * N, -0.7 * N])
    a = complex(wr_h[1], wr_h[2]) / wr_h[0]
    x_ref, r_ref = x64 + a * z64, r64 - a * w64
    res = []
    for rep in range(2):
        x, r = x64.to(ct, copy=True), rk.clone()
        o = torch.zeros(1, dtype=torch.float64, device="cuda")
        slot = torch.zeros(1, dtype=torch.float64, device="cuda")
        call("mg2d_gcr_step", P_(x), P_(r), P_(z64.to(ct)), P_(wk), P_(dev(wr_h)), P_(slot), N, dtype, P_(o), S_())
        res.append((x, r, o, slot))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][2], res[1][2])
    x, r, o, slot = res[0]
    assert rel(x, x_ref) < tol and rel(r, r_ref) < tol
    assert abs(float(o.item()) / float((r.to(torch.complex128).abs() ** 2).sum()) - 1) < TOL
    assert abs(float(o.item()) / float((r_ref.abs() ** 2).sum()) - 1) < tol
    assert float(slot.item()) == wr_h[0]
    del res, x, r, x_ref, r_ref
    # lazy step over a whole restart cycle (nj = 0..7), x updated once from the accumulated g (every nj)
    coef = torch.zeros(144, dtype=torch.float64, device="cuda")
    bs, as_ = [], []
    r = rk.clone()
    r_ref = r64.clone()
    wn2_slot = torch.zeros(8, dtype=torch.float64, device="cuda")
    for nj in range(8):
        wr_j = np.array([0.0 if nj == 5 else (1.0 + nj) * N, rng.normal() * N, rng.normal() * N])   # a = 0 guard at nj = 5
        a_j = complex(wr_j[1], wr_j[2]) / wr_j[0] if wr_j[0] > 0 else 0.0
        wj = W[nj]
        o = torch.zeros(1, dtype=torch.float64, device="cuda")
        call("mg2d_gcr_step_lazy", P_(r), P_(wj), P_(dev(wr_j)), P_(wn2_slot[nj:]), P_(dots), P_(wn2), nj, P_(coef), N, dtype, P_(o), S_())
        r_ref = r_ref - a_j * W64[nj]
        bs.append(np.array([dots_h[i] / wn2_h[i] if wn2_h[i] > 0 else 0.0 for i in range(nj)]))
        as_.append(a_j)
        C, gv = lazy_coefficients(bs, as_)
        ch = coef.cpu().numpy()
        got_C = (ch[0:128:2] + 1j * ch[1:128:2]).reshape(8, 8)
        got_g = ch[128:144:2] + 1j * ch[129:144:2]
        assert np.max(np.abs(got_C[:, :nj + 1] - C[:, :nj + 1])) < TOL * np.max(np.abs(C)), nj
        assert np.max(np.abs(got_g - gv)) < TOL * np.max(np.abs(gv)), nj
        assert rel(r, r_ref) < tol, nj
        assert abs(float(o.item()) / float((r_ref.abs() ** 2).sum()) - 1) < tol, nj
        assert float(wn2_slot[nj].item()) == wr_j[0]
        gd = torch.tensor(gv[:nj + 1], dtype=torch.complex128, device="cuda")
        x_ref = x64 + gd @ Z64[:nj + 1]
        xs = []
        for rep in range(2):
            x = x64.to(ct, copy=True)
            call("mg2d_gcr_xupdate", P_(x), P_(Z), N, nj + 1, P_(coef), N, dtype, S_())
            xs.append(x)
        assert torch.equal(xs[0], xs[1])
        assert rel(xs[0], x_ref) < tol, nj
        del xs, x_ref
