"""The strip-halo code of the multi-GPU benchmark at its strip shapes, on one GPU.

On 2, 4 and 8 GPUs every level of the benchmark down to MIN_ROWS rows per rank is a strip of rows, and the smoothers move
halo rows between ranks themselves: after one standalone exchange (mg2d_halo_exchange) each red-black launch of a relax
call reads its neighbours' boundary rows from halo buffer set A or B, pushes the boundary rows it produces into the other
set, and its last boundary warp / CTA publishes epoch + 1 while the interior still runs (Comm.fused_link, Level.relax).
Reductions are summed over the ranks by the last CTA of the producing kernel (mg2d_comm_reduce) through a two-parity
mailbox.  `Comm.single` makes the rank its own strip neighbour, so all of this runs on one GPU, and an Lx x Ly strip is
then the periodic Lx x Ly torus: a linked sweep must equal the unlinked kernel given explicit wrap-around halo rows BIT
FOR BIT (same arithmetic, only the source of the halo rows differs), an exchange must return the strip's own last / first
rows, and a reduction summed over one rank must equal the plain one (0.0 + x).

Every case asserts, from the launcher's own formula and the device's SM count, the regime it reaches and prints it.
One shape per sweep kernel is also held to the fp64 torch restatement of the sweep (test_gpu_bench_shapes), relative in
the max-norm: 1e-12 in complex128, 2e-5 against the fp64 reference of the rounded inputs in complex64.

Not covered: the ntail = 2 branch of wilson_rb2_kernel (a last row chunk of one row) needs an odd Ly, which no strip plan
produces; two ranks on two GPUs are test_gpu_dist.py's.
"""
import ctypes
import importlib
import importlib.util
import os
import sys

import pytest
import torch

import mg2d
from test_clover import links, self_ref
from test_gpu_bench_shapes import (C64, C128, CT, TOL, TOL32, P_, S_, _periodic_halos, assert_capped, call, crandn, ctx, gen,
                                   gpu_mem, hop_dense, hop_lowrank, neighbours, rb_half, rounded, rel, sms)
from test_twisted_mass import rb2_tm, twist

dmod = importlib.import_module("2d_multigrid_b200.dist")
mgmod = importlib.import_module("2d_multigrid_b200.mg")

# Lx x Ly per rank of levels 0..3 of the 4096^2 benchmark (None: replicated on every rank), from dist.plan_strips
SHAPES = {
    2: [(4096, 2048), (1024, 512), (256, 128), (64, 32)],
    4: [(4096, 1024), (1024, 256), (256, 64), None],
    8: [(4096, 512), (1024, 128), (256, 32), None],
}
POST = [4, 2, 6, 4]              # the benchmark's post-smoothing sweeps on levels 0..3 (bench.post_sweeps)
MASS, MU = -0.05, 0.0173
RB2_W, RB2_WARPS = 62, 4         # csrc/wilson_rb2.cu: stored columns per warp tile, warps per CTA
ST_GPB = 8                       # csrc/stencil.cu: 16-dof sites per 256-thread CTA (one warp each)
HX_WORDS = 4096                  # mg2d_halo_exchange: more 16-byte words than this -> 8 CTAs
L0_SHAPES = sorted({s[0] for s in SHAPES.values()}, reverse=True)
L1_SHAPES = sorted({s[1] for s in SHAPES.values()}, reverse=True)
L23_SHAPES = sorted({s[k] for s in SHAPES.values() for k in (2, 3) if s[k] is not None}, reverse=True)


def _bench(monkeypatch):
    """bench.py as a module (loading it prepends the repository to sys.path and turns off bytecode writing: undone later)"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    monkeypatch.setattr(sys, "path", list(sys.path))
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


# ================================================================================================================
# CPU: the shapes are the benchmark's
# ================================================================================================================
def test_shapes_are_the_benchmarks_strip_plan(monkeypatch):
    """SHAPES and POST are what bench.py's workload and dist.plan_strips give on 2, 4 and 8 ranks: a change of the cycle or
    of MIN_ROWS fails here instead of leaving the GPU tests on stale shapes."""
    bench = _bench(monkeypatch)
    p = bench.workload_params(mg2d, 4096, MASS)
    assert p.size == [4096, 1024, 256, 64, 16] and p.n_dof[1:] == [16] * 4 and p.blocks == [4] * 4
    assert p.post[:4] == POST and p.pre == [0] * 5 and p.smoother == "rbgs" and p.matrix_free
    for world, want in SHAPES.items():
        plan = dmod.plan_strips(p, world)
        got = [(L, rows) if d else None for L, (d, rows) in zip(p.size, plan)]
        assert got[:4] == want and got[4] is None, (world, got)
    assert all(Lx % RB2_W for Lx, _ in L0_SHAPES)     # the last rb2 tile of every level-0 strip is partial


# ================================================================================================================
# GPU fixtures and helpers
# ================================================================================================================
@pytest.fixture(scope="module")
def comm():
    """One rank that is its own strip neighbour: IPC slab, halo slots, A/B buffers and the reduction mailbox on this GPU."""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device (sm_100a)")
    if not dmod.FUSED:
        pytest.skip("MG2D_FUSED=0: the smoothers do not push their halo rows, the linked paths are not what runs")
    if dmod.LINK_DEBUG:
        pytest.skip(f"MG2D_LINK_DEBUG={dmod.LINK_DEBUG}: the linked kernels neither push nor wait as in production")
    c = dmod.Comm.single(ctx(), torch.device("cuda", 0), slab_bytes=256 << 20)
    assert c.fused and c.xdesc is not None
    yield c
    call("mg2d_comm_reduce", 0)


def _healthy(comm):
    assert comm.p2p_errors() == 0
    m = ctypes.c_longlong(-1)
    call("mg2d_comm_error", comm.xdesc, ctypes.byref(m))
    assert m.value == 0


def _rb2_regime(Lx, Ly):
    """launch_rb2 (csrc/wilson_rb2.cu) and the linked item order of wilson_rb2_kernel"""
    ntx = -(-Lx // RB2_W)
    RY = 128
    while RY > 8 and ntx * -(-Ly // RY) < sms() * 12:
        RY >>= 1
    nchunks = -(-Ly // RY)
    nitems = ntx * nchunks
    wstride = min(-(-nitems // RB2_WARPS), sms() * 4) * RB2_WARPS
    ntail = (1 if nchunks >= 2 else 0) + (1 if nchunks >= 3 and (nchunks - 1) * RY + 2 > Ly else 0)
    nbi = ntx * (1 + ntail)
    return dict(RY=RY, nitems=nitems, wstride=wstride, ntail=ntail, nbi=nbi, bctas=-(-min(nbi, wstride) // RB2_WARPS),
                last_tile=Lx - (ntx - 1) * RB2_W)


def _stencil_regime(Lx, Ly):
    """launch_rb_pm / launch_rb_lr (16 dof, NV = nvec for nvec in {1, 4}): steps of 8 sites, grid capped at 32 CTAs per SM;
    the two boundary rows are the first 2 * Lx/2 sites"""
    nsteps = -(-(Lx // 2) * Ly // ST_GPB)
    gx = min(nsteps, sms() * 32)
    return dict(nsteps=nsteps, grid=gx, per_cta=-(-nsteps // gx), bctas=min(-(-Lx // ST_GPB), gx))


# ---- level 0: the two-colour Wilson sweep --------------------------------------------------------------------------
class _Wilson:
    """Seeded level-0 inputs of one strip: links, clover field, phi, r (rounded to the kernel's precision)."""

    def __init__(self, Lx, Ly, dtype, seed):
        g = gen(seed)
        self.Lx, self.Ly, self.dtype = Lx, Ly, dtype
        rt = torch.float64 if dtype == C128 else torch.float32
        self.Ug = links(g, Ly, Lx, dtype)
        self.Fg = (torch.randn((Ly, Lx), dtype=torch.float64, device="cuda", generator=g) * 0.3).to(rt).double()
        self.pg = rounded(crandn(g, Ly, Lx, 2), dtype)
        self.rg = rounded(crandn(g, Ly, Lx, 2), dtype)
        k = lambda t: t.to(CT[dtype]).reshape(Lx * Ly, -1).contiguous()
        self.U, self.phi0, self.r = k(self.Ug), k(self.pg), k(self.rg)
        self.F = self.Fg.to(rt).reshape(-1).contiguous()

    def relax(self, comm, variant, with_r, nsweeps, linked, phi=None):
        """Level.relax's two-colour branch on this strip: out-of-place ping-pong, an even sweep count ends in phi.  Linked:
        one standalone depth-2 exchange, then fused_link phase k for launch k (pushing except in the last); unlinked: the
        periodic wrap rows of the current input as explicit halos.  Link rows and the clover field are the periodic wrap."""
        Lx, Ly, dt = self.Lx, self.Ly, self.dtype
        phi = self.phi0.clone() if phi is None else phi
        tmp = torch.empty_like(phi)
        row = Lx * 2 * phi.element_size()
        U_lo2, U_hi = P_(self.U) + (Ly - 2) * row, P_(self.U)
        F_lo, F_hi = P_(self.F) + (Ly - 1) * Lx * self.F.element_size(), P_(self.F)
        r = self.r if with_r else None
        if r is None:
            r_lo = r_hi = None
        elif linked:
            lo, hi = comm.exchange_rows(r, Lx, Ly, 2, 1, key=("rb2 r",), depth=1)
            r_lo, r_hi = lo.data_ptr(), hi.data_ptr()
        else:
            r_lo, r_hi = P_(r) + (Ly - 1) * row, P_(r)
        cur, nxt = phi, tmp
        for it in range(nsweeps):
            link = None
            if linked:
                if it == 0:
                    comm.exchange_rows(cur, Lx, Ly, 2, 1, key=("rb2",), depth=2)
                lk, lo2, hi2 = comm.fused_link(cur, Lx, Ly, 2, 1, ("rb2",), 2, it, push=(it < nsweeps - 1))
                link = ctypes.byref(lk)
            else:
                lo2, hi2 = P_(cur) + (Ly - 2) * row, P_(cur)
            if variant == "tm":
                call("mg2d_wilson_tm_relax_rb2", P_(nxt), P_(cur), lo2, hi2, P_(self.U), U_lo2, U_hi, None, None, None, P_(r), r_lo,
                     r_hi, MASS, MU, Lx, Ly, 0, dt, link, S_())
            elif variant == "sw":
                call("mg2d_wilson_sw_relax_rb2", P_(nxt), P_(cur), lo2, hi2, P_(self.U), U_lo2, U_hi, P_(self.F), F_lo, F_hi, P_(r),
                     r_lo, r_hi, MASS, Lx, Ly, 0, dt, link, S_())
            else:
                call("mg2d_wilson_relax_rb2", P_(nxt), P_(cur), lo2, hi2, P_(self.U), U_lo2, U_hi, P_(r), r_lo, r_hi, MASS, Lx, Ly,
                     0, dt, link, S_())
            cur, nxt = nxt, cur
        assert nsweeps % 2 == 0 and cur is phi
        return phi

    def reference(self, variant, with_r, nsweeps):
        """nsweeps of the fp64 two-colour sweep on the periodic Lx x Ly torus"""
        F = self.Fg if variant == "sw" else torch.zeros_like(self.Fg)
        dgE = self_ref(torch.cat([F[-1:], F, F[:1]], dim=0), MASS) + twist(MU if variant == "tm" else 0.0, "cuda")
        Ug, rg = self.Ug, (self.rg if with_r else None)
        cur = self.pg
        for _ in range(nsweeps):
            cur = rb2_tm(cur, cur[-2:], cur[:2], Ug, Ug[-2:], Ug[:1], dgE, rg, None if rg is None else rg[-1:],
                         None if rg is None else rg[:1], 0)
        return cur


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("Lx,Ly", L0_SHAPES + [(4096, 400)])
def test_wilson_rb2_linked_equals_unlinked(Lx, Ly, dtype, comm, gpu_mem):
    """The level-0 post-smoothing (4 two-colour sweeps, halo sets A, B, A, B) of mg2d_wilson{,_sw,_tm}_relax_rb2 with the
    halo link equals the same sweeps with explicit periodic halos, with and without r.  4096 x 400 is not a strip of any
    plan: it is the shape where RY reaches its floor of 8 and warps loop over two items."""
    rg = _rb2_regime(Lx, Ly)
    print(f"\nwilson_rb2 {Lx}x{Ly}: RY {rg['RY']}, {rg['nitems']} items on {rg['wstride']} warps, {rg['nbi']} boundary items on "
          f"{rg['bctas']} CTAs, last tile {rg['last_tile']} of {RB2_W} columns")
    assert rg["ntail"] == 1 and rg["bctas"] >= 2 and rg["last_tile"] < RB2_W
    if (Lx, Ly) == (4096, 400):
        assert rg["RY"] == 8 and rg["nitems"] > rg["wstride"]
    else:
        assert rg["nitems"] <= rg["wstride"]
    w = _Wilson(Lx, Ly, dtype, 1000 + Ly + dtype)
    anchor = (Lx, Ly) == (4096, 512)
    for variant in ("plain", "sw", "tm"):
        for with_r in (True, False):
            got = w.relax(comm, variant, with_r, POST[0], linked=True)
            want = w.relax(comm, variant, with_r, POST[0], linked=False)
            _healthy(comm)
            assert torch.equal(got, want), (variant, with_r)
            assert not torch.equal(got, w.phi0) and bool(torch.isfinite(torch.view_as_real(got)).all())
            if anchor:
                err = rel(got, w.reference(variant, with_r, POST[0]))
                assert err < (TOL if dtype == C128 else TOL32), (variant, with_r, err)
            del got, want


# ---- coarse levels: pre-multiplied (levels 2, 3) and low-rank (level 1) half sweeps -----------------------------------------
class _Coarse:
    """Seeded 16-dof operator of one strip: D0^-1, and either hopping blocks D_k with M_k = -D0^-1 D_k (kind 'pm') or rank-4
    factors A, B of D_k = sum_b A_b B_b^dagger packed into F by mg2d_lowrank_pack (kind 'lr'); rounded to the kernel's precision."""
    n, R = 16, 4

    def __init__(self, kind, Lx, Ly, dtype, seed):
        n, S = self.n, Lx * Ly
        self.kind, self.Lx, self.Ly, self.dtype, self.g = kind, Lx, Ly, dtype, gen(seed)
        g = self.g
        eye = torch.eye(n, dtype=torch.complex128, device="cuda")
        self.D0inv = rounded(eye / 3.0 + crandn(g, S, n, n) * 0.02, dtype)                 # math layout
        Dk = self.D0inv.transpose(-1, -2).contiguous()                                     # device layout
        if kind == "pm":
            self.Dh = rounded(crandn(g, S, 4, n, n) * 0.05, dtype)                        # math layout, slots 1..4
            M = -torch.einsum("sij,skjl->skil", self.D0inv, self.Dh)
            self.Op = M.transpose(-1, -2).to(CT[dtype]).contiguous()
        else:
            Q = 4 * self.R
            self.A, self.B = rounded(crandn(g, S, Q, n) * 0.15, dtype), rounded(crandn(g, S, Q, n) * 0.15, dtype)
            F = torch.empty((S, 2, n * self.R // 8, 32), dtype=torch.complex128, device="cuda")
            call("mg2d_lowrank_pack", P_(F), P_(self.A), P_(self.B), P_(Dk), n, self.R, S, C128, S_())
            self.Op = F.to(CT[dtype])
            del F
        self.Dinv = Dk.to(CT[dtype])

    def fields(self, nvec, with_r):
        S, n = self.Lx * self.Ly, self.n
        phi0 = rounded(crandn(self.g, nvec, S, n), self.dtype).to(CT[self.dtype])
        r = rounded(crandn(self.g, nvec, S, n), self.dtype).to(CT[self.dtype]) if with_r else None
        return (phi0[0], None if r is None else r[0]) if nvec == 1 else (phi0, r)

    def relax(self, comm, phi0, r, nsweeps, linked):
        """Level.relax's rbgs branch for stored operators: cmode 0 without r, else 1 on the first sweep and 2 after; linked:
        one standalone exchange, then fused_link phase k = 2 * sweep + colour (depth 1, pushing except in the last launch)
        and halo stride L*n between the vectors of a batch; unlinked: the periodic wrap rows of phi, halo stride S*n."""
        Lx, Ly, n = self.Lx, self.Ly, self.n
        phi = phi0.clone()
        nvec = 1 if phi.dim() == 2 else phi.shape[0]
        vs = Lx * Ly * n
        cbuf = None if r is None else torch.zeros_like(phi)
        key = (self.kind, nvec)
        nk = 2 * nsweeps
        for it in range(nsweeps):
            cmode = 0 if r is None else (1 if it == 0 else 2)
            for colour in (0, 1):
                k = 2 * it + colour
                link = None
                if linked:
                    if k == 0:
                        comm.exchange_rows(phi, Lx, Ly, n, nvec, key=key, depth=1)
                    lk, lo, hi = comm.fused_link(phi, Lx, Ly, n, nvec, key, 1, k, push=(k < nk - 1))
                    link, hs = ctypes.byref(lk), (Lx * n if nvec > 1 else vs)
                else:
                    lo, hi, hs = P_(phi) + (Ly - 1) * Lx * n * phi.element_size(), P_(phi), vs
                if self.kind == "pm":
                    call("mg2d_relax_rb_pm", P_(phi), lo, hi, P_(self.Op), P_(self.Dinv), P_(r), P_(cbuf), cmode, n, Lx, Ly, colour,
                         0, self.dtype, nvec, vs, hs, link, S_())
                else:
                    call("mg2d_relax_rb_lr", P_(phi), lo, hi, P_(self.Op), P_(self.Dinv), P_(r), P_(cbuf), cmode, n, self.R, Lx, Ly,
                         colour, 0, self.dtype, nvec, vs, hs, link, S_())
        return phi

    def reference(self, phi0, r, nsweeps):
        """the fp64 sweeps on the periodic torus: phi <- -D0^-1 (hop(phi) - r) on one colour at a time"""
        Lx, Ly, n = self.Lx, self.Ly, self.n
        want = phi0.to(torch.complex128).reshape(-1, Ly, Lx, n)
        rr = None if r is None else r.to(torch.complex128).reshape(-1, Ly, Lx, n)
        D0i = self.D0inv.reshape(Ly, Lx, n, n)
        if self.kind == "pm":
            Dg = torch.cat([torch.zeros_like(self.Dh[:, :1]), self.Dh], dim=1).reshape(Ly, Lx, 5, n, n)
            hop = lambda f: hop_dense(Dg, neighbours(f, *_periodic_halos(f)))
        else:
            Ag, Bg = self.A.reshape(Ly, Lx, 4 * self.R, n), self.B.reshape(Ly, Lx, 4 * self.R, n)
            hop = lambda f: hop_lowrank(Ag, Bg, neighbours(f, *_periodic_halos(f)))
        for _ in range(nsweeps):
            for colour in (0, 1):
                want = rb_half(want, hop(want), D0i, rr, colour, 0)
        return want.reshape(phi0.shape)


def _coarse_case(comm, kind, Lx, Ly, dtype, nsweeps, anchor):
    st = _stencil_regime(Lx, Ly)
    print(f"\nrelax_rb_{kind} {Lx}x{Ly}: {st['nsteps']} steps on {st['grid']} CTAs ({st['per_cta']} per CTA), boundary rows on "
          f"{st['bctas']} CTAs, {nsweeps} sweeps")
    if st["nsteps"] > st["grid"]:
        assert_capped(st["nsteps"], st["grid"], f"stencil_rb_{kind}_kernel {Lx}x{Ly}")
    assert st["bctas"] >= 2
    c = _Coarse(kind, Lx, Ly, dtype, 2000 + Lx + Ly + dtype)
    for nvec in (1, 4):
        for with_r in (True, False):
            phi0, r = c.fields(nvec, with_r)
            got = c.relax(comm, phi0, r, nsweeps, linked=True)
            want = c.relax(comm, phi0, r, nsweeps, linked=False)
            _healthy(comm)
            assert torch.equal(got, want), (kind, Lx, Ly, nvec, with_r)
            assert not torch.equal(got, phi0) and bool(torch.isfinite(torch.view_as_real(got)).all())
            if anchor:
                err = rel(got, c.reference(phi0, r, nsweeps))
                assert err < (TOL if dtype == C128 else TOL32), (kind, nvec, with_r, err)
            del got, want


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("Lx,Ly", L1_SHAPES)
def test_lowrank_sweep_linked_equals_unlinked(Lx, Ly, dtype, comm, gpu_mem):
    """mg2d_relax_rb_lr (16 dof, rank 4) on the level-1 strips, the benchmark's 2 sweeps: nvec 1 and 4, cmode 0 / 1+2."""
    _coarse_case(comm, "lr", Lx, Ly, dtype, POST[1], anchor=(Ly == 128))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("Lx,Ly", L23_SHAPES)
def test_premultiplied_sweep_linked_equals_unlinked(Lx, Ly, dtype, comm, gpu_mem):
    """mg2d_relax_rb_pm (16 dof) on the level-2 and level-3 strips with the benchmark's sweeps there (6 and 4)."""
    _coarse_case(comm, "pm", Lx, Ly, dtype, POST[2] if Lx == 256 else POST[3], anchor=((Lx, Ly) == (256, 32)))


# ---- graph replay ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_linked_relax_replays_from_a_graph(comm, gpu_mem):
    """One linked relax call on a strip (the r exchange, the standalone exchange and 4 linked launches; and a low-rank relax
    of 4 half sweeps with nvec 4) captured as mg.py captures its cycle, replayed twice and then run once eagerly, equals three
    unlinked relax calls: the epochs live in device memory, so every replay continues the sequence."""
    w = _Wilson(4096, 512, C128, 3001)
    c = _Coarse("lr", 1024, 128, C128, 3002)
    phi0, r = c.fields(4, True)
    pw, pc = w.phi0.clone(), phi0.clone()
    out = {}
    w.relax(comm, "plain", True, POST[0], linked=True, phi=pw.clone())                  # warm-up outside the capture
    graph = torch.cuda.CUDAGraph()
    with mgmod._capture(graph):
        w.relax(comm, "plain", True, POST[0], linked=True, phi=pw)
        out["lr"] = c.relax(comm, pc, r, POST[1], linked=True)
    for _ in range(2):
        graph.replay()
        pc.copy_(out["lr"])
    torch.cuda.synchronize()
    w.relax(comm, "plain", True, POST[0], linked=True, phi=pw)
    got_c = c.relax(comm, pc, r, POST[1], linked=True)
    want_w, want_c = w.phi0.clone(), phi0
    for _ in range(3):
        want_w = w.relax(comm, "plain", True, POST[0], linked=False, phi=want_w)
        want_c = c.relax(comm, want_c, r, POST[1], linked=False)
    _healthy(comm)
    assert torch.equal(pw, want_w) and torch.equal(got_c, want_c)
    del graph


# ---- through DistMG ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_distmg_relax_equals_single_gpu_1024(comm, monkeypatch, gpu_mem):
    """Level.relax on the strips of a DistMG (the benchmark's cycle at 1024^2: levels 0-2 striped, level 3 replicated) equals
    the same call on a single-GPU MG holding the same synthetic operators, bit for bit: the two-colour sweep on level 0,
    low-rank on level 1, pre-multiplied on level 2; one vector with r and a batch of 4 without (near-null generation)."""
    p = _bench(monkeypatch).workload_params(mg2d, 1024, MASS)
    dmg = dmod.DistMG(p, comm)
    ref = mgmod.MG(p)
    ref.persistent_sites = 0          # level 2 (64^2) through the same half-sweep kernel as the strip, not the cooperative one
    try:
        assert [d for d, _ in dmg.plan] == [True, True, True, False]
        g = gen(4000)
        L = p.L
        U = links(g, L, L).reshape(L * L, 2).contiguous()
        for m in (dmg, ref):
            m.LVL[0].compute_lvl0_matrix(U, store=False)
        c1 = _Coarse("lr", 256, 256, C128, 4001)
        c2 = _Coarse("pm", 64, 64, C128, 4002)
        D1 = torch.zeros((256 * 256, 5, 16, 16), dtype=torch.complex128, device="cuda")
        D1[:, 0] = torch.linalg.inv(c1.D0inv).transpose(-1, -2)
        D2 = torch.cat([torch.linalg.inv(c2.D0inv)[:, None], c2.Dh], dim=1).transpose(-1, -2).contiguous()
        for m in (dmg, ref):
            lv1, lv2 = m.LVL[1], m.LVL[2]
            lv1.D, lv1.D0inv, lv1.M, lv1.F, lv1._lr_AB, lv1.lr_rank = D1.clone(), None, None, None, (c1.A.clone(), c1.B.clone()), 4
            lv2.D, lv2.D0inv, lv2.M = D2.clone(), None, None
        assert all(lv.distributed for lv in dmg.LVL[:3]) and not dmg.LVL[3].distributed
        for lvl in range(3):
            a, b = dmg.LVL[lvl], ref.LVL[lvl]
            for nvec, with_r in ((1, True), (4, False)):
                shape = (a.S, a.n) if nvec == 1 else (nvec, a.S, a.n)
                v = crandn(g, *shape)
                rr = crandn(g, *shape) if with_r else None
                strip, whole = v.clone(), v.clone()
                a.relax(4, phi=strip, r=rr)
                b.relax(4, phi=whole, r=rr)
                assert torch.equal(strip, whole), (lvl, nvec)
                assert not torch.equal(whole, v)
        _healthy(comm)
    finally:
        dmg.close()
        ref.close()


# ================================================================================================================
# GPU: the standalone exchange
# ================================================================================================================
def _read(ptr, nbytes):
    """nbytes of device memory at ptr (a halo buffer of the slab), through the library's own copy kernel"""
    out = torch.empty(nbytes // 8, dtype=torch.complex64, device="cuda")
    call("mg2d_copy", P_(out), ptr, nbytes // 8, C64, S_())
    return out.view(torch.uint8)


# (Lx, Ly, width, dtype, nvec, depth): both sides of the 1-CTA / 8-CTA switch, the benchmark's rows, batches of near-null vectors
_EXCHANGES = [
    (4096, 8, 1, C128, 1, 1), (4097, 8, 1, C128, 1, 1),           # 4096 words exactly / 4097
    (1024, 8, 1, C128, 4, 1), (1025, 8, 1, C128, 4, 1),           # batched: 4096 / 4100
    (2048, 8, 1, C64, 4, 1), (2050, 8, 1, C64, 4, 1),             # complex64 (float2) rows: 4096 / 4100
    (1024, 8, 2, C128, 1, 2), (1026, 8, 2, C128, 1, 2),           # two rows deep: 4096 / 4104
    (4096, 512, 2, C128, 1, 2), (4096, 512, 2, C64, 1, 2),        # level 0 (two-colour sweep)
    (4096, 2048, 2, C128, 1, 1),                                  # level 0, r
    (1024, 128, 16, C128, 4, 1), (1024, 128, 16, C64, 8, 1),      # level 1 batches
    (256, 32, 16, C64, 1, 1), (256, 32, 16, C128, 8, 1),          # level 2: the half-precision sweep's complex64 rows, a batch
    (64, 32, 16, C64, 8, 2), (64, 32, 16, C128, 1, 1),            # level 3
]


@pytest.mark.gpu
def test_halo_exchange_returns_the_current_rows(comm, gpu_mem):
    """Comm.exchange_rows (mg2d_halo_exchange) with the rank as its own neighbour: lo holds the strip's last `depth` rows and hi
    its first, bit for bit, for every vector of a batch (source stride Ly*Lx*width).  Every key is exchanged three times with new
    contents, interleaved with the other keys: each result is the current one, never a stale one."""
    g = gen(5000)
    seen = {}
    for rnd in range(3):
        for i, (Lx, Ly, width, dtype, nvec, depth) in enumerate(_EXCHANGES):
            t = crandn(g, nvec, Ly * Lx, width, dtype=CT[dtype])
            t = t[0] if nvec == 1 else t
            row = Lx * width * t.element_size() * depth
            words = nvec * row // 16
            if rnd == 0:
                print(f"\nexchange {Lx}x{Ly} width {width} {CT[dtype]} nvec {nvec} depth {depth}: {words} words, "
                      f"{8 if words > HX_WORDS else 1} CTA(s)")
            lo, hi = comm.exchange_rows(t, Lx, Ly, width, nvec, key=("x", i), depth=depth)
            assert isinstance(lo, dmod._Ptr) and isinstance(hi, dmod._Ptr)
            b = t.reshape(nvec, Ly, Lx * width).view(torch.uint8).reshape(nvec, Ly, -1)
            got_lo, got_hi = _read(lo.data_ptr(), nvec * row), _read(hi.data_ptr(), nvec * row)
            assert torch.equal(got_lo, b[:, Ly - depth:].reshape(-1)), (rnd, i, "lo")
            assert torch.equal(got_hi, b[:, :depth].reshape(-1)), (rnd, i, "hi")
            if i in seen:
                assert not torch.equal(got_lo, seen[i])
            seen[i] = got_lo
    _healthy(comm)


# ================================================================================================================
# GPU: reductions summed over the ranks inside the kernels
# ================================================================================================================
class _Reduce:
    """The same calls with mg2d_comm_reduce 0 and 1 on one context (always left at 0)."""

    def __init__(self, c):
        self.c = c

    def both(self, fn):
        try:
            self.c.call("mg2d_comm_reduce", 0)
            off = fn(self.c)
            self.c.call("mg2d_comm_reduce", 1)
            on = fn(self.c)
        finally:
            self.c.call("mg2d_comm_reduce", 0)
        return off, on


def _same(off, on, what):
    for k, (a, b) in enumerate(zip(off, on)):
        assert torch.equal(a, b), (what, k)


def _f64(n):
    return torch.zeros(n, dtype=torch.float64, device="cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [C128, C64])
@pytest.mark.parametrize("N", [4096 * 2048 * 2, 1024 * 128 * 16])
def test_fused_reductions_one_rank(N, dtype, comm, gpu_mem):
    """mg2d_norm2, gcr_dots (nj 1..8), gcr_ortho (z and lazy forms, nj 0..8), gcr_step and gcr_step_lazy (a whole restart
    cycle) on the level-0 (2 ranks) and level-1 (8 ranks) strip vectors: with the sums made global in the last CTA they are
    bit-identical to the plain kernels, vectors and sums.  The reductions run back to back, so the mailbox parity alternates."""
    ct = CT[dtype]
    g = gen(6000 + dtype)
    W, Z = crandn(g, 8, N, dtype=ct), crandn(g, 8, N, dtype=ct)
    w, z, x, r = (crandn(g, N, dtype=ct) for _ in range(4))
    dots = torch.randn(16, dtype=torch.float64, device="cuda", generator=g) * N
    wn2 = torch.rand(8, dtype=torch.float64, device="cuda", generator=g) * N + 1.0
    red = _Reduce(ctx())
    S = lambda: torch.cuda.current_stream().cuda_stream

    def norm(c):
        o = _f64(1)
        c.call("mg2d_norm2", P_(w), N, dtype, P_(o), S())
        return (o,)
    _same(*red.both(norm), "norm2")
    for nj in range(1, 9):
        def gd(c, nj=nj):
            o = _f64(16)
            c.call("mg2d_gcr_dots", P_(W), N, nj, P_(w), N, dtype, P_(o), S())
            return (o,)
        _same(*red.both(gd), ("gcr_dots", nj))
    for with_z in (True, False):
        for nj in range(9):
            def go(c, nj=nj, with_z=with_z):
                wo, zo, o = w.clone(), z.clone(), _f64(4)
                c.call("mg2d_gcr_ortho", P_(wo), P_(zo) if with_z else None, P_(r), P_(W), P_(Z) if with_z else None, N, nj,
                       P_(dots), P_(wn2), N, dtype, P_(o), S())
                return wo, zo, o
            _same(*red.both(go), ("gcr_ortho", with_z, nj))

    def step(c):
        xo, ro, o, slot = x.clone(), r.clone(), _f64(1), _f64(1)
        wr = torch.tensor([float(N), 0.3 * N, -0.7 * N], dtype=torch.float64, device="cuda")
        c.call("mg2d_gcr_step", P_(xo), P_(ro), P_(z), P_(w), P_(wr), P_(slot), N, dtype, P_(o), S())
        return xo, ro, o, slot
    _same(*red.both(step), "gcr_step")

    def lazy(c):
        ro, coef, slots, outs = r.clone(), _f64(144), _f64(8), []
        for nj in range(8):
            wr = torch.tensor([(1.0 + nj) * N, 0.1 * nj * N, -0.2 * N], dtype=torch.float64, device="cuda")
            o = _f64(1)
            c.call("mg2d_gcr_step_lazy", P_(ro), P_(W[nj]), P_(wr), P_(slots[nj:]), P_(dots), P_(wn2), nj, P_(coef), N, dtype,
                   P_(o), S())
            outs += [o, coef.clone()]
        return [ro, slots] + outs
    _same(*red.both(lazy), "gcr_step_lazy")
    _healthy(comm)


@pytest.mark.gpu
def test_fused_reductions_in_a_graph_and_from_a_second_context(comm, gpu_mem):
    """Back-to-back fused reductions captured in a CUDA graph and replayed twice, then interleaved with reductions of a second
    context attached to the same descriptor (Comm.attach, as the complex64 shadow hierarchy does): every sum equals the plain
    kernel's, so no reduction ever reads the other mailbox half."""
    N = 4096 * 512 * 2
    g = gen(7000)
    W = crandn(g, 8, N)
    vs = [crandn(g, N) for _ in range(3)]
    v32 = [crandn(g, N, dtype=torch.complex64) for _ in range(2)]

    def seq(c, outs):
        for k, v in enumerate(vs):
            c.call("mg2d_norm2", P_(v), N, C128, P_(outs[2 * k]), S_())
            c.call("mg2d_gcr_dots", P_(W), N, 3 + k, P_(v), N, C128, P_(outs[2 * k + 1]), S_())

    want = [_f64(16) for _ in range(6)]
    seq(ctx(), want)
    got = [_f64(16) for _ in range(6)]
    graph = torch.cuda.CUDAGraph()
    try:
        with mgmod._capture(graph):
            call("mg2d_comm_reduce", 1)
            seq(ctx(), got)
            call("mg2d_comm_reduce", 0)
        for _ in range(2):
            for o in got:
                o.zero_()
            graph.replay()
            torch.cuda.synchronize()
            for a, b in zip(got, want):
                assert torch.equal(a, b)
    finally:
        call("mg2d_comm_reduce", 0)
    del graph
    c2 = mg2d._lib.Context(0)
    comm.attach(c2)
    want2 = [_f64(1) for _ in v32]
    for o, v in zip(want2, v32):
        c2.call("mg2d_norm2", P_(v), N, C64, P_(o), S_())
    try:
        c2.call("mg2d_comm_reduce", 1)
        call("mg2d_comm_reduce", 1)
        for rep in range(2):
            got, got2 = [_f64(16) for _ in range(6)], [_f64(1) for _ in v32]
            for k, v in enumerate(vs):
                call("mg2d_norm2", P_(v), N, C128, P_(got[2 * k]), S_())
                if k < len(v32):
                    c2.call("mg2d_norm2", P_(v32[k]), N, C64, P_(got2[k]), S_())
                call("mg2d_gcr_dots", P_(W), N, 3 + k, P_(v), N, C128, P_(got[2 * k + 1]), S_())
            torch.cuda.synchronize()
            assert all(torch.equal(a, b) for a, b in zip(got, want)), rep
            assert all(torch.equal(a, b) for a, b in zip(got2, want2)), rep
    finally:
        call("mg2d_comm_reduce", 0)
        c2.call("mg2d_comm_reduce", 0)
        c2.close()
    _healthy(comm)


@pytest.mark.gpu
def test_allreduce_entry_point(comm):
    """mg2d_allreduce (the standalone mailbox kernel for reductions that are not fused) with one rank returns its input for
    n = 1, 17 and 64, leaves the rest of the buffer alone, and refuses n = 0 and n = 65."""
    g = gen(8000)
    prev = None
    for n in (1, 17, 64, 17, 1):
        buf = torch.randn(65, dtype=torch.float64, device="cuda", generator=g) + 2.0
        before = buf.clone()
        call("mg2d_allreduce", P_(buf), n, S_())
        torch.cuda.synchronize()
        assert torch.equal(buf, before), n
        if prev is not None:
            assert not torch.equal(buf[:1], prev[:1])
        prev = before
    for n in (0, 65):
        with pytest.raises(mg2d._lib.MG2DError):
            call("mg2d_allreduce", P_(buf), n, S_())
    _healthy(comm)
