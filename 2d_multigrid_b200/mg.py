"""Host-side mirror of the reference's solver objects, driving the sm_100a kernels of libmg2d_sm100.so.

Reference -> here (S6 = code/6_ntl-mg_new_code/3_combining_laplace_and_wilson/):
  class Level : Near_null  (S6/level.h, S6/near_null.h)      -> class Level   (same method names, f_ prefix dropped)
  free functions of S6/modules_main.h                       -> module functions of the same names
  main()                   (S6/mgrid_ntl.cpp:29-73)         -> setup() / solve() / run_reference_flow()

Every numerical operation is a CUDA kernel behind the C ABI (include/mg2d.h); torch supplies device memory,
streams and (multi-GPU) torch.distributed.  There is no CPU path: constructing an MG without the library or
without an sm_100 device raises.

Layouts (device): fields [S, n]; links U [S, 2]; projector phi_null [S, nc, nf] (reference layout);
operator D [S, 5, n, n] with COLUMN-major n x n blocks, i.e. D[s, k, j, i] = D_ref(s, k)(i, j).
"""
from __future__ import annotations

import contextlib
import ctypes
import gc
import math
import os

import numpy as np
import torch

from . import _lib
from ._lib import Context, MG2DError
from .params import MGParams
from .rng import StdMT19937

GCR_PAD = int(os.environ.get("MG2D_GCR_PAD", "0"))     # extra elements between stored FGCR directions (A/B knob; measured: no effect)

_DT = {"complex128": (torch.complex128, _lib.C128), "complex64": (torch.complex64, _lib.C64)}


def _ptr(t):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


@contextlib.contextmanager
def _capture(graph):
    """torch.cuda.graph with Python's cycle collector held off.  A dead hierarchy (MG <-> Level reference cycles) collected
    mid-capture destroys its CUDA graphs and library context (cudaGraphExecDestroy, cudaFree), which invalidates the capture."""
    enabled = gc.isenabled()
    gc.disable()
    try:
        with torch.cuda.graph(graph):
            yield
    finally:
        if enabled:
            gc.enable()


def D_to_reference_layout(D: torch.Tensor) -> torch.Tensor:
    """[S,5,j,i] (device layout) <-> [S,5,i,j] (D(s,k)(i,j) of the reference).  Involution."""
    return D.transpose(-1, -2).contiguous()


class _GlobalSums:
    def __init__(self, lv, t, fusable):
        self.lv, self.t = lv, t
        self.fuse = bool(lv.distributed and fusable and lv.mg.comm is not None and lv.mg.comm.fused)

    def __enter__(self):
        if self.fuse:
            self.lv.mg.ctx.call("mg2d_comm_reduce", 1)
        return self

    def __exit__(self, *exc):
        if self.fuse:
            self.lv.mg.ctx.call("mg2d_comm_reduce", 0)
        elif exc[0] is None:
            self.lv.allreduce(self.t)
        return False


class Level:
    """class Level : public Near_null (S6/level.h:3-39, S6/near_null.h:9-22): phi, r, D, phi_null of one
    multigrid level, plus the kernel workspace (MR residual / direction, D0^-1, reduction slots)."""

    def __init__(self, mg: "MG", lvl: int):
        self.mg, self.lvl = mg, lvl
        p = mg.p
        self.L = p.size[lvl]       # global width (x); rows are strip-local
        self.Ly = self.L           # locally owned rows [y0, y0+Ly)
        self.y0 = 0
        self.distributed = False   # True: 1-D strip in y with halo exchange; False: whole lattice on this GPU
        self.n = p.n_dof[lvl]
        self.S = self.L * self.Ly  # local sites
        self.nc = p.n_dof[lvl + 1] if lvl < p.nlevels else None
        self.block = p.blocks[lvl] if lvl < p.nlevels else None      # aggregate size towards the next coarser level
        self.phi = None
        self.r = None
        self.D = None          # [S,5,n,n] column-major blocks; None on a matrix-free level 0
        self.D0inv = None
        self.M = None          # [S,4,n,n]: pre-multiplied hopping blocks -D0^-1 D_k of the red-black smoother
        self.F = None          # low-rank factors of the hopping blocks (first coarse level), lane-ordered for mg2d_relax_rb_lr
        self.lr_rank = 0       # rank of those factors (= aggregate size of the level below); 0: dense blocks only
        self._lr_AB = None     # unpacked factors (A, B) until the first sweep needs F
        self.Dh = None         # optional half-precision copies (__half2) of D / D0inv for the complex64 preconditioner
        self.D0inv_h = None
        self.phi_null = None   # [S,nc,nf]
        self.phi_null_c = None # [S,nc,nf/2]: chirality-compacted copy used by restriction / prolongation (wilson)
        self.U = None          # level 0 only: links [S,2]
        self.clover = None     # level 0 with csw != 0: real clover field f [S] (float64 / float32 with the field precision)
        self._clover_halos = None
        self.matrix_free = False
        self._work = {}

    # ---- plumbing -------------------------------------------------------------------------------------
    def new_field(self, nvec: int | None = None, zero: bool = True):
        shape = (self.S, self.n) if nvec is None else (nvec, self.S, self.n)
        f = torch.zeros if zero else torch.empty
        return f(shape, dtype=self.mg.tdtype, device=self.mg.device)

    def work(self, name: str, nvec: int | None = None):
        key = (name, nvec)
        if key not in self._work:
            self._work[key] = self.new_field(nvec)
        return self._work[key]

    def flat_work(self, key, nelem: int):
        """A flat work buffer of `nelem` field elements (callers carve padded vectors out of it)."""
        if key not in self._work:
            self._work[key] = torch.zeros(nelem, dtype=self.mg.tdtype, device=self.mg.device)
        return self._work[key]

    def dots(self, name: str = "dots"):
        if name not in self._work:
            self._work[name] = torch.zeros(64 * 4, dtype=torch.float64, device=self.mg.device)
        return self._work[name]

    def set_strip(self, y0: int, Ly: int):
        self.y0, self.Ly, self.distributed = y0, Ly, True
        self.S = self.L * Ly

    def _halo(self, t: torch.Tensor, nvec: int = 1, width: int | None = None, depth: int = 1):
        """(lo, hi) pointers to the `depth` rows below local row 0 (rows -depth..-1) and above the last local row
        (rows Ly..Ly+depth-1) of a field [S, width] (or a batch [nvec, S, width]) of this level: the periodic wrap
        rows on one GPU, the exchanged neighbour rows on a strip."""
        width = self.n if width is None else width
        if self.distributed:
            lo, hi = self.mg.comm.exchange_rows(t, self.L, self.Ly, width, nvec, key=(self.lvl, width, nvec, depth), depth=depth)
            return lo.data_ptr(), hi.data_ptr()
        t0 = t if nvec == 1 else t[0]
        es = t0.element_size() * width
        base = t0.data_ptr()
        return base + (self.Ly - depth) * self.L * es, base

    def allreduce(self, t, op: str = "sum"):
        if self.distributed:
            self.mg.comm.allreduce(t, op)

    def global_sums(self, t, fusable: bool = True):
        """Context for kernels that write partial sums into `t`: on a distributed level the sums are made global either
        inside the kernel itself (mg2d_comm_reduce: the last CTA exchanges with all ranks over NVLink) or, when the kernel
        cannot (batched reductions) or the comm has no peer mailboxes, by an all-reduce of `t` afterwards."""
        return _GlobalSums(self, t, fusable)

    def init_level(self, gen: StdMT19937 | None):
        """f_init_level (S6/level.h:42-53): phi, r, phi_null drawn in this order (gen None -> ones, rand=0)."""
        mg, p = self.mg, self.mg.p
        draw = (lambda k: gen.uniform_pm_pi(k)) if gen is not None else (lambda k: np.ones(k))
        self.phi = mg.to_device(draw(self.S * self.n).reshape(self.S, self.n))
        self.r = mg.to_device(draw(self.S * self.n).reshape(self.S, self.n))
        if self.lvl != p.nlevels:
            self.phi_null = mg.to_device(draw(self.S * self.nc * self.n).reshape(self.S, self.nc, self.n))

    def define_source(self):
        """f_define_source (S6/level.h:55-59): r(site 2 + 2L)(0) = 5 -- a GLOBAL site; on a strip only its owner writes."""
        s = 2 + 2 * self.mg.p.L - self.y0 * self.L
        if 0 <= s < self.S:
            self.r[s, 0] = 5.0

    # ---- operators ------------------------------------------------------------------------------------
    def compute_lvl0_matrix(self, U: torch.Tensor, store: bool = True):
        """f_compute_lvl0_matrix (S6/level.h:131-175).  With store=False only the links are kept and the
        Wilson operator is applied matrix-free."""
        mg, p = self.mg, self.mg.p
        assert self.lvl == 0
        self.U = U
        self.bind_link_halos(None)
        self.clover = None
        if p.csw != 0.0:
            # clover self term (2+m) 1 + f sigma3: f of the local rows from the links (and their halo rows)
            rdt = torch.float64 if mg.dcode == _lib.C128 else torch.float32
            self.clover = torch.empty(self.S, dtype=rdt, device=mg.device)
            mg.ctx.call("mg2d_clover_field", _ptr(self.clover), _ptr(U), self.U_lo_ptr, self.U_hi_ptr, float(p.csw), self.L,
                        self.Ly, mg.dcode, _stream())
            self.bind_clover_halos(None)
        if store:
            self.D = torch.empty((self.S, 5, self.n, self.n), dtype=mg.tdtype, device=mg.device)
            mg.ctx.call("mg2d_lvl0_matrix", _ptr(self.D), _ptr(U), self.U_lo_ptr, float(p.mass),
                        0 if p.stencil == "wilson" else 1, self.L, self.Ly, mg.dcode, _stream())
            if self.clover is not None:
                mg.ctx.call("mg2d_clover_add", _ptr(self.D), _ptr(self.clover), self.S, mg.dcode, _stream())
            if p.mu != 0.0:
                # twisted mass: + i mu sigma3 on the self blocks; the Galerkin products carry it to every coarse level
                mg.ctx.call("mg2d_twist_add", _ptr(self.D), float(p.mu), self.S, mg.dcode, _stream())
            self.D0inv = None
            self.M = None
        self.matrix_free = not store

    def bind_link_halos(self, halos):
        """Link rows outside the strip: two below (U_lo2: rows -2, -1; the two-colour smoother recomputes one row of
        the neighbour's red sites) and one above (U_hi).  Exchanged once per gauge field (halos None) or taken from
        `halos` = (lo2, hi) tensors (precision copies); on one GPU they are the periodic wrap rows of U itself."""
        U = self.U
        row = self.L * 2 * U.element_size()
        if self.distributed:
            if halos is None:
                lo2, hi2 = self.mg.comm.exchange_rows(U, self.L, self.Ly, 2, 1, key=("U",), as_tensor=True, depth=2)
                halos = (lo2.clone(), hi2[:self.L].clone())
            self._U_halos = halos
            self.U_lo2_ptr, self.U_hi_ptr = halos[0].data_ptr(), halos[1].data_ptr()
        else:
            self._U_halos = None
            self.U_lo2_ptr, self.U_hi_ptr = U.data_ptr() + (self.Ly - 2) * row, U.data_ptr()
        self.U_lo_ptr = self.U_lo2_ptr + row          # row -1

    def bind_clover_halos(self, halos):
        """Rows -1 and Ly of the clover field (the two-colour sweep recomputes red sites there).  Exchanged once per gauge
        field (halos None) or taken from `halos` = (lo, hi) tensors (precision copies); on one GPU the periodic wrap rows."""
        F = self.clover
        if self.distributed:
            if halos is None:
                lo, hi = self.mg.comm.exchange_rows(F, self.L, self.Ly, 1, 1, key=("clover",), as_tensor=True, depth=1)
                halos = (lo.clone(), hi.clone())
            self._clover_halos = halos
            self.clover_lo_ptr, self.clover_hi_ptr = halos[0].data_ptr(), halos[1].data_ptr()
        else:
            self._clover_halos = None
            self.clover_lo_ptr, self.clover_hi_ptr = F.data_ptr() + (self.Ly - 1) * self.L * F.element_size(), F.data_ptr()

    def _stencil(self, out, vin, b, mode, dots, nvec=1):
        mg = self.mg
        _lib.TRACE_TAG = self.lvl
        if out.data_ptr() == vin.data_ptr():
            raise ValueError("stencil output must not alias its input")
        if self.matrix_free:
            if nvec != 1:
                for v in range(nvec):
                    self._stencil(out[v], vin[v], None if b is None else b[v], mode,
                                  None if dots is None else dots[4 * v:], 1)
                return
            lo, hi = self._halo(vin)
            if mg.p.mu != 0.0:
                mg.ctx.call("mg2d_wilson_tm_apply", _ptr(out), _ptr(vin), lo, hi, _ptr(self.U), self.U_lo_ptr, _ptr(self.clover),
                            _ptr(b), float(mg.p.mass), float(mg.p.mu), self.L, self.Ly, mode, mg.dcode, _ptr(dots), _stream())
            elif self.clover is None:
                mg.ctx.call("mg2d_wilson_apply", _ptr(out), _ptr(vin), lo, hi, _ptr(self.U), self.U_lo_ptr, _ptr(b),
                            float(mg.p.mass), self.L, self.Ly, mode, mg.dcode, _ptr(dots), _stream())
            else:
                mg.ctx.call("mg2d_wilson_sw_apply", _ptr(out), _ptr(vin), lo, hi, _ptr(self.U), self.U_lo_ptr, _ptr(self.clover),
                            _ptr(b), float(mg.p.mass), self.L, self.Ly, mode, mg.dcode, _ptr(dots), _stream())
        else:
            vs = self.S * self.n
            lo, hi = self._halo(vin, nvec)
            hs = self.L * self.n if (self.distributed and nvec > 1) else vs
            mg.ctx.call("mg2d_stencil_apply", _ptr(out), _ptr(vin), lo, hi, _ptr(self.D), _ptr(b), self.n,
                        self.L, self.Ly, mode, mg.dcode, nvec, vs, hs, _ptr(dots), _stream())

    def apply_D(self, v_out, v_in):
        """f_apply_D (S6/level.h:251-265): v_out = D v_in."""
        self._stencil(v_out, v_in, None, _lib.MODE_APPLY, None)

    def residue(self, rtemp):
        """f_residue (S6/level.h:61-77): rtemp = r - D phi."""
        self._stencil(rtemp, self.phi, self.r, _lib.MODE_RESID, None)

    def residue_mag_async(self):
        """Launch the fused residual + norms of f_get_residue_mag; returns the device dots tensor
        ([0] = |r - D phi|^2, [3] = |r|^2).  No host sync."""
        d = self.dots("resmag")
        with self.global_sums(d[:4]):
            self._stencil(self.work("rtemp"), self.phi, self.r, _lib.MODE_RESID, d)
        return d

    def get_residue_mag(self) -> float:
        """f_get_residue_mag (S6/level.h:79-98): |r - D phi| / |r|."""
        d = self.residue_mag_async().cpu()
        return math.sqrt(d[0].item()) / math.sqrt(d[3].item())

    def make_half_blocks(self):
        """__half2 copies of the stored operator and of D0^-1 (complex64 levels with n in {8,16,32}) for
        mg2d_relax_rb_half."""
        if self.D is None or self.mg.p.dtype != "complex64" or self.n not in (8, 16, 32):
            return
        if self.lr_rank and self.mg.lowrank:      # complex64 low-rank factors are already fewer bytes than half-precision blocks
            return
        self._ensure_D0inv()
        mg = self.mg
        self.Dh = torch.empty(self.D.shape, dtype=torch.float32, device=mg.device)            # 4 bytes per complex
        self.D0inv_h = torch.empty(self.D0inv.shape, dtype=torch.float32, device=mg.device)
        mg.ctx.call("mg2d_to_half", _ptr(self.Dh), _ptr(self.D), self.D.numel(), _stream())
        mg.ctx.call("mg2d_to_half", _ptr(self.D0inv_h), _ptr(self.D0inv), self.D0inv.numel(), _stream())

    def _ensure_D0inv(self):
        if self.D0inv is None:
            if self.D is None:
                raise MG2DError("Gauss-Seidel / Jacobi need the stored operator (matrix_free=False)")
            self.D0inv = torch.empty((self.S, self.n, self.n), dtype=self.mg.tdtype, device=self.mg.device)
            self.mg.ctx.call("mg2d_block_inverse", _ptr(self.D0inv), _ptr(self.D), self.n, self.S, self.mg.dcode, _stream())

    def _ensure_M(self):
        """M[s][k-1] = -D0(s)^-1 D_k(s): the hopping blocks with f_relax's inverse (S6/level.h:116) folded in."""
        if self.M is None:
            self._ensure_D0inv()
            self.M = torch.empty((self.S, 4, self.n, self.n), dtype=self.mg.tdtype, device=self.mg.device)
            self.mg.ctx.call("mg2d_premultiply", _ptr(self.M), _ptr(self.D), _ptr(self.D0inv), self.n, self.S, self.mg.dcode, _stream())

    def _ensure_F(self):
        """Lane-ordered low-rank factors (conj(B), -D0^-1 A) of the hopping blocks for mg2d_relax_rb_lr."""
        if self.F is None and self._lr_AB is not None:
            self._ensure_D0inv()
            A, B = self._lr_AB
            self.F = torch.empty((self.S, 2, self.n * self.lr_rank // 8, 32), dtype=self.mg.tdtype, device=self.mg.device)
            self.mg.ctx.call("mg2d_lowrank_pack", _ptr(self.F), _ptr(A), _ptr(B), _ptr(self.D0inv), self.n, self.lr_rank, self.S,
                             self.mg.dcode, _stream())
            self._lr_AB = None
        if self.F is not None:
            self._ensure_D0inv()       # (a precision copy receives F but builds its own D0^-1 for the c = D0^-1 r pass)
        return self.F is not None

    def hop_factors(self, lvl_f: "Level", P: torch.Tensor, p_lo: int, p_hi: int):
        """Rank-`block` factors of this level's hopping blocks from the fine operator and projector (mg2d_hop_factors);
        `self` is the coarse level.  status[1] != 0 (a fine hopping block that is not rank one) is read by the caller."""
        mg = self.mg
        Q = 4 * lvl_f.block
        A = torch.empty((self.S, Q, self.n), dtype=mg.tdtype, device=mg.device)
        B = torch.empty_like(A)
        mg.ctx.call("mg2d_hop_factors", _ptr(A), _ptr(B), _ptr(lvl_f.D), _ptr(P), p_lo, p_hi, lvl_f.n, self.n, lvl_f.L, lvl_f.Ly,
                    lvl_f.block, mg.dcode, _ptr(mg.status[1:]), _stream())
        self._lr_AB, self.F, self.lr_rank = (A, B), None, lvl_f.block

    def relax(self, num_iter: int, gs_flag: int | None = None, phi=None, r="self", smoother: str | None = None):
        """f_relax (S6/level.h:100-128).  gs_flag 1 = lexicographic Gauss-Seidel, 0 = Jacobi (reference);
        smoother='mr' = minimal residual (north_star).  phi may be a batch [nvec, S, n]; r=None means r=0."""
        mg = self.mg
        _lib.TRACE_TAG = self.lvl
        if smoother is None:
            smoother = mg.p.smoother if gs_flag is None else ("gs" if gs_flag == 1 else "jacobi")
        phi = self.phi if phi is None else phi
        r = self.r if isinstance(r, str) else r
        nvec = 1 if phi.dim() == 2 else phi.shape[0]
        vs = self.S * self.n
        if num_iter <= 0:
            return
        if smoother == "gs" and self.distributed:
            # the reference's own smoother on strips: global anti-diagonal fronts, one flag hop per front (parity mode)
            if mg.comm.p2p is None:
                raise MG2DError("lexicographic Gauss-Seidel on strips needs the peer-to-peer halo path (MG2D_HALO=p2p)")
            self._ensure_D0inv()
            key = (self.lvl, self.n, 1, 1)
            for v in range(nvec):
                ph = phi if nvec == 1 else phi[v]
                rv = None if r is None else (r if nvec == 1 else r[v])
                for _ in range(num_iter):
                    lo, hi = self._halo(ph)                     # the neighbours' OLD boundary rows
                    g = mg.comm.gs_links(ph, self.L, self.n, key)
                    mg.ctx.call("mg2d_relax_gs_strip", _ptr(ph), lo, hi, _ptr(self.D), _ptr(self.D0inv), _ptr(rv), self.n, self.L,
                                self.Ly, self.y0, self.L, mg.dcode, g["slot_mine"], g["slot_next"], g["slot_last"],
                                g["push_next_lo"], g["push_last_hi"], g["first"], g["last"], _stream())
        elif smoother == "gs":
            self._ensure_D0inv()
            mg.ctx.call("mg2d_relax_gs", _ptr(phi), _ptr(self.D), _ptr(self.D0inv), _ptr(r), self.n, self.L,
                        num_iter, mg.dcode, nvec, vs, _stream())
        elif smoother == "jacobi":
            self._ensure_D0inv()
            tmp = self.work("jacobi_tmp", None if nvec == 1 else nvec)
            cur, nxt = phi, tmp
            for _ in range(num_iter):
                lo, hi = self._halo(cur, nvec)
                hs = self.L * self.n if (self.distributed and nvec > 1) else vs
                mg.ctx.call("mg2d_relax_jacobi", _ptr(nxt), _ptr(cur), lo, hi, _ptr(self.D), _ptr(self.D0inv),
                            _ptr(r), self.n, self.L, self.Ly, mg.dcode, nvec, vs, hs, _stream())
                cur, nxt = nxt, cur
            if cur.data_ptr() != phi.data_ptr():
                mg.ctx.call("mg2d_copy", _ptr(phi), _ptr(cur), phi.numel(), mg.dcode, _stream())
        elif smoother == "mr":
            key = None if nvec == 1 else nvec
            res, t, d = self.work("mr_res", key), self.work("mr_t", key), self.dots("mr")
            b = r if r is not None else self.work("zero_rhs", key)
            self._stencil(res, phi, b, _lib.MODE_RESID, None, nvec)
            for _ in range(num_iter):
                with self.global_sums(d[:4 * nvec], fusable=(nvec == 1)):
                    self._stencil(t, res, None, _lib.MODE_APPLY, d, nvec)
                mg.ctx.call("mg2d_mr_update", _ptr(phi), _ptr(res), _ptr(t), _ptr(d), float(mg.p.mr_omega),
                            vs, mg.dcode, nvec, vs, _stream())
        elif smoother == "rbgs" and self.matrix_free and mg.two_colour and self.Ly >= 2:
            # both colours per pass, out of place (mg2d_wilson_relax_rb2): ping-pong between phi and a work buffer
            tmp = self.work("rb2_tmp", None if nvec == 1 else nvec)
            fused = self.distributed and mg.comm.fused
            for v in range(nvec):
                cur, nxt = (phi, tmp) if nvec == 1 else (phi[v], tmp[v])
                rv = None if r is None else (r if nvec == 1 else r[v])
                r_lo, r_hi = (None, None) if rv is None else self._halo(rv)
                for it in range(num_iter):
                    link = None
                    if fused:
                        # one standalone exchange in front; afterwards every sweep pushes the two boundary rows it
                        # produces into the neighbours' (alternating) halo buffers itself and waits only in its boundary chunks
                        if it == 0:
                            self._halo(cur, depth=2)
                        lk, lo2, hi2 = mg.comm.fused_link(cur, self.L, self.Ly, self.n, 1, (self.lvl, self.n, 1, 2), 2, it,
                                                          push=(it < num_iter - 1))
                        link = ctypes.byref(lk)
                    else:
                        lo2, hi2 = self._halo(cur, depth=2)
                    if mg.p.mu != 0.0:
                        F_lo, F_hi = (None, None) if self.clover is None else (self.clover_lo_ptr, self.clover_hi_ptr)
                        mg.ctx.call("mg2d_wilson_tm_relax_rb2", _ptr(nxt), _ptr(cur), lo2, hi2, _ptr(self.U), self.U_lo2_ptr,
                                    self.U_hi_ptr, _ptr(self.clover), F_lo, F_hi, _ptr(rv), r_lo, r_hi, float(mg.p.mass),
                                    float(mg.p.mu), self.L, self.Ly, self.y0 & 1, mg.dcode, link, _stream())
                    elif self.clover is None:
                        mg.ctx.call("mg2d_wilson_relax_rb2", _ptr(nxt), _ptr(cur), lo2, hi2, _ptr(self.U), self.U_lo2_ptr,
                                    self.U_hi_ptr, _ptr(rv), r_lo, r_hi, float(mg.p.mass), self.L, self.Ly, self.y0 & 1,
                                    mg.dcode, link, _stream())
                    else:
                        mg.ctx.call("mg2d_wilson_sw_relax_rb2", _ptr(nxt), _ptr(cur), lo2, hi2, _ptr(self.U), self.U_lo2_ptr,
                                    self.U_hi_ptr, _ptr(self.clover), self.clover_lo_ptr, self.clover_hi_ptr, _ptr(rv), r_lo,
                                    r_hi, float(mg.p.mass), self.L, self.Ly, self.y0 & 1, mg.dcode, link, _stream())
                    cur, nxt = nxt, cur
                if num_iter & 1:
                    mg.ctx.call("mg2d_copy", _ptr(nxt), _ptr(cur), vs, mg.dcode, _stream())
        elif (smoother == "rbgs" and not self.matrix_free and not self.distributed and nvec == 1 and mg.premul and self.n <= 16
              and mg.persistent_sites >= self.S and self.Ly == self.L and not (self.Dh is not None and mg.use_half)):
            # small level: every sweep of this call in one cooperative launch (grid barriers instead of kernel boundaries)
            self._ensure_M()
            cbuf = None if r is None else self.work("pm_c")
            mg.ctx.call("mg2d_relax_rb_pm_sweeps", _ptr(phi), _ptr(self.M), _ptr(self.D0inv), _ptr(r), _ptr(cbuf), self.n, self.L,
                        num_iter, mg.dcode, _stream())
        elif smoother == "rbgs":
            hs = self.L * self.n if (self.distributed and nvec > 1) else vs
            for it in range(num_iter):
                for colour in (0, 1):
                    if self.matrix_free:
                        for v in range(nvec):
                            ph = phi if nvec == 1 else phi[v]
                            rv = None if r is None else (r if nvec == 1 else r[v])
                            lo, hi = self._halo(ph)
                            if mg.p.mu != 0.0:
                                mg.ctx.call("mg2d_wilson_tm_relax_rb", _ptr(ph), lo, hi, _ptr(self.U), self.U_lo_ptr,
                                            _ptr(self.clover), _ptr(rv), float(mg.p.mass), float(mg.p.mu), self.L, self.Ly, colour,
                                            self.y0 & 1, mg.dcode, _stream())
                            elif self.clover is None:
                                mg.ctx.call("mg2d_wilson_relax_rb", _ptr(ph), lo, hi, _ptr(self.U), self.U_lo_ptr, _ptr(rv),
                                            float(mg.p.mass), self.L, self.Ly, colour, self.y0 & 1, mg.dcode, _stream())
                            else:
                                mg.ctx.call("mg2d_wilson_sw_relax_rb", _ptr(ph), lo, hi, _ptr(self.U), self.U_lo_ptr,
                                            _ptr(self.clover), _ptr(rv), float(mg.p.mass), self.L, self.Ly, colour, self.y0 & 1,
                                            mg.dcode, _stream())
                    elif self.lr_rank and mg.premul and mg.lowrank and self._ensure_F():
                        # first coarse level: rank-`block` factors of the pre-multiplied hopping blocks (half the bytes);
                        # batches of 4 vectors share one stream of the factors (near-null generation)
                        cmode = 0 if r is None else (1 if it == 0 else 2)
                        cbuf = None if r is None else self.work("pm_c", None if nvec == 1 else nvec)
                        link = None
                        if self.distributed and mg.comm.fused:
                            k = 2 * it + colour
                            if k == 0:
                                self._halo(phi, nvec)
                            lk, lo, hi = mg.comm.fused_link(phi, self.L, self.Ly, self.n, nvec, (self.lvl, self.n, nvec, 1), 1, k,
                                                            push=(k < 2 * num_iter - 1))
                            link = ctypes.byref(lk)
                        else:
                            lo, hi = self._halo(phi, nvec)
                        mg.ctx.call("mg2d_relax_rb_lr", _ptr(phi), lo, hi, _ptr(self.F), _ptr(self.D0inv), _ptr(r), _ptr(cbuf), cmode,
                                    self.n, self.lr_rank, self.L, self.Ly, colour, self.y0 & 1, mg.dcode, nvec, vs, hs, link, _stream())
                    elif self.Dh is not None and nvec == 1 and mg.use_half:
                        lo, hi = self._halo(phi)
                        mg.ctx.call("mg2d_relax_rb_half", _ptr(phi), lo, hi, _ptr(self.Dh), _ptr(self.D0inv_h), _ptr(r),
                                    self.n, self.L, self.Ly, colour, self.y0 & 1, _stream())
                    elif mg.premul and self.n <= 16:
                        # pre-multiplied blocks M_k = -D0^-1 D_k: 4 blocks per updated site instead of 5
                        self._ensure_M()
                        cmode = 0 if r is None else (1 if it == 0 else 2)
                        cbuf = None if r is None else self.work("pm_c", None if nvec == 1 else nvec)
                        link = None
                        if self.distributed and mg.comm.fused:
                            k = 2 * it + colour        # one standalone exchange, then the half sweeps push / wait themselves
                            if k == 0:
                                self._halo(phi, nvec)
                            lk, lo, hi = mg.comm.fused_link(phi, self.L, self.Ly, self.n, nvec, (self.lvl, self.n, nvec, 1), 1, k,
                                                            push=(k < 2 * num_iter - 1))
                            link = ctypes.byref(lk)
                        else:
                            lo, hi = self._halo(phi, nvec)
                        mg.ctx.call("mg2d_relax_rb_pm", _ptr(phi), lo, hi, _ptr(self.M), _ptr(self.D0inv), _ptr(r), _ptr(cbuf),
                                    cmode, self.n, self.L, self.Ly, colour, self.y0 & 1, mg.dcode, nvec, vs, hs, link, _stream())
                    else:
                        self._ensure_D0inv()
                        lo, hi = self._halo(phi, nvec)
                        mg.ctx.call("mg2d_relax_rb", _ptr(phi), lo, hi, _ptr(self.D), _ptr(self.D0inv), _ptr(r),
                                    self.n, self.L, self.Ly, colour, self.y0 & 1, mg.dcode, nvec, vs, hs, _stream())
        else:
            raise ValueError(smoother)

    # ---- near-null vectors (class Near_null) -------------------------------------------------------------
    def near_null(self, null_iters: int | None = None, warm: bool = False):
        """f_near_null (S6/level.h:177-249): null_iters relaxation sweeps on D v = 0 in chunks of null_chunk
        with a global renormalisation (f_g_norm, S6/modules_indiv.h:70-92) after each chunk, all vectors
        batched; then conjugate (+ chirality split for wilson) into the rows of phi_null.
        warm=True starts each vector from the current projector (MG.refresh): for wilson the sum of its two chirality rows,
        which undoes the split of the previous pack; otherwise from rows d1 of the random start."""
        mg, p = self.mg, self.mg.p
        nf, nc = self.n, self.nc
        wilson = p.stencil == "wilson"
        nvec = nc // 2 if wilson else nc
        num = max((p.null_iters if null_iters is None else null_iters) // p.null_chunk, 1)
        if warm and wilson:
            V = (self.phi_null[:, :nvec, :] + self.phi_null[:, nc // 2:nc // 2 + nvec, :]).conj().permute(1, 0, 2).contiguous()
        elif warm:
            V = self.phi_null[:, :nvec, :].conj().permute(1, 0, 2).contiguous()
        else:
            V = self.phi_null[:, :nvec, :].permute(1, 0, 2).contiguous()     # rows d1 of the random start
        vs = self.S * nf
        nrm = self.dots("nullnorm")
        # level 0 of a matrix-free run: relax through the link field (160 B/site/sweep) instead of the stored 2x2-block
        # operator (~400 B/site/sweep); the stored copy is only kept for the Galerkin product
        stored = self.matrix_free
        if self.lvl == 0 and p.matrix_free and self.U is not None:
            self.matrix_free = True
        for _ in range(num):
            self.relax(p.null_chunk, phi=V, r=None)
            with self.global_sums(nrm[:nvec]):
                for v in range(nvec):
                    mg.ctx.call("mg2d_norm2", _ptr(V[v]), vs, mg.dcode, _ptr(nrm[v:]), _stream())
            for v in range(nvec):
                mg.ctx.call("mg2d_scale_inv_norm", _ptr(V[v]), _ptr(nrm[v:]), vs, mg.dcode, _stream())
        self.matrix_free = stored
        mg.ctx.call("mg2d_pack_null", _ptr(self.phi_null), _ptr(V), nvec, vs, nf, nc, self.S, int(wilson),
                    mg.dcode, _stream())

    def norm_nn(self, quad: int):
        """f_norm_nn (S6/near_null.h:24-48); a NaN or tiny block norm sets status[0] (read by compute_near_null)."""
        mg = self.mg
        mg.ctx.call("mg2d_norm_nn", _ptr(self.phi_null), self.n, self.nc, self.L, self.Ly, self.block, quad, mg.dcode,
                    _ptr(mg.status), _stream())

    def ortho(self, quad: int):
        """f_ortho (S6/near_null.h:97-173)."""
        mg = self.mg
        mg.ctx.call("mg2d_ortho", _ptr(self.phi_null), self.n, self.nc, self.L, self.Ly, self.block, quad, mg.dcode,
                    _ptr(mg.status), _stream())

    def check_ortho(self, quad: int) -> float:
        """f_check_ortho (S6/near_null.h:175-214): worst |<null_d1, null_d2>| over aggregates."""
        mg = self.mg
        out = self.dots("ortho_check")
        mg.ctx.call("mg2d_check_ortho", _ptr(self.phi_null), self.n, self.nc, self.L, self.Ly, self.block, quad,
                    mg.dcode, _ptr(out), _stream())
        self.allreduce(out[:1], "max")
        return float(out[0].item())

    def compact_projector(self, drop_dense: bool = False, check: bool = False):
        """Wilson levels: keep the non-zero chirality half of every row of phi_null (S6/level.h:236-245) in
        phi_null_c[s][ic][jf'] so that restriction / prolongation stream half the bytes."""
        if self.phi_null is None or self.mg.p.stencil != "wilson":
            return
        nc, nf = self.nc, self.n
        P = self.phi_null
        if check:
            # supplied vectors (gen_null = 0) need not have f_near_null's chirality structure: keep the dense projector
            # (as the reference's f_restriction / f_prolongation do) unless the halves to be dropped are exactly zero
            dropped = torch.stack([P[:, :nc // 2, nf // 2:].abs().max(), P[:, nc // 2:, :nf // 2].abs().max()]).max()
            if self.distributed:
                self.mg.comm.allreduce(dropped, "max")
            if float(dropped.item()) != 0.0:
                self.phi_null_c = None
                return
        self.phi_null_c = torch.cat([P[:, :nc // 2, :nf // 2], P[:, nc // 2:, nf // 2:]], dim=1).contiguous()
        if drop_dense:
            self.phi_null = None

    def restriction(self, vec_c, vec_f, quad: int):
        """f_restriction (S6/near_null.h:217-240): vec_c = P vec_f."""
        mg = self.mg
        _lib.TRACE_TAG = self.lvl
        gather = self.distributed and not self._coarse_distributed()
        if self.distributed and quad != 1:
            raise MG2DError("shifted aggregates (quad != 1) need the whole lattice on one GPU")
        dst = vec_c
        if gather:   # the coarse level is replicated: restrict the local strip, then all-gather the strips
            dst = self.work_coarse_strip()
        if self.phi_null_c is not None:
            mg.ctx.call("mg2d_restrict_chiral", _ptr(dst), _ptr(vec_f), _ptr(self.phi_null_c), self.n, self.nc, self.L,
                        self.Ly, self.block, quad, mg.dcode, _stream())
        else:
            mg.ctx.call("mg2d_restrict", _ptr(dst), _ptr(vec_f), _ptr(self.phi_null), self.n, self.nc, self.L, self.Ly,
                        self.block, quad, mg.dcode, _stream())
        if gather:
            mg.comm.allgather(vec_c, dst)

    def prolongation(self, vec_f, vec_c, quad: int, zero_vc: bool = False, accumulate: bool = True):
        """f_prolongation (S6/near_null.h:242-264): vec_f += P^dagger vec_c.  `self` is the FINE level.
        accumulate=False writes vec_f = P^dagger vec_c (caller knows vec_f == 0; chirality-compacted path only)."""
        mg = self.mg
        blk = self.block
        _lib.TRACE_TAG = self.lvl

        def launch(vc_ptr, zv):
            if self.phi_null_c is not None:
                mg.ctx.call("mg2d_prolong_chiral", _ptr(vec_f), vc_ptr, _ptr(self.phi_null_c), self.n, self.nc, self.L,
                            self.Ly, blk, quad, zv, int(accumulate), mg.dcode, _stream())
            else:
                if not accumulate:
                    mg.ctx.call("mg2d_zero", _ptr(vec_f), vec_f.numel(), mg.dcode, _stream())
                mg.ctx.call("mg2d_prolong_add", _ptr(vec_f), vc_ptr, _ptr(self.phi_null), self.n, self.nc, self.L, self.Ly,
                            blk, quad, zv, mg.dcode, _stream())

        if self.distributed and not self._coarse_distributed():
            # replicated coarse level: every rank prolongs from its rows of the full coarse field
            Lc = self.L // blk
            view = vec_c[(self.y0 // blk) * Lc:(self.y0 // blk + self.Ly // blk) * Lc]
            launch(_ptr(view), 0)
            if zero_vc:
                mg.ctx.call("mg2d_zero", _ptr(vec_c), vec_c.numel(), mg.dcode, _stream())
            return
        launch(_ptr(vec_c), int(zero_vc))

    def _coarse_distributed(self) -> bool:
        nxt = self.mg.LVL[self.lvl + 1] if self.lvl + 1 < len(self.mg.LVL) else None
        return bool(nxt is not None and nxt.distributed)

    def work_coarse_strip(self):
        blk = self.block
        key = ("coarse_strip", None)
        if key not in self._work:
            self._work[key] = torch.zeros(((self.Ly // blk) * (self.L // blk), self.nc), dtype=self.mg.tdtype, device=self.mg.device)
        return self._work[key]


# ==========================================================================================================
class MG:
    """The LVL[] / NTL[][4] arrays of main() (S6/mgrid_ntl.cpp:38-45) on one GPU."""

    def __init__(self, params: MGParams, device: int | None = None):
        if not torch.cuda.is_available():
            raise MG2DError("2d_multigrid_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.p = params
        self.device_index = torch.cuda.current_device() if device is None else device
        self.device = torch.device("cuda", self.device_index)
        self.ctx = Context(self.device_index)
        self.tdtype, self.dcode = _DT[params.dtype]
        self.status = torch.zeros(4, dtype=torch.int32, device=self.device)
        self.LVL = [Level(self, l) for l in range(params.nlevels + 1)]
        self.NTL = [[Level(self, l) for _ in range(4)] for l in range(params.nlevels + 1)]
        self.info = {}
        self.use_half = False      # complex64 preconditioner copy: smooth with the half-precision operator blocks
        self.premul = True         # red-black sweeps on stored operators use the pre-multiplied blocks -D0^-1 D_k
        self.lowrank = True        # first coarse level: red-black sweeps stream rank-`block` factors of the hopping blocks
        self.lazy_gcr = True       # outer FGCR: raw stored directions + one solution update per restart cycle (mg2d_gcr_step_lazy)
        self.persistent_sites = 8192   # levels with at most this many sites relax all sweeps of a call in one cooperative launch
        self.two_colour = True     # level-0 matrix-free red-black sweeps through the one-pass two-colour kernel
        self.comm = None           # set by dist.DistMG: strip decomposition over torch.distributed (NCCL)
        self.min_rows = 0
        self.graph_launches = 0    # kernels executed through CUDA-graph replays (not seen by ctx.launches)
        self.capture_launches = 0  # launches recorded (not executed) while capturing iteration graphs

    def _ctxs(self):
        """The handles whose launch counters a solve on this hierarchy advances (its own + the complex64 shadow's)."""
        sh = self.info.get("single")
        return [self.ctx] + ([sh.ctx] if isinstance(sh, MG) else [])

    @property
    def launches(self) -> int:
        """Kernels of libmg2d_sm100.so launched so far (eager + replayed from graphs, minus capture-only)."""
        cap = sum(g.nlaunch for g in self.info.values() if isinstance(g, CycleGraph)) + self.capture_launches
        return sum(c.launches for c in self._ctxs()) - cap + self.graph_launches

    def _ntl_fields(self, level: int):
        """The phi of NTL[level][0..3] live in one [4,S,n] buffer so that the Gram matrix is one batched launch."""
        key = ("ntl_phi", level)
        if key not in self.info:
            lv = self.LVL[level]
            buf = lv.new_field(4)
            for q in range(4):
                old = self.NTL[level][q].phi
                if old is not None:
                    buf[q].copy_(old)
                self.NTL[level][q].phi = buf[q]
            self.info[key] = buf
        return self.info[key]

    def close(self):
        """Drop every device buffer and break the Level <-> MG reference cycles so that the memory returns to the
        allocator immediately (hierarchies are tens of GB)."""
        for lv in self.LVL + [nt for row in self.NTL for nt in row]:
            lv.__dict__.update(phi=None, r=None, D=None, D0inv=None, M=None, F=None, _lr_AB=None, Dh=None, D0inv_h=None, phi_null=None, phi_null_c=None,
                               U=None, _U_halos=None, clover=None, _clover_halos=None, _work={}, mg=None)
        for v in list(self.info.values()):
            if isinstance(v, MG):
                v.close()
        self.info.clear()
        self.LVL, self.NTL = [], []

    def to_device(self, a) -> torch.Tensor:
        return torch.as_tensor(np.ascontiguousarray(a)).to(self.tdtype).to(self.device)

    def allreduce(self, t, op: str = "sum"):
        """Global reduction of level-0 partial sums (no-op on one GPU)."""
        self.LVL[0].allreduce(t, op)

    # ---- main() steps ------------------------------------------------------------------------------------
    def init_reference_fields(self):
        """The draws of main() (S6/mgrid_ntl.cpp:38-48) in the reference's order (SURVEY A.2)."""
        gen = StdMT19937(self.p.seed)
        for lv in self.LVL:
            lv.init_level(gen)
        init_NTL(self, gen)
        self.LVL[0].define_source()

    def init_fields(self, generator_seed: int | None = None):
        """Device-side initialisation for lattices too large for the host RNG stream: phi = 0, r = 0 and near-null
        seeds phi_null ~ U(-pi, pi) (f_init_near_null_vector, S6/modules_indiv.h:52-68) from the COUNTER-based generator
        (mg2d_fill_uniform) keyed on (seed, level, GLOBAL element index): a strip draws exactly the numbers the
        single-GPU field holds at the same sites, so the hierarchy does not depend on the partition
        (mirrored by oracle build_device_problem)."""
        seed = self.p.seed if generator_seed is None else generator_seed
        for lv in self.LVL:
            lv.phi, lv.r = lv.new_field(), lv.new_field()
            if lv.lvl != self.p.nlevels:
                lv.phi_null = torch.empty((lv.S, lv.nc, lv.n), dtype=self.tdtype, device=self.device)
                per_site = lv.nc * lv.n
                self.ctx.call("mg2d_fill_uniform", _ptr(lv.phi_null), lv.S * per_site, lv.y0 * lv.L * per_site, seed, lv.lvl,
                              -math.pi, math.pi, self.dcode, _stream())
        if self.p.ntl and self.p.nlevels > 0:       # the copies of f_init_NTL (S6/modules_main.h:7-37), zero instead of random starts
            for lvl in (self.p.nlevels - 1, self.p.nlevels):
                for q in range(self.p.n_copies):
                    self.NTL[lvl][q].phi, self.NTL[lvl][q].r = self.NTL[lvl][q].new_field(), self.NTL[lvl][q].new_field()

    def set_gauge(self, U):
        """U: the full link field [L*L, 2] (each strip keeps its own rows) or already the local rows."""
        lv0 = self.LVL[0]
        U = torch.as_tensor(U)
        if lv0.distributed and U.shape[0] == lv0.L * lv0.L:
            U = U[lv0.y0 * lv0.L:(lv0.y0 + lv0.Ly) * lv0.L]
        U = U.to(self.tdtype).to(self.device).contiguous()
        lv0.compute_lvl0_matrix(U, store=True)

    # ---- moving a built hierarchy to a new gauge field (HMC) -----------------------------------------------
    def _check_updatable(self, what: str):
        p = self.p
        if self.comm is not None:
            raise MG2DError(f"{what}: strip-decomposed hierarchies (DistMG) cannot be updated in place")
        if not p.matrix_free or p.stencil != "wilson":
            raise MG2DError(f"{what}: the level-0 operator is stored (smoother {p.smoother!r}); it needs the matrix-free "
                            "Wilson operator, which reads the links directly")
        if p.csw != 0.0:
            raise MG2DError(f"{what}: the clover field is derived from the links once; csw != 0 is not supported")

    def _drop_graphs(self):
        """Forget every captured graph and the complex64 shadow (closed now: a dead hierarchy collected during a later
        capture would invalidate it)."""
        sh = self.info.pop("single", None)
        if isinstance(sh, MG):
            sh.close()
        for k in [k for k, v in self.info.items() if isinstance(v, CycleGraph) or (isinstance(k, tuple) and k[0] == "iter_graphs")]:
            del self.info[k]

    def update_links(self, U):
        """Copy new links U[L*L, 2] into the level-0 link tensor (and the complex64 shadow's) in place: captured graphs
        stay valid and replay on the new field.  The coarse levels are left as they are; inside FGCR the cycle is only a
        preconditioner, so a stale coarse hierarchy costs iterations, not accuracy (the outer residual uses the new links).
        The first call replaces a link tensor the caller may own (set_gauge keeps the caller's tensor when it can) by a
        copy and drops the graphs captured on it, so the caller's input is never written."""
        self._check_updatable("update_links")
        lv0 = self.LVL[0]
        U = torch.as_tensor(U)
        if tuple(U.shape) != tuple(lv0.U.shape):
            raise ValueError(f"links must have shape {tuple(lv0.U.shape)}")
        if not self.info.get("own_links"):
            lv0.U = lv0.U.clone()
            lv0.bind_link_halos(None)
            self._drop_graphs()
            self.info["own_links"] = True
        lv0.U.copy_(U)
        sh = self.info.get("single")
        if isinstance(sh, MG):
            sh.LVL[0].U.copy_(lv0.U)

    def refresh(self, null_iters: int = 0):
        """Rebuild the coarse hierarchy for the current links: the stored level-0 operator is rebuilt transiently, the current
        near-null vectors are relaxed `null_iters` sweeps on the new operators (in whole chunks of p.null_chunk, at least one,
        as setup does; each vector warm-started from its two chirality rows), re-orthonormalised, and the Galerkin operators, D0^-1, M, F and the compacted projectors are rebuilt.  The
        complex64 shadow and every captured graph are dropped.  null_iters=0 gives exactly what
        setup(U, p, null_vectors=<current vectors>) gives."""
        self._check_updatable("refresh")
        if null_iters < 0:
            raise ValueError("null_iters must be >= 0")
        if self.p.ntl:
            raise MG2DError("refresh: non-telescoping hierarchies are not supported")
        self._drop_graphs()
        for lv in self.LVL:
            lv.Dh = lv.D0inv_h = None
        if self.p.nlevels == 0:
            return
        lv0 = self.LVL[0]
        lv0.compute_lvl0_matrix(lv0.U, store=True)
        if null_iters == 0:
            compute_near_null(self, self.p.quad, gen_null=0)
        else:
            compute_near_null(self, self.p.quad, gen_null=1, null_iters=null_iters, warm=True)


def make_single_precision(mg: "MG") -> "MG":
    """complex64 shadow of a set-up hierarchy (links, clover field, stored operators, projectors), used as the preconditioner
    of the fp64 outer GCR: every V-cycle kernel then moves half the bytes.  The outer residual, the GCR vectors
    and the convergence test stay in complex128, so the 1e-10 TRUE residual is unaffected."""
    import dataclasses
    if mg.p.dtype != "complex128":
        raise ValueError("make_single_precision expects a complex128 hierarchy")
    p32 = dataclasses.replace(mg.p, dtype="complex64", size=[], n_dof=[])
    if mg.comm is not None:
        from .dist import DistMG
        m32 = DistMG(p32, mg.comm, min_rows=mg.min_rows, plan=mg.plan)
    else:
        m32 = MG(p32, mg.device_index)
    c64 = torch.complex64
    for lv, l32 in zip(mg.LVL, m32.LVL):
        l32.phi, l32.r = l32.new_field(), l32.new_field()
        if lv.phi_null_c is not None:
            l32.phi_null_c = lv.phi_null_c.to(c64)      # the cycle only needs the compacted projector
        elif lv.phi_null is not None:
            l32.phi_null = lv.phi_null.to(c64)
        if lv.D is not None:
            l32.D = lv.D.to(c64)
        if lv.lr_rank and mg.lowrank and lv._ensure_F():
            l32.F, l32.lr_rank = lv.F.to(c64), lv.lr_rank
        l32.matrix_free = lv.matrix_free
        if lv.U is not None:
            l32.U = lv.U.to(c64)
            l32.bind_link_halos(None if lv._U_halos is None else tuple(h.to(c64) for h in lv._U_halos))
        if lv.clover is not None:
            l32.clover = lv.clover.to(torch.float32)
            l32.bind_clover_halos(None if lv._clover_halos is None else tuple(h.to(torch.float32) for h in lv._clover_halos))
    return m32


# ---- modules_main.h --------------------------------------------------------------------------------------
def init_NTL(mg: MG, gen: StdMT19937 | None):
    """f_init_NTL (S6/modules_main.h:7-37)."""
    p = mg.p
    if not (p.ntl and p.nlevels > 0):
        return
    draw = (lambda k: gen.uniform_pm_pi(k)) if gen is not None else (lambda k: np.ones(k))
    lo = p.nlevels - 1
    for q in range(p.n_copies):
        lv = mg.NTL[lo][q]
        lv.phi = mg.to_device(draw(lv.S * lv.n).reshape(lv.S, lv.n))
        lv.r = mg.to_device(draw(lv.S * lv.n).reshape(lv.S, lv.n))
        lv.phi_null = mg.to_device(draw(lv.S * lv.nc * lv.n).reshape(lv.S, lv.nc, lv.n))
    for q in range(p.n_copies):
        lv = mg.NTL[p.nlevels][q]
        lv.phi = mg.to_device(draw(lv.S * lv.n).reshape(lv.S, lv.n))
        lv.r = mg.to_device(draw(lv.S * lv.n).reshape(lv.S, lv.n))


def compute_coarse_matrix(lvl_c: Level, lvl_f: Level, lvl_P: Level, quad: int):
    """f_compute_coarse_matrix (S6/modules_main.h:81-185): lvl_c.D = P D_f P^dagger with P = lvl_P.phi_null."""
    mg = lvl_f.mg
    nf, nc = lvl_f.n, lvl_P.nc
    if lvl_f.D is None:
        raise MG2DError("compute_coarse_matrix needs the stored fine operator")
    lvl_c.D = torch.empty((lvl_c.S, 5, nc, nc), dtype=mg.tdtype, device=mg.device)
    lvl_c.D0inv = None
    lvl_c.M = None
    lvl_c.F, lvl_c._lr_AB, lvl_c.lr_rank = None, None, 0
    P = lvl_P.phi_null
    p_lo, p_hi = lvl_f._halo(P, 1, nc * nf)          # projector rows below / above the strip (or the periodic wrap)
    if (mg.lowrank and nf <= 2 and quad == 1 and lvl_P is lvl_f and lvl_c.Ly * lvl_f.block == lvl_f.Ly
            and 2 * lvl_f.block < nc and mg.ctx.lib.mg2d_lowrank_supported(nc, lvl_f.block)):
        lvl_c.hop_factors(lvl_f, P, p_lo, p_hi)
        # (read now, not at the end of the setup: the next level's near-null relaxation already runs on the factors)
        if mg.comm is not None:
            mg.comm.allreduce(mg.status, "max")
        if int(mg.status[1].item()) != 0:      # a fine hopping block that is not rank one: keep the dense blocks
            lvl_c.F, lvl_c._lr_AB, lvl_c.lr_rank = None, None, 0
            mg.status[1] = 0
    if lvl_f.distributed and not lvl_c.distributed:
        # first replicated level: every rank builds its strip of D_c, then the strips are all-gathered
        blk = lvl_f.block
        strip = torch.empty(((lvl_f.Ly // blk) * (lvl_f.L // blk), 5, nc, nc), dtype=mg.tdtype, device=mg.device)
        mg.ctx.call("mg2d_coarse_matrix", _ptr(strip), _ptr(lvl_f.D), _ptr(P), p_lo, p_hi, nf, nc, lvl_f.L, lvl_f.Ly,
                    blk, quad, mg.dcode, _stream())
        mg.comm.allgather(lvl_c.D, strip)
        return
    mg.ctx.call("mg2d_coarse_matrix", _ptr(lvl_c.D), _ptr(lvl_f.D), _ptr(P), p_lo, p_hi, nf, nc, lvl_f.L, lvl_f.Ly,
                lvl_f.block, quad, mg.dcode, _stream())


def compute_near_null(mg: MG, quad: int | None = None, gen_null: int = 1, null_iters: int | None = None, warm: bool = False):
    """f_compute_near_null (S6/modules_main.h:187-222).  gen_null=0: phi_null rows are already supplied.  null_iters / warm:
    the relaxation sweeps and start of Level.near_null (default p.null_iters from the rows of phi_null as drawn)."""
    p = mg.p
    quad = p.quad if quad is None else quad
    worst = []
    marks = []          # CUDA events around the phases of every level (resolved below, after the status read has synchronised)

    def mark():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e
    for lvl in range(p.nlevels):
        lv = mg.LVL[lvl]
        m = [mark()]
        if gen_null == 1:
            lv.near_null(null_iters, warm)
        m.append(mark())
        lv.norm_nn(quad)
        lv.ortho(quad)
        lv.ortho(quad)
        worst.append(lv.check_ortho(quad))
        m.append(mark())
        compute_coarse_matrix(mg.LVL[lvl + 1], lv, lv, quad)
        m.append(mark())
        marks.append(m)
    if p.ntl:
        lo = p.nlevels - 1
        for q in range(p.n_copies):
            nt = mg.NTL[lo][q]
            nt.phi_null = mg.LVL[lo].phi_null.clone()
            nt.norm_nn(quad)
            nt.ortho(q + 1)
            nt.ortho(q + 1)
            worst.append(nt.check_ortho(q + 1))
            compute_coarse_matrix(mg.NTL[p.nlevels][q], mg.LVL[lo], nt, q + 1)
    if mg.comm is not None:
        mg.comm.allreduce(mg.status, "max")
    st = mg.status.cpu()
    if int(st[1]) != 0:       # a fine hopping block that is not rank one: keep the dense blocks
        for lv in mg.LVL:
            lv.F, lv._lr_AB, lv.lr_rank = None, None, 0
        mg.status[1] = 0
    for lv in mg.LVL:
        if lv.lr_rank and lv.M is not None and lv._ensure_F():
            lv.M = None       # the dense pre-multiplied blocks were only needed by the batched near-null relaxation
    if int(st[0]) != 0:
        raise FloatingPointError(f"near-null orthonormalisation failed (status {int(st[0])}): NaN or tiny norm "
                                 "(S6/modules_indiv.h:119-126, S6/near_null.h:149-159)")
    mg.info["ortho_worst"] = worst
    torch.cuda.synchronize()
    mg.info["setup_phases"] = [{"level": l, "sites": mg.LVL[l].S, "near_null_ms": m[0].elapsed_time(m[1]),
                                "ortho_ms": m[1].elapsed_time(m[2]), "coarse_matrix_ms": m[2].elapsed_time(m[3])}
                               for l, m in enumerate(marks)]
    if p.stencil == "wilson" and p.chiral_transfer:
        for lvl in range(p.nlevels):
            mg.LVL[lvl].compact_projector(check=(gen_null != 1))
    if p.matrix_free:   # the stored level-0 operator was only needed for the Galerkin product
        mg.LVL[0].D = None
        mg.LVL[0].D0inv = None
        mg.LVL[0].M = None
        mg.LVL[0].matrix_free = True


def restriction_res(res_c, L_residue: Level, L_restrict: Level, quad: int):
    """f_restriction_res (S6/modules_main.h:224-241): res_c = P (r - D phi)."""
    rtemp = L_residue.work("rtemp")
    L_residue.residue(rtemp)
    L_restrict.restriction(res_c, rtemp, quad)


def prolongate_phi(phi_f, phi_c, LVLP: Level, quad: int, accumulate: bool = True):
    """f_prolongate_phi (S6/modules_main.h:243-252): phi_f += P^dagger phi_c ; phi_c = 0."""
    LVLP.prolongation(phi_f, phi_c, quad, zero_vc=True, accumulate=accumulate)


def MG_simple(mg: MG, zero_start: bool = False):
    """f_MG_simple (S6/modules_main.h:255-280).  p.pre / p.post give the sweeps per level (the reference uses one
    count everywhere).  zero_start: the caller guarantees phi = 0 on every level at entry (preconditioner use);
    a level without pre-smoothing then restricts r directly, since r - D*0 = r exactly."""
    p, LVL = mg.p, mg.LVL
    if p.nlevels > 0:
        for lvl in range(p.nlevels):
            LVL[lvl].relax(p.pre[lvl])
            if zero_start and p.pre[lvl] == 0:
                LVL[lvl].restriction(LVL[lvl + 1].r, LVL[lvl].r, p.quad)
            else:
                restriction_res(LVL[lvl + 1].r, LVL[lvl], LVL[lvl], p.quad)
        for lvl in range(p.nlevels, -1, -1):
            LVL[lvl].relax(p.post[lvl])
            if lvl > 0:
                # phi of the finer level is still exactly zero when it was not pre-smoothed: overwrite, do not add
                fresh = zero_start and p.pre[lvl - 1] == 0 and LVL[lvl - 1].phi_null_c is not None
                prolongate_phi(LVL[lvl - 1].phi, LVL[lvl].phi, LVL[lvl - 1], p.quad, accumulate=not fresh)
    else:
        LVL[0].relax(p.post[0])


def _coarse_gcr(mg: MG, lvl: int):
    """K-cycle coarse solve (ours; SURVEY 8f N3): p.k_inner steps of flexible GCR on D_lvl phi = r_lvl from phi = 0, each
    preconditioned by the K-cycle of this level (recursion).  A fixed number of steps: no residual test, no host sync.
    Mirrors oracle _coarse_gcr."""
    p = mg.p
    lv = mg.LVL[lvl]
    vs = lv.S * lv.n
    kin = p.k_inner
    call, dc, st = mg.ctx.call, mg.dcode, _stream
    x, Z, W, sc = lv.work("k_x"), lv.work("k_Z", kin), lv.work("k_W", kin), lv.dots("kcyc")
    call("mg2d_zero", _ptr(x), vs, dc, st())
    keep = lv.phi
    for j in range(kin):
        z, w = Z[j], W[j]
        call("mg2d_zero", _ptr(z), vs, dc, st())
        lv.phi = z                       # the cycle writes its result in place; lv.r is the current residual
        try:
            MG_kcycle(mg, lvl)
        finally:
            lv.phi = keep
        lv._stencil(w, z, None, _lib.MODE_APPLY, None)
        if j > 0:
            with lv.global_sums(sc[16:16 + 2 * j]):
                call("mg2d_gcr_dots", _ptr(W), vs, j, _ptr(w), vs, dc, _ptr(sc[16:]), st())
        with lv.global_sums(sc[0:4]):
            call("mg2d_gcr_ortho", _ptr(w), _ptr(z), _ptr(lv.r), _ptr(W), _ptr(Z), vs, j, _ptr(sc[16:]), _ptr(sc[40:]), vs, dc,
                 _ptr(sc[0:]), st())
        with lv.global_sums(sc[4:5]):
            call("mg2d_gcr_step", _ptr(x), _ptr(lv.r), _ptr(z), _ptr(w), _ptr(sc[0:]), _ptr(sc[40 + j:]), vs, dc, _ptr(sc[4:]), st())
    call("mg2d_copy", _ptr(lv.phi), _ptr(x), vs, dc, st())


def MG_kcycle(mg: MG, lvl: int = 0, zero_start: bool = False):
    """One K-cycle on level `lvl` (acts on LVL[lvl].phi / .r like f_MG_simple's body, S6/modules_main.h:255-280): pre-smooth,
    restrict the residual, solve the coarse system with p.k_inner Krylov (FGCR) steps preconditioned by the K-cycle of the next
    level instead of ONE recursive visit, prolong, post-smooth.  The coarsest level is only relaxed, as in the reference."""
    p, LVL = mg.p, mg.LVL
    lv = LVL[lvl]
    if lvl == p.nlevels:
        lv.relax(p.post[lvl])
        return
    lv.relax(p.pre[lvl])
    if zero_start and p.pre[lvl] == 0:
        lv.restriction(LVL[lvl + 1].r, lv.r, p.quad)
    else:
        restriction_res(LVL[lvl + 1].r, lv, lv, p.quad)
    if lvl + 1 == p.nlevels:
        MG_kcycle(mg, lvl + 1)              # bottom: smoothing only, no Krylov wrapper around a stationary smoother
    else:
        _coarse_gcr(mg, lvl + 1)
    prolongate_phi(lv.phi, LVL[lvl + 1].phi, lv, p.quad)
    lv.relax(p.post[lvl])


def cycle_once(mg: MG, zero_start: bool = False):
    """One multigrid cycle of the configured kind on (LVL[0].phi, LVL[0].r): f_MG_ntl, f_MG_simple (V) or the K-cycle.
    Returns the NTL weights tensor (or None)."""
    p = mg.p
    if p.ntl and p.nlevels > 0:
        return MG_ntl(mg)
    if p.cycle == "K" and p.nlevels > 0:
        MG_kcycle(mg, 0, zero_start)
    else:
        MG_simple(mg, zero_start)
    return None


def min_res(mg: MG, num_copies: int, level: int) -> torch.Tensor:
    """f_min_res (S6/modules_main.h:283-373): weights a_q (device tensor, 2*num_copies doubles)."""
    p = mg.p
    lv = mg.LVL[level]
    E = mg._ntl_fields(level)           # [4, S, n] contiguous views of NTL[level][q].phi
    T = lv.work("minres_t", 4)
    for q in range(num_copies):
        lv.apply_D(T[q], E[q])
    vs = lv.S * lv.n
    buf = lv.dots("minres")
    gram, src, a = buf[0:32], buf[32:40], buf[40:48]
    mg.ctx.call("mg2d_cdot_batch", _ptr(E), vs, num_copies, _ptr(T), vs, num_copies, vs, mg.dcode, _ptr(gram), _stream())
    if p.stencil == "laplace":   # src_i = <e_i, r>   (:336-340)
        mg.ctx.call("mg2d_cdot_batch", _ptr(E), vs, num_copies, _ptr(lv.r), vs, 1, vs, mg.dcode, _ptr(src), _stream())
    else:                        # src_i = <r, D e_i> (:358-366)
        mg.ctx.call("mg2d_cdot_batch", _ptr(lv.r), vs, 1, _ptr(T), vs, num_copies, vs, mg.dcode, _ptr(src), _stream())
    lv.allreduce(buf[0:40])
    mg.ctx.call("mg2d_minres_solve", _ptr(gram), _ptr(src), num_copies, _ptr(a), _stream())
    return a


def scale_phi(mg: MG, L1: Level, a, num_copies: int, lvl: int):
    """f_scale_phi (S6/modules_main.h:375-384)."""
    E = mg._ntl_fields(lvl)
    vs = L1.S * L1.n
    mg.ctx.call("mg2d_scale_phi", _ptr(L1.phi), _ptr(E), vs, _ptr(a), num_copies, vs, mg.dcode, _stream())


def MG_ntl(mg: MG):
    """f_MG_ntl (S6/modules_main.h:386-439).  Returns the device tensor of the 4 complex copy weights."""
    p, LVL, NTL = mg.p, mg.LVL, mg.NTL
    a = None
    for lvl in range(p.nlevels):
        LVL[lvl].relax(p.pre[lvl])
        if lvl != p.nlevels - 1:
            restriction_res(LVL[lvl + 1].r, LVL[lvl], LVL[lvl], p.quad)
        else:
            rtemp = LVL[lvl].work("rtemp")
            LVL[lvl].residue(rtemp)
            for q in range(p.n_copies):
                NTL[lvl][q].restriction(NTL[lvl + 1][q].r, rtemp, q + 1)
    for lvl in range(p.nlevels, -1, -1):
        if lvl == p.nlevels:
            mg._ntl_fields(lvl - 1)
            for q in range(p.n_copies):
                NTL[lvl][q].relax(p.post[lvl])
                prolongate_phi(NTL[lvl - 1][q].phi, NTL[lvl][q].phi, NTL[lvl - 1][q], q + 1)
            if p.min_res_flag == 1:
                a = min_res(mg, p.n_copies, lvl - 1)
            else:
                a = LVL[lvl - 1].dots("minres")[40:48]
                a.zero_()
                a[0:2 * p.n_copies:2] = 1.0 / p.n_copies
            scale_phi(mg, LVL[lvl - 1], a, p.n_copies, lvl - 1)
        else:
            LVL[lvl].relax(p.post[lvl])
            if lvl > 0:
                prolongate_phi(LVL[lvl - 1].phi, LVL[lvl].phi, LVL[lvl - 1], p.quad)
    return a


class CycleGraph:
    """One multigrid cycle (f_MG_simple / f_MG_ntl) + the fused residual norm, captured into a CUDA graph so
    that a cycle costs one launch on the host.  Smoothers 'gs' (cooperative wavefront kernel) stay eager."""

    def __init__(self, mg: MG, with_resmag: bool = True, zero_start: bool = False):
        self.mg = mg
        self.zero_start = zero_start
        self.ntl = mg.p.ntl and mg.p.nlevels > 0
        self.with_resmag = with_resmag
        self.graph = None
        self.weights = None
        self.nlaunch = 0
        self.ptrs = None
        self.enabled = mg.p.smoother != "gs"

    def _body(self):
        mg = self.mg
        w = cycle_once(mg, self.zero_start)
        if self.ntl:
            self.weights = w
        if self.with_resmag:
            mg.LVL[0].residue_mag_async()

    def run(self):
        if not self.enabled:
            self._body()
            return
        ptrs = tuple((lv.phi.data_ptr(), lv.r.data_ptr()) for lv in self.mg.LVL)
        if self.graph is not None and ptrs != self.ptrs:
            self.graph = None          # a caller rebound phi / r of a level: the captured pointers are stale, capture again
        if self.graph is None:
            # warm-up on a side stream (allocates every lazily created work buffer), then capture
            mg = self.mg
            self.ptrs = ptrs
            saved = [(lv, lv.phi.clone(), lv.r.clone()) for lv in mg.LVL]
            saved += [(nt, nt.phi.clone(), nt.r.clone()) for row in mg.NTL for nt in row if nt.phi is not None and nt.r is not None]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                self._body()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            for lv, ph, r in saved:
                lv.phi.copy_(ph); lv.r.copy_(r)
            self.graph = torch.cuda.CUDAGraph()
            n0 = mg.ctx.launches
            with _capture(self.graph):
                self._body()
            self.nlaunch = mg.ctx.launches - n0
            for lv, ph, r in saved:      # capture does not execute, but keep the state explicit
                lv.phi.copy_(ph); lv.r.copy_(r)
        self.graph.replay()
        self.mg.graph_launches += self.nlaunch


def perform_MG(mg: MG, tol: float | None = None, max_iters: int | None = None, check_every: int = 1,
               record_phi: bool = False, use_graph: bool = False, on_iteration=None):
    """f_perform_MG; see _perform_MG.  On strips a peer time-out during the solve raises instead of returning fields
    computed from stale halo rows."""
    info = _perform_MG(mg, tol, max_iters, check_every, record_phi, use_graph, on_iteration)
    if mg.comm is not None:
        mg.comm.check_errors()
    return info


def _perform_MG(mg: MG, tol: float | None = None, max_iters: int | None = None, check_every: int = 1,
                record_phi: bool = False, use_graph: bool = False, on_iteration=None):
    """f_perform_MG (S6/modules_main.h:442-481): cycles until |r - D phi|/|r| < tol; diverged if > 1e6.
    The residual norms are produced on the device by the fused residual kernel; the host reads them every
    `check_every` cycles (1 = the reference's behaviour)."""
    p = mg.p
    tol = p.tol if tol is None else tol
    max_iters = p.max_iters if max_iters is None else max_iters
    info = {"iters": 0, "resnorms": [], "ntl_weights": [], "converged": False, "diverged": False, "phi_hist": []}
    hist = torch.zeros((max(check_every, 1), 4), dtype=torch.float64, device=mg.device)
    whist = torch.zeros((max(check_every, 1), 8), dtype=torch.float64, device=mg.device)
    ntl = p.ntl and p.nlevels > 0
    cyc = None
    if use_graph:
        cyc = mg.info.get("cycle_graph")
        if cyc is None:
            cyc = mg.info["cycle_graph"] = CycleGraph(mg)
    it = 0
    while it < max_iters:
        nb = min(check_every, max_iters - it)
        for k in range(nb):
            if record_phi:
                info["phi_hist"].append(mg.LVL[0].phi.clone())
            if on_iteration is not None:
                on_iteration(it + k, mg)          # the reference's per-iteration writers (S6/modules_main.h:446-458)
            if cyc is not None:
                cyc.run()
                if ntl:
                    whist[k].copy_(cyc.weights[:8])
                hist[k].copy_(mg.LVL[0].dots("resmag")[:4])
                continue
            a = cycle_once(mg)
            if ntl:
                whist[k].copy_(a[:8])
            d = mg.LVL[0].residue_mag_async()
            hist[k].copy_(d[:4])
        h = hist[:nb].cpu()
        wh = whist[:nb].cpu() if ntl else None
        for k in range(nb):
            resmag = math.sqrt(h[k, 0].item()) / math.sqrt(h[k, 3].item()) if h[k, 3].item() > 0 else float("nan")
            info["resnorms"].append(resmag)
            if ntl:
                w = wh[k].numpy()
                info["ntl_weights"].append(w[0::2] + 1j * w[1::2])
            info["iters"] = it + k + 1
            if resmag < tol:
                info["converged"] = True
                return info
            if resmag > 1e6 or math.isnan(resmag):
                info["diverged"] = True
                return info
        it += nb
    return info


class IterGraph:
    """One whole outer iteration (cycle + operator apply + the three fused GCR passes, every reduction on the device)
    captured into a CUDA graph: one host launch per iteration.  There is one graph per number of stored directions
    (`slot`), because the stored vectors the iteration reads and the buffers it writes depend on it."""

    def __init__(self, body, state):
        self.body, self.state, self.graph, self.nlaunch = body, state, None, 0

    def run(self, mg: "MG", slot: int):
        if self.graph is None:
            saved = [t.clone() for t in self.state]
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):          # warm-up: allocates every lazily created work buffer
                self.body(slot)
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            for t, c in zip(self.state, saved):
                t.copy_(c)
            self.graph = torch.cuda.CUDAGraph()
            n0 = sum(c.launches for c in mg._ctxs())
            with _capture(self.graph):
                self.body(slot)
            self.nlaunch = sum(c.launches for c in mg._ctxs()) - n0
            for t, c in zip(self.state, saved):
                t.copy_(c)
            mg.capture_launches += self.nlaunch
        self.graph.replay()
        mg.graph_launches += self.nlaunch


def gcr_MG(mg: MG, tol: float | None = None, max_iters: int | None = None, restart: int = 8, check_every: int = 1,
           use_graph: bool = False, precond: "MG | None" = None):
    """Flexible GCR(restart) around one multigrid cycle as preconditioner (mirrors oracle gcr_MG; the reference
    itself only iterates the cycle stationarily).  On entry LVL[0].phi / LVL[0].r hold x0 / b; on exit the
    solution is in LVL[0].phi.  All scalars (Gram-Schmidt coefficients, step lengths, residual norms; on strips their
    sums over the ranks) stay on the device; the host reads |r|^2 after every `check_every` iterations (1: no cycle is
    executed past convergence).  use_graph: each iteration is ONE graph launch (IterGraph)."""
    p = mg.p
    tol = p.tol if tol is None else tol
    max_iters = p.max_iters if max_iters is None else max_iters
    if restart > 8 or restart < 1:
        raise ValueError("1 <= restart <= 8 (mg2d_gcr_dots / mg2d_gcr_ortho handle up to 8 stored directions)")
    check_every = max(1, min(check_every, restart))
    lv0 = mg.LVL[0]
    vs = lv0.S * lv0.n
    call, dc, st = mg.ctx.call, mg.dcode, _stream
    x, b = lv0.work("gcr_x"), lv0.work("gcr_b")
    r = lv0.work("gcr_r")
    # stored directions `stride` elements apart (MG2D_GCR_PAD: a 4096^2 field is exactly 2^29 bytes and up to 10 such streams are
    # read at the same offset at the same time; padding the stride was measured to make no difference on B200)
    stride = vs + GCR_PAD
    Zb, Wb = lv0.flat_work(("gcr_Z", restart, GCR_PAD), restart * stride), lv0.flat_work(("gcr_W", restart, GCR_PAD), restart * stride)
    Z = [Zb[j * stride:j * stride + vs].view(lv0.S, lv0.n) for j in range(restart)]
    W = [Wb[j * stride:j * stride + vs].view(lv0.S, lv0.n) for j in range(restart)]
    lazy = bool(mg.lazy_gcr)
    coef = lv0.dots("gcr_coef")     # lazy update: coefficients of the orthogonalised directions in the raw z_i (mg2d_gcr_step_lazy)
    sc = lv0.dots("gcr")            # [0:4] |w|^2,<w,r> ; [4] |r|^2 ; [5] |b|^2 ; [16:32] <W_j,w> ; [40+j] |w_j|^2 ; [48+j] |r|^2 after slot j
    call("mg2d_copy", _ptr(x), _ptr(lv0.phi), vs, dc, st())
    call("mg2d_copy", _ptr(b), _ptr(lv0.r), vs, dc, st())
    lv0._stencil(r, x, b, _lib.MODE_RESID, None)
    with lv0.global_sums(sc[5:6]):
        call("mg2d_norm2", _ptr(b), vs, dc, _ptr(sc[5:]), st())
    pm = mg if precond is None else precond      # hierarchy that runs the cycle (may be the complex64 shadow)
    pl0 = pm.LVL[0]
    for lv in pm.LVL[1:]:
        pm.ctx.call("mg2d_zero", _ptr(lv.phi), lv.S * lv.n, pm.dcode, st())
    ntl = p.ntl and p.nlevels > 0
    fresh_top = p.nlevels > 0 and pm.p.pre[0] == 0 and pl0.phi_null_c is not None and not ntl
    alias = pm is mg and not ntl     # the cycle reads the GCR residual as its right-hand side and writes z in place

    def body(slot):
        z, w = Z[slot], W[slot]
        # z = M(r): one cycle from phi = 0 on the preconditioner hierarchy
        if alias:
            keep = (pl0.phi, pl0.r)
            pl0.phi, pl0.r = z, r
        else:
            pm.ctx.call("mg2d_convert", _ptr(pl0.r), pm.dcode, _ptr(r), dc, vs, st())
        try:
            if not fresh_top:      # (with no pre-smoothing the first write to phi is the overwriting prolongation)
                pm.ctx.call("mg2d_zero", _ptr(pl0.phi), vs, pm.dcode, st())
            cycle_once(pm, zero_start=True)
        finally:
            if alias:
                pl0.phi, pl0.r = keep
        if not alias:
            pm.ctx.call("mg2d_convert", _ptr(z), dc, _ptr(pl0.phi), pm.dcode, vs, st())
        lv0._stencil(w, z, None, _lib.MODE_APPLY, None)
        # classical Gram-Schmidt against the stored directions, then the minimal-residual step (3 fused passes)
        if slot > 0:
            with lv0.global_sums(sc[16:16 + 2 * slot]):
                call("mg2d_gcr_dots", _ptr(Wb), stride, slot, _ptr(w), vs, dc, _ptr(sc[16:]), st())
        if lazy:
            # the z_i stay raw and x is updated once per restart cycle: (2j+9) instead of (3j+14) vector passes
            with lv0.global_sums(sc[0:4]):
                call("mg2d_gcr_ortho", _ptr(w), None, _ptr(r), _ptr(Wb), None, stride, slot, _ptr(sc[16:]), _ptr(sc[40:]),
                     vs, dc, _ptr(sc[0:]), st())
            with lv0.global_sums(sc[48 + slot:49 + slot]):
                call("mg2d_gcr_step_lazy", _ptr(r), _ptr(w), _ptr(sc[0:]), _ptr(sc[40 + slot:]), _ptr(sc[16:]), _ptr(sc[40:]), slot,
                     _ptr(coef), vs, dc, _ptr(sc[48 + slot:]), st())
            if slot == restart - 1:
                call("mg2d_gcr_xupdate", _ptr(x), _ptr(Zb), stride, restart, _ptr(coef), vs, dc, st())
            return
        with lv0.global_sums(sc[0:4]):
            call("mg2d_gcr_ortho", _ptr(w), _ptr(z), _ptr(r), _ptr(Wb), _ptr(Zb), stride, slot, _ptr(sc[16:]), _ptr(sc[40:]),
                 vs, dc, _ptr(sc[0:]), st())
        with lv0.global_sums(sc[48 + slot:49 + slot]):
            call("mg2d_gcr_step", _ptr(x), _ptr(r), _ptr(z), _ptr(w), _ptr(sc[0:]), _ptr(sc[40 + slot:]), vs, dc,
                 _ptr(sc[48 + slot:]), st())

    graphs = None
    if use_graph and pm.p.smoother != "gs":
        gkey = ("iter_graphs", id(pm), lazy, pm.use_half, pm.lowrank, pm.premul, pm.persistent_sites, restart, tuple(pm.p.pre), tuple(pm.p.post))
        graphs = mg.info.setdefault(gkey, {})
    info = {"iters": 0, "resnorms": [], "ntl_weights": [], "converged": False, "diverged": False}
    bn2 = None
    it, slot, pending = 0, 0, 0
    done = False
    while it < max_iters and not done:
        nb = min(check_every, max_iters - it, restart - slot)
        slots = []
        for k in range(nb):
            if graphs is not None:
                g = graphs.get(slot)
                if g is None:
                    g = graphs[slot] = IterGraph(body, [x, r, sc, coef])
                g.run(mg, slot)
            else:
                body(slot)
            slots.append(slot)
            slot = (slot + 1) % restart
            pending = slot          # iterations whose contribution to x is still held in `coef` (flushed when the cycle wraps)
        h = sc[48:56].cpu()
        if bn2 is None:
            bn2 = float(sc[5].item())
        for k, sl in enumerate(slots):
            resmag = math.sqrt(h[sl].item()) / math.sqrt(bn2) if bn2 > 0 else float("nan")
            info["resnorms"].append(resmag)
            info["iters"] = it + k + 1
            if resmag < tol:
                info["converged"] = True; done = True; break
            if resmag > 1e6 or math.isnan(resmag):
                info["diverged"] = True; done = True; break
        it += nb
    info["executed_iters"] = it
    if lazy and pending > 0:
        call("mg2d_gcr_xupdate", _ptr(x), _ptr(Zb), stride, pending, _ptr(coef), vs, dc, st())
    call("mg2d_copy", _ptr(lv0.phi), _ptr(x), vs, dc, st())
    call("mg2d_copy", _ptr(lv0.r), _ptr(b), vs, dc, st())
    info["true_resnorm"] = lv0.get_residue_mag()
    if mg.comm is not None:
        mg.comm.check_errors()
    return info
