"""2d_multigrid_b200 -- B200-native (sm_100a) solver hot path of vmos1/2d_multigrid.

Public API (SURVEY.md section 8b; argument order follows the reference functions, S6 = code/6_ntl-mg_new_code/
3_combining_laplace_and_wilson/).  Arrays are torch CUDA tensors (complex128 or complex64):

    p  = make_params(L, mass, stencil='wilson', nlevels=2, block=2, n_null=2, n_smooth=3, smoother='gs', ...)
         # csw=1.0: Wilson-clover level 0, self block (2+m) 1 + f(s) sigma3 with f(s) = (csw/8) sum of Im U_P over the four
         # plaquettes at s (stored and matrix-free paths, every smoother; the coarse levels inherit it through the Galerkin product)
         # mu=1e-3: twisted mass, + i mu gamma5 (gamma5 = sigma3) on the level-0 self block, with or without clover; D^dag D gains
         # mu^2, so the solve stays well posed at m = m_crit (estimate m_crit with critical.estimate_critical_mass at mu = 0).
         # The coarse levels inherit i mu Gamma5_c through the Galerkin product of the chirality-split projector
    mg = setup(U, p, null_vectors=None)          # f_compute_lvl0_matrix + f_compute_near_null
    x, info = solve(mg, rhs, x0=None, tol=1e-10) # f_perform_MG
    apply_D(v_out, v_in, level, mg)              # Level::f_apply_D        S6/level.h:251-265
    residue(r_out, level, mg)                    # Level::f_residue        S6/level.h:61-77
    residue_mag(level, mg) -> float              # Level::f_get_residue_mag S6/level.h:79-98
    relax(level, num_iter, mg, gs_flag)          # Level::f_relax          S6/level.h:100-128
    restriction(vec_c, vec_f, level, mg, quad)   # Near_null::f_restriction S6/near_null.h:217-240
    prolongation(vec_f, vec_c, level, mg, quad)  # Near_null::f_prolongation S6/near_null.h:242-264 (level = coarse)
    near_null(level, mg) / norm_nn(level, quad, mg) / ortho(level, quad, mg) / compute_coarse_matrix(level, quad, mg)

Gauge-field updates and HMC (matrix-free complex128 Wilson hierarchies on one GPU, csw = 0):

    mg.update_links(U)                           # new links copied into the hierarchy in place; captured graphs replay on them
    mg.refresh(null_iters=0)                     # coarse hierarchy rebuilt for the current links from the current near-null
                                                 # vectors (relaxed null_iters sweeps first); 0 = setup(U, p, null_vectors=...)
    h = HMC(p, theta, beta, tau=1.0, n_md=10, flavours=2, seed=1, md_tol=1e-10, accept_tol=1e-12,
            refresh_null_iters=8, precond_dtype=None, use_graph=True)
    h.trajectory() -> dict(dH, accepted, plaquette, iters_md, iters_accept, times_ms, ...)
                                                 # two-flavour Wilson HMC (leapfrog), fermion force from two multigrid solves;
                                                 # flavours=0 is pure-gauge HMC; h.theta holds the phases

The compute path is libmg2d_sm100.so (C ABI in include/mg2d.h) and nothing else: importing this package on a
machine without the library is allowed (so that host logic can be tested), but creating an MG raises.
"""
from __future__ import annotations

import torch

from . import _lib, diagnostics, gauge, mg as _mg, refio
from ._lib import MG2DError, Context
from .mg import MG, Level, D_to_reference_layout, MG_simple, MG_ntl, perform_MG, compute_near_null, init_NTL
from .params import MGParams, make_params, from_argv
from .rng import StdMT19937
from .scalar import ScalarMG, solve_scalar, solve_scalar_s1
from .hmc import HMC

__all__ = ["make_params", "from_argv", "MGParams", "MG", "Level", "setup", "solve", "apply_D", "residue",
           "residue_mag", "relax", "restriction", "prolongation", "near_null", "norm_nn", "ortho",
           "compute_coarse_matrix", "run_reference_flow", "ScalarMG", "solve_scalar", "solve_scalar_s1", "gauge", "refio", "diagnostics", "MG2DError", "D_to_reference_layout", "HMC"]


def apply_D(v_out, v_in, level: int, mg: MG):
    mg.LVL[level].apply_D(v_out, v_in)


def residue(r_out, level: int, mg: MG):
    mg.LVL[level].residue(r_out)


def residue_mag(level: int, mg: MG) -> float:
    return mg.LVL[level].get_residue_mag()


def relax(level: int, num_iter: int, mg: MG, gs_flag: int | None = None):
    mg.LVL[level].relax(num_iter, gs_flag)


def restriction(vec_c, vec_f, level: int, mg: MG, quad: int = 1):
    mg.LVL[level].restriction(vec_c, vec_f, quad)


def prolongation(vec_f, vec_c, level: int, mg: MG, quad: int = 1):
    """level = COARSE level index, as in the reference (uses phi_null of level-1)."""
    mg.LVL[level - 1].prolongation(vec_f, vec_c, quad)


def near_null(level: int, mg: MG):
    mg.LVL[level].near_null()


def norm_nn(level: int, quad: int, mg: MG):
    mg.LVL[level].norm_nn(quad)


def ortho(level: int, quad: int, mg: MG):
    mg.LVL[level].ortho(quad)


def compute_coarse_matrix(level: int, quad: int, mg: MG):
    """D[level+1] = P D[level] P^dagger."""
    _mg.compute_coarse_matrix(mg.LVL[level + 1], mg.LVL[level], mg.LVL[level], quad)


def setup(U, params: MGParams, null_vectors=None, init: str = "reference", device: int | None = None) -> MG:
    """Build the multigrid hierarchy for links U[L*L,2]: level-0 operator, near-null vectors (generated by
    relaxation, or supplied as a list of phi_null[L_l^2, nc, nf] tensors), per-aggregate orthonormalisation
    and the Galerkin coarse operators (f_compute_near_null, S6/modules_main.h:187-222).

    init='reference' draws phi / r / phi_null exactly as main() does (bit-identical std::mt19937 stream);
    init='device' starts from phi = 0 and torch-generated random null-vector seeds (large lattices)."""
    mg = MG(params, device)
    if init == "reference":
        mg.init_reference_fields()
    elif init == "device":
        mg.init_fields()
    else:
        raise ValueError("init must be 'reference' or 'device'")
    mg.set_gauge(U)
    gen_null = 1
    if null_vectors is not None:
        if len(null_vectors) != params.nlevels:
            raise ValueError("null_vectors needs one tensor per fine level")
        for lv, P in zip(mg.LVL, null_vectors):
            P = torch.as_tensor(P).to(mg.tdtype).to(mg.device).contiguous()
            if tuple(P.shape) != (lv.S, lv.nc, lv.n):
                raise ValueError(f"null vectors of level {lv.lvl} must have shape {(lv.S, lv.nc, lv.n)}")
            lv.phi_null = P.clone()
        gen_null = 0
    if params.nlevels > 0:
        compute_near_null(mg, params.quad, gen_null)
    elif params.matrix_free:
        mg.LVL[0].D = None
        mg.LVL[0].matrix_free = True
    return mg


def solve(mg: MG, rhs=None, x0=None, tol: float | None = None, max_iters: int | None = None, check_every: int = 1,
          record_phi: bool = False, outer: str = "stationary", restart: int = 8, use_graph: bool = False,
          precond_dtype: str | None = None):
    """f_perform_MG (S6/modules_main.h:442-481).  rhs / x0 None keep the fields already in LVL[0] (the
    reference's random start); otherwise they are copied in and every coarse phi is cleared.
    outer='stationary' iterates the cycle as the reference does; outer='gcr' wraps it as the preconditioner of
    a flexible GCR(restart); precond_dtype='complex64' runs that preconditioner cycle on a complex64 copy of the
    hierarchy (half the HBM traffic) while residuals and the convergence test stay complex128; 'complex64+half'
    additionally stores the coarse operators of that copy in half precision for the red-black smoother.  use_graph replays the cycle from a CUDA graph (one host launch per cycle).
    Returns (x, info) with info = dict(iters, resnorms, ntl_weights, converged, diverged)."""
    lv0 = mg.LVL[0]
    if rhs is not None:
        lv0.r.copy_(torch.as_tensor(rhs).to(mg.tdtype).reshape(lv0.S, lv0.n))
    if x0 is not None or rhs is not None:
        if x0 is None:
            lv0.phi.zero_()
        else:
            lv0.phi.copy_(torch.as_tensor(x0).to(mg.tdtype).reshape(lv0.S, lv0.n))
        for lv in mg.LVL[1:]:
            lv.phi.zero_()
        for row in mg.NTL:
            for nt in row:
                if nt.phi is not None:
                    nt.phi.zero_()
    if outer == "stationary":
        info = perform_MG(mg, tol, max_iters, check_every, record_phi, use_graph)
    elif outer == "gcr":
        pm = None
        if precond_dtype in ("complex64", "complex64+half") and mg.p.dtype == "complex128":
            pm = mg.info.get("single")
            if pm is None:
                pm = mg.info["single"] = _mg.make_single_precision(mg)
            pm.use_half = precond_dtype.endswith("+half")
            if pm.use_half and not pm.info.get("half_built"):
                for lv in pm.LVL[1:]:
                    lv.make_half_blocks()
                pm.info["half_built"] = True
        elif precond_dtype not in (None, mg.p.dtype):
            raise ValueError("precond_dtype must be None, 'complex64' or 'complex64+half' (on a complex128 hierarchy)")
        info = _mg.gcr_MG(mg, tol, max_iters, restart, check_every, use_graph, pm)
    else:
        raise ValueError("outer must be 'stationary' (f_perform_MG) or 'gcr'")
    return lv0.phi, info


def run_reference_flow(params: MGParams, U, record_phi: bool = False):
    """main() of the reference (S6/mgrid_ntl.cpp:29-73): random fields, source, links, setup, solve."""
    mg = setup(U, params, init="reference")
    x, info = solve(mg, record_phi=record_phi)
    return mg, info
