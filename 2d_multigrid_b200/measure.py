"""Measurements on a gauge ensemble of the two-flavour Schwinger model: topological charge, Wilson loops, meson correlators
with the PCAC quark mass, and the chiral condensate.

Conventions (DESIGN section 4): sites s = x + y L, time is y; gamma_x = sigma1, gamma_y = sigma2, gamma5 = sigma3.  The gauge
observables are one reduction kernel each (csrc/measure.cu).  The fermionic ones run complex128 FGCR(8) + multigrid solves
through solve(), one source at a time, on a one-GPU hierarchy (Wilson, clover or twisted mass; a hierarchy an HMC has moved
in place with stale coarse levels costs iterations, not accuracy):

    meson_correlators: two point-source solves psi_be = D^-1 e_{s0,be}, then mg2d_meson_contract
        G_ab(t) = sum_x tr[s_a S(x, y0+t) s_b s3 S(x, y0+t)^dag s3],  S_{al,be} = psi_be_al.
        gamma5-hermiticity (gamma5 D(mu) gamma5 = D(-mu)^dag for the twisted doublet) makes -G_ab the connected correlator
        <psibar1 s_a psi2(x) psibar2 s_b psi1(x0)>, so
        pp = G_33 = sum |S|^2 (the pion),  ap = Re(i G_13) (A_y = psibar gamma_y gamma5 psi, gamma_y gamma5 = i sigma1),
        m_eff(t) = arccosh[(pp(t-1) + pp(t+1)) / (2 pp(t))],  m_pcac(t) = [ap(t+1) - ap(t-1)] / (4 pp(t)).
    chiral_condensate: U(1) noise eta_e = e^{i alpha_e} (one phase per component), alpha from mg2d_fill_uniform keyed on
        (seed, noise index) so every noise is reproducible on its own; per noise (1/L^2) eta^dag D^-1 eta, whose expectation
        is Tr D^-1 / L^2.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib
from ._lib import MG2DError
from .mg import MG, _ptr, _stream

_CTX: dict = {}


def _ctx(dev: int) -> _lib.Context:
    if dev not in _CTX:
        _CTX[dev] = _lib.Context(dev)
    return _CTX[dev]


def _links(U, L: int) -> torch.Tensor:
    """U[L*L, 2] as a contiguous complex128 device tensor (complex64 links are converted)."""
    U = torch.as_tensor(U)
    if U.numel() != 2 * L * L:
        raise ValueError(f"links must have {2 * L * L} elements ([L*L, 2]), got shape {tuple(U.shape)}")
    dev = U.device if U.is_cuda else torch.device("cuda", torch.cuda.current_device())
    return U.to(device=dev, dtype=torch.complex128).reshape(L * L, 2).contiguous()


def topological_charge(U, L: int) -> float:
    """Q = (1/2 pi) sum_P arg U_P with arg in (-pi, pi] (the geometric charge; an integer up to rounding on a torus)."""
    U = _links(U, L)
    out = torch.zeros(1, dtype=torch.float64, device=U.device)
    with torch.cuda.device(U.device):
        _ctx(U.device.index).call("mg2d_topo_charge", _ptr(U), L, _ptr(out), _stream())
        return float(out.item()) / (2.0 * math.pi)


def wilson_loops(U, L: int, r_max: int, t_max: int) -> np.ndarray:
    """W[T-1, R-1] = mean over base sites of the anticlockwise R x T loop (R along x, T along y), 1 <= R <= r_max,
    1 <= T <= t_max; W[0, 0] is the mean plaquette.  Needs 1 <= r_max, t_max <= 32 and < L (MG2DError otherwise)."""
    U = _links(U, L)
    out = torch.zeros(2 * 32 * 32, dtype=torch.float64, device=U.device)
    with torch.cuda.device(U.device):
        _ctx(U.device.index).call("mg2d_wilson_loops", _ptr(U), L, int(r_max), int(t_max), _ptr(out), _stream())
        w = out[:2 * r_max * t_max].cpu().numpy()
    return (w[0::2] + 1j * w[1::2]).reshape(t_max, r_max) / (L * L)


def _check(mg: MG):
    if getattr(mg, "comm", None) is not None:
        raise MG2DError("measurements need a one-GPU hierarchy: strip-decomposed hierarchies (DistMG) are not supported")
    if mg.p.stencil != "wilson":
        raise ValueError("measurements need the Wilson stencil")
    if mg.p.dtype != "complex128":
        raise ValueError("measurements need a complex128 hierarchy (precond_dtype='complex64' runs the cycle in complex64)")


def _solve(mg: MG, rhs, tol, precond_dtype, use_graph):
    from . import solve
    x, info = solve(mg, rhs=rhs, tol=tol, outer="gcr", restart=8, use_graph=use_graph, check_every=1,
                    precond_dtype=precond_dtype)
    if not info["converged"]:
        raise MG2DError(f"measurement solve did not converge (iterations {info['iters']}, residual {info['resnorms'][-1]:.3g})")
    return x, info


def meson_correlators(mg: MG, site=(0, 0), tol: float = 1e-10, precond_dtype: str | None = None,
                      use_graph: bool = True) -> dict:
    """Point-source meson correlators from site = (x0, y0) on the links of the hierarchy mg.  Returns dict(G [L, 4, 4]
    complex with t = y - y0, pp, ap, m_eff, m_pcac [L] (periodic in t), iters [2], true_resnorms [2])."""
    _check(mg)
    L = mg.p.L
    x0, y0 = (int(v) for v in site)
    if not (0 <= x0 < L and 0 <= y0 < L):
        raise ValueError(f"source site {site} is outside the {L} x {L} lattice")
    cols, iters, res = [], [], []
    for be in (0, 1):
        rhs = torch.zeros((L * L, 2), dtype=torch.complex128, device=mg.device)
        rhs[x0 + y0 * L, be] = 1.0
        x, info = _solve(mg, rhs, tol, precond_dtype, use_graph)
        cols.append(x.clone())                 # solve() returns the hierarchy's own phi
        iters.append(info["iters"])
        res.append(info["true_resnorm"])
    out = torch.empty((L, 4, 4, 2), dtype=torch.float64, device=mg.device)
    mg.ctx.call("mg2d_meson_contract", _ptr(cols[0]), _ptr(cols[1]), L, _ptr(out), _stream())
    o = out.cpu().numpy()
    G = np.roll(o[..., 0] + 1j * o[..., 1], -y0, axis=0)
    pp = G[:, 3, 3].real.copy()
    ap = (1j * G[:, 1, 3]).real
    with np.errstate(invalid="ignore", divide="ignore"):
        m_eff = np.arccosh((np.roll(pp, 1) + np.roll(pp, -1)) / (2.0 * pp))
        m_pcac = (np.roll(ap, -1) - np.roll(ap, 1)) / (4.0 * pp)
    return {"G": G, "pp": pp, "ap": ap, "m_eff": m_eff, "m_pcac": m_pcac, "iters": iters, "true_resnorms": res}


def chiral_condensate(mg: MG, n_noise: int, seed: int = 1, tol: float = 1e-10, precond_dtype: str | None = None,
                      use_graph: bool = True) -> dict:
    """Stochastic (1/L^2) Tr D^-1 from n_noise U(1) noise vectors: noise k has the phases alpha = mg2d_fill_uniform(seed,
    stream k) in [-pi, pi).  Returns dict(mean complex, stderr of the real part (nan for one noise), values [n_noise] complex,
    iters [n_noise])."""
    _check(mg)
    if n_noise < 1:
        raise ValueError("n_noise must be >= 1")
    L, ctx, dev = mg.p.L, mg.ctx, mg.device
    S = L * L
    draw = torch.empty(2 * S, dtype=torch.complex128, device=dev)
    eta = torch.empty((S, 2), dtype=torch.complex128, device=dev)
    dot = torch.zeros(2, dtype=torch.float64, device=dev)
    vals, iters = [], []
    for k in range(n_noise):
        ctx.call("mg2d_fill_uniform", _ptr(draw), 2 * S, 0, seed, k, -math.pi, math.pi, _lib.C128, _stream())
        alpha = draw.real.contiguous()        # the generator writes (alpha, 0) pairs
        ctx.call("mg2d_phases_to_links", _ptr(eta), _ptr(alpha), 2 * S, _lib.C128, _stream())
        x, info = _solve(mg, eta, tol, precond_dtype, use_graph)
        ctx.call("mg2d_cdot_batch", _ptr(eta), 2 * S, 1, _ptr(x), 2 * S, 1, 2 * S, _lib.C128, _ptr(dot), _stream())
        d = dot.cpu().tolist()
        vals.append(complex(d[0], d[1]) / S)
        iters.append(info["iters"])
    v = np.array(vals)
    err = float(v.real.std(ddof=1) / math.sqrt(len(v))) if len(v) > 1 else float("nan")
    return {"mean": complex(v.mean()), "stderr": err, "values": v, "iters": iters}
