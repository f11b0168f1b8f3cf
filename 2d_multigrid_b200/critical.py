"""Locate the critical mass of a gauge configuration with the multigrid solver itself.

D(m) = D(0) + m, so "near-critical" means m = m_crit + delta with m_crit = -min Re lambda(D(0)) (SURVEY 8d).
For lattices too large for a dense/ARPACK eigen-solve the lowest eigenvalue is found by shifted inverse iteration
x <- D(m_k)^-1 x, each solve done by the MG-preconditioned FGCR; the shift moves towards the eigenvalue in stages
(a new hierarchy per stage), and the eigenvalue is read off the gamma5-symmetric quotient
    lambda ~ <g5 x, D(0) x> / <g5 x, x>        (D is gamma5-hermitian, so g5 x is the LEFT eigenvector: second-order accurate;
                                                 falls back to the plain Rayleigh quotient when <g5 x, x> ~ 0)
Input preparation, not part of the timed hot path.  The operator must be untwisted (mu == 0): the twisted-mass solve at
maximal twist takes the m_crit found here.
"""
from __future__ import annotations

import torch


def _quotients(x, Dx, wilson: bool):
    """(two-sided gamma5 quotient or None, plain Rayleigh quotient) of D for the vector x."""
    xf, Df = x.reshape(-1), Dx.reshape(-1)
    rq = (torch.vdot(xf, Df) / torch.vdot(xf, xf)).item()
    if not wilson or x.shape[-1] != 2:
        return None, rq
    g5x = x.clone()
    g5x[:, 1] = -g5x[:, 1]                       # gamma5 = sigma_3 on the two spin components
    den = torch.vdot(g5x.reshape(-1), xf).item()
    if abs(den) < 1e-3 * float(torch.vdot(xf, xf).real):
        return None, rq
    return (torch.vdot(g5x.reshape(-1), Df) / den).item(), rq


def _untwisted(p):
    if getattr(p, "mu", 0.0) != 0.0:
        raise ValueError("estimate_critical_mass needs mu == 0: the gamma5 quotient relies on gamma5-hermiticity, which the "
                         "twisted mass breaks; estimate m_crit at mu = 0 and pass it to the twisted solve")
    return p


def estimate_critical_mass(U, params_factory, m0: float = 0.0, iters: int = 4, refine: int = 3, tol: float = 1e-8,
                           margins=(0.02, 0.004), target: float = 2e-5, max_refine: int = 12, verbose: bool = False):
    """params_factory(mass) -> MGParams.  Returns (m_crit_estimate, history of eigenvalue estimates of D(0)).
    Stage 0: `iters` inverse-iteration steps at mass m0.  Stage k >= 1: shift to -Re(lambda) + margins[k-1] and iterate until the
    estimate moves by less than `target` (at least `refine`, at most `max_refine` steps).  estimate_critical_mass.info holds the
    quality of the result: eigen-residual |D x - lambda x| / |x|, the last change of the estimate, the number of solves."""
    from . import setup, solve
    hist = []
    x = None
    lam = None
    nsolves = 0
    stages = [(m0, iters, iters)] + [(None, refine, max_refine)] * len(margins)
    _untwisted(params_factory(m0))
    for stage, (m, nmin, nmax) in enumerate(stages):
        if m is None:
            m = -lam.real + margins[stage - 1]
        p = _untwisted(params_factory(m))
        mg = setup(U, p, init="device")
        lv = mg.LVL[0]
        wilson = p.stencil == "wilson"
        if x is None:
            g = torch.Generator(device=mg.device); g.manual_seed(99)
            x = torch.randn((lv.S, lv.n), generator=g, dtype=torch.float64, device=mg.device).to(mg.tdtype)
        Dx = torch.empty_like(x)
        for k in range(nmax):
            x = x / torch.linalg.vector_norm(x)
            y, info = solve(mg, rhs=x, tol=tol, max_iters=200, outer="gcr", restart=8)
            nsolves += 1
            x = y.clone()
            lv.apply_D(Dx, x)
            q5, rq = _quotients(x, Dx, wilson)
            mu = q5 if q5 is not None else rq                       # eigenvalue estimate of D(m)
            lam_new = complex(mu) - m                               # ... of D(0)
            res = float(torch.linalg.vector_norm(Dx - mu * x) / torch.linalg.vector_norm(x))
            change = abs(lam_new - lam) if lam is not None else None
            lam = lam_new
            hist.append(lam)
            estimate_critical_mass.info = {"eig_residual": res, "last_change": change, "solves": nsolves, "imag": lam.imag,
                                           "quotient": "gamma5" if q5 is not None else "rayleigh", "last_shift_margin": m + lam.real}
            if verbose:
                print(f"  stage {stage} m={m:+.6f} solve iters={info['iters']} lambda(D0)~{lam:.7f} |Dx-lx|/|x|={res:.2e}")
            if k + 1 >= nmin and change is not None and change < target:
                break
        mg.close()          # tens of GB at 4096^2: give them back before the next hierarchy is built
        del mg, lv, y
        import gc
        gc.collect()
        torch.cuda.empty_cache()
    return -lam.real, hist


estimate_critical_mass.info = {}
