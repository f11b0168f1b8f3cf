"""Multi-shift CG for (M + sigma_k) x_k = phi, M = D^dag D, on the level-0 Wilson operator of a hierarchy (one-flavour RHMC).

Jegerlehner's multi-shift CG (hep-lat/9612014): one Krylov space for every shift, the base system being the smallest shift.  An
iteration is two existing Wilson applies and mg2d_gamma5 for M p_0 = gamma5 D gamma5 D p_0 (D^dag = gamma5 D gamma5), then the
two vector passes of csrc/rhmc.cu; the scalar recurrences run on the device and the host reads one residual norm per
iteration.  Every x_k starts from 0.  The coarse levels of the hierarchy are never touched.
"""
from __future__ import annotations

import math

import torch

from . import _lib
from ._lib import MG2DError
from .mg import _ptr, _stream


def multishift_cg(mg, rhs, shifts, tol: float, max_iters: int, weights=None):
    """Solve (D^dag D + shifts[k]) x_k = rhs for every k on the level-0 links and mass of `mg`.

    rhs[L*L, 2] complex128; shifts: N <= 64 numbers >= 0.  Every shift iterates until its residual |rhs - (M + s_k) x_k| is
    below tol |rhs| (by the recurrence), then stops being updated.  Returns (X, info): X[N, L*L, 2] in the order of `shifts`, or,
    with `weights`, y = sum_k weights[k] x_k[L*L, 2] without storing the x_k.  info: iters, converged, residuals (recurrence,
    relative), true_residuals (relative |rhs - (M + s_k) x_k| / |rhs| computed once at the end; None with weights), ritz (the
    smallest and largest Ritz values of M from the Lanczos tridiagonal of the base system)."""
    lv = mg.LVL[0]
    p = mg.p
    if p.stencil != "wilson" or p.dtype != "complex128" or not lv.matrix_free or p.mu != 0.0 or lv.clover is not None:
        raise ValueError("multishift_cg needs a matrix-free complex128 Wilson level 0 without clover or twist")
    if getattr(lv, "distributed", False):
        raise ValueError("multishift_cg runs on one GPU (whole lattice)")
    shifts = [float(s) for s in shifts]
    N = len(shifts)
    if not 1 <= N <= _lib.MSC_MAX_SHIFTS or not all(s >= 0.0 and math.isfinite(s) for s in shifts):
        raise ValueError(f"need 1 to {_lib.MSC_MAX_SHIFTS} finite shifts >= 0")
    if weights is not None and len(weights) != N:
        raise ValueError("weights needs one number per shift")
    if not tol > 0.0 or max_iters < 1:
        raise ValueError("need tol > 0 and max_iters >= 1")
    ctx, S = mg.ctx, lv.S
    dev = lv.U.device
    order = sorted(range(N), key=lambda k: shifts[k])
    sig = [shifts[k] for k in order]
    sigma0 = sig[0]
    phi = torch.as_tensor(rhs).to(torch.complex128).to(dev).reshape(S, 2)
    acc = weights is not None
    Pk = torch.empty((N, S, 2), dtype=torch.complex128, device=dev)
    X = None if acc else torch.empty_like(Pk)
    y = torch.empty_like(phi) if acc else None
    r, t, u, w = (torch.empty_like(phi) for _ in range(4))
    dots = torch.zeros(_lib.NDOTS, dtype=torch.float64, device=dev)
    nsc = _lib.MSC_SHIFTS + 6 * N
    sc = torch.zeros(nsc + 2 * max_iters, dtype=torch.float64, device=dev)
    st = _stream()
    ctx.call("mg2d_norm2", _ptr(phi), 2 * S, _lib.C128, _ptr(dots), st)
    b2 = float(dots[0].item())
    if not b2 > 0.0:
        raise ValueError("multishift_cg: rhs is zero")
    init = [0.0] * nsc
    init[_lib.MSC_RR] = init[_lib.MSC_PP] = b2
    init[_lib.MSC_ALPHA_PREV] = 1.0
    init[_lib.MSC_NACT_NEXT] = N
    init[_lib.MSC_THRESH] = tol * tol * b2
    o = _lib.MSC_SHIFTS
    init[o:o + N] = [s - sigma0 for s in sig]
    init[o + N:o + 3 * N] = [1.0] * (2 * N)                                  # zeta, zeta_prev
    if acc:
        init[o + 5 * N:o + 6 * N] = [float(weights[k]) for k in order]
    sc[:nsc].copy_(torch.tensor(init, dtype=torch.float64))
    ctx.call("mg2d_copy", _ptr(r), _ptr(phi), 2 * S, _lib.C128, st)
    for k in range(N):
        ctx.call("mg2d_copy", _ptr(Pk[k]), _ptr(phi), 2 * S, _lib.C128, st)
    ctx.call("mg2d_zero", _ptr(X if X is not None else y), (N if X is not None else 1) * 2 * S, _lib.C128, st)
    p0 = Pk[0]
    converged, it = False, 0
    while it < max_iters:
        lv._stencil(t, p0, None, _lib.MODE_APPLY, dots)                        # t = D p_0, dots[0] = <p_0, M p_0>
        ctx.call("mg2d_gamma5", _ptr(u), _ptr(t), S, st)
        lv._stencil(w, u, None, _lib.MODE_APPLY, None)                        # M p_0 = gamma5 w
        ctx.call("mg2d_msc_pass_a", _ptr(r), _ptr(w), _ptr(p0), _ptr(dots), _ptr(sc), sigma0, N, S, st)
        ctx.call("mg2d_msc_pass_b", _ptr(X), _ptr(Pk), _ptr(y), _ptr(r), _ptr(sc), sigma0, N, S, st)
        it += 1
        h = sc[:_lib.MSC_SHIFTS].tolist()
        if not math.isfinite(h[_lib.MSC_RR]):
            raise MG2DError(f"multishift_cg: residual is not finite at iteration {it}")
        if h[_lib.MSC_NACT_NEXT] == 0:
            converged = True
            break
    rr = float(sc[_lib.MSC_RR].item())
    zeta = sc[o + N:o + 2 * N].tolist()
    res_sorted = [abs(z) * math.sqrt(rr / b2) for z in zeta]
    hist = sc[nsc:nsc + 2 * it].view(it, 2).cpu().double().numpy()
    info = {"iters": it, "converged": converged, "ritz": _ritz(hist, sigma0), "true_residuals": None}
    inv = [0] * N
    for j, k in enumerate(order):
        inv[k] = j
    info["residuals"] = [res_sorted[inv[k]] for k in range(N)]
    if acc:
        return y, info
    # true residuals, once: rhs - (M + s_k) x_k
    out = torch.zeros(N, dtype=torch.float64, device=dev)
    for j in range(N):
        lv._stencil(t, X[j], None, _lib.MODE_APPLY, None)
        ctx.call("mg2d_gamma5", _ptr(u), _ptr(t), S, st)
        lv._stencil(w, u, None, _lib.MODE_APPLY, None)
        ctx.call("mg2d_gamma5", _ptr(w), _ptr(w), S, st)
        ctx.call("mg2d_copy", _ptr(t), _ptr(phi), 2 * S, _lib.C128, st)
        ctx.call("mg2d_axpy", _ptr(t), _ptr(w), -1.0, 0.0, None, 2 * S, _lib.C128, st)
        ctx.call("mg2d_axpy", _ptr(t), _ptr(X[j]), -sig[j], 0.0, None, 2 * S, _lib.C128, st)
        ctx.call("mg2d_norm2", _ptr(t), 2 * S, _lib.C128, _ptr(out[j:]), st)
    tr = [math.sqrt(v / b2) for v in out.tolist()]
    info["true_residuals"] = [tr[inv[k]] for k in range(N)]
    if order != list(range(N)):
        X = X[torch.tensor(inv, device=dev)]
    return X, info


def _ritz(hist, sigma0):
    """(min, max) Ritz values of M from the CG coefficients of the base system A = M + sigma0: the Lanczos tridiagonal
    T_ii = 1/alpha_i + beta_{i-1}/alpha_{i-1}, T_i,i+1 = sqrt(beta_i)/alpha_i."""
    from scipy.linalg import eigvalsh_tridiagonal
    al, be = hist[:, 0], hist[:, 1]
    n = len(al)
    d = 1.0 / al
    d[1:] += be[:-1] / al[:-1]
    e = (be[:-1] ** 0.5) / al[:-1]
    if n == 1:
        return (float(d[0]) - sigma0, float(d[0]) - sigma0)
    ev = eigvalsh_tridiagonal(d, e, select="i", select_range=(0, 0))[0], eigvalsh_tridiagonal(d, e, select="i", select_range=(n - 1, n - 1))[0]
    return (float(ev[0]) - sigma0, float(ev[1]) - sigma0)
