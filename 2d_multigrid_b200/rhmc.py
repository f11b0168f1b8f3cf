"""Multi-shift CG for (M + sigma_k) x_k = phi, M = D^dag D, on the level-0 Wilson operator of a hierarchy (one-flavour RHMC).

Jegerlehner's multi-shift CG (hep-lat/9612014): one Krylov space for every shift, the base system being the smallest shift.  An
iteration is two existing Wilson applies and mg2d_gamma5 for M p_0 = gamma5 D gamma5 D p_0 (D^dag = gamma5 D gamma5), then the
two vector passes of csrc/rhmc.cu; the scalar recurrences run on the device and the host reads one residual norm per
iteration.  Every x_k starts from 0.  The coarse levels of the hierarchy are never touched.

normal_solve solves the same systems with the multigrid hierarchy instead: D_tm(mu)^dag D_tm(mu) = D^dag D + mu^2 and
D_tm(mu)^dag = gamma5 D_tm(-mu) gamma5 give, for sigma = mu^2,
    (D^dag D + sigma)^-1 = D_tm(+mu)^-1 gamma5 D_tm(-mu)^-1 gamma5,
two FGCR solves on one hierarchy whose twist MG.set_twist changes in place.
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
    tr = _true_residuals(mg, phi, X, sig, b2, (t, u, w))
    info["true_residuals"] = [tr[inv[k]] for k in range(N)]
    if order != list(range(N)):
        X = X[torch.tensor(inv, device=dev)]
    return X, info


def _true_residuals(mg, phi, X, sig, b2, work):
    """|phi - (D^dag D + sig[j]) X[j]| / |phi| for every j, computed once (b2 = |phi|^2; work: three fields)."""
    lv, ctx, st = mg.LVL[0], mg.ctx, _stream()
    S = lv.S
    t, u, w = work
    out = torch.zeros(len(sig), dtype=torch.float64, device=phi.device)
    for j in range(len(sig)):
        lv._stencil(t, X[j], None, _lib.MODE_APPLY, None)
        ctx.call("mg2d_gamma5", _ptr(u), _ptr(t), S, st)
        lv._stencil(w, u, None, _lib.MODE_APPLY, None)
        ctx.call("mg2d_gamma5", _ptr(w), _ptr(w), S, st)
        ctx.call("mg2d_copy", _ptr(t), _ptr(phi), 2 * S, _lib.C128, st)
        ctx.call("mg2d_axpy", _ptr(t), _ptr(w), -1.0, 0.0, None, 2 * S, _lib.C128, st)
        ctx.call("mg2d_axpy", _ptr(t), _ptr(X[j]), -sig[j], 0.0, None, 2 * S, _lib.C128, st)
        ctx.call("mg2d_norm2", _ptr(t), 2 * S, _lib.C128, _ptr(out[j:]), st)
    return [math.sqrt(v / b2) for v in out.tolist()]


def operator_norm_bound(p, mu: float) -> float:
    """An upper bound on the operator norm of D_tm(mu) = D + i mu gamma5: |2+m| + |c_sw|/2 for the self term (the clover field is
    at most |c_sw|/2), 2 sqrt 2 for the four hops and |mu|."""
    return abs(2.0 + p.mass) + abs(p.csw) / 2.0 + 2.0 * math.sqrt(2.0) + abs(mu)


def second_solve_tol(tol: float, rhs_norm: float, z_norm: float, p, mu: float) -> float:
    """Relative tolerance of the second solve D_tm(+mu) x = gamma5 z.  With r1 = gamma5 rhs - D_tm(-mu) z and
    r2 = gamma5 z - D_tm(+mu) x the normal residual is rhs - (D^dag D + mu^2) x = gamma5 r1 + D_tm(mu)^dag r2, so |r1| <= tol/2 |rhs|
    and |r2| <= this value times |z| bound it by tol |rhs|."""
    return tol * rhs_norm / (2.0 * operator_norm_bound(p, mu) * z_norm)


_SOLVE_KW = ("precond_dtype", "use_graph", "max_iters", "restart", "check_every")


def normal_solve(mg, rhs, shifts, tol: float, **solve_kw):
    """Solve (D^dag D + shifts[k]) x_k = rhs for every k with multigrid: x = D_tm(+mu)^-1 gamma5 D_tm(-mu)^-1 gamma5 rhs with
    mu = sqrt(shifts[k]), each a solve(outer="gcr") from x0 = 0 with solve_kw (precond_dtype, use_graph, max_iters, restart,
    check_every) on the hierarchy `mg`, whose twist set_twist changes in place.  The first solve runs to tol/2, the second to
    second_solve_tol, so that the true residual of the normal equations is at most tol.

    mg: a one-GPU Wilson or Wilson-clover hierarchy at twist 0 (p.mu == 0), left at twist 0.  rhs[L*L, 2] complex128;
    shifts: numbers >= 0 (0 is the two-flavour composition D^-1 gamma5 D^-1 gamma5).  Returns (X[N, L*L, 2] in the order of
    shifts, info) with info: iters (the (-mu, +mu) FGCR iterations per shift), converged, true_residuals (relative
    |rhs - (D^dag D + s_k) x_k| / |rhs|, computed once at the end) and twist_ms (device time spent in set_twist).
    Raises MG2DError when an inner solve does not converge."""
    from . import solve
    p = mg.p
    if p.stencil != "wilson" or p.dtype != "complex128":
        raise ValueError("normal_solve needs a complex128 Wilson hierarchy")
    if p.mu != 0.0:
        raise ValueError(f"normal_solve needs the hierarchy at twist 0 (D itself); it is at mu = {p.mu}")
    if mg.comm is not None:
        raise ValueError("normal_solve runs on one GPU (whole lattice)")
    lv = mg.LVL[0]
    shifts = [float(s) for s in shifts]
    if not shifts or not all(s >= 0.0 and math.isfinite(s) for s in shifts):
        raise ValueError("need at least one finite shift >= 0")
    if not tol > 0.0:
        raise ValueError("need tol > 0")
    bad = sorted(set(solve_kw) - set(_SOLVE_KW))
    if bad:
        raise ValueError(f"normal_solve: unknown solve arguments {bad} (allowed: {', '.join(_SOLVE_KW)})")
    ctx, S, st = mg.ctx, lv.S, _stream()
    dev = mg.device
    phi = torch.as_tensor(rhs).to(torch.complex128).to(dev).reshape(S, 2)
    nrm = torch.zeros(2, dtype=torch.float64, device=dev)
    ctx.call("mg2d_norm2", _ptr(phi), 2 * S, _lib.C128, _ptr(nrm), st)
    b2 = float(nrm[0].item())
    if not b2 > 0.0:
        raise ValueError("normal_solve: rhs is zero")
    X = torch.empty((len(shifts), S, 2), dtype=torch.complex128, device=dev)
    g = torch.empty_like(phi)
    ctx.call("mg2d_gamma5", _ptr(g), _ptr(phi), S, st)
    events = []

    def twist(mu):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        mg.set_twist(mu)
        e1.record()
        events.append((e0, e1))

    def inner(b, t, what):
        x, info = solve(mg, rhs=b, tol=t, outer="gcr", **solve_kw)
        if not info["converged"]:
            raise MG2DError(f"normal_solve: the {what} solve did not converge (iterations {info['iters']}, residual "
                            f"{info['resnorms'][-1] if info['resnorms'] else float('nan'):.3g})")
        return x, info["iters"]
    iters = []
    gz = torch.empty_like(phi)
    try:
        for k, s in enumerate(shifts):
            mu = math.sqrt(s)
            twist(-mu)
            z, n1 = inner(g, 0.5 * tol, "D_tm(-mu)")
            ctx.call("mg2d_norm2", _ptr(z), 2 * S, _lib.C128, _ptr(nrm[1:]), st)
            ctx.call("mg2d_gamma5", _ptr(gz), _ptr(z), S, st)
            z2 = float(nrm[1].item())
            twist(mu)
            t2 = second_solve_tol(tol, math.sqrt(b2), math.sqrt(z2), p, mu) if z2 > 0.0 else 1.0
            x, n2 = inner(gz, t2, "D_tm(+mu)")
            ctx.call("mg2d_copy", _ptr(X[k]), _ptr(x), 2 * S, _lib.C128, st)
            iters.append((n1, n2))
    finally:
        twist(0.0)
    work = (g, gz, torch.empty_like(phi))
    tr = _true_residuals(mg, phi, X, shifts, b2, work)
    torch.cuda.synchronize()
    info = {"iters": iters, "converged": True, "true_residuals": tr,
            "twist_ms": sum(e0.elapsed_time(e1) for e0, e1 in events)}
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
