"""Two-flavour Wilson Hybrid Monte Carlo for compact U(1) in two dimensions, with the multigrid solver in the fermion force.

H(theta, P) = 1/2 sum P^2 + S_g + S_f,  S_g = beta sum_P (1 - cos theta_P),  S_f = phi^dag (D^dag D)^-1 phi,  phi = D^dag eta,
eta complex Gaussian with <|eta|^2> = 1 per component.  Leapfrog in theta with the momenta P (real N(0,1) per link); every
kernel is in libmg2d_sm100.so (csrc/hmc.cu, mg2d_fill_gaussian, mg2d_plaquette, mg2d_norm2, the Wilson apply and the
FGCR + multigrid solve).  With gamma5 D gamma5 = D^dag the pseudofermion is kept as chi = gamma5 phi = D gamma5 eta, so
every solve is one with D on the same hierarchy:
    Y = D^-dag phi = gamma5 D^-1 chi,   X = (D^dag D)^-1 phi = D^-1 Y,   S_f = |D^-1 chi|^2.
The hierarchy follows the links: mg2d_hmc_links writes e^{i theta} into its level-0 link tensor (and the complex64 shadow's)
in place, so the captured solve graphs replay on the new field; the coarse levels are refreshed (MG.refresh) at the start of
every trajectory that follows an accepted one.  Every solve starts from x0 = 0, so a trajectory is reversible to the solver
tolerance.  Random numbers come from the counter generator keyed on (seed, 3 k + {0: momenta, 1: eta, 2: accept draw}) for
trajectory k, so a trajectory is reproducible from (seed, k) alone.
"""
from __future__ import annotations

import math
import time

import torch

from . import _lib
from ._lib import MG2DError
from .mg import MG, _ptr, _stream
from .params import MGParams


class HMC:
    """HMC(params, theta, beta, ...).trajectory() -> dict.

    params: a complex128, matrix-free (smoother 'rbgs' or 'mr') Wilson MGParams without clover, twist or NTL; the hierarchy is
    built once by setup() at theta.  theta[L*L, 2]: float64 link phases (copied).  tau / n_md: trajectory length and leapfrog
    steps.  flavours: 2 (det D^dag D) or 0 (pure gauge).  md_tol: relative residual of the force solves; accept_tol: of the
    final action's solve.  refresh_null_iters: sweeps of MG.refresh after an accepted trajectory (None: never refresh;
    default 8, measured in DESIGN section 4).
    precond_dtype / use_graph: passed to solve() (outer FGCR(8))."""

    def __init__(self, params: MGParams, theta, beta: float, tau: float = 1.0, n_md: int = 10, flavours: int = 2, seed: int = 1,
                 md_tol: float = 1e-10, accept_tol: float = 1e-12, refresh_null_iters: int | None = 8,
                 precond_dtype: str | None = None, use_graph: bool = True, device: int | None = None):
        from . import setup
        p = params
        if p.stencil != "wilson":
            raise ValueError("HMC needs the Wilson stencil")
        if p.mu != 0.0:
            raise ValueError("HMC: mu != 0 is not supported (D(mu)^dag needs the D(-mu) hierarchy)")
        if p.csw != 0.0:
            raise ValueError("HMC: csw != 0 is not supported (the clover force is not implemented)")
        if p.dtype != "complex128":
            raise ValueError("HMC needs a complex128 hierarchy (precond_dtype='complex64' runs the cycle in complex64)")
        if p.ntl:
            raise ValueError("HMC: non-telescoping hierarchies are not supported")
        if not p.matrix_free:
            raise ValueError("HMC needs the matrix-free level 0 (smoother 'rbgs' or 'mr'): the links change at every step")
        if flavours not in (0, 2):
            raise ValueError("flavours must be 0 (pure gauge) or 2")
        if n_md < 1 or not tau > 0.0:
            raise ValueError("need n_md >= 1 and tau > 0")
        if refresh_null_iters is not None and refresh_null_iters < 0:
            raise ValueError("refresh_null_iters must be None or >= 0")
        self.p, self.L = p, p.L
        self.beta, self.tau, self.n_md, self.flavours, self.seed = float(beta), float(tau), int(n_md), int(flavours), int(seed)
        self.md_tol, self.accept_tol, self.refresh_null_iters = md_tol, accept_tol, refresh_null_iters
        self.precond_dtype, self.use_graph = precond_dtype, use_graph
        dev = torch.cuda.current_device() if device is None else device
        self.device = torch.device("cuda", dev)
        S = self.L * self.L
        self.theta = torch.as_tensor(theta).to(torch.float64).to(self.device).reshape(S, 2).clone()
        U = torch.empty((S, 2), dtype=torch.complex128, device=self.device)
        with torch.cuda.device(dev):
            c = _lib.Context(dev)
            c.call("mg2d_phases_to_links", _ptr(U), _ptr(self.theta), 2 * S, _lib.C128, _stream())
            torch.cuda.synchronize()
            c.close()
            self.mg = setup(U, p, init="device", device=dev)
        self.ctx = self.mg.ctx
        self.mg.update_links(U)              # the hierarchy now owns its link tensor: the MD writes into it in place
        self.P = torch.empty((S, 2), dtype=torch.float64, device=self.device)
        self.theta0 = torch.empty_like(self.theta)
        self.eta = torch.empty((S, 2), dtype=torch.complex128, device=self.device)
        self.chi = torch.empty_like(self.eta)
        self.Y = torch.empty_like(self.eta)
        self.red = torch.zeros(8, dtype=torch.float64, device=self.device)
        self.u = torch.zeros(1, dtype=torch.complex128, device=self.device)
        self.k = 0                           # trajectories run
        self.stale = False                   # the links moved since the coarse hierarchy was last built for them

    # ---- pieces --------------------------------------------------------------------------------------------
    def _solve(self, rhs, tol):
        from . import solve
        x, info = solve(self.mg, rhs=rhs, tol=tol, outer="gcr", restart=8, use_graph=self.use_graph, check_every=1,
                        precond_dtype=self.precond_dtype)
        if not info["converged"]:
            raise MG2DError(f"HMC: solve did not converge (iterations {info['iters']}, residual {info['resnorms'][-1]:.3g})")
        return x, info["iters"]

    def _links_c64(self):
        sh = self.mg.info.get("single")
        return None if not isinstance(sh, MG) else sh.LVL[0].U

    def _action(self, out):
        """out[0] = S_g (with the fermion part added by the caller): beta (V - Re sum_P U_P) from mg2d_plaquette."""
        self.ctx.call("mg2d_plaquette", _ptr(self.mg.LVL[0].U), self.L, _lib.C128, _ptr(out), _stream())

    def _norm2(self, t, out):
        """out[0] = sum |t|^2 of a complex128 field or of a float64 one (read as complex pairs)."""
        n = t.numel() if t.is_complex() else t.numel() // 2
        self.ctx.call("mg2d_norm2", _ptr(t), n, _lib.C128, _ptr(out), _stream())

    def force_step(self, eps: float, iters: list, timer=None):
        """P -= eps dS/dtheta at the current links (two solves for flavours = 2)."""
        mg, S = self.mg, self.L * self.L
        timer = timer or _NullTimer
        x = None
        if self.flavours:
            with timer("solves"):
                yt, n1 = self._solve(self.chi, self.md_tol)                           # D^-1 chi
            with timer("momentum"):
                self.ctx.call("mg2d_gamma5", _ptr(self.Y), _ptr(yt), S, _stream())     # Y = gamma5 D^-1 chi = D^-dag phi
            with timer("solves"):
                x, n2 = self._solve(self.Y, self.md_tol)                              # X = D^-1 Y
            iters += [n1, n2]
        with timer("momentum"):
            self.ctx.call("mg2d_hmc_momentum", _ptr(self.P), _ptr(mg.LVL[0].U), _ptr(x), None if x is None else _ptr(self.Y),
                          self.beta, float(eps), self.L, _stream())

    def link_step(self, eps: float):
        self.ctx.call("mg2d_hmc_links", _ptr(self.theta), _ptr(self.P), float(eps), _ptr(self.mg.LVL[0].U), _ptr(self._links_c64()),
                      self.theta.numel(), _stream())

    def leapfrog(self, eps: float, n_md: int, iters: list, timer=None):
        """P(eps/2) [Q(eps) P(eps)]^(n_md-1) Q(eps) P(eps/2)."""
        timer = timer or _NullTimer
        self.force_step(0.5 * eps, iters, timer)
        for i in range(n_md):
            with timer("links"):
                self.link_step(eps)
            self.force_step(eps if i < n_md - 1 else 0.5 * eps, iters, timer)

    def draw(self, k: int):
        """The random start of trajectory k: momenta P ~ N(0, 1) per link, eta with <|eta|^2> = 1 per component, and the
        pseudofermion chi = gamma5 phi = D gamma5 eta at the current links."""
        ctx, S = self.ctx, self.L * self.L
        ctx.call("mg2d_fill_gaussian", _ptr(self.P), 2 * S, 0, self.seed, 3 * k, 1.0, _stream())
        if self.flavours:
            ctx.call("mg2d_fill_gaussian", _ptr(self.eta), 4 * S, 0, self.seed, 3 * k + 1, 0.5, _stream())
            ctx.call("mg2d_gamma5", _ptr(self.Y), _ptr(self.eta), S, _stream())
            self.mg.LVL[0].apply_D(self.chi, self.Y)

    # ---- one trajectory ------------------------------------------------------------------------------------
    def trajectory(self) -> dict:
        """One HMC trajectory.  Returns dict(dH, accepted, plaquette, H0, H1, iters_md, iters_accept, times_ms, refreshed)."""
        mg, ctx, S, k = self.mg, self.ctx, self.L * self.L, self.k
        tm = _Timer(self.flavours)
        t_start = time.perf_counter()
        refreshed = False
        if self.stale and self.refresh_null_iters is not None and self.flavours:
            with tm("refresh"):
                mg.refresh(self.refresh_null_iters)
            refreshed = True
            self.stale = False
        red = self.red
        red.zero_()
        with tm("energies"):
            self.theta0.copy_(self.theta)
            self.draw(k)
            self._norm2(self.P, red[0:])
            self._action(red[1:])
            if self.flavours:
                self._norm2(self.eta, red[3:])                                    # S_f(start) = |eta|^2
        iters_md = []
        self.leapfrog(self.tau / self.n_md, self.n_md, iters_md, tm)
        it_acc = 0
        with tm("energies"):
            self._norm2(self.P, red[4:])
            self._action(red[5:])
        if self.flavours:
            with tm("solves"):
                yt, it_acc = self._solve(self.chi, self.accept_tol)
            with tm("energies"):
                self._norm2(yt, red[7:])                                          # S_f(end) = |D^-1 chi|^2
        ctx.call("mg2d_fill_uniform", _ptr(self.u), 1, 0, self.seed, 3 * k + 2, 0.0, 1.0, _lib.C128, _stream())
        r = red.cpu().tolist()
        u = float(self.u.real.cpu().item())
        V = 2 * S
        H0 = 0.5 * r[0] + self.beta * (S - r[1]) + (r[3] if self.flavours else 0.0)
        H1 = 0.5 * r[4] + self.beta * (S - r[5]) + (r[7] if self.flavours else 0.0)
        dH = H1 - H0
        accepted = bool(math.isfinite(dH) and u < math.exp(min(0.0, -dH)))
        if accepted:
            self.stale = True
            plaq = r[5] / S
        else:
            self.theta.copy_(self.theta0)
            ctx.call("mg2d_phases_to_links", _ptr(mg.LVL[0].U), _ptr(self.theta), V, _lib.C128, _stream())
            u32 = self._links_c64()
            if u32 is not None:
                ctx.call("mg2d_phases_to_links", _ptr(u32), _ptr(self.theta), V, _lib.C64, _stream())
            plaq = r[1] / S
        torch.cuda.synchronize()
        self.k += 1
        return {"trajectory": k, "dH": dH, "accepted": accepted, "exp_minus_dH": math.exp(-dH) if dH > -700 else float("inf"),
                "plaquette": plaq, "H0": H0, "H1": H1, "iters_md": iters_md, "iters_accept": it_acc, "refreshed": refreshed,
                "times_ms": dict(tm.totals(), total=1e3 * (time.perf_counter() - t_start))}


class _NullTimer:
    def __init__(self, name=None):
        pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


class _Timer:
    """Device time of the phases of a trajectory (CUDA events, resolved once at the end).  The two solves of a force step are
    counted under 'solves'; the rest of that step is the momentum kernel."""

    def __init__(self, flavours):
        self.ev, self.flavours = [], flavours

    def __call__(self, name):
        t = self

        class _Ctx:
            def __enter__(self_):
                self_.e0 = torch.cuda.Event(enable_timing=True)
                self_.e0.record()
                return self_

            def __exit__(self_, *exc):
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record()
                t.ev.append((name, self_.e0, e1))
                return False
        return _Ctx()

    def totals(self):
        torch.cuda.synchronize()
        out = {}
        for name, e0, e1 in self.ev:
            out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
        return out
