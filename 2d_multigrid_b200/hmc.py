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

flavours = 1 (RHMC): S_f = phi^dag r_{-1/2}(M) phi with M = D^dag D and r_p(x) = alpha0 + sum_k alpha_k / (x + beta_k) ~ x^p on the
spectral range [a, b] (rational.py).  The heat bath draws eta as above and sets phi = r_{+1/4}(M) eta, so S_f(start) = |eta|^2;
the force is sum_k alpha_k (-2 Re[Y_k^dag dD/dtheta X_k]) with X_k = (M + beta_k)^-1 phi from one multi-shift CG (rhmc.py) and
Y_k = D X_k, one mg2d_hmc_momentum call per pole; the accept step is S_f(end) = alpha0 |phi|^2 + Re <phi, sum_k alpha_k x_k>.
The multi-shift solves use the level-0 links only, so the coarse hierarchy is never refreshed.
"""
from __future__ import annotations

import math
import time

import torch

from . import _lib
from ._lib import MG2DError
from .mg import MG, _ptr, _stream
from .params import MGParams
from .rational import MD_TOL, PRECISE_TOL, rational_approx
from .rhmc import multishift_cg

_INV_ITER_STREAM = 2 ** 63 - 1       # counter stream of the start vector of the lambda_min estimate (trajectories use 3k + j)


class HMC:
    """HMC(params, theta, beta, ...).trajectory() -> dict.

    params: a complex128, matrix-free (smoother 'rbgs' or 'mr') Wilson MGParams without clover, twist or NTL; the hierarchy is
    built once by setup() at theta.  theta[L*L, 2]: float64 link phases (copied).  tau / n_md: trajectory length and leapfrog
    steps.  flavours: 2 (det D^dag D), 1 (|det D| = det (D^dag D)^(1/2), RHMC) or 0 (pure gauge).  md_tol: relative residual of
    the force solves; accept_tol: of the final action's solve (and of the flavours = 1 heat bath).  spectrum = (a, b): the
    range of D^dag D the rational approximations of flavours = 1 cover (default: b = (|2+m| + 2 sqrt 2)^2, a rigorous bound, and
    a = 1/4 of lambda_min estimated at construction by inverse iteration with multigrid solves).  refresh_null_iters: sweeps of MG.refresh after an accepted trajectory (None: never refresh;
    default 8, measured in DESIGN section 4).
    precond_dtype / use_graph: passed to solve() (outer FGCR(8))."""

    def __init__(self, params: MGParams, theta, beta: float, tau: float = 1.0, n_md: int = 10, flavours: int = 2, seed: int = 1,
                 md_tol: float = 1e-10, accept_tol: float = 1e-12, refresh_null_iters: int | None = 8,
                 precond_dtype: str | None = None, use_graph: bool = True, device: int | None = None, spectrum=None):
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
        if flavours not in (0, 1, 2):
            raise ValueError("flavours must be 0 (pure gauge), 1 or 2")
        if spectrum is not None:
            a, b = (float(v) for v in spectrum)
            if not (math.isfinite(a) and math.isfinite(b) and 0.0 < a < b):
                raise ValueError(f"spectrum must be (a, b) with 0 < a < b, got {spectrum}")
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
        if self.flavours == 1:
            self._setup_rational(spectrum)

    # ---- one flavour ---------------------------------------------------------------------------------------
    MSC_MAX_ITERS = 100000

    def lambda_min_estimate(self, steps: int = 6, tol: float = 1e-8) -> float:
        """Rayleigh quotient 1 / <x, M^-1 x> (an upper bound on lambda_min(M)) after `steps` inverse-iteration steps
        x <- M^-1 x / |M^-1 x|, M^-1 = D^-1 gamma5 D^-1 gamma5, with multigrid solves from a counter-generator start."""
        S = self.L * self.L
        x = torch.empty((S, 2), dtype=torch.complex128, device=self.device)
        g = torch.empty_like(x)
        self.ctx.call("mg2d_fill_gaussian", _ptr(x), 4 * S, 0, self.seed, _INV_ITER_STREAM, 0.5, _stream())
        lam = float("inf")
        for _ in range(steps):
            x /= torch.linalg.vector_norm(x)
            self.ctx.call("mg2d_gamma5", _ptr(g), _ptr(x), S, _stream())
            z, _ = self._solve(g, tol)
            self.ctx.call("mg2d_gamma5", _ptr(g), _ptr(z), S, _stream())
            y, _ = self._solve(g, tol)
            lam = 1.0 / float(torch.vdot(x.reshape(-1), y.reshape(-1)).real)
            x = y.clone()
        return lam

    def _setup_rational(self, spectrum):
        if spectrum is None:
            b = (abs(2.0 + self.p.mass) + 2.0 * math.sqrt(2.0)) ** 2
            a = 0.25 * self.lambda_min_estimate()
            if not a < b:
                raise MG2DError(f"HMC: the lambda_min estimate {4 * a:.6g} is not below the bound {b:.6g}")
        else:
            a, b = (float(v) for v in spectrum)
        self.spectrum = (a, b)
        self.r_md = rational_approx(-0.5, a, b, MD_TOL)
        self.r_acc = rational_approx(-0.5, a, b, PRECISE_TOL)
        self.r_hb = rational_approx(0.25, a, b, PRECISE_TOL)
        self.phi = torch.empty_like(self.eta)
        self.red1 = torch.zeros(2, dtype=torch.float64, device=self.device)

    def _msc(self, rhs, r, tol, accumulate):
        out, info = multishift_cg(self.mg, rhs, r.beta, tol, self.MSC_MAX_ITERS, weights=r.alpha if accumulate else None)
        if not info["converged"]:
            raise MG2DError(f"HMC: multi-shift solve did not converge in {info['iters']} iterations")
        return out, info

    def _heatbath(self):
        """phi = r_{+1/4}(M) eta (precise, accumulate mode); returns the iterations."""
        y, info = self._msc(self.eta, self.r_hb, self.accept_tol, True)
        self.phi.copy_(y)
        self.ctx.call("mg2d_axpy", _ptr(self.phi), _ptr(self.eta), self.r_hb.alpha0, 0.0, None, self.phi.numel(), _lib.C128,
                      _stream())
        return info["iters"]

    def _force_one(self, eps, iters, timer):
        mg, S, r = self.mg, self.L * self.L, self.r_md
        with timer("solves"):
            X, info = self._msc(self.phi, r, self.md_tol, False)
        iters.append(info["iters"])
        with timer("momentum"):
            U = _ptr(mg.LVL[0].U)
            for k in range(r.n):
                mg.LVL[0].apply_D(self.Y, X[k])
                self.ctx.call("mg2d_hmc_momentum", _ptr(self.P), U, _ptr(X[k]), _ptr(self.Y), 0.0, float(eps) * r.alpha[k], self.L,
                              _stream())
            self.ctx.call("mg2d_hmc_momentum", _ptr(self.P), U, None, None, self.beta, float(eps), self.L, _stream())

    def _trajectory_one(self) -> dict:
        mg, ctx, S, k = self.mg, self.ctx, self.L * self.L, self.k
        tm = _Timer(self.flavours)
        t_start = time.perf_counter()
        red = self.red
        red.zero_()
        with tm("energies"):
            self.theta0.copy_(self.theta)
            self.draw(k, heatbath=False)
        with tm("solves"):
            it_hb = self._heatbath()
        with tm("energies"):
            self._norm2(self.P, red[0:])
            self._action(red[1:])
            self._norm2(self.eta, red[3:])                                       # S_f(start) = |eta|^2
        iters_md = []
        self.leapfrog(self.tau / self.n_md, self.n_md, iters_md, tm)
        with tm("energies"):
            self._norm2(self.P, red[4:])
            self._action(red[5:])
        with tm("solves"):
            y, info = self._msc(self.phi, self.r_acc, self.accept_tol, True)
        with tm("energies"):
            self._norm2(self.phi, red[6:])
            ctx.call("mg2d_cdot_batch", _ptr(self.phi), 0, 1, _ptr(y), 0, 1, 2 * S, _lib.C128, _ptr(self.red1), _stream())
        ctx.call("mg2d_fill_uniform", _ptr(self.u), 1, 0, self.seed, 3 * k + 2, 0.0, 1.0, _lib.C128, _stream())
        r = red.cpu().tolist()
        phi_y = float(self.red1[0].item())
        u = float(self.u.real.cpu().item())
        if info["ritz"][0] < self.spectrum[0]:
            raise MG2DError(f"HMC: the smallest Ritz value {info['ritz'][0]:.6g} of D^dag D is below the spectrum's a = "
                            f"{self.spectrum[0]:.6g}: the rational approximations no longer cover the spectrum")
        H0 = 0.5 * r[0] + self.beta * (S - r[1]) + r[3]
        H1 = 0.5 * r[4] + self.beta * (S - r[5]) + self.r_acc.alpha0 * r[6] + phi_y     # S_f(end) = a0 |phi|^2 + Re <phi, y>
        dH = H1 - H0
        accepted = bool(math.isfinite(dH) and u < math.exp(min(0.0, -dH)))
        if accepted:
            plaq = r[5] / S
        else:
            self.theta.copy_(self.theta0)
            ctx.call("mg2d_phases_to_links", _ptr(mg.LVL[0].U), _ptr(self.theta), 2 * S, _lib.C128, _stream())
            u32 = self._links_c64()
            if u32 is not None:
                ctx.call("mg2d_phases_to_links", _ptr(u32), _ptr(self.theta), 2 * S, _lib.C64, _stream())
            plaq = r[1] / S
        torch.cuda.synchronize()
        self.k += 1
        return {"trajectory": k, "dH": dH, "accepted": accepted, "exp_minus_dH": math.exp(-dH) if dH > -700 else float("inf"),
                "plaquette": plaq, "H0": H0, "H1": H1, "iters_md": iters_md, "iters_accept": info["iters"],
                "iters_heatbath": it_hb, "poles": (self.r_md.n, self.r_acc.n), "spectrum": self.spectrum, "ritz": info["ritz"],
                "refreshed": False, "times_ms": dict(tm.totals(), total=1e3 * (time.perf_counter() - t_start))}

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
        """P -= eps dS/dtheta at the current links (two solves for flavours = 2, one multi-shift solve for flavours = 1)."""
        mg, S = self.mg, self.L * self.L
        timer = timer or _NullTimer
        if self.flavours == 1:
            return self._force_one(eps, iters, timer)
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

    def draw(self, k: int, heatbath: bool = True):
        """The random start of trajectory k: momenta P ~ N(0, 1) per link, eta with <|eta|^2> = 1 per component, and the
        pseudofermion chi = gamma5 phi = D gamma5 eta at the current links (flavours = 1: phi = r_{+1/4}(M) eta, unless
        heatbath is False)."""
        ctx, S = self.ctx, self.L * self.L
        ctx.call("mg2d_fill_gaussian", _ptr(self.P), 2 * S, 0, self.seed, 3 * k, 1.0, _stream())
        if self.flavours:
            ctx.call("mg2d_fill_gaussian", _ptr(self.eta), 4 * S, 0, self.seed, 3 * k + 1, 0.5, _stream())
        if self.flavours == 1:
            if heatbath:
                self._heatbath()
            return
        if self.flavours:
            ctx.call("mg2d_gamma5", _ptr(self.Y), _ptr(self.eta), S, _stream())
            self.mg.LVL[0].apply_D(self.chi, self.Y)

    # ---- one trajectory ------------------------------------------------------------------------------------
    def trajectory(self) -> dict:
        """One HMC trajectory.  Returns dict(dH, accepted, plaquette, H0, H1, iters_md, iters_accept, times_ms, refreshed);
        flavours = 1 adds iters_heatbath, poles (MD, precise), spectrum (a, b) and ritz (the extreme Ritz values of D^dag D from
        the accept solve) and raises MG2DError when the smallest Ritz value is below a."""
        if self.flavours == 1:
            return self._trajectory_one()
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
