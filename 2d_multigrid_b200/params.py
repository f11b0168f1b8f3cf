"""MGParams -- the reference's `class params` (S6/params.h:38-128) as a frozen-ish dataclass.

The reference is driven by 8 positional CLI arguments
    ./a.out L num_iters block gen_null m nlevels t_flag n_copies          (S6/params.h:42-50)
plus compile-time constants (gs_flag, quad, res_threshold, stencil ...).  `make_params` keeps those names and
meanings; `from_argv` accepts the reference's argv order.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field


@dataclass
class MGParams:
    L: int
    mass: float                      # argv[5] "m"; used linearly (it is m^2 for laplace)
    stencil: str = "wilson"          # S6/params.h:68-69
    nlevels: int = 2                 # argv[6]: number of coarse levels; levels are 0..nlevels
    block: object = 2                # argv[3]: block_x = block_y; an int, or one block size per coarsening step
                                     # (S5L/setup.h:2-10 `block_x[level]`: e.g. [4, 2, 2] = 4x4 aggregates on the fine lattice)
    n_smooth: int = 3                # argv[2] num_iters: smoother sweeps per visit
    smoother: str = "gs"             # 'gs' (gs_flag=1, S6/params.h:61) | 'jacobi' (gs_flag=0) | 'mr' (north_star)
                                     # | 'rbgs' (red-black ordering of the GS update)
    ntl: bool = False                # argv[7] t_flag
    n_copies: int = 4                # argv[8]
    tol: float = 1.0e-13             # res_threshold, S6/params.h:67
    max_iters: int = 50000           # S6/params.h:64
    quad: int = 1                    # S6/params.h:63
    n_null: int | None = None        # near-null vectors per chirality (wilson) / total (laplace);
                                     # coarse dof = n_dof_scale = 2*n_null (wilson) | n_null (laplace).
                                     # default 2 -> n_dof_scale 4 | 2 as S6/params.h:75,81
    null_iters: int = 500            # S6/modules_main.h:193
    null_chunk: int = 4              # iters_per_norm, S6/level.h:190
    seed: int = 4302529              # S6/mgrid_ntl.cpp:35
    dtype: str = "complex128"        # 'complex128' | 'complex64'
    mr_omega: float = 1.0
    min_res_flag: int = 1            # S6/modules_main.h:391
    n_pre: object = None             # pre-smoothing sweeps: int or list per level (default n_smooth, as the reference)
    n_post: object = None            # post-smoothing sweeps: int or list per level (default n_smooth); the coarsest
                                     # level is relaxed once per cycle with n_post (S6/modules_main.h:270-273)
    cycle: str = "V"                 # 'V' = f_MG_simple (one recursive visit per level) | 'K' = Krylov-accelerated coarse
                                     # solves (k_inner FGCR steps per coarse level; SURVEY 8f N3, no reference counterpart)
    k_inner: int = 2
    chiral_transfer: bool = True     # wilson: restriction / prolongation on the chirality-compacted projector
    matrix_free: bool | None = None  # level-0 Wilson operator applied from the links (no D0 stored).
                                     # default: True for smoother 'mr', False for 'gs'/'jacobi' (they need D0)
    csw: float = 0.0                 # clover (Sheikholeslami-Wohlert) coefficient of the level-0 Wilson operator: self block
                                     # (2+m) 1 + f(s) sigma3, f(s) = (csw/8) sum of Im U_P over the 4 plaquettes at s; 1 = tree level
    mu: float = 0.0                  # twisted mass of the level-0 Wilson(-clover) operator: + i mu gamma5 = i mu sigma3 on the self
                                     # block, so D^dag D gains mu^2 and no singular value is below |mu| (solvable at m = m_crit)
    size: list = field(default_factory=list)
    n_dof: list = field(default_factory=list)

    def __post_init__(self):
        if self.stencil not in ("wilson", "laplace"):
            raise ValueError(f"Incorrect stencil: {self.stencil}. Need either 'laplace' or 'wilson'")
        if self.smoother not in ("gs", "jacobi", "mr", "rbgs"):
            raise ValueError("smoother must be 'gs', 'jacobi', 'mr' or 'rbgs'")
        if self.cycle not in ("V", "K") or not (1 <= self.k_inner <= 8):
            raise ValueError("cycle must be 'V' or 'K' with 1 <= k_inner <= 8")
        if self.dtype not in ("complex128", "complex64"):
            raise ValueError("dtype must be complex128 or complex64")
        if self.ntl and self.nlevels < 2:
            raise ValueError(f"Need at least 2 levels for non-telescoping. Have {self.nlevels}")  # S6/params.h:52-55
        if self.n_null is None:
            self.n_null = 2
        n0 = 2 if self.stencil == "wilson" else 1
        self.n_dof_scale = 2 * self.n_null if self.stencil == "wilson" else self.n_null
        if isinstance(self.block, (list, tuple)):
            self.blocks = [int(b) for b in self.block]
            if len(self.blocks) != self.nlevels or any(b < 1 for b in self.blocks):
                raise ValueError("a per-level block list needs one entry >= 1 per coarsening step (nlevels)")
            self.block = self.blocks[0] if self.blocks else 1
        else:
            self.block = int(self.block)
            self.blocks = [self.block] * self.nlevels
            max_levels = math.ceil(math.log2(self.L) / math.log2(self.block)) if self.block > 1 else 0
            if self.nlevels > max_levels:                                               # S6/params.h:100-106
                raise ValueError(f"Too many levels {self.nlevels}. Can only have {max_levels} levels for block size "
                                 f"{self.block} for lattice of size {self.L}")
        self.size, self.n_dof = [self.L], [n0]
        for lvl in range(self.nlevels):
            if self.size[-1] % self.blocks[lvl] or self.size[-1] // self.blocks[lvl] < 1:
                raise ValueError("lattice size must be divisible by the block size on every level")
            self.size.append(self.size[-1] // self.blocks[lvl])
            self.n_dof.append(self.n_dof_scale)
        def per_level(v):
            if v is None:
                return [self.n_smooth] * (self.nlevels + 1)
            if isinstance(v, int):
                return [v] * (self.nlevels + 1)
            v = list(v)
            if len(v) != self.nlevels + 1:
                raise ValueError("n_pre / n_post lists need one entry per level (nlevels + 1)")
            return v
        self.pre, self.post = per_level(self.n_pre), per_level(self.n_post)
        if self.matrix_free is None:
            self.matrix_free = self.stencil == "wilson" and self.smoother in ("mr", "rbgs")
        if self.matrix_free and (self.stencil != "wilson" or self.smoother not in ("mr", "rbgs")):
            raise ValueError("matrix_free needs stencil='wilson' and smoother 'mr' or 'rbgs'")
        self.csw = float(self.csw)
        if self.csw != 0.0 and self.stencil != "wilson":
            raise ValueError("the clover term (csw != 0) exists for stencil='wilson' only")
        if self.csw != 0.0 and not 2.0 + self.mass - abs(self.csw) / 2.0 > 0.0:
            # |f| <= |csw|/2, so this bound keeps every clover self block diag(2+m+f, 2+m-f) invertible
            raise ValueError(f"clover self blocks may be singular: need 2 + mass - |csw|/2 > 0 (mass {self.mass}, csw {self.csw})")
        self.mu = float(self.mu)
        if not math.isfinite(self.mu):
            raise ValueError(f"the twisted mass must be finite (mu {self.mu})")
        if self.mu != 0.0 and self.stencil != "wilson":
            raise ValueError("the twisted mass (mu != 0) exists for stencil='wilson' only")

    @property
    def diag(self) -> float:
        """D0 of level 0: 1/scale[0] (S6/params.h:76,82), with the sign of S6/level.h:148,165."""
        return (2.0 + self.mass) if self.stencil == "wilson" else -(4.0 + self.mass)


def make_params(L, mass, stencil="wilson", nlevels=2, block=2, n_null=None, n_smooth=3, smoother="gs", ntl=False,
                n_copies=4, tol=1e-13, max_iters=50000, quad=1, null_iters=500, null_chunk=4, seed=4302529,
                dtype="complex128", **kw) -> MGParams:
    return MGParams(L=L, mass=mass, stencil=stencil, nlevels=nlevels, block=block, n_null=n_null, n_smooth=n_smooth,
                    smoother=smoother, ntl=ntl, n_copies=n_copies, tol=tol, max_iters=max_iters, quad=quad,
                    null_iters=null_iters, null_chunk=null_chunk, seed=seed, dtype=dtype, **kw)


def from_argv(argv, stencil="wilson", **kw) -> MGParams:
    """The reference CLI: L num_iters block gen_null m nlevels t_flag n_copies (S6/params.h:42-50)."""
    L, num_iters, block, _gen_null = int(argv[0]), int(argv[1]), int(argv[2]), int(argv[3])
    m, nlevels, t_flag, n_copies = float(argv[4]), int(argv[5]), int(argv[6]), int(argv[7])
    return make_params(L, m, stencil=stencil, nlevels=nlevels, block=block, n_smooth=num_iters, ntl=bool(t_flag),
                       n_copies=n_copies, **kw)
