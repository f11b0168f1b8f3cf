"""ctypes binding of libmg2d_sm100.so (C ABI: include/mg2d.h).

There is NO fallback: if the shared library is missing, does not load, or the device is not sm_100, every
entry point raises.  PyTorch is used only for device memory, streams and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmg2d_sm100.so")

C128, C64 = 0, 1
MODE_APPLY, MODE_RESID = 0, 1
DOT_OUT2, DOT_OUTIN_RE, DOT_OUTIN_IM, DOT_B2, NDOTS = 0, 1, 2, 3, 4
MSC_RR, MSC_ALPHA_PREV, MSC_BETA_PREV, MSC_PP, MSC_NACT, MSC_NACT_NEXT, MSC_ITER, MSC_THRESH, MSC_SHIFTS = range(9)
MSC_MAX_SHIFTS = 64

_vp, _i, _d, _ll, _ull = C.c_void_p, C.c_int, C.c_double, C.c_longlong, C.c_ulonglong

# name -> argtypes (after the leading mg2d_ctx*); mirrors include/mg2d.h one to one
SIGNATURES = {
    "mg2d_wilson_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp],
    "mg2d_lvl0_matrix": [_vp, _vp, _vp, _d, _i, _i, _i, _i, _vp],
    "mg2d_wilson_sw_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp],
    "mg2d_wilson_sw_relax_rb": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _i, _vp],
    "mg2d_wilson_sw_relax_rb2": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp],
    "mg2d_clover_add": [_vp, _vp, _ll, _i, _vp],
    "mg2d_wilson_tm_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _vp, _vp],
    "mg2d_wilson_tm_relax_rb": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _i, _vp],
    "mg2d_wilson_tm_relax_rb2": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _vp, _vp],
    "mg2d_twist_add": [_vp, _d, _ll, _i, _vp],
    "mg2d_stencil_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _ll, _ll, _vp, _vp],
    "mg2d_block_inverse": [_vp, _vp, _i, _ll, _i, _vp],
    "mg2d_relax_jacobi": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _ll, _ll, _vp],
    "mg2d_relax_gs": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _ll, _vp],
    "mg2d_relax_gs_strip": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp],
    "mg2d_relax_rb": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _ll, _ll, _vp],
    "mg2d_wilson_relax_rb": [_vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _i, _vp],
    "mg2d_wilson_relax_rb2": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _i, _vp, _vp],
    "mg2d_premultiply": [_vp, _vp, _vp, _i, _ll, _i, _vp],
    "mg2d_relax_rb_pm": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _ll, _ll, _vp, _vp],
    "mg2d_relax_rb_pm_sweeps": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "mg2d_hop_factors": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "mg2d_lowrank_pack": [_vp, _vp, _vp, _vp, _i, _i, _ll, _i, _vp],
    "mg2d_relax_rb_lr": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _ll, _ll, _vp, _vp],
    "mg2d_relax_rb_half": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    "mg2d_to_half": [_vp, _vp, _ll, _vp],
    "mg2d_axpy_ratio2": [_vp, _vp, _vp, _vp, _vp, _vp, _d, _ll, _i, _vp],
    "mg2d_gcr_dots": [_vp, _ll, _i, _vp, _ll, _i, _vp, _vp],
    "mg2d_gcr_ortho": [_vp, _vp, _vp, _vp, _vp, _ll, _i, _vp, _vp, _ll, _i, _vp, _vp],
    "mg2d_gcr_step": [_vp, _vp, _vp, _vp, _vp, _vp, _ll, _i, _vp, _vp],
    "mg2d_gcr_step_lazy": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _ll, _i, _vp, _vp],
    "mg2d_gcr_xupdate": [_vp, _vp, _ll, _i, _vp, _ll, _i, _vp],
    "mg2d_mr_update": [_vp, _vp, _vp, _vp, _d, _ll, _i, _i, _ll, _vp],
    "mg2d_axpy": [_vp, _vp, _d, _d, _vp, _ll, _i, _vp],
    "mg2d_zero": [_vp, _ll, _i, _vp],
    "mg2d_copy": [_vp, _vp, _ll, _i, _vp],
    "mg2d_convert": [_vp, _i, _vp, _i, _ll, _vp],
    "mg2d_norm2": [_vp, _ll, _i, _vp, _vp],
    "mg2d_cdot_batch": [_vp, _ll, _i, _vp, _ll, _i, _ll, _i, _vp, _vp],
    "mg2d_scale_inv_norm": [_vp, _vp, _ll, _i, _vp],
    "mg2d_restrict": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mg2d_prolong_add": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mg2d_restrict_chiral": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mg2d_prolong_chiral": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mg2d_pack_null": [_vp, _vp, _i, _ll, _i, _i, _ll, _i, _i, _vp],
    "mg2d_norm_nn": [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "mg2d_ortho": [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "mg2d_check_ortho": [_vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp],
    "mg2d_coarse_matrix": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "mg2d_minres_solve": [_vp, _vp, _i, _vp, _vp],
    "mg2d_scale_phi": [_vp, _vp, _ll, _vp, _i, _ll, _i, _vp],
    "mg2d_comm_create": [_i, _i, C.POINTER(_vp), C.POINTER(_vp)],
    "mg2d_comm_attach": [_vp],
    "mg2d_comm_reduce": [_i],
    "mg2d_comm_error": [_vp, C.POINTER(_ll)],
    "mg2d_allreduce": [_vp, _i, _vp],
    "mg2d_halo_errors": [_vp, _i, C.POINTER(_ll)],
    "mg2d_ipc_alloc": [_ll, C.POINTER(_vp), _vp],
    "mg2d_ipc_open": [_vp, C.POINTER(_vp)],
    "mg2d_halo_exchange": [_vp, _vp, _ll, _ll, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "mg2d_fill_uniform": [_vp, _ll, _ll, _ull, _ull, _d, _d, _i, _vp],
    "mg2d_gauge_metropolis": [_vp, _i, _d, _d, _i, _i, _ull, _ull, _vp],
    "mg2d_plaquette": [_vp, _i, _i, _vp, _vp],
    "mg2d_clover_field": [_vp, _vp, _vp, _vp, _d, _i, _i, _i, _vp],
    "mg2d_phases_to_links": [_vp, _vp, _ll, _i, _vp],
    "mg2d_fill_gaussian": [_vp, _ll, _ll, _ull, _ull, _d, _vp],
    "mg2d_hmc_momentum": [_vp, _vp, _vp, _vp, _d, _d, _i, _vp],
    "mg2d_hmc_links": [_vp, _vp, _d, _vp, _vp, _ll, _vp],
    "mg2d_gamma5": [_vp, _vp, _ll, _vp],
    "mg2d_msc_pass_a": [_vp, _vp, _vp, _vp, _vp, _d, _i, _ll, _vp],
    "mg2d_msc_pass_b": [_vp, _vp, _vp, _vp, _vp, _d, _i, _ll, _vp],
    "mg2d_meson_contract": [_vp, _vp, _i, _vp, _vp],
    "mg2d_topo_charge": [_vp, _i, _vp, _vp],
    "mg2d_wilson_loops": [_vp, _i, _i, _i, _vp, _vp],
    "mg2d_s2_relax": [_vp, _vp, _i, _d, _d, _i, _i, _vp],
    "mg2d_s2_project": [_vp, _vp, _vp, _i, _d, _d, _i, _vp],
    "mg2d_s2_interpolate": [_vp, _vp, _i, _i, _vp],
    "mg2d_s2_residue_mag": [_vp, _vp, _i, _d, _d, _vp, _vp],
    "mg2d_s2_scale": [_vp, _d, _ll, _vp],
}
PLAIN = {  # entry points without the uniform (ctx, ...) -> int shape
    "mg2d_version": ([], _i),
    "mg2d_create": ([C.POINTER(_vp), _i], _i),
    "mg2d_destroy": ([_vp], _i),
    "mg2d_last_error": ([_vp], C.c_char_p),
    "mg2d_launch_count": ([_vp], _i),
    "mg2d_comm_mailbox_bytes": ([], _i),
    "mg2d_lowrank_supported": ([_i, _i], _i),
}


class HaloLink(C.Structure):
    """mg2d_halo_link of include/mg2d.h."""
    _fields_ = [("slot_mine", _vp), ("slot_prev", _vp), ("slot_next", _vp), ("push_next_lo", _vp), ("push_prev_hi", _vp),
                ("wait", _i)]


_lib = None
TRACE_TAG = "-"                                          # multigrid level of the launches that follow (set by Level)
TRACE = [] if os.environ.get("MG2D_TRACE") else None     # list of (entry point, start event, end event) when tracing


def trace_begin():
    global TRACE
    TRACE = []


def trace_report(reset: bool = True):
    """{entry point: (calls, total ms)} of the traced launches (synchronises)."""
    global TRACE
    import torch
    torch.cuda.synchronize()
    out = {}
    for name, e0, e1 in TRACE or []:
        c, t = out.get(name, (0, 0.0))
        out[name] = (c + 1, t + e0.elapsed_time(e1))
    if reset:
        TRACE = None
    return out


class MG2DError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises MG2DError when it is absent -- there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MG2DError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C 2d_multigrid_b200/csrc).  This package has no CPU/PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (args, res) in PLAIN.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = args, res
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = [_vp] + args, _i
    _lib = lib
    return lib


class Context:
    """One mg2d_ctx per GPU / stream of work (mg2d_create / mg2d_destroy)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = _vp()
        rc = self.lib.mg2d_create(C.byref(h), device)
        if rc != 0:
            raise MG2DError(f"mg2d_create(device={device}) failed with code {rc} "
                            "(needs a CUDA device of compute capability 10.x; no fallback exists)")
        self.h = h
        self.device = device

    def call(self, name: str, *args):
        if TRACE is not None:
            return self._traced_call(name, *args)
        rc = getattr(self.lib, name)(self.h, *args)
        if rc != 0:
            raise MG2DError(f"{name} failed ({rc}): {self.lib.mg2d_last_error(self.h).decode()}")

    def _traced_call(self, name: str, *args):
        """MG2D_TRACE=1 (or trace_begin()): bracket every entry point with CUDA events on the current stream; trace_report()
        sums the device time per entry point.  Eager launches only (events cannot be recorded into a graph capture)."""
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(self.lib, name)(self.h, *args)
        e1.record()
        if rc != 0:
            raise MG2DError(f"{name} failed ({rc}): {self.lib.mg2d_last_error(self.h).decode()}")
        TRACE.append((f"{name}@L{TRACE_TAG}", e0, e1))

    @property
    def launches(self) -> int:
        return int(self.lib.mg2d_launch_count(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.mg2d_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
