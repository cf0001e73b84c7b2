"""ctypes binding of libgglasso_b200.so (C ABI declared in include/gglasso_b200.h).

There is deliberately no CPU fallback: if the shared library is missing or a call fails the
caller gets an exception.  Build with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C gglasso_b200/csrc``.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# GGLASSO_B200_LIB: alternative build of the same library (instrumented diagnostics builds, scripts/gpu_tr_timing.sh)
LIB_PATH = os.environ.get("GGLASSO_B200_LIB") or os.path.join(_HERE, "libgglasso_b200.so")

CTRL_STRIDE = 16
HIST_STRIDE = 5
NPART = 5
C_RHO, C_XSCALE, C_DONE, C_ITER, C_R, C_S, C_EPRI, C_EDUAL, C_STATUS, C_LAM1, C_LAM2 = range(11)

_vp, _i, _d, _sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_size_t

# name -> (restype, argtypes); mirrors include/gglasso_b200.h one to one
SIGNATURES = {
    "gg_version": (_i, []),
    "gg_launch_count": (ctypes.c_longlong, []),
    "gg_build_w": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "gg_eigh_workspace_bytes": (_sz, [_i, _i]),
    "gg_eigh": (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _sz, _i, _i, _d, _i, _d, ctypes.POINTER(_i), _vp, _vp]),
    "gg_sytrd_profile": (_i, [_vp, _vp, _i, _i, _vp, _sz, _i, _vp]),
    "gg_sytrd_write_depth": (_i, []),
    "gg_sytrd_phase_clock": (_i, [ctypes.POINTER(ctypes.c_ulonglong)]),
    "gg_recon": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "gg_sgl_nparts": (_i, [_i, _i]),
    "gg_prox_sgl": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _vp, _i, _i, _vp, _vp, _vp]),
    "gg_prox_fsgl": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _i, _i, _i, _vp, _vp, _vp]),
    "gg_mgl_ntile": (_i, [_i]),
    "gg_mgl_upper_nparts": (_i, [_i]),
    "gg_jacobi_max": (_i, []),
    "gg_prox_mgl_upper": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _vp, _vp]),
    "gg_build_w_upper": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "gg_mirror_upper": (_i, [_vp, _vp, _i, _i, _vp]),
    "gg_prox_mgl": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _vp, _vp]),
    "gg_prox_mgl_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _vp, _vp]),
    "gg_prox_mgl_upper_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _vp, _vp]),
    "gg_prox_mgl_ragged": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _vp, _vp, _vp]),
    "gg_mgl_screen": (_i, [_vp, _vp, _d, _d, _i, _i, _i, _vp, _vp]),
    "gg_build_w_upper_batch": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "gg_add3": (_i, [_vp, _vp, _vp, _vp, _sz, _vp]),
    "gg_pack_bands": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "gg_pack_bands_p2p": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "gg_prox_band_p2p": (_i, [_vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _i, _i, _vp]),
    "gg_unpack_dual": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "gg_prox_band": (_i, [_vp, _vp, _vp, _d, _d, _i, _i, _i, _i, _i, _vp]),
    "gg_ext_theta": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "gg_ext_lambda": (_i, [_vp, _vp, _vp, _i, _i, _i, _d, _vp, _vp, _vp]),
    "gg_ext_dual": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp]),
    "gg_dual_update": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "gg_stop_update": (_i, [_vp, _i, _vp, _vp, _i, _vp, _d, _d, _i, _i, _vp]),
    "gg_scale_pending": (_i, [_vp, _vp, _i, _i, _i, _vp]),
    "gg_objective_nparts": (_i, [_i]),
    "gg_objective": (_i, [_vp, _vp, _vp, _d, _d, _i, _i, _i, _vp, _vp]),
    "gg_asym_max": (_i, [_vp, _i, _i, _vp, _vp]),
    "gg_gershgorin_min": (_i, [_vp, _i, _i, _vp, _sz, _vp, _vp]),
    "gg_host_tv1d": (None, [ctypes.POINTER(_d), _i, _i, _d]),
    "gg_ppdna_build": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "gg_ppdna_spectral": (_i, [_vp, _vp, _d, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gg_ppdna_nparts": (_i, [_i]),
    "gg_ppdna_prox": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _d, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gg_ppdna_jp_nparts": (_i, [_i]),
    "gg_ppdna_jp": (_i, [_vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "gg_ppdna_hess": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gg_ppdna_cg_init": (_i, [_vp, _i, _i, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "gg_ppdna_cg": (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _d, _d, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                         _vp]),
    "gg_subsample_cov": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "gg_edge_count": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "gg_stars_instability": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
}

_LIB = None


class GGLassoB200Error(RuntimeError):
    pass


def load():
    """Load the CUDA extension; raises if it has not been built (no fallback path exists)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise GGLassoB200Error(
                f"{LIB_PATH} not found: the CUDA extension is required (build it with "
                "`make -C gglasso_b200/csrc` or __graft_entry__.build()); there is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = lib
    return _LIB


def check(rc, what):
    if rc != 0:
        raise GGLassoB200Error(f"{what} failed with code {rc}"
                               + (" (CUDA error)" if rc > 0 else " (invalid argument)"))
