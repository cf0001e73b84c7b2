"""gglasso_b200 -- B200 (sm_100a) implementation of GGLasso's ADMM hot path.

Drop-in replacements for ``gglasso.solver.admm_solver.ADMM_MGL``,
``gglasso.solver.single_admm_solver.ADMM_SGL`` and ``block_SGL``, and of the second-order solvers
``gglasso.solver.ppdna_solver.PPDNA`` / ``warmPPDNA`` (same call signatures and return dicts), backed by hand-written CUDA kernels behind a C ABI (include/gglasso_b200.h).
``install()`` rebinds those names inside an importable ``gglasso`` package so that
``glasso_problem`` and ``grid_search`` run unmodified on top of the GPU path.
``ADMM_MGL_batch`` (no counterpart in the reference, so ``install()`` leaves it alone) solves many MGL problems of the
same shape in one device loop.  ``stability_selection`` (also without counterpart) chooses lambda1 of SGL or MGL by
StARS from raw samples, on the device.  ``block_MGL`` (also without counterpart) solves GGL / FGL component by
component of an exact screening graph computed on the device, small components in ragged device batches.
"""
from .solver.admm_solver import ADMM_MGL, ADMM_MGL_batch, block_MGL, mgl_connected_components  # noqa: F401
from .solver.single_admm_solver import ADMM_SGL, block_SGL, get_connected_components  # noqa: F401
from .solver.functional_sgl_admm import ADMM_FSGL  # noqa: F401
from .solver.ext_admm_solver import ext_ADMM_MGL  # noqa: F401
from .solver.ppdna_solver import PPDNA, warmPPDNA  # noqa: F401
from .stability import stability_selection  # noqa: F401
from ._lib import GGLassoB200Error, LIB_PATH  # noqa: F401

__version__ = "0.1.0"


def install():
    """Patch an importable ``gglasso`` so its façade and model selection call the B200 solvers.

    The reference binds the solver names at import time (src/gglasso/problem.py:10-11,
    src/gglasso/helper/model_selection.py:13), so every holder of the name is rebound.
    """
    import importlib
    patched = []
    uninstall()
    targets = {
        "gglasso.solver.admm_solver": {"ADMM_MGL": ADMM_MGL},
        "gglasso.solver.single_admm_solver": {"ADMM_SGL": ADMM_SGL, "block_SGL": block_SGL},
        "gglasso.problem": {"ADMM_MGL": ADMM_MGL, "ADMM_SGL": ADMM_SGL, "block_SGL": block_SGL,
                            "ext_ADMM_MGL": ext_ADMM_MGL},
        "gglasso.helper.model_selection": {"ADMM_SGL": ADMM_SGL, "block_SGL": block_SGL},
        "gglasso.solver.ppdna_solver": {"ADMM_MGL": ADMM_MGL, "PPDNA": PPDNA, "warmPPDNA": warmPPDNA},
        "gglasso.solver.functional_sgl_admm": {"ADMM_FSGL": ADMM_FSGL},
        "gglasso.solver.ext_admm_solver": {"ext_ADMM_MGL": ext_ADMM_MGL},
    }
    for modname, names in targets.items():
        try:
            mod = importlib.import_module(modname)
        except Exception:
            continue
        for n, fn in names.items():
            if hasattr(mod, n):
                _ORIGINALS.append((mod, n, getattr(mod, n)))
                setattr(mod, n, fn)
                patched.append(f"{modname}.{n}")
    return patched


_ORIGINALS = []


def uninstall():
    """undo ``install()``: restore the reference's own solver callables (used by tests that run both paths)."""
    while _ORIGINALS:
        mod, n, fn = _ORIGINALS.pop()
        setattr(mod, n, fn)
