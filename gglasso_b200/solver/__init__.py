from .admm_solver import ADMM_MGL, ADMM_MGL_batch  # noqa: F401
from .single_admm_solver import ADMM_SGL, block_SGL, get_connected_components  # noqa: F401
from .functional_sgl_admm import ADMM_FSGL  # noqa: F401
