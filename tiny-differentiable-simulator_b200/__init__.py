"""tds_b200: B200-native batched rigid-body env-step behind the reference's plugin boundary.

Host-side mirror of the reference's interface for the hot path (names follow
python/pytinydiffsim*.{cc,inl,h} and examples/ars/ars_vectorized_environment.h); all compute
happens in libtds_b200.so (hand-written sm_100a CUDA, C-ABI in include/tds_b200.h).  There is no
CPU fallback: creating a simulator without the library or without a GPU raises.
"""
from ._lib import lib, lib_path, LibraryMissing  # noqa: F401
from .model import compile_urdf, load_model, save_model, model_dims, merge_models  # noqa: F401
from .rigid import RigidWorld  # noqa: F401
from . import rigid  # noqa: F401
from .sim import BatchSim, MODE_FD, MODE_NOCONTACT, MODE_FULL, MODE_WORLD, PREC_MIXED, PREC_F64, PREC_F32, PREC_AUTO  # noqa: F401
from .envs import (VectorizedLaikagoEnv, VectorizedLaikagoEnvOutput, VectorizedAntEnv, CudaModelV1, laikago_sim,  # noqa: F401
                   ant_sim)


def __getattr__(name):   # tds_b200.autograd (torch.autograd through the steps) imports torch: loaded on first use
    if name == "autograd":
        import importlib
        return importlib.import_module(__name__ + ".autograd")
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
