"""B200-native batched cached-graph navigation environments (hot path of a2cat-vn-pytorch).

The directory name carries a hyphen (it mirrors the reference repo name), so import it with
``importlib.import_module("a2cat-vn-pytorch_b200")`` or through the ``vn_b200`` alias module at
the repository root.
"""
from . import scenes, tables, spaces  # noqa: F401
from .tables import (FAMILIES, GYM_GRAPH, GRAPH_ENV_ORIENTED, GRAPH_ENV_ORIENTED_POSITION, SIMPLE_GRAPH,  # noqa: F401
                     THOR_CACHED, compile_world)


def __getattr__(name):
    # torch / CUDA dependent modules are imported lazily so that the host-side compiler and the
    # synthetic scenes stay usable (and testable) without torch being imported.
    import importlib
    if name in ("lib", "store", "vec_env", "rollout", "build", "loaders", "single_env", "evaluation",
                "nn"):
        return importlib.import_module("." + name, __name__)
    if name in ("GraphVecEnv", "shard_range", "gather_plane", "reduce_stats"):
        return getattr(importlib.import_module(".vec_env", __name__), name)
    if name == "GraphEnv":
        return importlib.import_module(".single_env", __name__).GraphEnv
    if name == "DeviceWorld":
        return importlib.import_module(".store", __name__).DeviceWorld
    raise AttributeError(name)

__version__ = "0.1.0"
