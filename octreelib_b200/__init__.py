"""
octreelib_b200 -- a from-scratch, B200-native (sm_100a) implementation of the data-parallel grid
pipeline of prime-slam/octreelib: `Grid.insert_points` -> `subdivide` -> `filter` /
`get_leaf_points` -> per-leaf batched RANSAC, behind the reference's unchanged Python API.

    from octreelib_b200.grid import Grid, GridConfig          # instead of octreelib.grid
    import octreelib_b200; octreelib_b200.install_as("octreelib")   # or alias the whole package

Importing the package needs neither a GPU nor the native library; the first operation that
touches point data does (there is no CPU fallback).
"""
import importlib
import sys

__version__ = "0.1.0"
__all__ = ["install_as", "release_cached_memory", "grid", "octree", "octree_manager", "internal", "ransac", "criteria", "leaf_maps"]

_SUBMODULES = ["internal", "internal.interfaces", "internal.point", "internal.typing", "internal.voxel", "octree",
               "octree.octree_base", "octree.octree", "octree_manager", "octree_manager.octree_manager", "ransac",
               "ransac.cuda_ransac", "grid", "grid.grid_base", "grid.grid"]


def install_as(name: str = "octreelib"):
    """Register this package (and its sub-modules) in `sys.modules` under `name`, so that existing
    `import octreelib...` statements resolve to the B200 build."""
    pkg = importlib.import_module(__name__)
    sys.modules[name] = pkg
    for sub in _SUBMODULES:
        sys.modules[f"{name}.{sub}"] = importlib.import_module(f"{__name__}.{sub}")
    return pkg


def release_cached_memory() -> int:
    """Return the device memory the native library keeps cached between grids to torch's allocator (bytes released)."""
    from .forest import release_cached_memory as _release

    return _release()


def __getattr__(attr):
    if attr in ("grid", "octree", "octree_manager", "internal", "ransac", "criteria", "leaf_maps"):
        return importlib.import_module(f"{__name__}.{attr}")
    raise AttributeError(attr)
