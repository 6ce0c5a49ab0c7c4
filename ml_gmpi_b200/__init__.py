"""B200-native multiplane-image renderer: drop-in for the render path of apple/ml-gmpi
(gmpi/core/mpi.py MPI.forward + homography, driven by MPIRenderer.render)."""
from . import _lib  # noqa: F401
from ._build import build_library  # noqa: F401
from .mpi import (MPI, MPIOutOfPlaneError, check_range, expand_factored, occupancy_map, render_frames, render_views,  # noqa: F401
                  render_views_factored)

__all__ = ["MPI", "MPIOutOfPlaneError", "render_views", "render_views_factored", "render_frames", "expand_factored", "check_range",
           "occupancy_map", "build_library"]
