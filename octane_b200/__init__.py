"""octane_b200 -- B200-native implementation of OCTANE's dense variational
optical-flow path (pyramid -> coefficient build -> Jacobi-PCG -> prolongation ->
pixel-to-u/v navigation) behind the reference's operator surface.

The product is csrc/ (hand-written sm_100a CUDA + the C ABI of
include/octane_b200.h, built into lib/liboctane_b200.so); this package binds it.
"""
from .api import (Context, OctaneError, band_minmax, band_plan, batch_workspace_bytes, default_params, goes_cal,  # noqa: F401
                  goes_nav, level_dims)
from ._lib import Cal, Nav, Params, Stats  # noqa: F401

__all__ = ["Context", "OctaneError", "Params", "Nav", "Cal", "Stats", "default_params", "goes_nav", "goes_cal",
           "band_minmax", "level_dims", "band_plan", "batch_workspace_bytes"]
