"""StencilStream-B200: a B200-native backend for the StencilStream generation loop.

The product is the header-only C++ backend in `stencilstream_b200/include/StencilStream` (drop-in for
the reference's `stencil::cuda::{Grid, StencilUpdate}`) plus two C-ABI shared libraries. This Python
package is the host-side mirror of that interface over the C ABI (`api`), the recipes for the
reference's example experiments (`workloads`), and the build script (`_build`).
"""
from .api import (Grid, GridBatch, Params, RangeError, StencilStreamError, StencilUpdate, workload_info,
                  workload_names)

__all__ = ["Grid", "GridBatch", "Params", "RangeError", "StencilStreamError", "StencilUpdate", "workload_info",
           "workload_names"]
