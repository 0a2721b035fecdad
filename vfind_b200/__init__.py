"""vfind_b200 — B200-native implementation of vFind's per-read variant-recovery path.

`find_variants` is a drop-in for `vfind.find_variants` of nsbuitrago/vfind; everything
behind it runs as hand-written sm_100a CUDA kernels in libvfind_b200.so (see DESIGN.md).
"""
from .api import (Context, MultiContext, PanicException, collapse_variants, find_variants,  # noqa: F401
                  find_variants_multi, read_diagnostics)

__all__ = ["find_variants", "find_variants_multi", "collapse_variants", "read_diagnostics", "Context", "MultiContext",
           "PanicException"]
