"""xsparse_b200 -- B200-native assembly hot path of ExtendableSparse.jl.

The directory is called `extendablesparse.jl_b200`; because of the dot it is imported
through the repo-root shim `xsparse_b200` (import xsparse_b200).
"""
from . import capi  # noqa: F401
from .capi import (  # noqa: F401
    ASSIGN, COMBINE_ADD, COMBINE_SEED, DETERMINISTIC, FAST, I32, I64, OP_ADD, OP_SUB, RAW, UPDATE, Handle, XsbBoundsError, XsbError,
    XsbIllegalError, XsbSizeError,
)
from .matrix import (  # noqa: F401
    ExtendableSparseMatrix, MTExtendableSparseMatrix, dropzeros, fdrand, flush, nnz, pointblock, rawupdateindex, reset, sparse,
    updateindex,
)
