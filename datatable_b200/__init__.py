"""
datatable_b200 -- B200-native groupby/sort engine behind h2oai/datatable's
DT[i, j, by(), sort()] hot path.  See DESIGN.md / INTEGRATION.md.

Importing this package loads libdtb200.so (sm_100a CUDA); it raises if the
library has not been built.  There is no CPU fallback.
"""
from . import _lib
from ._lib import (DtbError, DtbValueError, DtbNotImplError, DtbCudaError, DtbMemoryError)
from . import engine
from .frame import (Frame, f, by, sort, join, sum, mean, min, max, count, countna, first, last, sd, median,   # noqa: A004
                    unique, nunique, union, intersect, setdiff, symdiff,
                    cumsum, cumprod, cummin, cummax, cumcount, ngroup, shift, fillna)
from .jay import open_jay, save_jay

__all__ = ["engine", "Frame", "f", "by", "sort", "sum", "mean", "min", "max", "count", "countna", "first", "last", "sd", "median", "join", "unique", "nunique", "union", "intersect", "setdiff", "symdiff", "cumsum", "cumprod", "cummin", "cummax", "cumcount", "ngroup", "shift", "fillna", "open_jay", "save_jay", "DtbError", "DtbValueError", "DtbNotImplError", "DtbCudaError", "DtbMemoryError"]
