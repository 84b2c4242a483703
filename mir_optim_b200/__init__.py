"""mir_optim_b200 -- B200-native Levenberg-Marquardt / BOXCQP engine behind mir-optim's API.

The compute lives in ``libmir_optim_b200.so`` (hand-written sm_100a CUDA, C ABI declared in
``include/mir_optim_b200.h``).  This package is only the host-side mirror of the reference's
operator interface; it never computes and has no CPU fallback: the first use of ``mir_optim_b200.lib`` /
``mir_optim_b200.engine`` without the built library raises, and calling it without a CUDA device returns the
library's error.
"""
from __future__ import annotations

import ctypes as _C
import os as _os

from . import _abi
from ._abi import (BoxQPStatus, LeastSquaresStatus, ModelDesc, ModelId, BatchStats,  # noqa: F401
                   MODEL_FD_JACOBIAN, MODEL_GRID_PER_PROBLEM)

_HERE = _os.path.dirname(_os.path.abspath(__file__))
LIB_PATH = _os.environ.get("MIR_B200_LIB") or _os.path.join(_HERE, "libmir_optim_b200.so")   # env override: load the library from another path


class LibraryMissing(ImportError):
    pass


def load_library(path: str = LIB_PATH):
    if not _os.path.exists(path):
        raise LibraryMissing(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C mir_optim_b200/csrc`).  There is no CPU fallback.")
    lib = _C.CDLL(path, mode=_C.RTLD_LOCAL)
    _abi.bind_reference_abi(lib)
    _abi.bind_b200_abi(lib)
    return lib


# `lib` (the ctypes handle of libmir_optim_b200.so) and `engine` are created on first access, not at import: modules that
# only need the constants / workload generators (bench.py's CPU reference arm, the oracle-only tests) then never map the
# product library into their process, so a record of loaded libraries cannot mistake them for users of it.  Any use of
# the engine still fails loudly when the library is missing (LibraryMissing) -- there is no CPU fallback.
from .api import ReferenceAPI, LeastSquaresException  # noqa: E402
from .engine import Engine, B200Error, RESULT_DTYPES  # noqa: E402

# (`mir_optim_b200.engine` is the Engine OBJECT, as it always was; the submodule of the same name stays importable as
#  `from mir_optim_b200.engine import ...` through sys.modules)
globals().pop("engine", None)
_lazy = {}


def __getattr__(name):
    if name in ("lib", "engine"):
        if "lib" not in _lazy:
            _lazy["lib"] = load_library()
            _lazy["engine"] = Engine(_lazy["lib"])
        return _lazy[name]
    raise AttributeError(f"module 'mir_optim_b200' has no attribute {name!r}")


__all__ = ["lib", "engine", "Engine", "B200Error", "ReferenceAPI", "LeastSquaresException", "LeastSquaresStatus",
           "BoxQPStatus", "ModelId", "ModelDesc", "BatchStats", "MODEL_FD_JACOBIAN", "MODEL_GRID_PER_PROBLEM",
           "RESULT_DTYPES", "LIB_PATH"]
