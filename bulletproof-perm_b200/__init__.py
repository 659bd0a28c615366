"""bulletproof-perm B200 backend: hand-written sm_100a CUDA kernels behind a C ABI.

Import as `bpperm_b200` (the repo-root shim maps that name to this directory, whose own name
is not a valid Python identifier).
"""
from ._lib import BppError, LIB_PATH, SYMBOLS, load  # noqa: F401
from .backend import Backend, Points, FMT_AFFINE, FMT_COMPRESSED, FMT_DALEK_XYZT, scalars_to_bytes  # noqa: F401
from .util import Ops  # noqa: F401
from . import acproof, ipa, weights  # noqa: F401

try:  # torch is only needed for the multi-GPU plumbing
    from . import parallel  # noqa: F401
except ImportError:  # pragma: no cover
    parallel = None
