"""bspatom_b200 -- B200-native hot path of BspAtom (B-spline assembly + banded generalized
eigensolve + dipole contraction) behind a C-ABI (include/bspatom.h).

Only what the path needs lives here: ``csrc/`` (CUDA kernels + the C-ABI), ``_lib`` (ctypes
binding), ``host`` (mirror of the reference driver's interface), ``parallel`` (sharding of the
(instance, l) list over one-process-per-GPU ranks and the single eigenpair gather)."""
from ._lib import BspAtomError, LIB_PATH, load  # noqa: F401
from .host import (BspAtom, BspAtomMulti, BspAtomPipeline, BspInputs, Problem, Selection, dsbgv, dsygv, parse_namelists,  # noqa: F401
                   POT_COULOMB, POT_ROGERS, POT_SIMONS_FUES, POT_TABLE, POT_TIETZ, POT_YUKAWA)
from .parallel import gather_eigenpairs, gather_eigenpairs_device, shard_items  # noqa: F401

__version__ = "0.1.0"
