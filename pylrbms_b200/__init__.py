"""pylrbms_b200 -- the data-parallel hot path of the Localized Reduced Basis Multiscale Method on B200 (sm_100a).

Host side: a pyMOR-shaped Operator / VectorArray / ``LRBMSReductor`` API (Python, like the reference).  Device side:
hand-written CUDA behind the C ABI of ``include/lrbms_sm100.h`` (``liblrbms_sm100.so``, loaded with ctypes).
There is no CPU fallback: without the shared library or without an sm_100 device every entry point raises.
"""
from ._lib import LrbmsError, Handle, load_library                                   # noqa: F401
from .parameters import (ExpressionParameterFunctional, ProductParameterFunctional,     # noqa: F401
                         ProjectionParameterFunctional, ConstantParameterFunctional)
from .vectorarray import (GpuVectorSpace, GpuVectorArray, BlockVectorSpace, BlockVectorArray,  # noqa: F401
                          ReducedVectorArray)
from .operators import (CsrOperator, LincombOperator, BlockOperator, BlockDiagonalOperator, Concatenation,  # noqa: F401
                        BlockProjectionOperator, BlockRowOperator, VectorFunctional,
                        OswaldInterpolationErrorOperator, FluxReconstructionOperator)
from .estimators import EllipticEstimator                                            # noqa: F401
from .discretization import discretize, BlockSwipdgDiscretization                    # noqa: F401
from .reductor import LRBMSReductor, GenericRBSystemReductor, ExtensionError           # noqa: F401
from .reduced import ReducedModel, ReducedBlockOperator                               # noqa: F401

__version__ = '0.1.0'
from .online_enrichment import AdaptiveEnrichment, doerfler_marking                              # noqa: F401
from .error_analysis import reduction_error_analysis, ReductionErrorAnalysis                     # noqa: F401
from .greedy import greedy                                                                       # noqa: F401
