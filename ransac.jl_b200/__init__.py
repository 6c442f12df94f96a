"""ransac.jl_b200 -- B200 (sm_100a) hot path of efficient-RANSAC shape detection behind the public
surface of cserteGT3/RANSAC.jl.  Host layer in Python (Julia is not available in this image; the
Julia `ccall` binding is in julia/ and INTEGRATION.md), compute in libransac_b200.so (csrc/).

Import fails loudly when the CUDA library has not been built; a context cannot be created without
an sm_100 device.  There is no CPU fallback anywhere in this package.
"""
from . import _lib
from ._lib import Context, RscError
from .cloud import RANSACCloud, makesubsets
from .confidence import ConfidenceInterval, E, estimatescore, estimatescore_f64, isoverlap, notsoconfident, prob
from .fitting import (
    IterationCandidates,
    bitmap_filter,
    findhighestscore,
    fit,
    fit_batch,
    fit_points,
    invalidate_indexes,
    lsq_refit,
    refine_progressive,
    refit,
    sample_fit,
    sample_fit_cells,
    score_counts,
    score_counts_culled,
    scorecandidate,
    scorecandidates,
    unpack_mask,
    user_score_counts,
)
from .iterations import ransac
from .jsonyaml import dict2nt, exportJSON, readconfig, toDict
from .normals import estimate_normals, orient_normals
from .params import (
    DEFAULT_PARAMETERS,
    DEFAULT_SHAPE_DICT,
    DEFAULT_SHAPE_TYPES,
    defaultcommonparameters,
    defaultiterationparameters,
    defaultparameters,
    defaultshapeparameters,
    ransacparameters,
    setfloattype,
    to_c,
)
from .shapes import (
    ExtractedShape,
    FittedCone,
    FittedCylinder,
    FittedPlane,
    FittedShape,
    FittedSphere,
    from_cand,
    pack_cands,
    strt,
)

__all__ = [n for n in dir() if not n.startswith("_")]
