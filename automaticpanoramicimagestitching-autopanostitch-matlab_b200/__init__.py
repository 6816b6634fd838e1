"""apsmatch (B200): AutoPanoStitch's featureMatching/ hot path on sm_100a.

The package is a thin host-side mirror of the reference's MATLAB interface for this path
(`featureMatchingGlobal`, `featureMatchingPairwise`, `matchFeaturesScratch`, `flann_knn_win`,
`nearest2HammingExhaustiveMEX`, ...) over the C ABI in include/apsmatch.h (libapsmatch.so, built
from csrc/*.cu).  There is no CPU implementation in here: every call needs the CUDA library and
a B200, and fails loudly otherwise.
"""
from . import _lib  # noqa: F401
from ._lib import ApsError, Context, DeviceGroup, build_library, library_path  # noqa: F401
from .host import (  # noqa: F401
    ApsSemanticsWarning,
    GlobalPlan,
    PairwisePlan,
    RECORD_PAD,
    binaryFeatures,
    featureMatchingGlobal,
    featureMatchingGlobalDevice,
    featureMatchingGlobalSets,
    featureMatchingGlobalSetsDevice,
    featureMatchingPairwiseSets,
    featureMatchingPairwiseSetsDevice,
    featureMatchingPairwiseDevice,
    estimateTransformationRANSAC,
    featureMatchingPairwise,
    imageMatching,
    globalImageMatching,
    globalImageMatchingDevice,
    globalImageMatchingSets,
    globalImageMatchingSetsDevice,
    imageMatchingBatch,
    imageMatchingSets,
    pairwiseImageMatching,
    pairwiseImageMatchingDevice,
    pairwiseImageMatchingSets,
    pairwiseImageMatchingSetsDevice,
    ransacSampleTable,
    flann_knn_win,
    matchFeaturesScratch,
    merge_pairwise_csr,
    merge_pairwise_shards,
    nearest2HammingExhaustiveMEX,
    nearest2HammingExhaustiveOMPMEX,
    nearest2SSDExhaustive,
    selectImagePartners,
    selectImagePartnersSets,
)
from . import multigpu, synth  # noqa: F401
