"""zoe_b200 -- B200 (sm_100a) backend for zoe's striped Smith-Waterman path.

Host-side mirror of the zoe interface for this path (``alignment``), the data tables
(``matrices``), and the ctypes binding of the C-ABI CUDA library (``_lib``).
"""
from .alignment import (  # noqa: F401
    Alignment,
    BestHit,
    CudaProfiles,
    MaybeAligned,
    PairedHit,
    ProfileError,
    ScoreAndRanges,
    SeqSrc,
    Strand,
    ZoeCudaError,
    reverse_complement,
)
from .sneaky_snake import SneakySnake  # noqa: F401
from .matrices import (  # noqa: F401
    AA_ALL_AMBIG_PROFILE_MAP_WITH_STOP,
    BLOSUM_62,
    DNA_PROFILE_MAP,
    ByteIndexMap,
    WeightMatrix,
)
