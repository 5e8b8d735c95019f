"""anyseq_b200 -- B200-native (sm_100a CUDA) DP-relaxation hot path of DasNaCl/anyseq.

The package holds only what the path needs: ``csrc/`` (CUDA kernels + C ABI),
``build`` (nvcc recipe), ``capi`` (ctypes binding of include/anyseq.h) and ``api``
(the host-side mirror of the reference's operator surface).
"""
from .api import (  # noqa: F401
    Aligner, AlignmentResult, BatchAlignment, BatchStream, ScoringScheme, REFERENCE_SCORING,
    affine_scoring_scheme, linear_scoring_scheme, cigar, default_aligner, pack2, plan_launch,
    global_alignment_score, semiglobal_alignment_score, local_alignment_score,
    construct_global_alignment, construct_semiglobal_alignment, construct_local_alignment,
)
from .capi import AnyseqError, GLOBAL, SEMIGLOBAL, LOCAL  # noqa: F401

__version__ = "0.1.0"
