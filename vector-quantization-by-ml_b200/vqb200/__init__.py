"""vqb200 -- B200-native codebook hot path behind the module API of
MisterBourbaki/vector-quantization-by-ml (``vector_quantization``).

    from vqb200 import VectorQuantize, ResidualVQ, Codebook, CodebookParams, KmeansParameters

replaces

    from vector_quantization import VectorQuantize, ResidualVQ
    from vector_quantization.codebooks import Codebook, CodebookParams, KmeansParameters
"""
from .codebook import Codebook, CosineSimCodebook, EuclideanCodebook
from .params import AffineParameters, CodebookParams, GumbelParams, KmeansParameters
from .rvq import GroupedResidualVQ, ResidualVQ
from .simvq import ResidualSimVQ, SimVQ
from .vq import LossBreakdown, VectorQuantize

__all__ = ["Codebook", "EuclideanCodebook", "CosineSimCodebook", "CodebookParams", "KmeansParameters", "GumbelParams",
           "AffineParameters", "VectorQuantize", "LossBreakdown", "ResidualVQ", "GroupedResidualVQ", "SimVQ",
           "ResidualSimVQ"]
