"""universal_recommender_b200 -- Blackwell-native Correlated Cross-Occurrence (CCO) model builder:
the train hot path of actionml/universal-recommender (URAlgorithm.calcAll -> Mahout
SimilarityAnalysis) as hand-written sm_100a CUDA behind the C ABI of include/cco_b200.h.

Host-side mirror of the reference interface for this path:
  preparator.prepare                      <- Preparator.prepare           (Preparator.scala:44-87)
  preparator.prepare_on_device            <- the same from id strings on the B200 (cco_ingest_strings)
  IndexedDataset / BiDictionary           <- Mahout IndexedDataset
  DownsamplableCrossOccurrenceDataset     <- URAlgorithm.scala:336-340
  SimilarityAnalysis.cooccurrencesIDSs / crossOccurrenceDownsampled  <- URAlgorithm.scala:323,343
  ur_algorithm.calc_all                   <- URAlgorithm.calcAll          (URAlgorithm.scala:310-349)
  ur_algorithm.write_model                <- the documents calcAll hands to URModel.save (URAlgorithm.scala:351-367)
"""
from ._native import (CcoError, CcoInvalidArgument, FLAG_ASSUME_CANONICAL, FLAG_ENTROPY_VARARGS, FLAG_RESULT_NO_COUNT,
                      FLAG_RESULT_NO_LLR, FLAG_ROWRATE_INTDIV, LIB_PATH)
from .indexed_dataset import BiDictionary, IndexedDataset
from .preparator import prepare, prepare_on_device
from .similarity_analysis import (CcoContext, DownsamplableCrossOccurrenceDataset, SimilarityAnalysis,
                                  default_context)
from .ur_algorithm import (DefaultURAlgoParams, IndicatorParams, RankingParams, URAlgorithmParams, calc_all, resolve_rankings,
                           write_model)

__all__ = [
    "BiDictionary", "CcoContext", "CcoError", "CcoInvalidArgument", "DefaultURAlgoParams",
    "DownsamplableCrossOccurrenceDataset", "IndexedDataset", "IndicatorParams", "RankingParams", "SimilarityAnalysis",
    "URAlgorithmParams", "calc_all", "resolve_rankings", "write_model", "default_context", "prepare", "prepare_on_device", "FLAG_ASSUME_CANONICAL",
    "FLAG_ENTROPY_VARARGS", "FLAG_ROWRATE_INTDIV", "FLAG_RESULT_NO_COUNT", "FLAG_RESULT_NO_LLR", "LIB_PATH",
]
