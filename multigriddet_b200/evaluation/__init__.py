"""Drop-in for the matching / AP functions of the reference's ``multigriddet/evaluation``."""
from .metrics import (ConfusionMatrixAccumulator, ErrorAnalysisAccumulator, MapAccumulator, ShardedConfusionMatrixAccumulator,
                      ShardedErrorAnalysisAccumulator, ShardedMapAccumulator, calculate_ap_for_class, calculate_ap_for_class_cached, calculate_iou_matrix,
                      calculate_map, compute_average_precision, compute_iou_cache_for_class,
                      compute_precision_recall, match_predictions_to_gt,
                      match_predictions_to_gt_cached)

__all__ = ["calculate_iou_matrix", "match_predictions_to_gt", "match_predictions_to_gt_cached",
           "compute_precision_recall", "compute_average_precision", "calculate_ap_for_class",
           "calculate_ap_for_class_cached", "compute_iou_cache_for_class", "calculate_map",
           "MapAccumulator", "ShardedMapAccumulator", "ConfusionMatrixAccumulator",
           "ShardedConfusionMatrixAccumulator", "ErrorAnalysisAccumulator", "ShardedErrorAnalysisAccumulator"]
