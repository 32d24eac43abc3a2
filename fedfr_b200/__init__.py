"""fedfr_b200 -- B200-native (sm_100a) PartialFC CosFace head + FedAvg, drop-in for jackie840129/FedFR's
``partial_fc.PartialFC`` / ``losses.CosFace`` / ``server.FedPavg`` hot path.  See DESIGN.md.

IJB-C 1:N identification, once per gallery (G1, G2), on ``template_features`` rows with subjects from the protocol's
template -> subject table: ``rank, mate_score, _, top1_score = mate_ranks(tf[probe_rows], probe_subjects, tf[g1_rows],
g1_subjects)``, then ``cmc(rank)`` and ``tpir_at_fpir(rank, mate_score, top1_score)``."""
from . import _native  # noqa: F401  (fails loudly when the CUDA extension has not been built)
from .bce_head import BCE_module
from .dense_head import MarginSoftmaxHead, margin_cross_entropy
from .fedavg import FedAvg_on_FC, FedPavg, FedPavg_sharded, FlatStateDict, flatten_state_dict
from .hardneg import hard_negative_ids, similar_columns
from .losses import ArcFace, CosFace
from .partial_fc import PartialFC
from .roc import calc_ROC, roc_histogram, tpr_at_fpr
from .spreadout import SpreadOut_Module
from .verify import (cmc, kfold_accuracy, mate_ranks, pair_scores, roc_curve, tar_at_far, tar_at_far_nearest,
                     template_features, tpir_at_fpir)

__all__ = ["PartialFC", "CosFace", "ArcFace", "FedPavg", "FedAvg_on_FC", "FedPavg_sharded", "FlatStateDict", "flatten_state_dict", "margin_cross_entropy", "MarginSoftmaxHead", "SpreadOut_Module",
           "BCE_module", "similar_columns", "hard_negative_ids", "calc_ROC", "roc_histogram", "tpr_at_fpr",
           "template_features", "pair_scores", "tar_at_far", "roc_curve", "tar_at_far_nearest",
           "kfold_accuracy", "mate_ranks", "cmc", "tpir_at_fpir"]
