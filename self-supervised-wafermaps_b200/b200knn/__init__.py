"""b200knn — B200-native (sm_100a) drop-in for the kNN hot path of
faris-k/self-supervised-wafermaps (lightly's ``knn_predict`` as called from
``KNNBenchmarkModule.validation_step``, ``src/ssl_wafermap/models/knn.py:87-101``).

Public surface (mirrors the reference names for this path):
    knn_predict(feature, feature_bank, feature_labels, num_classes, knn_k=200, knn_t=0.1)
    knn_predict_multi(..., knn_ks, knn_ts)        -> knn_predict over a (k, t) grid, one search
    knn_predict_loo(feature_bank, feature_labels, num_classes, knn_ks, knn_ts, groups=None)
                                                  -> leave-one-out (or leave-one-group-out) grid of the
                                                     bank against itself
    knn_predict_multilabel(feature, feature_bank, label_matrix, knn_ks, knn_ts)
                                                  -> per-label scores of multi-hot banks over a (k, t) grid
    knn_topk(feature, feature_bank, k)            -> (sims, idx)
    install() / uninstall()                       -> rebind lightly's symbol
    ShardedBank                                   -> bank row-sharded over the GPUs of a node
    FeatureBank                                   -> fused normalise + bank build (knn.py:67-81)
    L2Index / l2_topk / knn_graph                 -> the notebooks' nearest-neighbour search, batched
    knn_radius / radius_graph                     -> every neighbour above a similarity threshold (CSR rows)
    near_duplicate_groups                         -> near-duplicate groups for knn_predict_loo(groups=)
    knn_metrics                                   -> macro accuracy / F1 / confusion matrix on the device
    knn_multilabel_metrics                        -> multi-label F1, subset accuracy, Hamming loss, AUC
"""
from .install import install, uninstall  # noqa: F401
from .knn import (  # noqa: F401
    ALL_MODES,
    CASCADES,
    LEVELS,
    RESCORED_MODES,
    bank_cache,
    decode_keys,
    get_default_mode,
    knn_predict,
    knn_predict_loo,
    knn_predict_multi,
    knn_predict_multilabel,
    knn_topk,
    merge_keys,
    pack_label_bits,
    plan_info,
    prepare_rows,
    set_default_mode,
    topk_keys,
    vote,
)
from .knn import normalize_rows, row_sqnorms, vote_packed  # noqa: F401
from .bank import FeatureBank  # noqa: F401
from .hooks import install_hooks, uninstall_hooks  # noqa: F401
from .metrics import (  # noqa: F401
    confusion_counts,
    knn_metrics,
    knn_multilabel_metrics,
    metrics_from_counts,
    multilabel_metrics_from_scores,
)
from .retrieval import (  # noqa: F401
    L2Index,
    RadiusNeighbors,
    knn_graph,
    knn_radius,
    l2_topk,
    load_embedding_table,
    near_duplicate_groups,
    radius_graph,
)
from .sharded import ShardedBank, shard_bounds  # noqa: F401

__version__ = "0.1.0"
