/*
 * ygg_b200.h — C ABI of libygg_b200.so, the B200-native GBT split-finding engine.
 *
 * Scope: the bucketised-feature (histogram) split finder of YDF's gradient-boosted-trees
 * learner, and nothing else (SURVEY.md §8).  The reference has no C ABI for this path; its
 * seam is C++ virtuals + protobuf messages.  Each entry point below names the reference
 * interface it stands in for (paths relative to /root/reference/yggdrasil_decision_forests).
 *
 * Conventions (mirroring the reference's ownership / error rules, SURVEY.md §8b):
 *  - every function returns an int status: 0 = OK, non-zero = error (absl::Status analogue);
 *    the message of the last error on the calling thread is ygg_last_error();
 *    no C++ exception ever crosses this boundary;
 *  - inputs are borrowed for the duration of the call only (the engine copies to HBM);
 *  - a handle is not thread-safe; distinct handles are independent;
 *  - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *    YGG_ERR_NO_DEVICE.
 */
#ifndef YGG_B200_H_
#define YGG_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YGG_ABI_VERSION 4

enum ygg_status {
  YGG_OK = 0,
  YGG_ERR_INVALID_ARGUMENT = 1, /* absl::InvalidArgumentError */
  YGG_ERR_NO_DEVICE = 2,        /* no CUDA device / extension built without one */
  YGG_ERR_CUDA = 3,             /* a CUDA runtime call failed (absl::InternalError) */
  YGG_ERR_UNIMPLEMENTED = 4,    /* absl::UnimplementedError: option outside the hot path */
  YGG_ERR_CANCELLED = 5,        /* stop flag raised (stop_training_trigger) */
  YGG_ERR_IO = 6
};

/* proto::Loss values the hot path covers
 * (learner/gradient_boosted_trees/gradient_boosted_trees.proto; loss/loss_imp_binomial.cc,
 * loss/loss_imp_mean_square_error.cc). */
enum ygg_loss {
  YGG_LOSS_BINOMIAL_LOG_LIKELIHOOD = 0,
  YGG_LOSS_SQUARED_ERROR = 1,
  /* K >= 2 classes, labels in 1..K, K trees per iteration, one per class
   * (loss_imp_multinomial.cc; gradient_boosted_trees.cc:1490-1511); cfg.num_classes = K */
  YGG_LOSS_MULTINOMIAL_LOG_LIKELIHOOD = 2
};

/* The proto fields the path reads, as a POD.  Defaults (ygg_gbt_config_init) are the proto
 * defaults: gradient_boosted_trees.proto:35-278, decision_tree.proto:32-108,
 * gradient_boosted_trees.cc:3238-3262 (max_depth 6, all attributes tested). */
typedef struct ygg_gbt_config {
  int32_t abi_version;          /* YGG_ABI_VERSION */
  int32_t loss;                 /* enum ygg_loss */
  int32_t num_trees;            /* 300 */
  float shrinkage;              /* 0.1 */
  int32_t max_depth;            /* 6; root has depth 1, depth >= max_depth => leaf */
  int32_t min_examples;         /* 5 */
  int32_t in_split_min_examples_check; /* 1 */
  int32_t use_hessian_gain;     /* 0 => variance-reduction gain (reference default) */
  float l1_regularization;      /* 0 */
  float l2_regularization;      /* 0 */
  float l2_regularization_categorical; /* 1 (reserved for categorical features) */
  float clamp_leaf_logit;       /* 5 */
  int32_t hessian_split_score_subtract_parent; /* 0 */
  uint32_t random_seed;         /* 123456; consumed by the hold-out draw (ygg_validation_split_mask) and the tie-break replay */
  float subsample;              /* must be 1.0 (row sampling is SURVEY §8f N3) */
  float validation_ratio;       /* 0: the engine trains on the rows it is given; validation rows are attached
                                   with ygg_gbt_set_validation_* (split helpers below).  Kept for hosts that
                                   forward GradientBoostedTreesTrainingConfig.validation_set_ratio */
  int32_t sibling_subtraction;  /* 1: build the smaller child's histogram, derive the other
                                   by exact integer subtraction (bit-identical results) */
  int32_t early_stopping;       /* enum ygg_early_stopping, 2 (LOSS_INCREASE); inert without validation rows */
  int32_t early_stopping_num_trees_look_ahead; /* 30 */
  int32_t early_stopping_initial_iteration;    /* 10 */
  int32_t num_classes;          /* multinomial loss: K (2..32); ignored otherwise */
  /* Tie-break between features whose best splits have EQUAL float scores: the reference takes the first one in the
   * order of its per-node std::shuffle of the candidate features on the learner's std::mt19937
   * (GetCandidateAttributes, learner/decision_tree/training.cc:4293-4306), visiting the nodes depth-first, positive
   * child first.  0 (default): lowest feature index.  1 / 2: replay that stream with libstdc++'s / libc++'s
   * std::shuffle algorithm (the reference's golden models follow libc++'s) and give tied nodes the feature the reference
   * picks; done on the finished trees, see DESIGN.md §9.  Single GPU only. */
  int32_t candidate_shuffle;
  uint32_t rng_words_consumed;     /* words of the learner's engine drawn before the first tree (the hold-out draw:
                                      one per row when validation_ratio > 0, gradient_boosted_trees.cc:2731-2738) */
  int32_t split_jobs_draw_seeds;   /* 1: FindBestConditionConcurrentManager (num_threads > 1) — one engine word per
                                      feature job after every shuffle (training.cc:1658, :1781); 0: single-thread manager */
  /* DecisionTreeTrainingConfig.growing_strategy (decision_tree.proto:205-232).  0: growing_strategy_local (default).
   * 1: growing_strategy_best_first_global (GrowTreeBestFirstGlobal, training.cc:4499-4656): the node with the largest
   * split_score * num_examples is split next until max_num_nodes leaves exist; the root has depth 0 there, so a tree may be
   * one level deeper than with the local growth and the same max_depth.  The engine grows the full tree level-wise and
   * replays the priority queue on it (DESIGN.md §17): the scores of a node do not depend on the order of growth. */
  int32_t growing_strategy;
  int32_t max_num_nodes;           /* best-first growth: 31; -1 = unlimited */
  /* GradientOneSideSampling (gradient_boosted_trees.proto:317-335; SampleTrainingExamplesWithGoss,
   * gradient_boosted_trees.cc:2958-3007), on when alpha > 0 or beta > 0 (both 0 = off; the reference's defaults are 0.2 / 0.1):
   * every iteration the ceil(alpha * rows) rows with the largest |gradient| are kept, every other row with probability beta
   * (one word of the learner's engine each, in decreasing-|gradient| order) and weight (1 - alpha) / beta.  Rows with EQUAL
   * |gradient| are ordered by row index (the reference: whatever its std::sort does; DESIGN.md §19).  Variance gain,
   * binomial / squared error, single GPU, not with subsample < 1 or example weights.  (These 8 bytes were `reserved`, zero.) */
  float goss_alpha;
  float goss_beta;
} ygg_gbt_config;

/* GradientBoostedTreesTrainingConfig.EarlyStopping (gradient_boosted_trees.proto:150-169). */
enum ygg_early_stopping {
  YGG_EARLY_STOPPING_NONE = 0,
  YGG_EARLY_STOPPING_MIN_LOSS_FINAL = 1, /* MIN_VALIDATION_LOSS_ON_FULL_MODEL: train every tree, keep the best prefix */
  YGG_EARLY_STOPPING_LOSS_INCREASE = 2   /* VALIDATION_LOSS_INCREASE: stop when the best loss is look_ahead trees old */
};

/* One tree node, flat.  Trees are emitted in the reference's serialization order
 * (model/decision_tree/decision_tree.cc:609-646): node, negative subtree, positive subtree.
 * Mirrors proto::Node + proto::NodeCondition (model/decision_tree/decision_tree.proto). */
enum ygg_feature_type {
  YGG_FEATURE_DISCRETIZED_NUMERICAL = 0, /* condition: bin >= threshold_bin */
  YGG_FEATURE_CATEGORICAL = 1            /* condition: category in cat_mask (CART, < 300 values) */
};

typedef struct ygg_node {
  int32_t feature;          /* NodeCondition.attribute (dataset feature index); -1 for a leaf */
  int32_t threshold_bin;    /* Condition.DiscretizedHigher.threshold: bin >= threshold => positive
                               (0 for a categorical condition) */
  int32_t na_value;         /* NodeCondition.na_value */
  int32_t depth;            /* root = 1 */
  int32_t neg_child;        /* index in the emitted array, -1 for a leaf */
  int32_t pos_child;
  float split_score;        /* NodeCondition.split_score */
  float leaf_value;         /* NodeRegressorOutput.top_value (set on every node, as the reference does) */
  int64_t num_examples;     /* num_training_examples_without_weight of the node */
  int64_t num_pos_examples; /* num_pos_training_examples_without_weight of the split */
  /* Label statistics saved in the node (loss_utils.cc:109-117):
   *   variance gain: stat[0]=sum, stat[1]=sum_squares, stat[2]=count
   *   hessian gain : stat[0]=sum_gradients, stat[1]=sum_hessians (floored at 1e-3), stat[2]=sum_weights */
  double stat[3];
  /* Categorical condition (Condition.ContainsVector / ContainsBitmap,
   * learner/decision_tree/utils.cc:31-63): bit c set => category c goes to the positive child. */
  int32_t condition_type;   /* enum ygg_feature_type of the split feature; 0 for a leaf */
  float threshold_value;    /* Condition.Higher.threshold of the EXACT numerical splitter for features with bucket values
                               (ygg_dataset_set_bucket_values); NaN otherwise (discretized rule: threshold_bin only) */
  uint32_t cat_mask[8];
} ygg_node;

typedef struct ygg_dataset ygg_dataset;
typedef struct ygg_gbt ygg_gbt;

/* ---- library ------------------------------------------------------------------------- */
int ygg_abi_version(void);
const char* ygg_last_error(void);
/* Number of visible CUDA devices (0 if none; never fails). */
int ygg_device_count(void);

/* ---- dataset: the engine's input contract ----------------------------------------------
 * Replaces dataset::VerticalDataset with DISCRETIZED_NUMERICAL columns
 * (dataset/vertical_dataset.h:377-378) as consumed by
 * FeatureDiscretizedNumericalBucket::Filler (learner/decision_tree/splitter_accumulator.h:253-338).
 *  bins        : column-major, bins[f * column_stride + r], one byte per value, value < num_bins[f].
 *                The reference stores uint16 with 65535 = missing; here missing values are
 *                already folded into na_bin[f], which is what GetBucketIndex
 *                (splitter_accumulator.h:288-299) and EvalConditionDiscretizedHigher
 *                (model/decision_tree/decision_tree.cc:724-743, with na_value = na_bin >= threshold)
 *                do with them.
 *  num_bins[f] : boundaries_size()+1, 2..256.
 *  na_bin[f]   : NumericalToDiscretizedNumerical(column mean) (training.cc:917-922).
 * Categorical columns (dataset/vertical_dataset.h:416; ygg_dataset_set_feature_types) use the same
 * byte layout: value = integerised category (0 = out-of-dictionary), num_bins[f] =
 * number_of_unique_values <= 256, na_bin[f] = most_frequent_value (the NA replacement,
 * training.cc:3262-3314); they are split with the CART rule (buckets sorted by label mean /
 * hessian priority, then scanned).  Columns with >= 300 values (random-mask algorithm,
 * decision_tree.proto:576) do not fit one byte and are rejected.
 *  device      : CUDA ordinal this handle lives on (one process per GPU).
 */
int ygg_dataset_create(ygg_dataset** out, int64_t n_rows, int32_t n_features,
                       const uint8_t* bins, int64_t column_stride,
                       const int32_t* num_bins, const int32_t* na_bin, int32_t device);
/* feature_types[f]: enum ygg_feature_type (default: all DISCRETIZED_NUMERICAL). */
int ygg_dataset_set_feature_types(ygg_dataset* ds, const int32_t* feature_types, int32_t n_features);
/* Exact numerical splits through lossless buckets (one bucket per distinct value, DESIGN.md §14): `values[b]` = the value
 * of bucket b of `feature` (ascending, n = its number of bins).  For such a feature the engine places thresholds like the
 * reference's exact splitter: the middle of the two values PRESENT in the node around the cut
 * (FeatureNumericalBucket::Filler::SetConditionFinal, splitter_accumulator.h:213-232; MidThreshold, utils.h:103-109)
 * instead of the middle of the empty buckets (bucket interpolation) — the same partition of the training rows, the
 * reference's side for a held-out value inside the gap — and reports the float threshold in ygg_node.threshold_value.
 * `na_replacement` = the column mean the exact splitter imputes missing values with: na_value = na_replacement >= threshold
 * (splitter_accumulator.h:218). */
int ygg_dataset_set_bucket_values(ygg_dataset* ds, int32_t feature, const float* values, int32_t n, float na_replacement);
int ygg_dataset_destroy(ygg_dataset* ds);
int64_t ygg_dataset_num_rows(const ygg_dataset* ds);
int32_t ygg_dataset_num_features(const ygg_dataset* ds);

/* ---- learner -----------------------------------------------------------------------------
 * Replaces GradientBoostedTreesLearner::TrainWithStatusImpl
 * (learner/gradient_boosted_trees/gradient_boosted_trees.cc:1154-1732) for configurations
 * whose features are all DISCRETIZED_NUMERICAL. */
void ygg_gbt_config_init(ygg_gbt_config* cfg);
int ygg_gbt_create(ygg_gbt** out, ygg_dataset* ds, const ygg_gbt_config* cfg);
int ygg_gbt_destroy(ygg_gbt* h);

/* Labels.  i32: integerised categorical label as the reference stores it (1 = negative,
 * 2 = positive; loss_imp_binomial.cc:133).  f32: regression target. */
int ygg_gbt_set_labels_i32(ygg_gbt* h, const int32_t* labels, int64_t n);
int ygg_gbt_set_labels_f32(ygg_gbt* h, const float* labels, int64_t n);

/* Example weights (TrainingConfig.weight_definition -> dataset::GetWeights, learner/abstract_learner.cc; consumed as the
 * `weights` spans of InitialPredictions / Loss (loss_imp_binomial.cc:65-99, :204-234; loss_imp_mean_square_error.cc:56-88;
 * metric/metric.cc:2097-2115), of the bucket filler (LabelNumericalBucket<weighted=true>, splitter_accumulator.h:1552-1560)
 * and of SetLeafValueWithNewtonRaphsonStep<true> (loss_utils.cc:81-89)).  One non-negative float per training row, host
 * memory; call BEFORE ygg_gbt_set_labels_* (the initial predictions are weighted).  min_examples keeps counting rows.
 * Row shards: every rank passes its rows' weights (before ygg_gbt_set_row_shard*, which reduces the scales and the weight sum).
 * YGG_ERR_UNIMPLEMENTED with use_hessian_gain (the reference's weighted hessian filler sums UNWEIGHTED gradients into the buckets
 * it compares with a WEIGHTED parent, splitter_accumulator.h:1806-1814: neither reproduced nor silently corrected). */
int ygg_gbt_set_weights_f32(ygg_gbt* h, const float* weights, int64_t n);

/* ---- validation rows and early stopping (SURVEY.md §8f N2) ------------------------------------
 * The reference holds out validation rows before training (ExtractValidationDataset,
 * gradient_boosted_trees.cc:2718-2746: row r trains iff uniform_real_distribution<float>(mt19937(seed)) >
 * ratio, the first use of the learner's random engine), evaluates the loss on them after every
 * iteration (:1610-1626), feeds EarlyStopping (early_stopping/early_stopping.cc:30-62) and finally
 * truncates the model to the best number of trees (FinalizeModelWithValidationDataset, :212-272).
 * Here: ygg_validation_split_mask reproduces the row draw (libstdc++ semantics), ygg_dataset_split_rows
 * gathers the two row sets on the device, ygg_gbt_set_validation_* attaches the held-out rows (same
 * features and binning as the training dataset).  ygg_gbt_train then applies cfg.early_stopping;
 * afterwards ygg_gbt_num_trees is the truncated model size and ygg_gbt_num_iterations the number of
 * iterations that have log entries (training stopped there).  Not combined with sharding. */
int ygg_validation_split_mask(uint32_t random_seed, int64_t n_rows, float validation_ratio,
                              uint8_t* out_in_training /* [n_rows] 1 = training row */);
int ygg_dataset_split_rows(const ygg_dataset* ds, const uint8_t* select, ygg_dataset** selected,
                           ygg_dataset** rest);
int ygg_gbt_set_validation_i32(ygg_gbt* h, const ygg_dataset* valid, const int32_t* labels, int64_t n);
int ygg_gbt_set_validation_f32(ygg_gbt* h, const ygg_dataset* valid, const float* labels, int64_t n);
/* Weights of the validation rows (the hold-out is cut from the weighted dataset, gradient_boosted_trees.cc:1262-1280):
 * validation loss and accuracy become weighted.  After ygg_gbt_set_validation_*, before training. */
int ygg_gbt_set_validation_weights_f32(ygg_gbt* h, const float* weights, int64_t n);
/* Validation loss / secondary metric after iteration `iter` (TrainingLogs.Entry.validation_loss). */
int ygg_gbt_validation_loss(ygg_gbt* h, int32_t iter, float* loss, float* secondary);
/* Iterations with log entries; > ygg_gbt_num_trees when the model was truncated. */
int32_t ygg_gbt_num_iterations(const ygg_gbt* h);
/* Header.validation_loss and Header.early_stopping_triggered of the final model. */
int ygg_gbt_final_validation(ygg_gbt* h, float* validation_loss, int32_t* early_stopping_triggered);

/* Feature sharding across the GPUs of one box (SURVEY.md §8e; the reference's model is
 * distributed_decision_tree: workers own feature subsets).  This rank histograms and scans
 * features [feature_begin, feature_end) only; all ranks hold all columns so the row partition
 * is local.  `exchange` is called once per tree level with this rank's packed best-split
 * records (device pointer, `bytes` bytes) and must all-gather them into `recv` (device pointer,
 * world*bytes) on `stream` (a cudaStream_t) — NCCL in production, see INTEGRATION.md. */
typedef int (*ygg_allgather_fn)(void* ctx, const void* send, void* recv, int64_t bytes,
                                void* stream);
int ygg_gbt_set_feature_shard(ygg_gbt* h, int32_t feature_begin, int32_t feature_end,
                              int32_t rank, int32_t world, ygg_allgather_fn exchange, void* ctx);

/* Row sharding (data parallel): this rank holds n_rows of n_rows_global rows of ALL features.  Per
 * tree level the engine fills its local integer histograms and calls `allreduce` ONCE on the level
 * buffer (sum, u64) — the "NCCL all-reduce of per-node histograms"; integer sums make the result
 * exact and independent of the reduction order, so trees are identical for any world size.  Child
 * statistics ride in the same buffer.  `allreduce(ctx, buf, count, dtype, op, stream)` must reduce
 * `count` elements in place on `stream`: dtype 0 = u32, 1 = u64, 2 = f64; op 0 = sum, 1 = max.
 * Call after ygg_gbt_set_labels_*; `initial_prediction` is the job-wide value (the harness owns
 * the global label statistics, loss_imp_binomial.cc:65-99). */
typedef int (*ygg_allreduce_fn)(void* ctx, void* buf, int64_t count, int32_t dtype, int32_t op, void* stream);
int ygg_gbt_set_row_shard(ygg_gbt* h, int32_t rank, int32_t world, int64_t n_rows_global,
                          float initial_prediction, ygg_allreduce_fn allreduce, void* ctx);

/* Row sharding with a reduce-scatter: the level buffer is cut into `world` chunks by feature
 * (chunk r = features [r*c, (r+1)*c), c = ceil(F / world), plus a copy of the node statistics), ONE
 * reduce-scatter per level gives rank r the summed histograms of its features only, every rank scans its
 * chunk and the best splits are all-gathered like in feature sharding (<= 3.5 KB): half the collective
 * bytes of the all-reduce and no replicated scan.  `reducescatter(ctx, buf, count_per_rank, dtype, op,
 * stream)` reduces world*count_per_rank elements in place, rank r's result at buf + r*count_per_rank;
 * `allreduce` is still used for a few scalars per iteration. */
typedef int (*ygg_reducescatter_fn)(void* ctx, void* buf, int64_t count_per_rank, int32_t dtype, int32_t op,
                                    void* stream);
int ygg_gbt_set_row_shard_scatter(ygg_gbt* h, int32_t rank, int32_t world, int64_t n_rows_global,
                                  float initial_prediction, ygg_allreduce_fn allreduce,
                                  ygg_reducescatter_fn reducescatter, ygg_allgather_fn allgather, void* ctx);

/* Contiguous feature range of `rank` (the shard layout every rank must agree on). */
int ygg_feature_shard(int32_t n_features, int32_t rank, int32_t world, int32_t* begin, int32_t* end);

/* The record exchanged per (level, node): this rank's best split over its features. */
typedef struct ygg_shard_best {
  float score;      /* split_score as float; only meaningful if feature >= 0 */
  int32_t feature;  /* global feature index, -1 = no valid split in this shard */
  int32_t threshold_bin;
  int32_t num_pos_examples;
  int32_t condition_type; /* ygg_feature_type of `feature` */
  int32_t na_value;       /* categorical splits: 1 if the NA replacement category is positive */
  uint32_t cat_mask[8];   /* categorical splits: positive categories */
} ygg_shard_best;
/* Host restatement of the on-device merge (records: [world][nodes], out: [nodes]): the first strictly
 * greater float score in rank order, i.e. the ordered consumption of
 * FindBestConditionConcurrentManager (learner/decision_tree/training.cc:1728-1746). */
int ygg_merge_shard_best(const ygg_shard_best* records, int32_t world, int32_t nodes, ygg_shard_best* out);

/* loss->InitialPredictions (loss_imp_binomial.cc:65-99, loss_imp_mean_square_error.cc:56-88). */
int ygg_gbt_initial_prediction(ygg_gbt* h, float* out);

/* Runs `num_iters` boosting iterations (gradient_boosted_trees.cc:1428-1571).  `stop_flag`
 * (may be NULL) is polled between iterations like stop_training_trigger
 * (gradient_boosted_trees.cc:1430-1433). */
int ygg_gbt_train(ygg_gbt* h, int32_t num_iters, const volatile int32_t* stop_flag);
/* One iteration, asynchronous on the handle's stream; ygg_gbt_sync waits for it. */
int ygg_gbt_step(ygg_gbt* h);
int ygg_gbt_sync(ygg_gbt* h);

/* `num_iters` iterations (including the final prediction update) bracketed by CUDA events on the
 * handle's stream; *device_ms receives the elapsed device time, *kernel_launches (may be NULL)
 * the number of kernels this library launched in between.  Used by bench.py. */
int ygg_gbt_train_timed(ygg_gbt* h, int32_t num_iters, double* device_ms, int64_t* kernel_launches);

int32_t ygg_gbt_num_trees(const ygg_gbt* h);
/* Best-split exchange over peer memory instead of the all-gather callback (feature shards and row shards with the
 * reduce-scatter layout): `peer_windows[r]` = this process's mapping of rank r's window of
 * ygg_gbt_best_split_window_bytes(h) zeroed bytes (ygg_comm_window_create of ygg_b200_comm.h).  k_select_global then
 * stores this rank's ShardBest records of a level straight into every rank's window over NVLink, publishes an epoch
 * flag and waits for the other ranks' flags in its own window: no collective call, no extra kernel per level. */
int64_t ygg_gbt_best_split_window_bytes(const ygg_gbt* h);
int ygg_gbt_set_best_split_window(ygg_gbt* h, void* const* peer_windows, int32_t world);

/* Tie-break replay (cfg.candidate_shuffle != 0; GetCandidateAttributes, training.cc:4293-4306): resolves the ties of
 * every tree trained so far and reports how many tied nodes were given the reference's feature (`renamed`) and how many
 * could not be (`unresolved`: the tied candidates cut the node's rows differently, or more than 3 features tied). */
int ygg_gbt_tie_stats(ygg_gbt* h, int64_t* renamed, int64_t* unresolved);
/* Positions the tie-break stream `words` engine words after the seed: for callers of ygg_tree_train_on_gradients (the
 * decision_tree::Train seam), whose trees are not grown in the handle's own boosting loop. */
int ygg_gbt_set_tie_rng_position(ygg_gbt* h, uint64_t words);

/* Copies tree `iter` (pre-order: node, neg subtree, pos subtree).  *n_nodes receives the node
 * count; fails with INVALID_ARGUMENT if capacity is too small. */
int ygg_gbt_get_tree(ygg_gbt* h, int32_t iter, ygg_node* out, int32_t capacity, int32_t* n_nodes);
/* Training loss / secondary metric after iteration `iter` (loss->Loss,
 * gradient_boosted_trees.cc:1575-1580): binomial => (2x mean log-loss, accuracy);
 * squared error => (rmse, rmse). */
int ygg_gbt_train_loss(ygg_gbt* h, int32_t iter, float* loss, float* secondary);
/* Current raw predictions (logits / regression values), N floats to host. */
int ygg_gbt_get_predictions(ygg_gbt* h, float* out, int64_t n);
/* Raw scores (before the loss' activation) of the trained model — the trees kept after early stopping — on ANY dataset that
 * has the training dataset's features and binning: out[k * n_rows + r], k < classes (1 unless multinomial).  The device
 * counterpart of ComputePredictions (gradient_boosted_trees.cc:2872-2930), e.g. to resume training from a model
 * (ygg_gbt_set_predictions) or to evaluate a test fold without leaving the GPU. */
int ygg_gbt_predict(ygg_gbt* h, const ygg_dataset* ds, float* out, int64_t n);

/* Overwrites the current predictions (warm start from another model; also the teacher-forcing hook of the parity tests). */
int ygg_gbt_set_predictions(ygg_gbt* h, const float* pred, int64_t n);

/* decision_tree::Train seam (learner/decision_tree/training.h:1012-1021): grows ONE regression
 * tree on caller-provided per-example gradients / hessians (host pointers) with the handle's
 * tree hyper-parameters; does not touch the boosting state. */
int ygg_tree_train_on_gradients(ygg_gbt* h, const float* gradients, const float* hessians,
                                ygg_node* out, int32_t capacity, int32_t* n_nodes);

/* Histogram capture, for tests of the histogram kernels (FillExampleBucketSet, learner/decision_tree/
 * splitter_scanner.h:859-909): while enabled, every tree grown (ygg_gbt_step / _train / ygg_tree_train_on_gradients)
 * copies each level's slot histograms, as the level's histogram launches left them on this rank (before any
 * collective), into a buffer of the handle.  Off: one host-side branch per level. */
int ygg_gbt_debug_capture_histograms(ygg_gbt* h, int32_t enabled);

/* Which histogram kernel / shared-memory layout filled a level (DESIGN.md §3, csrc/ygg_hist.cuh). */
enum ygg_hist_layout {
  YGG_HIST_LAYOUT_ROOT_SUM = 0,           /* k_hist at the root: low word + carry plane; counts from k_root_counts */
  YGG_HIST_LAYOUT_PACKED = 1,             /* k_hist: 13-bit count + 19-bit coarse sum, sum mod 2^32 */
  YGG_HIST_LAYOUT_SHARED = 2,             /* k_hist: 20-bit count + 12 carry bits, low word */
  YGG_HIST_LAYOUT_SHARED_HESS = 3,        /* YGG_HIST_LAYOUT_SHARED + the second plane (hessians or weights) */
  YGG_HIST_LAYOUT_PACKED_MULTI = 4,       /* the windowed instantiations: `passes` launches over windows of slots */
  YGG_HIST_LAYOUT_SHARED_MULTI = 5,
  YGG_HIST_LAYOUT_SHARED_HESS_MULTI = 6
};

typedef struct ygg_hist_level_info {
  int32_t layout;             /* enum ygg_hist_layout */
  int32_t features_per_item;  /* k_hist: G features per work item */
  int32_t smem_slots;         /* k_hist: slots in shared memory (windowed: window + 1 dummy slot) */
  int32_t passes;             /* launches of the level (> 1: windowed) */
  int32_t chunk_blocks;       /* 8192-row blocks per work item */
  int32_t reserved;           /* always 0 */
  int32_t num_slots;          /* histogram slots of the level */
  int32_t feature_begin;      /* histogrammed features of this rank: [feature_begin, feature_begin + num_features) */
  int32_t num_features;
  int32_t has_hsum;           /* 1: the level has the second plane */
  float g_pow2;               /* P: q = rint(g * 2^23 / P) + 2^23, clamped to [0, 2^24 - 1] */
  float h2_pow2;              /* second plane: hq = min(rint(v * 2^24 / h2_pow2), 2^24) */
  int64_t n_rows;             /* rows of this rank */
  /* in (may be NULL): host buffers of n_rows entries that receive the quantiser's float inputs of the captured tree:
   * the gradients, the second plane's values (hessians or weights; 1 when the loss has none) and the rows of the
   * iteration's sample (all 1 without sampling) */
  float* g;
  float* h2;
  uint8_t* selected;
} ygg_hist_level_info;

/* The capture of level `level` of the last tree grown with the capture on.  Fills `info` (see above).  With any
 * array non-NULL, they receive num_slots <= capacity slots: sum / hsum (u64) / cnt (u32) as [slot][feature][256]
 * over the rank's histogrammed features (sum = sum of q, hsum = sum of hq), slot_node[slot] = the index of the
 * slot's node in the array ygg_gbt_get_tree / ygg_tree_train_on_gradients return for that tree. */
int ygg_gbt_debug_level_histograms(ygg_gbt* h, int32_t level, ygg_hist_level_info* info, uint64_t* sum, uint64_t* hsum,
                                   uint32_t* cnt, int32_t* slot_node, int32_t capacity);

/* SplitExamplesInPlace seam (learner/decision_tree/training.cc:5243-5305 ->
 * model/decision_tree/decision_tree.cc:957-1012): stable two-way partition of a row-id list by
 * `bin(feature,row) >= threshold_bin`; positives then negatives, both ascending-stable.
 * rows_in/rows_out are host pointers of n entries; *n_pos receives the positive count. */
int ygg_partition_rows(ygg_dataset* ds, const uint32_t* rows_in, int64_t n, int32_t feature,
                       int32_t threshold_bin, uint32_t* rows_out, int64_t* n_pos);

/* Per-kernel device time of the last ygg_gbt_step/train call, in milliseconds, summed over
 * launches, measured with CUDA events on the handle's stream when profiling is enabled.
 * names: "grad", "hist", "scan", "select", "partition", "total". */
int ygg_gbt_set_profiling(ygg_gbt* h, int32_t enabled);
int ygg_gbt_get_profile(ygg_gbt* h, const char* name, double* ms, int64_t* launches);

/* model::SaveModel analogue (model/gradient_boosted_trees/gradient_boosted_trees.cc:111-139):
 * writes header.pb, data_spec.pb, gradient_boosted_trees_header.pb, nodes-00000-of-00001, done.
 * data_spec_pb / n: an already-serialised dataset::proto::DataSpecification (built by the host
 * harness, which owns column names and boundaries). */
int ygg_gbt_save_ydf(ygg_gbt* h, const char* directory, const char* label_name,
                     const uint8_t* data_spec_pb, int64_t data_spec_len, int32_t label_col_idx,
                     const int32_t* feature_col_idx);

#ifdef __cplusplus
}
#endif
#endif /* YGG_B200_H_ */
