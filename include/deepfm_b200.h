/*
 * deepfm_b200.h — C ABI of libdeepfm_b200.so: the B200-native (sm_100a) DeepFM / wide&deep
 * train step that sits directly beneath the reference's Estimator `model_fn`.
 *
 * The reference (leotimus/recommender-tensorflow) has no native seam of its own: every op of
 *   trainers/deep_fm.py:11-125      model_fn(features, labels, mode, params)
 *   trainers/linear_deep.py:32-39   DNNLinearCombinedClassifier(...)
 *   trainers/ml_100k.py:18-39       get_feature_columns()
 *   trainers/model_utils.py:57-66   get_optimizer()
 * is a TensorFlow-1.12 graph op.  This header is the seam a TF custom op (or the ctypes host in
 * recommender_tensorflow_b200/) binds: one handle = one model instance on one device.
 *
 * Conventions
 *  - plain C types only; every function returns an int status (0 = DFM_OK, negative = error) and
 *    never throws or aborts; dfm_last_error() gives the text of the last failure on a handle.
 *  - the caller owns every batch / output buffer; the handle owns tables, optimizer slots and
 *    workspaces.  Device-pointer entry points enqueue on the caller's cudaStream_t (passed as
 *    void*) and do not synchronise; *_host entry points take host pointers, copy inside and return
 *    after the result is on the host.
 *  - calls on one handle must be serialised by the caller.
 *  - categorical fields are processed in the order given in dfm_config.cat ("model order"; the
 *    host passes them sorted by column name exactly like tf.feature_column.input_layer /
 *    linear_model do, see SURVEY.md §8a row 2).
 */
#ifndef DEEPFM_B200_H_
#define DEEPFM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFM_OK                 0
#define DFM_ERR_INVALID_ARG   -1
#define DFM_ERR_CUDA          -2
#define DFM_ERR_OUT_OF_RANGE  -3   /* identity column value outside [0, num_buckets) */
#define DFM_ERR_UNSUPPORTED   -4
#define DFM_ERR_NCCL          -5
#define DFM_ERR_NOT_FOUND     -6
#define DFM_ERR_PARSE         -7   /* malformed CSV record (dfm_csv_decode) */

#define DFM_MAX_CAT     64
#define DFM_MAX_NUM     64
#define DFM_MAX_HIDDEN   8

/* column kinds — tf.feature_column.categorical_column_with_* (trainers/ml_100k.py:19-35) */
enum { DFM_COL_HASH = 0, DFM_COL_BUCKETIZED = 1, DFM_COL_VOCAB = 2, DFM_COL_IDENTITY = 3,
       /* tf.feature_column.crossed_column: model column whose ids are sparse_cross_hashed over source columns */
       DFM_COL_CROSSED = 4,
       /* a raw int32 / string feature used as it is; allowed only among dfm_config.src */
       DFM_COL_RAW = 5 };
#define DFM_MAX_CROSS_KEYS 8   /* constituents of one crossed column */
/* raw column dtypes — what tf.decode_csv yields (trainers/ml_100k.py:11-15,45) */
enum { DFM_INT32 = 0, DFM_FLOAT32 = 1, DFM_STRING = 2 };
/* optimizers — trainers/model_utils.py:57-66 */
enum { DFM_OPT_ADAM = 0, DFM_OPT_ADAGRAD = 1, DFM_OPT_FTRL = 2, DFM_OPT_SGD = 3, DFM_OPT_RMSPROP = 4 };
/* loss reduction — contrib binary head (mean, trainers/deep_fm.py:118) vs canned head (sum) */
enum { DFM_LOSS_MEAN = 0, DFM_LOSS_SUM = 1 };

/* One categorical feature column.  Replaces the _HashedCategoricalColumn / _BucketizedColumn /
 * _VocabularyListCategoricalColumn / _IdentityCategoricalColumn objects built at
 * trainers/ml_100k.py:19-35. */
typedef struct {
    const char*        name;          /* column name (model-order key) */
    int32_t            kind;          /* DFM_COL_* */
    int32_t            dtype;         /* DFM_INT32 | DFM_FLOAT32 | DFM_STRING of the raw column */
    int64_t            num_buckets;   /* hash / identity: N.  bucketized / vocab: derived, may be 0 */
    const float*       boundaries;    /* bucketized: ascending float32 boundaries */
    int32_t            n_boundaries;
    const char* const* vocab;         /* vocab: NUL-terminated strings */
    int32_t            vocab_size;
    int32_t            num_oov;       /* vocab: OOV hash buckets appended after the list */
    /* multivalent ("multi-hot") column: every sample carries `width` value slots (raw column = [B, width]
     * row-major; int32 slots padded with -1, string slots with ''); the embedding of the field is the MEAN of
     * the present slots (embedding_column combiner='mean'), the linear term their SUM (linear_model
     * sparse_combiner='sum'); an empty bag contributes zeros.  0 or 1 = single-valued. */
    int32_t            width;
    /* crossed column (kind DFM_COL_CROSSED, tf.feature_column.crossed_column): for every combination of one value of each
     * constituent, id = FingerprintCat64 chain over the constituents' values seeded with hash_key, mod num_buckets
     * (TF-1.12 sparse_cross_hashed).  keys[n_keys] index dfm_config.src in HASHING order (sparse constituents first:
     * categorical and multivalent raw sources, then single-valued raw sources; the caller orders them, the library
     * does not).  2 <= n_keys <= DFM_MAX_CROSS_KEYS.  hash_key 0 = TF's default 0xDECAFCAFFE.  width is derived: the
     * product of the constituents' widths.  The column's own cat_data entry is not read and may be NULL. */
    int32_t            n_keys;
    const int32_t*     keys;
    uint64_t           hash_key;
    /* vocabulary column, packed (tf.feature_column.categorical_column_with_vocabulary_list / _file).  dtype DFM_STRING:
     * entry j is the bytes vocab_data[vocab_offsets[j] .. vocab_offsets[j + 1]) (vocab_offsets has vocab_size + 1
     * monotone entries, total bytes < 2^31); used when `vocab` is NULL.  dtype DFM_INT32: vocab_int[vocab_size] int64
     * keys, matched against the sign-extended raw value (-1 is dropped before the lookup).  vocab_size >= 1.  A lookup
     * probes a device hash table keyed on the 64-bit fingerprint (strings: Fingerprint64, confirmed by a byte compare)
     * or on the key itself (ints); on duplicated entries the first occurrence wins. */
    const uint8_t*     vocab_data;
    const int64_t*     vocab_offsets;
    const int64_t*     vocab_int;
    /* has_default != 0: vocabulary column - an unknown key maps to default_value (-1 = dropped, else in
     * [0, vocab_size); not together with num_oov > 0); identity column - a value outside [0, num_buckets) maps to
     * default_value (in [0, num_buckets)) instead of failing with DFM_ERR_OUT_OF_RANGE.  0: unknown vocabulary keys
     * are dropped (-1), out-of-range identity values are an error. */
    int64_t            default_value;
    int32_t            has_default;
} dfm_column;

/* tf.train.*Optimizer(learning_rate) hyper-parameters (trainers/model_utils.py:57-66; TF defaults) */
typedef struct {
    int32_t kind;       /* DFM_OPT_* */
    float   lr;
    float   beta1, beta2, eps;   /* Adam: 0.9 0.999 1e-8.  RMSProp: beta1 = momentum (0), beta2 = decay (0.9), eps = 1e-10 */
    float   init_acc;            /* Adagrad / FTRL accumulators: 0.1.  RMSProp rms slot: 1.0 */
} dfm_optimizer;

/* params of model_fn (trainers/deep_fm.py:13-26) + the column lists it receives */
typedef struct {
    int32_t           n_cat;
    const dfm_column* cat;            /* categorical_columns, model order */
    int32_t           n_num;          /* numeric_columns (float32 inputs), model order */
    int32_t           embedding_size; /* k: multiple of 4 dividing 128 */
    int32_t           n_hidden;
    const int32_t*    hidden_units;
    int32_t           use_linear, use_mf, use_dnn;
    int32_t           loss_reduction; /* DFM_LOSS_* */
    dfm_optimizer     opt_deep;       /* embeddings, numeric_embeddings, DNN tower */
    dfm_optimizer     opt_linear;     /* linear tables, numeric linear weights, bias */
    int32_t           max_batch;      /* workspaces are sized for this many samples */
    int32_t           device;         /* CUDA device ordinal */
    /* row sharding (SURVEY.md §8e): this handle owns global rows {g : g mod world == rank} */
    int32_t           rank, world;
    void*             nccl_comm;      /* reserved (the host owns the communicator); pass NULL */
    /* tf.layers.dropout(net, rate=dropout, training=True) after every hidden layer in TRAIN mode
     * (trainers/deep_fm.py:102-103).  Own counter-based generator keyed on (seed, step, layer, element);
     * TF's RNG stream is not reproducible, the oracle restates this one. */
    float             dropout;
    /* the head (TF 1.12 contrib binary_classification_head / regression_head, canned *Classifier / *Regressor):
     * DFM_HEAD_LOGISTIC (0, a zeroed config): l_b = sigmoid cross-entropy, dz_b = sigmoid(z_b) - y_b, y in {0, 1}.
     * DFM_HEAD_SQUARED: l_b = (y_b - z_b)^2, dz_b = 2 (z_b - y_b), y any float32 (label_dimension 1, identity inverse
     * link: the prediction is the logit).  Then the loss_reduction scale, then the weight, as for the logistic head.
     * Any other value -> DFM_ERR_INVALID_ARG.  It fills the alignment gap before dropout_seed, so the size of the
     * struct and the offset of every other field are what they were without it. */
    int32_t           head;
    uint64_t          dropout_seed;
    /* params["activation"] (trainers/deep_fm.py:22,100; default tf.nn.relu): DFM_ACT_*.  Anything but ReLU runs the
     * general CUDA-core tower (the fused and tensor-core towers are built around the ReLU mask). */
    int32_t           activation;
    /* source columns: the inputs of crossed columns.  Kinds DFM_COL_RAW (int32 or string value, crossed as it is; width
     * > 1 makes it a sparse multivalent key whose -1 / '' padding slots are absent), DFM_COL_BUCKETIZED, DFM_COL_VOCAB,
     * DFM_COL_IDENTITY.  They own no table and have no place in model order; their raw data is
     * dfm_raw_batch.cat_data[n_cat + s] / cat_offsets[n_cat + s].  n_cat + n_src <= DFM_MAX_CAT. */
    int32_t           n_src;
    const dfm_column* src;
    /* weight_column of the canned estimators / binary head: nonzero makes every TRAIN batch carry per-example weights
     * (dfm_raw_batch.weights).  The per-sample loss and its gradient are multiplied by the weight:
     * SUM: loss = sum_b w_b l_b, dz_b = w_b (sigmoid(z_b) - y_b); MEAN: both divided by the (global) batch size, not by
     * sum w.  Zero, negative and fractional weights are accepted, as in TF.  0 = unweighted: weights is never read. */
    int32_t           weighted;
} dfm_config;

#define DFM_HEAD_LOGISTIC 0
#define DFM_HEAD_SQUARED  1

/* One batch of raw (un-hashed) feature columns = what input_fn's parse_csv yields
 * (trainers/ml_100k.py:44-49) for the columns the model consumes. */
typedef struct {
    int32_t               batch_size;
    const void* const*    cat_data;     /* [n_cat + n_src]: int32[B] | float32[B] | uint8 bytes (strings); the entry
                                           of a crossed column is ignored (may be NULL), source columns follow cat */
    const int32_t* const* cat_offsets;  /* [n_cat + n_src]: int32[B+1] byte offsets for string columns, else NULL */
    const float* const*   num_data;     /* [n_num]: float32[B] */
    const float*          labels;       /* [B] float32 labels; NULL for forward.  The logistic head takes 0/1 (rating >=
                                           cutoff, trainers/ml_100k.py:48), the squared head any value (the rating) */
    /* [B] float32 per-example weights, on the same side (host / device) as labels.  Read only by a handle created with
     * dfm_config.weighted != 0, and only by train steps and dfm_evaluate / dfm_evaluate_host (required there: NULL ->
     * DFM_ERR_INVALID_ARG); forward, PREDICT and layer_summary ignore it.  An unweighted handle never reads this field. */
    const float*          weights;
} dfm_raw_batch;

#define DFM_ACT_RELU 0
#define DFM_ACT_TANH 1
#define DFM_ACT_SIGMOID 2
#define DFM_ACT_IDENTITY 3

typedef struct dfm_handle dfm_handle;

/* Build a model instance: replaces graph construction inside model_fn (trainers/deep_fm.py:36-125).
 * Tables are zero-initialised; load weights with dfm_set_tensor or dfm_init_random. */
int dfm_create(const dfm_config* cfg, dfm_handle** out);
void dfm_destroy(dfm_handle* h);
const char* dfm_last_error(const dfm_handle* h);   /* h may be NULL: last dfm_create failure */

/* Variable access = tf.train.Saver / checkpoint surface (trainers/conf_utils.py:6-10).
 * Names: "emb" [R,k], "lin" [R], "num_emb" [dn,k], "num_lin" [dn], "bias" [1], "W<i>" [in,out],
 * "b<i>" [out], "Wo" [h,1], "bo" [1]; optimizer slots "<name>/m", "<name>/v" (Adam),
 * "<name>/acc" (Adagrad, FTRL), "<name>/lin" (FTRL), "<name>/rms", "<name>/mom" (RMSProp).  R = sum of the per-field bucket counts,
 * fields concatenated in model order.  Row ranges are in elements of the leading dimension.
 * dfm_get_tensor materialises any deferred non-lazy-Adam work first (dfm_flush). */
int dfm_tensor_rows(dfm_handle* h, const char* name, int64_t* rows, int64_t* row_elems);
int dfm_set_tensor(dfm_handle* h, const char* name, int64_t row_begin, int64_t n_rows, const float* host_src);
int dfm_get_tensor(dfm_handle* h, const char* name, int64_t row_begin, int64_t n_rows, float* host_dst);
/* reference initialisers run on the device (SURVEY.md A.2): tables truncated-normal(0, 1/sqrt(k)),
 * dense kernels glorot-uniform, linear + biases zero.  Own counter-based generator. */
int dfm_init_random(dfm_handle* h, uint64_t seed);

/* K1 alone: feature-column transforms (hash / bucketize / vocab / identity) -> ids [B, n_slots]
 * int32 (n_slots = sum of the column widths = n_cat when every column is single-valued), -1 = empty slot.  Device pointers.  Replaces the _transform_feature calls under
 * tf.feature_column.linear_model / input_layer (trainers/deep_fm.py:39,54). */
int dfm_transform(dfm_handle* h, const dfm_raw_batch* dev_batch, int32_t* ids_out_dev, void* stream);

/* One session.run(train_op) (trainers/deep_fm.py:119-125): forward, sigmoid-CE loss, backward,
 * sparse + dense optimizer apply, global_step += 1.  loss_out_dev [1], logits_out_dev [B] or NULL. */
int dfm_train_step(dfm_handle* h, const dfm_raw_batch* dev_batch, float* loss_out_dev,
                   float* logits_out_dev, void* stream);
/* Input-pipeline lookahead: transform + sort + segments of the NEXT device batch on the handle's side stream while the
 * current step runs; the dfm_train_step that follows on that batch adopts them (matched by first column pointer and
 * batch size, otherwise the prefetch is dropped).  after_stream: the stream that produced the batch, or NULL. */
int dfm_prefetch_batch(dfm_handle* h, const dfm_raw_batch* dev_batch, void* after_stream);
/* Same, from host buffers (pinned preferred): H2D of the raw columns, the step, D2H of the loss
 * (and logits if non-NULL).  Returns after the loss is on the host. */
int dfm_train_step_host(dfm_handle* h, const dfm_raw_batch* host_batch, float* loss_out_host,
                        float* logits_out_host);
/* Pipelined variant: enqueue step i, return the loss of the previously enqueued step in
 * *prev_loss_host (NaN on the first call).  dfm_train_step_host_drain waits for the last one. */
int dfm_train_step_host_async(dfm_handle* h, const dfm_raw_batch* host_batch, float* prev_loss_host);
int dfm_train_step_host_drain(dfm_handle* h, float* last_loss_host);

/* mode == EVAL / PREDICT: logits only, no state change (device pointers). */
int dfm_forward(dfm_handle* h, const dfm_raw_batch* dev_batch, float* logits_out_dev, void* stream);
int dfm_forward_host(dfm_handle* h, const dfm_raw_batch* host_batch, float* logits_out_host);

/* ---- EVAL metrics streamed on the device (csrc/metrics.cuh, DESIGN.md §8.6).  Every handle keeps one metric state in
 * device memory; each batch adds to it, and the host finishes the metrics of the handle's head from the raw state (the
 * states of several ranks are combined by summing the fields, in rank order).  Logistic head, as TF 1.12
 * metrics_impl / head.py: p = 1.f / (1.f + expf(-z)) in float32; bin = number of TF's 200 float32 AUC thresholds t with
 * p > t; positive = label > 0.5; predicted class = z > 0.  Squared head: only n and the four sums.  An unweighted
 * batch counts with w = 1, so the weighted fields hold unit-weight totals.  Counts are exact; the float64 fields are
 * summed in a fixed order, so a rerun gives the same bits. */
#define DFM_METRIC_BINS 201
typedef struct {
    int64_t n;                                  /* samples accumulated */
    int64_t bin_count[2][DFM_METRIC_BINS];      /* [0] negatives, [1] positives per bin (logistic head) */
    int64_t tp, fp, fn, correct;                /* class z > 0 against label > 0.5 (logistic head) */
    double  bin_weight[2][DFM_METRIC_BINS];     /* the same, sums of the weights */
    double  w_tp, w_fp, w_fn, w_correct;
    double  sum_w, sum_wy;                      /* sum w, sum w y */
    double  sum_wpred;                          /* logistic: sum w p (p in float64); squared: sum w z */
    double  sum_wloss;                          /* logistic: sum w (max(z,0) - z y + log1p(exp(-|z|))) in float64; squared: sum w (y - z)^2 */
} dfm_metric_state;
/* zero the handle's metric state */
int dfm_metrics_reset(dfm_handle* h, void* stream);
/* add n samples whose logits the caller already has (device pointers; the row-sharded ranks use this on their
 * dfm_shard_forward / dfm_xchg_forward output).  weights_dev: read on a weighted handle only, and required there. */
int dfm_metrics_accumulate(dfm_handle* h, const float* logits_dev, const float* labels_dev, const float* weights_dev, int64_t n,
                           void* stream);
/* the forward pass of dfm_forward into a handle workspace, then the accumulation of dev_batch->labels (required) and, on
 * a weighted handle, dev_batch->weights (required there).  Does not synchronise.  Unsharded handles only. */
int dfm_evaluate(dfm_handle* h, const dfm_raw_batch* dev_batch, void* stream);
/* the same from host buffers (the copy path of dfm_forward_host); returns after the batch was accumulated */
int dfm_evaluate_host(dfm_handle* h, const dfm_raw_batch* host_batch);
/* copy the state to the host (enqueued on stream, NULL = the handle's own) and synchronise that stream */
int dfm_metrics_read(dfm_handle* h, dfm_metric_state* out_host, void* stream);

/* ---- layer_summary side outputs (reference: trainers/model_utils.py:4-6 `layer_summary`, called at trainers/deep_fm.py:43
 * (linear logit), :89 (MF logit), :105 (every hidden layer, after dropout in TRAIN mode), :110 (DNN logit), :115 (logits)).
 * One call recomputes those tensors for a device batch with a forward pass on the weights as of the latest step and
 * reduces each to tf.nn.zero_fraction + the fields of TensorFlow's HistogramProto over its default bucket limits.
 * Tensor order: linear (if use_linear), mf (if use_mf), hidden layer 0..L-1 and dnn logit (if use_dnn), logits.
 * bucket_counts: [max_tensors][n limits] (may be NULL); train_mode != 0 applies the dropout mask of the NEXT train step. */
typedef struct dfm_tensor_summary { double min, max, num, sum, sum_squares, zero_fraction; } dfm_tensor_summary;
int dfm_summary_bucket_limits(double* limits_out, int32_t* n_out);
int dfm_layer_summary(dfm_handle* h, const dfm_raw_batch* dev_batch, int32_t train_mode, dfm_tensor_summary* out, int64_t* bucket_counts,
                      int32_t max_tensors, int32_t* n_tensors);
/* host copy of a tensor summarised by the last call: 0 linear, 1 mf, 2 hidden [B, sum of hidden_units], 3 dnn logit, 4 logits */
int dfm_layer_summary_tensor(dfm_handle* h, int32_t which, int64_t n, float* out_host);

/* Materialise deferred non-lazy Adam decay on every table row (before checkpoint / compare). */
int dfm_flush(dfm_handle* h, void* stream);
/* Wait for the handle's work and report sticky device-side errors (e.g. DFM_ERR_OUT_OF_RANGE). */
int dfm_sync(dfm_handle* h);

int64_t dfm_global_step(const dfm_handle* h);
/* Order-independent checksum (sum of the 32-bit patterns mod 2^64) of the whole trained state on this handle: table
 * records (weights, optimizer slots, last_step; deferred decay materialised first) and dense parameters + slots.
 * bench.py's multi-GPU parity_check compares it between the collective and the fused exchange. */
int dfm_state_checksum(dfm_handle* h, uint64_t* out_host);
/* unique table rows touched by the last step's batch (synchronises) */
int64_t dfm_last_unique_rows(dfm_handle* h);
/* Checkpoint restore (trainers/deep_fm.py:147-148 --restore; tf.train.Saver restores global_step and the
 * Adam beta powers): call after loading every variable and slot with dfm_set_tensor. */
int dfm_set_global_step(dfm_handle* h, int64_t step);
/* number of kernels the last train step launched (bench.py's gpu_launches) */
int64_t dfm_last_step_launches(const dfm_handle* h);
/* train steps replayed as one CUDA graph so far (dfm_train_step with batch_size <= 131072 on an unsharded handle captures
 * the step's kernels and launches them as a single graph: one session.run(train_op) = one launch; DFM_NO_GRAPH=1 disables) */
int64_t dfm_graph_steps(const dfm_handle* h);
/* device time (ms) spent in the named phase during the last *timed* step; enable with
 * dfm_set_profiling(h, 1).  Phases: "transform","sort","segments","catchup","gather","mlp_fwd",
 * "loss","mlp_bwd","reduce","update","dense". Returns <0 if unknown. */
int dfm_set_profiling(dfm_handle* h, int32_t on);
float dfm_phase_ms(dfm_handle* h, const char* phase);

/* ---- Row sharding over the GPUs of one box (SURVEY.md 8e; BASELINE.json configs[3], configs[4]).
 * A handle created with world > 1 owns global rows {g : g % world == rank} (local index g / world) of
 * the concatenated embedding + linear tables; the dense tower is replicated.  One train step is the
 * four calls below on every rank, with the collectives between them done by the host over
 * NCCL / NVLink (torch.distributed): all_to_all(counts), all_to_all(row ids), all_to_all(rows),
 * all_to_all(gradient rows), all_reduce(dense gradients, loss).  Row payloads are K+4 floats
 * {emb[K], linear weight, pad} (dfm_shard_row_width).
 *   dfm_shard_requests          K1 + sort + unique rows of the local batch; req_rows_out_dev (capacity
 *                               batch*n_cat) receives the owner-major unique local-row ids, counts_host[world]
 *                               the number per owner.  Synchronises the stream (the host needs the counts).
 *   dfm_shard_serve             owner side: sort the received ids, bring those rows up to date (non-lazy
 *                               Adam), reply_dev[i] = row payload of recv_rows_dev[i]
 *   dfm_shard_forward_backward  forward / loss / backward of the local batch from rowbuf_dev[U, K+4];
 *                               writes gsum_dev[U, K+4] (per unique row, deterministic order), the local
 *                               dense gradients (dfm_dense_size floats) and loss = local sum / global_batch
 *   dfm_shard_apply             owner side: ordered reduction of grecv_dev[n_recv, K+4] by row + sparse
 *                               optimizer; dense optimizer with the all-reduced dense gradients; step += 1 */
int dfm_shard_row_width(const dfm_handle* h);
int dfm_num_slots(const dfm_handle* h);      /* value slots per sample = sum of the column widths */
int64_t dfm_dense_size(const dfm_handle* h);
int dfm_shard_requests(dfm_handle* h, const dfm_raw_batch* dev_batch, uint32_t* req_rows_out_dev, int32_t* counts_host, void* stream);
int dfm_shard_serve(dfm_handle* h, const uint32_t* recv_rows_dev, int64_t n_recv, float* reply_dev, void* stream);
int dfm_shard_forward_backward(dfm_handle* h, const dfm_raw_batch* dev_batch, const float* rowbuf_dev, int64_t global_batch,
                               float* loss_dev, float* logits_dev, float* gsum_dev, float* dense_grad_dev, void* stream);
int dfm_shard_apply(dfm_handle* h, const float* grecv_dev, const float* dense_grad_dev, void* stream);

/* EVAL / PREDICT on a row-sharded model (collective path): after requests -> serve (and the two exchanges) the
 * forward pass alone on rowbuf_dev. */
int dfm_shard_forward(dfm_handle* h, const dfm_raw_batch* dev_batch, const float* rowbuf_dev, float* logits_dev, void* stream);

/* ---- The same sharded step with the exchanges FUSED into the kernels over NVLink peer memory and synchronised by
 * flags in that memory (csrc/xchg.cuh): no collective, no host round trip, no count exchange.  Every rank owns one
 * exchange region (fixed-capacity id / gradient-row segments per (source, owner), a row buffer, dense-gradient slots,
 * flags) that is mapped into the other ranks through CUDA IPC (dfm_xchg_export / _import, handles exchanged by the host
 * ONCE).  Producer kernels store into the consumer's region and stamp its flag (st.release.sys); the consumer's
 * stream carries a one-warp wait kernel (ld.acquire.sys) in front of the kernel that reads the payload.
 *   dfm_xchg_begin              K1 + owner-major unique rows of the local batch; ids -> the owners' regions
 *   dfm_xchg_serve              | wait ids  | rows as of step t-1 -> the requesters' row buffers (train != 0: the
 *                                            received ids are also sorted, on the handle's side stream, for the apply)
 *   dfm_xchg_forward_backward   | wait rows | forward / loss / backward; per-unique-row gradient sums -> the owners'
 *                                            regions; dense gradients + loss share -> every rank's dense slots
 *   dfm_xchg_apply              | wait gradient rows | ordered reduction by row + sparse optimizer
 *                               | wait dense         | sum of the slots in rank order + dense optimizer; step += 1;
 *                                                      loss_out_dev [1] = global loss
 *   dfm_xchg_train_step         the four phases back to back (one process per GPU: launches only)
 *   dfm_xchg_forward            EVAL / PREDICT: after begin + serve(train = 0), the forward pass alone
 * A host that runs all ranks in one process on one GPU (the tests) calls the phases rank by rank, so that a flag is
 * always set before the kernel that waits for it starts.  A wait gives up after 4 s (a peer died): dfm_sync then
 * reports DFM_ERR_PEER. */
#define DFM_ERR_PEER          -8
int dfm_xchg_export(dfm_handle* h, unsigned char* handle_out /* 64 bytes */);
int dfm_xchg_import(dfm_handle* h, const unsigned char* all_handles /* world * 64 bytes, rank order */);
int dfm_xchg_buffer(dfm_handle* h, void** region_out);
int dfm_xchg_set_peers(dfm_handle* h, void* const* regions /* world, rank order */);
int dfm_xchg_begin(dfm_handle* h, const dfm_raw_batch* dev_batch, void* stream);
int dfm_xchg_serve(dfm_handle* h, int32_t train, void* stream);
int dfm_xchg_forward_backward(dfm_handle* h, const dfm_raw_batch* dev_batch, int64_t global_batch, float* logits_dev, void* stream);
int dfm_xchg_apply(dfm_handle* h, float* loss_out_dev, void* stream);
int dfm_xchg_train_step(dfm_handle* h, const dfm_raw_batch* dev_batch, int64_t global_batch, float* loss_out_dev, float* logits_dev,
                        void* stream);
/* the step + the requests of next_batch (may be NULL) issued beside this step's owner-side apply; the next call must train next_batch */
int dfm_xchg_train_step_next(dfm_handle* h, const dfm_raw_batch* dev_batch, const dfm_raw_batch* next_batch, int64_t global_batch,
                             float* loss_out_dev, float* logits_dev, void* stream);
int dfm_xchg_forward(dfm_handle* h, const dfm_raw_batch* dev_batch, float* logits_dev, void* stream);

/* Building-block entry points used by the parity tests (device pointers, synchronous). */
int dfm_test_sort_pairs(uint32_t* keys_dev, uint32_t* vals_dev, int64_t n, int32_t key_bits);
/* algo 0: multi-launch LSD radix sort; 1: one-sweep (decoupled look-back); 2: one-sweep with the element count read
 * from device memory by the kernels (the row-sharded owner side never tells the host how many requests arrived) */
int dfm_test_sort_pairs_algo(uint32_t* keys_dev, uint32_t* vals_dev, int64_t n, int32_t key_bits, int32_t algo);
int dfm_test_fingerprint64(const uint8_t* bytes_dev, const int32_t* offsets_dev, int64_t n,
                           uint64_t* out_dev);

/* Non-lazy Adam replay in isolation (csrc/replay.cuh): element i (device arrays) is taken from step last[i] to step
 * upto by `m *= b1; v *= b2; w -= alpha_t m / (sqrt(v) + eps)` per skipped step — in closed form, or step by step
 * when force_loop != 0 (the fallback used for hyper-parameters outside the closed form's range). */
int dfm_test_replay(const dfm_optimizer* opt, float* w_dev, float* m_dev, float* v_dev, const int32_t* last_dev, int64_t n,
                    int32_t upto, int32_t force_loop);

/* 3xTF32 tcgen05 GEMM of the DNN tower in isolation (device pointers, synchronous):
 * mode 0: C[M,N] = A[M,K] * B[N,K]^T;  mode 2: same, B pre-split into tf32 hi/lo (weight path);
 * mode 1: C[M,N] = A[K,M]^T * B[K,N] through `splits` ordered partials (weight-gradient path). */
int dfm_test_tc_gemm(int32_t mode, const float* A_dev, const float* B_dev, float* C_dev, int32_t M, int32_t N,
                     int32_t K, int32_t splits);

/* ---- GPU CSV record decoder: replaces tf.data.TextLineDataset(csv) + tf.decode_csv(value, DEFAULTS) of the
 * reference's input_fn (trainers/ml_100k.py:44-58; schema COLUMNS / DEFAULTS, trainers/ml_100k.py:3-15) for the
 * fields the model consumes.  The host hands over whole records (lines); field splitting, RFC-4180 unquoting
 * ('""' inside a quoted field), int32 and float32 parsing, default substitution for empty fields and the label
 * threshold (rating >= cutoff, trainers/ml_100k.py:47-48; or the raw rating with label_raw) run on the device.  The decoded columns stay in the
 * reader's device buffers in the layout dfm_raw_batch takes: int32[n] and float32[n] columns, Arrow-style string
 * columns (int32 offsets[n+1] + bytes), float labels[n].  Float32 fields follow TF 1.12's strings::safe_strtof,
 * correctly rounded (oracle/strtof.py states the grammar), except that hexadecimal is rejected.  Errors follow
 * tf.decode_csv: wrong field count, a field that is not a valid int32 or float32, a quote inside an unquoted field
 * or an unterminated quote -> DFM_ERR_PARSE, with the first offending record in dfm_csv_last_error. */
#define DFM_CSV_SKIP    0          /* parsed for structure only (15 of the 42 ML-100K fields are never consumed) */
#define DFM_CSV_INT32   1          /* record_defaults [0]      */
#define DFM_CSV_STRING  2          /* record_defaults ["null"] */
#define DFM_CSV_FLOAT32 3          /* record_defaults [0.0]    */
#define DFM_CSV_ERR_FIELDS 1
#define DFM_CSV_ERR_INT    2
#define DFM_CSV_ERR_QUOTE  3
#define DFM_CSV_ERR_FLOAT  4
typedef struct {
    int32_t            n_fields;       /* fields per record (42) */
    const int32_t*     kind;           /* [n_fields] DFM_CSV_* */
    const int32_t*     int_default;    /* [n_fields] value of an empty int32 field (NULL: 0) */
    const char* const* str_default;    /* [n_fields] value of an empty string field (NULL entries: "") */
    int32_t            label_field;    /* int32 field the label is derived from (float32 too with label_raw), -1: none */
    int32_t            label_min;      /* label = value >= label_min */
    int32_t            max_records;    /* per decode call */
    int64_t            max_bytes;      /* per decode call, < 4 GiB */
    int32_t            device;
    const float*       float_default;  /* [n_fields] value of an empty float32 field (NULL: 0.0f) */
    int32_t            field_delim;    /* field separator, one byte other than '"', '\n' and '\r' (0: ',') */
    const int32_t*     as_float;       /* [n_fields] nonzero on an int32 field: also write it as float32, rounded to
                                          nearest (tf.to_float of a numeric_column over an int field); NULL: none */
    int32_t            label_raw;      /* nonzero: the label is the label field's value as float32 (tf.to_float: an
                                          int32 field rounded to nearest, or a float32 field) and label_min is not
                                          used - the regression head's label.  0: label = value >= label_min */
} dfm_csv_config;
typedef struct dfm_csv_reader dfm_csv_reader;
int dfm_csv_create(const dfm_csv_config* cfg, dfm_csv_reader** out);
void dfm_csv_destroy(dfm_csv_reader* r);
const char* dfm_csv_last_error(const dfm_csv_reader* r);
/* text: whole records, '\n'-terminated ('\r\n' tolerated, the last record may lack the newline).  Device variant:
 * 16-byte aligned and readable up to the next multiple of 16.  Both return after the decode finished (the record
 * count and the parse status need one synchronisation of the stream). */
int dfm_csv_decode(dfm_csv_reader* r, const char* text_dev, int64_t n_bytes, int32_t* n_records_out, void* stream);
int dfm_csv_decode_host(dfm_csv_reader* r, const char* text_host, int64_t n_bytes, int32_t* n_records_out, void* stream);
/* File-resident mode: upload the whole CSV text once (it is split into lines on the device; line 0 is usually the
 * header), then decode batches given as lists of line numbers — what shuffle(16*B).repeat().batch(B) of the reference's
 * input_fn selects (trainers/ml_100k.py:53-58).  Per batch the host sends 4 bytes per record. */
int dfm_csv_load(dfm_csv_reader* r, const char* text_host, int64_t n_bytes, int64_t* n_lines_out);
int dfm_csv_decode_lines(dfm_csv_reader* r, const int32_t* line_idx_host, int32_t n, void* stream);
int32_t dfm_csv_num_records(const dfm_csv_reader* r);
const int32_t* dfm_csv_int_column(const dfm_csv_reader* r, int32_t field);     /* device int32[n_records] */
const char*    dfm_csv_str_bytes(const dfm_csv_reader* r, int32_t field);      /* device bytes */
const int32_t* dfm_csv_str_offsets(const dfm_csv_reader* r, int32_t field);    /* device int32[n_records + 1] */
/* device float32[n_records] of a float32 field or of an int32 field with as_float; NULL for any other field */
const float*   dfm_csv_float_column(const dfm_csv_reader* r, int32_t field);
const float*   dfm_csv_labels(const dfm_csv_reader* r);                        /* device float[n_records] */

const char* dfm_version(void);

#ifdef __cplusplus
}
#endif
#endif  /* DEEPFM_B200_H_ */
