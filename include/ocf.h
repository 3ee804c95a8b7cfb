/* ocf.h - C ABI of the B200-native training/scoring hot path (libocf_b200.so).
 *
 * The reference (Epist/omnidirectional_collaborative_filtering) has no FFI: its seam is two
 * Python classes and the Keras Model methods train.py calls. Each entry point below names the
 * reference interface it replaces (file:line in the reference tree); INTEGRATION.md shows the
 * ctypes binding a reference maintainer would add at those call sites.
 *
 * Conventions
 *   - every function returns 0 on success, a negative ocf_status otherwise;
 *     ocf_last_error() gives the message of the calling thread's last failure
 *   - plain pointers and sizes only; no C++ exceptions cross the boundary
 *   - HOST pointers unless a parameter is documented as a device pointer; the caller owns every
 *     host buffer, the library owns all device memory behind its handles
 *   - `stream` is a cudaStream_t passed as void* (NULL = the legacy default stream); calls
 *     enqueue work on it and return without synchronising unless they hand results back to a
 *     host buffer
 *   - a handle lives on the device that was current when it was created; handles are not
 *     thread-safe
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails
 */
#ifndef OCF_H
#define OCF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OCF_VERSION 101

typedef enum {
  OCF_OK = 0,
  OCF_ERR_INVALID = -1,   /* bad argument / unsupported configuration            */
  OCF_ERR_CUDA = -2,      /* a CUDA runtime call failed (message has the detail)  */
  OCF_ERR_NOMEM = -3,
  OCF_ERR_STATE = -4      /* call order (e.g. train step on an eval batch)        */
} ocf_status;

typedef enum { OCF_ACT_LINEAR = 0, OCF_ACT_SIGMOID, OCF_ACT_TANH, OCF_ACT_RELU,
               OCF_ACT_ELU, OCF_ACT_SELU, OCF_ACT_SOFTPLUS } ocf_activation;
/* auxilliary_mask_type, data_reader.py:341-361 */
typedef enum { OCF_AUX_NONE = 0, OCF_AUX_CAUSAL, OCF_AUX_DROPOUT, OCF_AUX_ZEROS, OCF_AUX_BOTH } ocf_aux;
/* model_loss, train.py:49 */
typedef enum { OCF_LOSS_MSE = 0, OCF_LOSS_MAE = 1 } ocf_loss;
/* optimizer, train.py:50-51 / train_jester.py:61 */
typedef enum { OCF_OPT_SGD = 0, OCF_OPT_ADAGRAD, OCF_OPT_RMSPROP, OCF_OPT_ADAM } ocf_optimizer;

typedef struct ocf_store ocf_store;   /* device-resident rating store (CSR)                  */
typedef struct ocf_pair ocf_pair;     /* (input store, target store) of a fixed-split set    */
typedef struct ocf_batch ocf_batch;   /* one batch: row ids, keep-flags, gathered tiles      */
typedef struct ocf_model ocf_model;   /* weights, optimizer state, workspaces                */
typedef struct ocf_rng ocf_rng;       /* NumPy's MT19937 stream, resident on the device      */
typedef struct ocf_comm ocf_comm;     /* one rank of an NCCL communicator (one process per GPU) */

const char* ocf_last_error(void);
int ocf_version(void);
/* Number of CUDA devices visible (0 without a GPU; never fails). */
int ocf_device_count(void);
/* Page-locked host memory for the [rows, n_cols] outputs of ocf_predict / ocf_score (a pageable
 * destination makes the device->host copy several times slower). */
int ocf_host_alloc(int64_t bytes, void** out);
int ocf_host_free(void* ptr);

/* ---- rating store ------------------------------------------------------------------------
 * Replaces the per-row (item, rating) lists the reader keeps after loading
 * (data_reader.py:46-70) together with the id->dense-column map (data_reader.py:24-28, applied
 * by the caller: `col` already holds dense columns). Rows keep their stored order: draw j of
 * the reciprocal dropout belongs to the j-th stored rating (data_reader.py:130-134).
 * Repeated columns inside a row are allowed and resolve last-write-wins like the dense fills
 * at data_reader.py:158-169.
 * Limits: nnz < 2^31, n_cols < 2^31. */
int ocf_store_create(int64_t n_rows, int64_t n_cols, const int64_t* rowptr, const int32_t* col,
                     const float* val, ocf_store** out);
int ocf_store_destroy(ocf_store* store);
/* info[0]=n_rows, [1]=n_cols, [2]=nnz, [3]=1 if any row repeats a column, [4]=device bytes held */
int ocf_store_info(const ocf_store* store, int64_t info[5]);

/* Fixed-split valid/test set: row r of `in_store` holds the inputs of row r of `tgt_store`
 * (user_dicts_valid[0]/[1], data_reader.py:372-380; a None input row is an empty row). */
int ocf_pair_create(const ocf_store* in_store, const ocf_store* tgt_store, ocf_pair** out);
int ocf_pair_destroy(ocf_pair* pair);

/* ---- batch construction (kernel K1) -------------------------------------------------------
 * A batch object owns pinned staging, device tiles and the row->slot map; create a few and
 * rotate them to overlap the next batch's upload with the current step. */
int ocf_batch_create(int32_t max_rows, int64_t max_entries, ocf_batch** out);
int ocf_batch_destroy(ocf_batch* batch);

/* build_sparse_batch, data_reader.py:95-200 (dense branch), without the dense arrays:
 * keep_flags[k] is the reference's random_dropout_split value of the k-th rating of the batch
 * (rows in batch order, ratings in stored order): 1 = input (and target too when
 * pass_through), 0 = target. n_flags must equal the total length of the listed rows.
 * One host->device copy + one kernel on `stream`. */
int ocf_batch_fill_split(ocf_batch* batch, const ocf_store* store, const int32_t* row_ids,
                         int32_t n_rows, const uint8_t* keep_flags, int64_t n_flags,
                         int pass_through, float aux_var_value, void* stream);
/* Same batch from the raw uniform draws instead of keep flags: u[k] is the k-th double the
 * reference's np.random.choice calls consume (one per rating of the FULL rows, batch order),
 * cdf0[r] = (1-s_r)/((1-s_r)+s_r) of batch row r; flag = (u >= cdf0) (data_reader.py:120,130).
 * For a column shard, orig_pos[e] is the position of the shard's store entry e inside its full
 * row and full_len[r] the full length of batch row r (both NULL for an unsharded store). */
int ocf_batch_fill_split_uniform(ocf_batch* batch, const ocf_store* store, const int32_t* row_ids,
                                 int32_t n_rows, const double* u, int64_t n_u, const double* cdf0,
                                 const int32_t* orig_pos, const int64_t* full_len, int pass_through,
                                 float aux_var_value, void* stream);
/* The reference draws its reciprocal-dropout split from NumPy's global MT19937 stream
 * (np.random.uniform at data_reader.py:120, np.random.choice at :130). An ocf_rng holds that
 * stream on the device: set_state takes RandomState.get_state()[1:3] (key[624], pos), get_state
 * returns them at the consumers' position. The stream is produced ahead of its consumers, in blocks of
 * `block_regens` regenerations of the 624-word array, by `workers` generator CTAs on their own CUDA
 * streams: worker j makes blocks j, j + workers, ... and skips the others' blocks with a GF(2)
 * polynomial jump - bit for bit the sequential stream, at `workers` times the rate of one chain.
 * The blocks live in a ring of at least ring_words_min words (+ room for the blocks in flight); a
 * batch larger than the ring makes it grow. */
int ocf_rng_create(ocf_rng** out);                        /* workers = $OCF_RNG_WORKERS or 2, blocks of 256 regenerations */
int ocf_rng_configure(ocf_rng* rng, int32_t workers, int32_t block_regens, int64_t ring_words_min);   /* <= 0: keep; keeps the stream state */
int ocf_rng_destroy(ocf_rng* rng);
int ocf_rng_set_state(ocf_rng* rng, const uint32_t* key, int32_t pos);
int ocf_rng_get_state(ocf_rng* rng, uint32_t* key, int32_t* pos);
/* Advances the consumers' position by n_draws doubles (a batch the generator drew but nobody consumed). */
int ocf_rng_skip(ocf_rng* rng, int64_t n_draws);
/* Makes sure the blocks holding the next n_draws doubles are being generated (as far as the ring has room). */
int ocf_rng_prefetch(ocf_rng* rng, int64_t n_draws);
/* info[0..5] = workers, block_regens, ring blocks, ring words, consumers' position (words), blocks enqueued. */
int ocf_rng_info(const ocf_rng* rng, int64_t info[6]);
/* SM cycles and nanoseconds the last block-generation kernel took (synchronises the workers). */
int ocf_rng_last_timing(ocf_rng* rng, int64_t* sm_cycles, int64_t* nanoseconds);
/* Host side of the jump (no GPU needed): poly624 = x^n_words mod phi(x) as 624 32-bit words (phi = the
 * characteristic polynomial of MT19937's word recurrence, recovered by Berlekamp-Massey), and the array n_words
 * further down the stream than key624, computed the way the device kernel does (word 0 exact in its top bit only,
 * the only bit of it MT19937 reads). */
int ocf_mt_jump_poly(int64_t n_words, uint32_t* poly624);
int ocf_mt_jump_apply_host(const uint32_t* key624, const uint32_t* poly624, uint32_t* out624);
/* Column shards: orig_pos[e] = position of the shard's store entry e inside its full row. */
int ocf_store_set_orig_pos(ocf_store* store, const int32_t* orig_pos);
/* build_sparse_batch (data_reader.py:95-200) with the random split drawn ON THE DEVICE, bit for
 * bit what the reference draws: the stream's next n_rows doubles are
 * np.random.uniform(lo, hi, size=n_rows) (:120), the following sum(len(row)) doubles are the
 * rows' np.random.choice draws in batch order (:130). Nothing but the row ids crosses PCIe.
 * full_len[r] (column shards, else NULL) = full length of batch row r.
 * slice (row-parallel ranks, else NULL): the listed rows are rows [row0, row0 + n_rows) of a
 * larger drawing unit of n_draw_rows rows (the global batch); draws_before = ratings of the
 * unit's rows before row0, draws_total = n_draw_rows + all its ratings. Every rank advances its
 * copy of the stream by the whole unit and reads its own rows' draws. */
typedef struct {
  int32_t n_draw_rows;
  int32_t row0;
  int64_t draws_before;
  int64_t draws_total;
} ocf_rng_slice;
int ocf_batch_fill_split_rng(ocf_batch* batch, const ocf_store* store, const int32_t* row_ids,
                             int32_t n_rows, ocf_rng* rng, double lo, double hi,
                             const int64_t* full_len, int pass_through, float aux_var_value,
                             const ocf_rng_slice* slice, void* stream);
/* The keep flags of a split batch as the device holds them (synchronises `stream`). */
int ocf_batch_read_flags(ocf_batch* batch, uint8_t* out, int64_t count, void* stream);
/* build_sparse_batch_fixed_split, data_reader.py:202-298. */
int ocf_batch_fill_fixed(ocf_batch* batch, const ocf_pair* pair, const int32_t* row_ids,
                         int32_t n_rows, float aux_var_value, void* stream);
/* Re-runs K1 on the row ids / keep flags already resident in the batch's device staging (no
 * host->device copy). */
int ocf_batch_regather(ocf_batch* batch, void* stream);
/* info[0]=rows, [1]=entries, [2]=work items, [3]=target_count (data_reader.py:268; ratings
 * listed as targets, repeats included), [4]=bytes of the last host->device copy */
int ocf_batch_info(const ocf_batch* batch, int64_t info[5]);
/* The dense [rows, n_cols] float64 arrays the reference generator yields (the scatter half of
 * K1; for parity tests and callers that still want Keras-style feeds). which: 0 = inputs
 * (ratings_batch_inputs), 1 = input mask, 2 = output mask, 3 = targets, 4 = missing-data mask
 * (data_reader.py:191-200). Synchronises `stream`. */
int ocf_batch_densify(const ocf_batch* batch, int which, double* out, void* stream);

/* ---- model --------------------------------------------------------------------------------
 * omni_model, model.py:33-99, plus compile(), train.py:131-133. */
typedef struct {
  int32_t n_cols;            /* input_shape: width of this rank's column slice (== n_cols_total unsharded) */
  int32_t n_cols_total;      /* catalogue width N the loss is normalised by (B*N, train.py:49) */
  int32_t n_layers;          /* numlayers (hidden Dense layers), 1..8 */
  int32_t widths[8];         /* num_hidden_units per hidden layer (the reference uses one width) */
  int32_t aux;               /* ocf_aux: which mask blocks are concatenated to the data (model.py:47-56) */
  int32_t activation;        /* ocf_activation, dense_activation */
  int32_t loss;              /* ocf_loss */
  float l2;                  /* l2_weight_regulatization, < 0 = None */
  float dropout_p;           /* dropout_probability, < 0 = None */
  float aux_var_value;       /* value masks carry (train.py:47) */
  float rating_range;        /* for nMAE (train.py:118-121) */
  int32_t max_rows;          /* largest batch */
  int64_t max_entries;       /* most ratings in one batch */
  int32_t sharded;           /* 1: column shard; z/dh/row statistics are partial until reduced */
} ocf_model_config;

int ocf_model_create(const ocf_model_config* cfg, ocf_model** out);
int ocf_model_destroy(ocf_model* model);
/* Grow the batch-sized workspaces (weights and optimizer state are kept). No-op when the model
 * already holds max_rows rows and max_entries ratings per batch. */
int ocf_model_reserve(ocf_model* model, int32_t max_rows, int64_t max_entries);
/* Keras get_weights()/set_weights() order and layout (model.py:102-107): for each Dense layer
 * kernel [fan_in, fan_out] row-major then bias [fan_out]; layer 0 has fan_in = k*n_cols
 * (data | aux | second mask blocks), the last layer fan_out = n_cols.
 * index = 2*layer (+1 for the bias). Setting a weight does not touch optimizer state. */
int ocf_model_num_weights(const ocf_model* model);
int ocf_model_weight_shape(const ocf_model* model, int index, int64_t shape[2]);
int ocf_model_set_weight(ocf_model* model, int index, const float* host, int64_t count);
int ocf_model_get_weight(const ocf_model* model, int index, float* host, int64_t count);
/* Optimizer (Keras 2.0.4 rules). p1 = rho (RMSprop) or beta_1 (Adam), p2 = beta_2.
 * Resets the optimizer state and the iteration counter. */
int ocf_model_set_optimizer(ocf_model* model, int kind, float lr, float p1, float p2,
                            float epsilon, float decay);
/* compile(loss=...), train.py:131-133; rating_range feeds nMAE (train.py:118-121). */
int ocf_model_set_loss(ocf_model* model, int loss, float rating_range);
/* Which mask the reader feeds into the auxiliary input block(s) (auxilliary_mask_type,
 * data_reader.py:341-361). Must keep the number of blocks the model was created with. */
int ocf_model_set_aux(ocf_model* model, int aux);
/* layer.trainable (model.py:125,136-140,162,167); layer in [0, n_layers]. */
int ocf_model_set_trainable(ocf_model* model, int layer, int trainable);
int ocf_model_reset_optimizer(ocf_model* model);

typedef struct {
  uint64_t dropout_seed;     /* Philox key of the hidden dropout masks (oracle/philox.py) */
  uint32_t step;             /* counter word; normally the running step index */
  int32_t row0;              /* global index of this batch's first row (multi-GPU row slices) */
  int32_t rows_total;        /* B of the loss normalisation; 0 = the batch's own row count */
  int32_t phase;             /* 0 = whole step; 1..3 = sharded phases (see below) */
} ocf_step_args;

/* Metrics of one step, train.py:102-121 + the Keras loss:
 * [0] loss (with the L2 term) [1] mean_absolute_error [2] accurate_MAE [3] nMAE
 * [4] accurate_RMSE [5] accurate_MSE [6] sum of squared errors [7] count_nonzero(t+y) */
#define OCF_N_METRICS 8

/* One optimisation step on a split batch: model.train_on_batch as driven by fit_generator,
 * train.py:157. Metrics are computed before the update with dropout active, as in Keras.
 * host_metrics may be NULL: the values stay in the device log (ocf_model_read_metrics) and
 * the call does not synchronise.
 * Sharded models run the step in three phases with a collective between them (the caller
 * reduces the buffer ocf_model_buffer() names, in place, over the column shards):
 *   phase 1: gather + encoder partial sums        -> all-reduce OCF_BUF_Z
 *   phase 2: activations, decoder, loss partials  -> all-reduce OCF_BUF_DH and OCF_BUF_ROWSTATS
 *   phase 3: backward, fused optimizer update, metrics
 * A phase-0 step of an unsharded model also enqueues, on the batch's own stream and right behind the batch's fill, the
 * grouping of the batch's ratings by catalogue column that the update walks (it depends on the batch alone): by the
 * time the caller's stream reaches the step the list is there. Stepping the same fill again reuses it. */
int ocf_train_step(ocf_model* model, ocf_batch* batch, const ocf_step_args* args,
                   float* host_metrics, void* stream);
/* model.test_on_batch as driven by evaluate_generator (train.py:208,218): forward only,
 * dropout off. Sharded: phases 1, 2 then 3 (metrics only). */
int ocf_eval_step(ocf_model* model, ocf_batch* batch, const ocf_step_args* args,
                  float* host_metrics, void* stream);
/* model.predict (train.py:239): out[rows, n_cols] = output_mask * full_predictions.
 * Sharded models: the caller runs ocf_eval_step phase 1 and the OCF_BUF_Z all-reduce first; the
 * output holds this shard's columns. The same holds for ocf_score. */
int ocf_predict(ocf_model* model, ocf_batch* batch, float* out, void* stream);
/* Full-catalogue scoring: out[rows, n_cols] = full_predictions (model.py:82-84, the tensor
 * before the mask multiply). `out_is_device` != 0: out is a device pointer and the call does
 * not synchronise. */
int ocf_score(ocf_model* model, ocf_batch* batch, float* out, int out_is_device, void* stream);
/* Top-k serving epilogue on top of ocf_score (SURVEY.md section 8f-4): for every batch row the k
 * (<= 512) highest full-catalogue scores and their columns, best first (ties: lower column first),
 * selected on the device so that k pairs per row cross PCIe instead of n_cols scores.
 * exclude_inputs != 0 drops the columns the row holds as inputs (what the user has rated already).
 * out_cols int32[rows, k], out_scores float[rows, k] (host). Slots beyond the available columns
 * hold column -1 / score -inf. Column shards return their own columns' top k (local ids). */
int ocf_score_topk(ocf_model* model, ocf_batch* batch, int32_t k, int exclude_inputs,
                   int32_t* out_cols, float* out_scores, void* stream);
/* Ranking evaluation on top of ocf_score (see DESIGN): for every batch entry that is a relevant
 * target, its 1-based rank among the row's candidate columns (score desc, column asc: the order of
 * ocf_score_topk). exclude_inputs != 0 removes the row's input columns from the candidates and from the
 * relevant set; min_value: targets with a stored value below it are not relevant (-INFINITY = all).
 * out_col[e], out_rank[e] for e < ocf_batch_info()[1] entries (rank 0 = not a relevant target),
 * out_row_ptr[rows + 1] = the rows' entry ranges, out_n_cand[rows]. Synchronises `stream`. */
int ocf_rank_targets(ocf_model* model, ocf_batch* batch, int exclude_inputs, float min_value,
                     int32_t* out_col, int32_t* out_rank, int32_t* out_row_ptr, int64_t* out_n_cand,
                     void* stream);
/* The dense contraction kernel of the training step (tcgen05 kind::tf32 with fp32 operands split hi/lo, TMEM
 * accumulators, split-K over a thread-block cluster reduced through distributed shared memory;
 * csrc/ocf_gemm_tc.cuh: hidden layers of model.py:64-71 forward / backward / weight gradient), on host arrays:
 *   out[n, m] = sum_k A(m, k) * B(n, k)        out is [n_len, m_len] row-major
 * a_mn != 0: A is stored [k_len, m_len] (m contiguous), else [m_len, k_len]; b_mn likewise for B with n_len.
 * m_len, n_len, k_len multiples of 4. terms: 3 = fp32-grade (hi*hi + hi*lo + lo*hi), 1 = plain tf32.
 * split: 0 = the library's choice, else the cluster size along the contraction (1, 2, 4 or 8). */
int ocf_gemm_tc(const float* a, int a_mn, const float* b, int b_mn, int32_t m_len, int32_t n_len, int32_t k_len,
                int terms, int split, float* out);
/* Diagnostic twin (scripts/gemm_tc_bench.py): `reps` back-to-back launches of the kernel on zeroed device operands with
 * epilogue `kind` (1 = backward, 2 = gradient + Adagrad update, 3 = store); CUDA-event milliseconds per launch and
 * eight %globaltimer stamps (ns from kernel entry) of one CTA: entry, set-up done, first operands landed, products
 * done, tile parked + cluster barrier, epilogue done, second cluster barrier, exit. */
int ocf_gemm_tc_profile(int a_mn, int b_mn, int32_t m_len, int32_t n_len, int32_t k_len, int split, int kind, int reps,
                        float* ms_per_launch, int64_t stamps_ns[8]);
/* Copies `count` metric records starting at step slot `first` of the device log to the host
 * (synchronises `stream`). The log keeps the last 4096 steps. */
int ocf_model_read_metrics(ocf_model* model, int64_t first, int32_t count, float* host,
                           void* stream);
/* Waits for one step (one of the last 64) to finish and copies its metric record; later steps
 * already enqueued keep running. Every step's record is copied to pinned host memory right
 * behind its kernels, so this is the per-step device->host read of a pipelined caller. */
int ocf_model_wait_metrics(ocf_model* model, int64_t step, float* host);
/* Number of steps logged so far (train + eval). */
int64_t ocf_model_steps_logged(const ocf_model* model);

/* ---- multi-GPU: one process per GPU, NCCL over NVLink / NVSwitch -------------------------------
 * (absent in the reference, train.py:125-129 runs one session on one GPU; SURVEY.md section 8e)
 * Rank 0 draws a 128-byte id and ships it to the other ranks by any means (torch.distributed,
 * MPI, a file); every rank then creates its communicator on its own device. libnccl.so.2 is
 * loaded at run time, so single-GPU use does not need it. */
int ocf_comm_unique_id(uint8_t id[128]);
int ocf_comm_create(const uint8_t id[128], int32_t rank, int32_t world, ocf_comm** out);
int ocf_comm_destroy(ocf_comm* comm);
/* info[0] = rank, [1] = world, [2] = 0 (reserved). The two activation exchanges of a column-sharded step are
 * ncclAllReduce calls captured in the step's CUDA graph. */
int ocf_comm_info(const ocf_comm* comm, int32_t info[3]);
typedef enum {
  OCF_PAR_COLUMNS = 1,   /* item-dimension sharding: the model holds columns [lo, hi) (created with sharded = 1);
                            a phase-0 step runs phases 1..3 with the two activation all-reduces inside */
  OCF_PAR_ROWS = 2       /* data parallel: replicated weights, every rank steps on its own rows of the global batch
                            (ocf_step_args.row0 / rows_total); gradients are summed with one all-reduce and applied by
                            a streaming optimizer pass; the metrics cover the global batch. comm may be NULL (world 1) */
} ocf_parallel;
int ocf_model_set_comm(ocf_model* model, ocf_comm* comm, int mode);

/* OCF_BUF_STATS_DH: the row statistics [max_rows, 4] immediately followed by dL/dh [max_rows, hp];
 * a shard all-reduces its prefix of 4*max_rows + rows*hp floats with one collective. */
typedef enum { OCF_BUF_Z = 0, OCF_BUF_DH = 1, OCF_BUF_ROWSTATS = 2, OCF_BUF_STATS_DH = 3 } ocf_buffer;
/* Device pointer + float count of a buffer a sharded step exchanges between phases. */
int ocf_model_buffer(ocf_model* model, int which, void** device_ptr, int64_t* count);
/* Device pointer of a weight (kernel or bias, Keras index) in the library's internal layout,
 * for collectives over replicated parameters; count in floats. */
int ocf_model_weight_device(ocf_model* model, int index, void** device_ptr, int64_t* count);
/* ---- on-disk formats (host only; no CUDA device needed) --------------------------------------
 * Ingest of the JSON files the reference's reader loads with json.load (data_reader.py:85-92) into
 * CSR arrays, without a Python object per rating.
 *
 * ocf_vocab: `unique_items_list.json` / `unique_users_list.json` (data_reader.py:20-28) - a JSON list of
 * ids (numbers or strings); position in the list = dense column. Ids compare like Python dict keys:
 * 153 and 153.0 are the same id, "153" is another; a repeated id keeps its LAST position. */
typedef struct ocf_vocab ocf_vocab;
int ocf_vocab_load_json(const char* path, ocf_vocab** out);
int ocf_vocab_size(const ocf_vocab* vocab, int64_t* n);
int ocf_vocab_destroy(ocf_vocab* vocab);
/* ocf_ratings: one rating-dict file.
 *   paired = 0: {"row key": [[id, rating], ...], ...} - `ratingsBy*_dict.json` (data_reader.py:55) and
 *               `ratingsBy*_dicts_train.json` (:67-68). Rows = keys in file order (json.load's dict order).
 *   paired = 1: [input dict, target dict] - `ratingsBy*_dicts_{valid,test}.json` (:69-70). Rows = keys of
 *               the TARGET dict in file order (:74-80); the input row of a key is the input dict's entry for
 *               it, `null` = the reference's None (a zero input row, :234,253-254).
 * Column ids are mapped through `cols` (data_reader.py:135; an unknown id fails with the KeyError the
 * reference would raise). Ratings inside a row keep file order; a repeated row key keeps its first
 * place and its last value, like a Python dict. Values are stored as float32.
 * info = {rows, total bytes of the row keys (UTF-8), ratings of store 0, ratings of store 1}. */
typedef struct ocf_ratings ocf_ratings;
int ocf_ratings_load_json(const char* path, const ocf_vocab* cols, int paired, ocf_ratings** out);
int ocf_ratings_info(const ocf_ratings* ratings, int64_t info[4]);
/* Row keys, concatenated UTF-8 (bytes[info[1]]) + offsets[rows + 1]. */
int ocf_ratings_keys(const ocf_ratings* ratings, char* bytes, int64_t* offsets);
/* Copies store `which` (0 = the only / the input store, 1 = the target store of a paired file) into
 * caller-owned arrays: rowptr[rows + 1], col[nnz], val[nnz], none[rows] (1 = the file held null; may be
 * NULL). The arrays are what ocf_store_create takes. */
int ocf_ratings_csr(const ocf_ratings* ratings, int which, int64_t* rowptr, int32_t* col, float* val, uint8_t* none);
int ocf_ratings_destroy(ocf_ratings* ratings);

/* The offline splitter (TrainValidTestSplit.py:31-219), native: ratings CSV -> per-rating train/valid/test
 * split -> per-row dicts with paired inputs, written as the same files with the same bytes the reference's
 * script writes (json.dump / DataFrame.to_csv formatting included).
 *   ocf_csv_load    pandas.read_csv of the ratings file (:34): header line dropped, n_columns = 4
 *                   (user, item, rating, timestamp) or 3 (the "netflix" schema, :64-69); per column int64 /
 *                   float64 / string as pandas infers them.
 *   ocf_split_write `order` = the caller's np.random.permutation(rows) (:74) - the NumPy stream stays the
 *                   caller's; fractions = trainvalidtest_split; out_dir = output_filepath (with the trailing
 *                   separator, the reverse_item-user/ part included, :27-29). Writes train_data_mml*.csv /
 *                   test_data_mml*.csv (:91-96), ratingsByUser_dicts[_withtimestamps]_{train,valid,test}.json
 *                   (:98-103,151-181) when build_data_for_omni, unique_{items,users}_list.json (:105-118) when
 *                   save_users_and_items. cast_user_to_int = the "movielens" schema's str(int(userId)) keys;
 *                   reverse_user_item_data swaps the first two columns' roles (:40-43). */
typedef struct ocf_csv ocf_csv;
int ocf_csv_load(const char* path, int n_columns, ocf_csv** out);
int ocf_csv_rows(const ocf_csv* csv, int64_t* n);
int ocf_csv_destroy(ocf_csv* csv);
int ocf_split_write(const ocf_csv* csv, const int64_t* order, int64_t n_order, const double fractions[3],
                    const char* out_dir, int cast_user_to_int, int build_data_for_omni, int include_timestamps,
                    int save_users_and_items, int reverse_user_item_data);

/* The same split without the files: CSV -> the row stores the reader would build from the splitter's output
 * (ocf_split_write followed by ocf_ratings_load_json, minus two passes over the JSON text). `csv` must outlive the
 * handle. Columns = the distinct items in first-appearance order of the file (the order of unique_items_list.json).
 *   info[0] = columns; for set s in {0 train, 1 valid, 2 test}: info[1+4s] = rows (the set's row keys in dict order),
 *   info[2+4s] = bytes of its keys, info[3+4s] = ratings of part 0, info[4+4s] = ratings of part 1.
 *   part 0 = the set's input rows (train: its own ratings; valid: the train rows of the same users; test: their
 *   train+valid rows; none[k] = 1 where the reference stores None), part 1 = the set's target rows (valid / test). */
typedef struct ocf_split ocf_split;
int ocf_split_build(const ocf_csv* csv, const int64_t* order, int64_t n_order, const double fractions[3],
                    int cast_user_to_int, int reverse_user_item_data, ocf_split** out);
int ocf_split_info(const ocf_split* split, int64_t info[13]);
int ocf_split_keys(const ocf_split* split, int set, char* bytes, int64_t* offsets);
int ocf_split_csr(const ocf_split* split, int set, int part, int64_t* rowptr, int32_t* col, float* val, uint8_t* none);
/* The column ids as the text of unique_items_list.json: *needed = its length; copied into buf when cap suffices. */
int ocf_split_columns_json(const ocf_split* split, char* buf, int64_t cap, int64_t* needed);
int ocf_split_destroy(ocf_split* split);

/* Per-kernel timing with CUDA events recorded on the launching stream around the named kernels
 * (tag 0 = K1 gather, 1 = K2 encoder, 2 = K3 decoder/loss, 3 = K4a column scan, 4 = scoring GEMM,
 * 5 = K4b row update, 6 = first collective of a parallel step (z all-reduce / streaming optimizer
 * pass), 7 = second collective (row statistics + dL/dh all-reduce / gradient all-reduce), 9 = ranking
 * evaluation kernels of ocf_rank_targets). Off by default; ocf_profile_read synchronises the device and sums the elapsed times
 * of the launches recorded since the last reset. */
int ocf_profile_enable(int on);
int ocf_profile_reset(void);
int ocf_profile_read(int tag, double* total_ms, int64_t* count);
/* Number of kernels of this library launched by the calling process so far. */
int64_t ocf_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* OCF_H */
