/*
 * g4r.h -- C ABI of libg4r.so: the B200 (sm_100a) GRU4Rec session-parallel training step.
 *
 * This is the drop-in boundary for the hot path of hidasib/GRU4Rec.  In the reference the boundary is
 * the set of compiled Theano functions that gru4rec.py / evaluation.py call once per mini-batch; each
 * entry point below names the reference interface (file:line under /root/reference) it replaces.
 * Plain pointers and sizes only; no torch / Python types.  All functions return 0 on success or a
 * negative g4r_status; g4r_last_error() gives the message.  A handle is not thread-safe; one handle per
 * process per device (reference: single Python thread, single CUDA context, .theanorc_gru4rec:3).
 *
 * Unless a parameter is documented as a device pointer, buffers are HOST memory; the library does the
 * host<->device copies on its own stream (these copies are what bench.py's "e2e" number includes).
 */
#ifndef G4R_H
#define G4R_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define G4R_MAX_LAYERS 8

typedef enum {
  G4R_OK = 0,
  G4R_ERR_INVALID = -1,        /* bad argument / unsupported configuration (reference: NotImplementedError) */
  G4R_ERR_INDEX = -2,          /* index out of bounds (reference: IndexError, custom_theano_ops.py:586-591) */
  G4R_ERR_CUDA = -3,           /* CUDA runtime failure (reference: RuntimeError "gpuarray error") */
  G4R_ERR_NAN = -4,            /* NaN cost detected (reference: gru4rec.py:626-629) */
  G4R_ERR_STATE = -5
} g4r_status;

typedef enum { G4R_LOSS_XE = 0, G4R_LOSS_BPR_MAX = 1, G4R_LOSS_TOP1_MAX = 2, G4R_LOSS_BPR = 3, G4R_LOSS_TOP1 = 4,
               G4R_LOSS_XE_LOGIT = 5 } g4r_loss;                       /* gru4rec.py:136-143 */
typedef enum { G4R_ACT_LINEAR = 0, G4R_ACT_RELU = 1, G4R_ACT_TANH = 2, G4R_ACT_LEAKY = 3, G4R_ACT_ELU = 4,
               G4R_ACT_SELU = 5, G4R_ACT_SOFTMAX = 6, G4R_ACT_SOFTMAX_LOGIT = 7 } g4r_act;   /* gru4rec.py:144-161 */
typedef enum { G4R_ADAPT_NONE = 0, G4R_ADAPT_ADAGRAD = 1, G4R_ADAPT_RMSPROP = 2, G4R_ADAPT_ADADELTA = 3, G4R_ADAPT_ADAM = 4 } g4r_adapt;  /* gru4rec.py:300-381,392-399 */

/* Mirrors the GRU4Rec constructor arguments that shape the compiled step (gru4rec.py:97-135). */
typedef struct g4r_config {
  int32_t n_items;
  int32_t n_layers;
  int32_t layers[G4R_MAX_LAYERS];
  int32_t batch_size;
  int32_t embedding;              /* 0: none; >0: separate item embedding E of this width (gru4rec.py:449-456) */
  int32_t constrained_embedding;  /* 1: Wy doubles as the input embedding (gru4rec.py:438-448) */
  int32_t loss;                   /* g4r_loss */
  int32_t final_act;              /* g4r_act */
  float final_act_p1, final_act_p2;
  int32_t hidden_act;             /* g4r_act (elementwise ones) */
  float hidden_act_p1, hidden_act_p2;
  float dropout_p_hidden, dropout_p_embed;
  float learning_rate, momentum, lmbd;
  int32_t n_sample;
  float sample_alpha;
  float smoothing, bpreg, logq;
  int32_t adapt;                  /* g4r_adapt */
  int32_t sample_store;           /* capacity of the negative-sample store in ids (gru4rec.py:515,547); 0 = none */
  uint32_t dropout_seed;
  uint32_t mrg_seed;              /* MRG_RandomStreams seed (Theano default 12345) */
  int32_t max_resident_steps;     /* capacity (in mini-batches) of the device-resident schedule window; 0 = default */
  int32_t device;                 /* CUDA device ordinal */
  int32_t world_size, rank;       /* data-parallel geometry (1,0 for single GPU) */
  int32_t eval_batch_size;        /* lanes reserved for the scoring path (evaluation.py batch_size); 0 = batch_size */
  int32_t step_mode;              /* 0: one kernel per phase (CUDA-graph replay); 1: persistent cooperative kernel;
                                     2: role-specialised persistent kernel where the shape allows, else 1;
                                     3: as 2, launched as thread-block clusters: the GRU phases run on one cluster with the
                                        dense weights and optimizer state resident in shared memory (else 1);
                                     4: tensor-core step (tcgen05 GEMMs) whenever the model allows it -- modes 1-3 pick it
                                        automatically for constrained-embedding models with a layer of >= 160 units */
  int32_t mg_replicated;          /* 1: multi-GPU with replicated tables + NCCL exchange instead of row sharding */
  int32_t eval_tc;                /* scoring path: 0 auto, 1 fp32 FFMA tiles only, 2 tcgen05 (3xTF32) tiles whenever the ranking is full-catalogue */
  float adapt_p1, adapt_p1c;      /* adapt_params[0] and 1 - adapt_params[0] (rmsprop / adadelta decay; adam beta1), gru4rec.py:301-304,342-343,368-369 */
  float adapt_p2, adapt_p2c;      /* adapt_params[1] and 1 - adapt_params[1] (adam beta2) */
  float grad_cap;                 /* > 0: gradients are scaled to this global L2 norm when they exceed it (gru4rec.py:386-389) */
} g4r_config;

typedef struct g4r_handle g4r_handle;
typedef struct g4r_schedule g4r_schedule;

/* ---- lifecycle ------------------------------------------------------------------------------------ */
int g4r_version(void);
/* Bytes of device memory the handle needs; the caller may allocate them (e.g. a torch uint8 tensor used
 * purely as an allocator) and pass the DEVICE pointer to g4r_create, or pass NULL to let the library
 * cudaMalloc.  Replaces: theano.shared(...) allocations in GRU4Rec.init (gru4rec.py:267-294,331,401,425,556-558). */
int g4r_workspace_bytes(const g4r_config* cfg, size_t* bytes);
int g4r_create(const g4r_config* cfg, void* device_workspace, size_t workspace_bytes, g4r_handle** out);
int g4r_destroy(g4r_handle* h);
const char* g4r_last_error(const g4r_handle* h);   /* h may be NULL: last creation error */
/* cudaStream_t the step kernels are launched on (for CUDA-event timing by the caller). */
void* g4r_stream(g4r_handle* h);

/* ---- parameters: shared-variable get_value/set_value (gru4rec.py:745-767, 590, 649-651) ----------- */
/* names: "Wx0".."Wx7","Wh*","Wrz*","Bh*","H*","Wy","By","E", and optimizer state "<name>.acc", "<name>.vel". */
int g4r_tensor_shape(g4r_handle* h, const char* name, int64_t* rows, int64_t* cols);
int g4r_set_tensor(g4r_handle* h, const char* name, const float* host, int64_t rows, int64_t cols);
int g4r_get_tensor(g4r_handle* h, const char* name, float* host, int64_t rows, int64_t cols);
int g4r_reset_hidden(g4r_handle* h);               /* gru4rec.py:589-590 */

/* ---- negative sampling (gru4rec.py:539-566) ------------------------------------------------------- */
int g4r_set_sampling_cdf(g4r_handle* h, const float* P, int64_t n);     /* P (gru4rec.py:556) */
int g4r_set_logq_support(g4r_handle* h, const float* P0, int64_t n);    /* P0 (gru4rec.py:541) */
/* generate_samples(): MRG31k3p uniforms + binary search into P; resets the sample pointer (gru4rec.py:559-564). */
int g4r_generate_samples(g4r_handle* h);
/* Same search on caller-supplied uniforms (parity at the K2 boundary; custom_theano_ops.py:318-349). */
int g4r_generate_samples_from_uniform(g4r_handle* h, const float* u, int64_t n);
int g4r_set_sample_store(g4r_handle* h, const int64_t* st, int64_t rows);   /* rows x n_sample */
int g4r_get_sample_store(g4r_handle* h, int64_t* st, int64_t rows);
int g4r_sample_store_rows(g4r_handle* h);                                    /* generate_length (gru4rec.py:547) */
int g4r_set_sample_pointer(g4r_handle* h, int64_t p);                        /* STI (gru4rec.py:558,583) */
int64_t g4r_get_sample_pointer(g4r_handle* h);
/* Raw MRG uniforms (theano.sandbox.rng_mrg restatement) for tests. */
int g4r_mrg_uniform(g4r_handle* h, float* out, int64_t n);

/* ---- stand-alone custom ops (custom_theano_ops.py) ------------------------------------------------ */
/* GpuBinarySearchSorted (custom_theano_ops.py:275-407): y[i] = index of x[i] in sorted d. */
int g4r_searchsorted(g4r_handle* h, const float* d, int64_t n_d, const float* x, int64_t n_x, int64_t* y);
/* GpuAdvancedSubtensor1_fast (custom_theano_ops.py:409-595): out[i,:] = table[idx[i],:], negative wrap,
 * out-of-range -> G4R_ERR_INDEX. */
int g4r_gather_rows(g4r_handle* h, const float* table, int64_t rows, int64_t cols, const int64_t* idx, int64_t n_idx, float* out);

/* ---- session-parallel schedule (gru4rec.py:585-651; evaluation.py:90-139) -------------------------- */
/* Builds every mini-batch of one epoch on the host: X/Y item indices, reset flags, batch sizes, lane slots.
 * mode 0 = training order semantics (reset-after flags), 1 = evaluation (zero-before flags).
 * session_order: n_sessions session ids (gru4rec.py:585/593; a rank's shard in the multi-GPU path) or NULL for identity;
 * offset_sessions must cover every id that occurs in it. */
int g4r_schedule_build(const int64_t* data_items, int64_t n_events, const int32_t* offset_sessions, int64_t n_sessions,
                       const int64_t* session_order, int32_t batch_size, int32_t n_sample, int32_t mode, g4r_schedule** out);
int g4r_schedule_free(g4r_schedule* s);
int64_t g4r_schedule_steps(const g4r_schedule* s);
int64_t g4r_schedule_events(const g4r_schedule* s);       /* sum of batch sizes */
/* Copies out step arrays (each step padded to batch_size entries; unused lanes = -1 / 0). Any pointer may be NULL. */
int g4r_schedule_export(const g4r_schedule* s, int32_t* X, int32_t* Y, uint8_t* flags, int32_t* M, int32_t* slots);

/* ---- the compiled step: train_function(X, Y, M, R) -> cost (gru4rec.py:584,623) ------------------- */
/* One mini-batch from host arrays; returns the cost (D2H) like the reference call. */
int g4r_train_step(g4r_handle* h, const int32_t* X, const int32_t* Y, int32_t M, const int8_t* R, float* cost);
/* Steps [first, first+n) of a schedule: uploads the window, runs every step on the device without host
 * round trips, regenerates the sample store when the pointer wraps (gru4rec.py:618-621), copies the n
 * costs back.  NaN cost -> G4R_ERR_NAN with *nan_step set (gru4rec.py:626-629). */
int g4r_train_steps(g4r_handle* h, const g4r_schedule* s, int64_t first, int64_t n, float* cost_out, int64_t* nan_step);
/* Two-phase variant used for device-resident timing: upload (H2D + per-step column plans) then run. */
int g4r_upload_steps(g4r_handle* h, const g4r_schedule* s, int64_t first, int64_t n);
int g4r_run_uploaded(g4r_handle* h, float* cost_out /* may be NULL */, float* device_ms /* may be NULL */);
/* Re-runs the uploaded window with CUDA events around every kernel launch; sums device time and launch counts
 * per phase (index i is named by g4r_phase_name(i); n_phases must be >= g4r_phase_count()).  For bench.py's
 * roofline: achieved bytes/s of the dominant kernel = its algorithmic bytes / its mean duration. */
int g4r_profile_uploaded(g4r_handle* h, float* phase_ms, int32_t* phase_launches, int32_t n_phases);
const char* g4r_phase_name(int32_t i);
/* step_mode 2: number of windows run by the role-specialised kernel, and (out) windows that fell back to the
 * generic persistent kernel because a chunk of score columns was wider than 16. */
int64_t g4r_fast_windows(const g4r_handle* h, int64_t* fallback_windows);
/* 1 if the handle trains with the tensor-core step (tcgen05 3xTF32 GEMMs with fused epilogues, csrc/g4r_tcstep.cuh): constrained
 * embedding, one layer, batch <= 256, SGD / Adagrad (+momentum); automatic for layers >= 160 units, forced with step_mode 4. */
int g4r_uses_tensor_cores(const g4r_handle* h);
/* Persistent mode (step_mode 1): enable %globaltimer stamps at the phase boundaries of every step and/or read
 * the stamps of the last window (16 uint64 slots per step; slots 0..5 used: start, after GRU forward, after scores,
 * after statistics, after loss-gradient/update, end). */
int g4r_persistent_stamps(g4r_handle* h, int32_t enable, unsigned long long* out, int64_t n_steps);
int g4r_phase_count(void);
/* Counters for bench.py: kernels launched by this handle so far. */
int64_t g4r_kernel_launches(const g4r_handle* h);

/* ---- multi-GPU (one process per GPU; SURVEY section 8e) -------------------------------------------------------
 * Handles created with world_size > 1 compute gradients only; g4r_train_steps then exchanges them over NCCL
 * (all-gather of row gradients, all-reduce of dense gradients) and applies the merged update on every rank.
 * Rank 0 obtains a 128-byte NCCL unique id, the caller broadcasts it (e.g. torch.distributed), every rank calls
 * g4r_mg_init.  All ranks must call g4r_train_steps with the same number of steps. */
int g4r_mg_unique_id(char* out128);
int g4r_mg_init(g4r_handle* h, const char* id128);
/* Row-sharded layout (the default for world_size > 1 when the role-specialised kernel covers the shape: no-embedding mode, one
 * layer of <= 120 units, batch <= 32; cfg.mg_replicated = 1 forces the replicated NCCL path above).  Row i of Wy / By / Wx0 and
 * of their optimizer state lives only on rank i % world_size (local row i / world_size) in a library-owned segment that the
 * peers map with cudaIpc; parameter rows are fetched from their owners and gradient rows are stored into the owners' inboxes
 * over NVLink INSIDE the persistent kernel, the owners apply the merged update to their 1/world_size of the rows, and the
 * dense GRU gradients are pushed to all peers and summed in rank order.  NCCL only carries the per-window all-gather of the
 * sorted column lists.  Call order: g4r_create -> g4r_mg_init -> g4r_mg_ipc_handle (all-gather the 64-byte handles in rank
 * order) -> g4r_mg_ipc_open.  g4r_set_tensor / g4r_get_tensor keep the single-GPU shapes ("Wy" is n_items x L): set scatters
 * the caller's full matrix to this rank's rows, get assembles the full matrix from all shards (all ranks idle).
 * There is no reference counterpart (the reference is single-device, .theanorc_gru4rec:3); SURVEY section 8e is the spec. */
int g4r_mg_sharded(const g4r_handle* h);                               /* 1 if the handle uses the row-sharded layout */
int g4r_mg_ipc_handle(g4r_handle* h, char* out64);                    /* cudaIpcMemHandle_t of this rank's segment */
int g4r_mg_ipc_open(g4r_handle* h, const char* handles, int32_t world);   /* world x 64 bytes, rank order */
/* Ownership arithmetic and buffer sizing of the sharded layout (pure host functions, usable without a device). */
int g4r_mg_owner(int64_t item, int32_t world);
int64_t g4r_mg_local_row(int64_t item, int32_t world);
int64_t g4r_mg_shard_rows(int64_t n_items, int32_t world, int32_t rank);
int g4r_mg_segment_bytes(const g4r_config* cfg, size_t* total, size_t* inbox_bytes, size_t* inbox_in_bytes, size_t* dense_bytes);

/* ---- scoring path: evaluate(X, Y, M) (evaluation.py:76,108) and predict (gru4rec.py:706-710) ------- */
/* Runs a whole evaluation schedule: full-catalogue scores, rank of the target, per-cutoff hit counts and
 * reciprocal-rank sums.  mode: 0 standard, 1 conservative, 2 median, 3 tiebreaking (evaluation.py:55,60-65; the tie-breaking noise U(0,1) * 1e-10 is a
 * counter hash here, Theano's MRG stream in the reference).
 * recall_sum/mrr_sum: n_cut doubles each (sums, not yet divided by the number of events). */
int g4r_eval_schedule(g4r_handle* h, const g4r_schedule* s, const int32_t* cut_off, int32_t n_cut, int32_t mode,
                      double* recall_sum, double* mrr_sum, int64_t* n_events);
/* evaluate_gpu(items=...) (evaluation.py:15,52-56,84-100): rank the targets against the `n` candidate item indices instead of
 * the whole catalogue for subsequent g4r_eval_schedule calls (the target's own score competes only if the target is listed,
 * as in the reference); n = 0 restores the full-catalogue ranking.  G4R_ERR_INDEX on an out-of-range index. */
int g4r_set_eval_items(g4r_handle* h, const int64_t* items, int64_t n);

/* predict_next_batch's device call: scores of all items for `batch` lanes; reset_mask zeroes lanes first
 * (gru4rec.py:712-717).  out: [batch x n_items] row-major. */
int g4r_predict(g4r_handle* h, const int32_t* X, int32_t batch, const uint8_t* reset_mask, float* out);
/* Top-k of the scores g4r_predict would return for the same call, without materialising them.  Advances the scoring-path
 * hidden state exactly like g4r_predict (one event per lane; reset_mask as there).  cand/n_cand: optional candidate item
 * indices (NULL/0 = whole catalogue; duplicates -> G4R_ERR_INVALID).  Out: items_out / scores_out [batch x k], each row
 * sorted by score descending, ties by item index ascending; softmax-family scores normalised over the candidates.
 * k must be in 1 .. min(256, number of candidates).  Out-of-range X or candidate index -> G4R_ERR_INDEX. */
int g4r_predict_topk(g4r_handle* h, const int32_t* X, int32_t batch, const uint8_t* reset_mask,
                     const int64_t* cand, int64_t n_cand, int32_t k, int32_t* items_out, float* scores_out);
/* Zero the scoring-path hidden state (gru4rec.py:696-697). */
int g4r_reset_eval_hidden(g4r_handle* h);

#ifdef __cplusplus
}
#endif
#endif
