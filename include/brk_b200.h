/*
 * brk_b200.h -- C ABI of the B200-native recommender hot path (libbrk_b200.so).
 *
 * The reference (leotimus/binary-recommendation) is pure Python over TensorFlow/Keras/TFRS and
 * has no FFI layer of its own; the interface this library replaces is the set of framework ops
 * its model/trainer code calls (SURVEY.md section 2.2, K1-K10).  Each entry point below cites the
 * reference call site(s) whose framework op it stands in for (paths relative to /root/reference).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; the caller owns all
 *     buffers; the library allocates nothing except the opaque context's small workspace;
 *   - ids are int32, tables are row-major contiguous fp32 [rows, d];
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), no hidden syncs,
 *     safe to capture into a CUDA graph;
 *   - return 0 on success, <0 for a bad argument (BRK_E_*), >0 for a cudaError_t; the message is
 *     available from brk_last_error() (thread-local);
 *   - there is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef BRK_B200_H
#define BRK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BRK_ABI_VERSION 2

#define BRK_E_ARG   (-1)   /* null pointer, negative size, unsupported dimension */
#define BRK_E_ALIGN (-2)   /* pointer / row stride not aligned as required */
#define BRK_E_STATE (-3)   /* context unusable */

typedef struct brk_ctx brk_ctx;

/* One embedding table (or one flat dense parameter when rows == 1) with its gradient
 * accumulator and optimizer slots.  g is a dense fp32 accumulator of the same shape that the
 * fused forward/backward kernels add row gradients into and the optimizer kernels consume and
 * zero.  touched is a bitmask over rows ((rows+31)/32 words, zero between steps) recording which
 * rows received a gradient this step; required by the row-sparse optimizers, may be NULL when
 * only dense optimizers are used. m, v: Adam moments; for Adagrad m is the accumulator. */
typedef struct brk_table {
  float*    w;
  float*    g;
  float*    m;
  float*    v;
  uint32_t* touched;
  int64_t   rows;
  int32_t   d;
  int32_t   _pad;
} brk_table;

struct brk_dp_peer;   /* defined below: peer-memory descriptor of the data-parallel optimizer */

typedef struct brk_adam_hyper {
  float lr, beta1, beta2, eps;   /* Keras defaults: 1e-3, 0.9, 0.999, 1e-7 */
} brk_adam_hyper;

/* ---- context ---------------------------------------------------------------------------- */
int         brk_abi_version(void);
const char* brk_last_error(void);
int         brk_create(brk_ctx** out, int device);
int         brk_destroy(brk_ctx* ctx);
int         brk_sm_count(const brk_ctx* ctx);

/* ---- K1: embedding row gather -------------------------------------------------------------
 * Stands in for keras Embedding(...)(ids) -> tf ResourceGather:
 *   src/models/NeuMFModel.py:58-63, src/models/BPRModel.py:55-61, src/models/bpr.py:178-184,
 *   trainers/twoTower.py:34,36.   out[b,:] = table[ids[b],:], b < n.  ids must be in [0,rows). */
int brk_gather_rows(brk_ctx* ctx, const float* table, int64_t rows, int32_t d,
                    const int32_t* ids, int64_t n, float* out, void* stream);

/* ---- K5: sparse embedding-gradient scatter-add -------------------------------------------
 * Stands in for the IndexedSlices gradient of the gathers above and the optimizer's duplicate
 * summation (tf UnsortedSegmentSum; inside model.fit src/models/RModel.py:130 and
 * tape.gradient trainers/twoTower.py:97).  acc[ids[b],:] += vals[b,:].
 * mode 0: vector atomics (red.global.add.v4.f32), one RED per occurrence and 16-byte chunk.
 * mode 1: sort-and-segment-reduce -- each CTA sorts a tile of 1024 (id, position) pairs in shared memory and
 *   sends one RED per run of up to 16 equal ids (d % 4 == 0, d <= 128, else mode 0 is taken); for small hot
 *   tables where the same rows are hit over and over (pick it when n / rows, the mean duplicate factor, is large).
 * touched (may be NULL) gets bit ids[b] set. */
int brk_scatter_add_rows(brk_ctx* ctx, float* acc, int64_t rows, int32_t d,
                         const int32_t* ids, int64_t n, const float* vals,
                         uint32_t* touched, int32_t mode, void* stream);

/* ---- K10: counter-based negative sampling (Philox4x32-10) ---------------------------------
 * Replaces the host-RNG sampling of src/models/NeuMFModel.py:104-105 and the exhaustive
 * enumeration of src/models/BPRModel.py:111-119 / src/models/bpr.py:96-107.  The stream is
 * defined in oracle/philox.py ("brk sampler v2") and reproduced bit-for-bit.
 * BPR: for sample first_index+b with user users[b], one draw picks a rank among the items that are
 * not in the user's sorted positive list (csr_indptr int64 [U+1], csr_items int32); that item is
 * written to neg[b] (uniform over the non-interacted items, one binary search, no rejection loop). */
int brk_philox_bpr_negatives(brk_ctx* ctx, const int32_t* users, int64_t n, int64_t first_index,
                             uint32_t seed, uint32_t epoch, int32_t num_items,
                             const int64_t* csr_indptr, const int32_t* csr_items,
                             int32_t* neg, void* stream);
/* NeuMF: neg_user[b] = pos_users[(w0*P)>>32], neg_item[b] = pos_items[(w1*P)>>32]. */
int brk_philox_neumf_negatives(brk_ctx* ctx, const int32_t* pos_users, const int32_t* pos_items,
                               int64_t num_pos, int64_t n, int64_t first_index,
                               uint32_t seed, uint32_t epoch,
                               int32_t* neg_users, int32_t* neg_items, void* stream);
/* Raw generator (known-answer tests): out[i,0..3] = philox4x32_10(ctr[i,0..3], key). */
int brk_philox4x32_10(brk_ctx* ctx, const uint32_t* ctr, int64_t n, uint32_t key0, uint32_t key1,
                      uint32_t* out, void* stream);

/* ---- K1+K4+K5 fused: BPR triplet forward + backward ----------------------------------------
 * Stands in for the graph of src/models/BPRModel.py:49-74 with bprTripletLoss/identityLoss
 * (:124-144; twin src/models/bpr.py:136-192) and its gradient inside model.fit (BPRModel.py:109):
 *   x = <u,p> - <u,n>;  l = 1 - sigmoid(x);  loss = mean(l);
 *   user.g[u] += g(p-n), item.g[p] += g u, item.g[n] -= g u,  g = -s(1-s)/B.
 * loss_out[0] receives the batch mean.  Row gradients are accumulated into user->g / item->g
 * (which must be zero on entry -- the optimizer calls below re-zero them).
 * global_batch (0 = batch): data-parallel replicas pass the summed batch of all replicas so that
 * the SUM of their accumulators (one all-reduce) is the gradient of the global mean loss -- the
 * synchronous mirrored training of src/models/RModel.py:119-121. */
int brk_bpr_fwd_bwd(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                    const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch,
                    int64_t global_batch, float* loss_out, void* stream);
/* n_steps x (brk_bpr_fwd_bwd + Adam) enqueued by one call: the inner loop of model.fit
 * (src/models/BPRModel.py:109, src/models/bpr.py:220-223).  u/p/n are device arrays of `total`
 * triplets cut into batches of `batch`; batch_index_host[k] (HOST array) names the batch step k
 * consumes; losses (device, [n_steps], may be NULL) receives each step's mean loss.
 * lazy_adam 0: exact Keras Adam (dense pass); 1: row-sparse lazy Adam. */
int brk_bpr_train_steps(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                        const int32_t* u, const int32_t* p, const int32_t* n, int64_t total,
                        int64_t batch, const int64_t* batch_index_host, int32_t n_steps,
                        brk_adam_hyper h, int32_t lazy_adam, int64_t* step_dev, float* losses,
                        void* stream);
/* The same loop fed from HOST memory (what a caller holding NumPy / pandas columns does): every step's
 * user and positive ids go H2D with their own cudaMemcpyAsync (copy stream, ring of staging slots), the
 * steps run in cooperative launches of up to 16 steps each (the kernel draws its own Philox negatives
 * while the previous step's Adam phase runs), every step's loss comes back D2H.
 * u_host / p_host / losses_host should be page-locked (then nothing here blocks).
 * host_batch_stride: int32 elements between consecutive batches in u_host / p_host (0 = batch, i.e. two flat
 * arrays); with the batch-major layout [n_batches][2][batch] (p_host == u_host + batch, stride 2*batch;
 * the last block padded to full size) each step's ids move with ONE copy.
 * d_stage: device int32 scratch [brk_bpr_host_stage_ints(batch)]; d_losses: device [n_steps].
 * dp (may be NULL): mirrored data parallelism as in brk_bpr_train_steps_dp -- every rank feeds its own host
 * batches, all ranks call with the same n_steps, full batches only. */
int64_t brk_bpr_host_stage_ints(int64_t batch);
int brk_bpr_train_steps_host(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                             const int32_t* u_host, const int32_t* p_host, int64_t total, int64_t batch,
                             int64_t host_batch_stride, const int64_t* batch_index_host, int32_t n_steps, uint32_t seed, uint32_t epoch,
                             int32_t num_items, const int64_t* csr_indptr, const int32_t* csr_items,
                             brk_adam_hyper h, int32_t lazy_adam, int64_t* step_dev, int32_t* d_stage,
                             float* d_losses, float* losses_host, const struct brk_dp_peer* dp, void* stream);
/* Zero-copy variant: u_host / p_host / losses_host are MAPPED page-locked host memory; ONE cooperative
 * launch runs all n_steps, every step's kernel phase pulls that step's ids over PCIe (8*batch bytes),
 * draws the negatives, trains, and stores the loss straight into losses_host[k].  Exact Keras Adam
 * only (the cooperative path). */
int brk_bpr_train_steps_mapped(brk_ctx* ctx, const brk_table* user, const brk_table* item,
                               const int32_t* u_host, const int32_t* p_host, int64_t total, int64_t batch,
                               const int64_t* batch_index_host, int32_t n_steps, uint32_t seed, uint32_t epoch,
                               int32_t num_items, const int64_t* csr_indptr, const int32_t* csr_items,
                               brk_adam_hyper h, int64_t* step_dev, float* losses_host, void* stream);
/* Forward only: x_out[b] = <u,p> - <u,n> (scores for evaluation, bpr.py:122-133). */
int brk_bpr_scores(brk_ctx* ctx, const float* user_w, const float* item_w, int32_t d,
                   const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch,
                   float* x_out, void* stream);

/* ---- K6: optimizers -----------------------------------------------------------------------
 * step_dev: device optimizer state of three 8-byte words: [0] int64 t = completed steps,
 * [1] double beta1^t, [2] double beta2^t (initialise to 0, 1.0, 1.0).  The kernels use step t+1
 * and, when advance_step != 0, the last block advances the state (so a whole epoch can be
 * enqueued or captured in a CUDA graph without host involvement).
 * brk_adam_dense_keras: exact Keras Adam (src/models/NeuMFModel.py:89, BPRModel.py:70,
 *   bpr.py:201, trainers/NFC_plain.py:153): every element of every listed table moves,
 *   alpha_t = lr*sqrt(1-b2^t)/(1-b1^t), w -= alpha_t*m/(sqrt(v)+eps); g is zeroed, touched cleared.
 * brk_adam_rows: lazy variant touching only rows whose touched bit is set (clears the bits).
 * brk_adagrad_rows: Keras Adagrad sparse apply (trainers/twoTower.py:278-279; accumulator in
 *   tab.m, initial value 0.1 set by the caller): acc += g^2, w -= lr*g/(sqrt(acc)+eps).
 * brk_adagrad_dense: same on whole tables (dense kernels/biases). */
int brk_adam_dense_keras(brk_ctx* ctx, const brk_table* tabs, int32_t n_tabs, brk_adam_hyper h,
                         int64_t* step_dev, int32_t advance_step, void* stream);
int brk_adam_rows(brk_ctx* ctx, const brk_table* tabs, int32_t n_tabs, brk_adam_hyper h,
                  int64_t* step_dev, int32_t advance_step, void* stream);
int brk_adagrad_rows(brk_ctx* ctx, const brk_table* tabs, int32_t n_tabs, float lr, float eps,
                     void* stream);
int brk_adagrad_dense(brk_ctx* ctx, const brk_table* tabs, int32_t n_tabs, float lr, float eps,
                      void* stream);

/* ---- K1+K2+K3+K4+K5 fused: NeuMF forward + backward --------------------------------------------
 * Stands in for the Keras graph of src/models/NeuMFModel.py:53-100 (class spec) and
 * trainers/NFC_plain.py:109-155 (script spec) inside model.fit / predict / evaluate
 * (src/models/RModel.py:130-147):
 *   x0 = [uMLP[u], iMLP[i]] -> dropout -> act(W1) -> BN -> dropout -> act(W2) -> BN -> dropout -> act(W3) = h3
 *   out = sigmoid([h3, <uMF[u], iMF[i]>] W4 + b4);   loss = mean squared error (0) | binary cross-entropy (1)
 * dense is ONE flat parameter block (brk_table with rows = 1) laid out as
 *   W1[2E,H1] b1[H1] gamma1[H1] beta1[H1] W2[H1,H2] b2[H2] gamma2[H2] beta2[H2] W3[H2,H3] b3[H3] W4[H3+1] b4[1]
 * (Keras Dense kernels are [in, out] row-major; W4 rows are ordered [h3..., mf]); its length is
 * brk_neumf_dense_floats().  bn_moving holds moving mean1[H1], var1[H1], mean2[H2], var2[H2]
 * (Keras: momentum 0.99, eps 1e-3, biased batch variance).  act: 0 relu, 1 sigmoid.  dropout != 0
 * applies the Philox-defined masks of oracle/neumf.py (keep 205/256) in training.
 * Any widths are accepted (numFactor is a free attribute of the reference model, RModel.py:35).  Tiled fp32 instances
 * (E; H1,H2,H3): (32;32,16,8) (64;64,32,16) (16;16,8,4) (8;8,4,2) (10;100,50,10); every other width runs on the
 * any-width kernels of csrc/neumf_generic.cu (correct, not tuned).  (32;32,16,8) and (64;64,32,16) also exist as
 * tensor-core kernels (tensor_cores = 1: every Dense product of the forward and backward pass is a tcgen05.mma with
 * TF32 operands out of shared memory and fp32 accumulators in TMEM): one cooperative launch for the whole step when
 * the batch fits on chip (csrc/neumf_fused.cu), five kernels otherwise (csrc/neumf_tc.cu); results agree with the
 * TF32-operand oracle (oracle/tf32.py) to ~1e-5 on predictions.
 * Workspace: h1,dy1 [H1*batch], h2,dy2 [H2*batch] floats, acc brk_neumf_acc_doubles() doubles that
 * must be ZERO before the first call (every call leaves them zero again).
 * training != 0: accumulates all gradients into the tables' g (to be consumed by the optimizer
 * calls), updates bn_moving, writes out[batch] (predictions) and loss_out[0].
 * training == 0: inference with the moving statistics; y may be NULL (then no loss).
 * global_batch (0 = batch) scales the loss gradient for data-parallel replicas; BatchNorm statistics
 * stay per replica (MirroredStrategy's default). */
typedef struct brk_neumf_model {
  brk_table uMLP, iMLP, uMF, iMF, dense;
  float*  bn_moving;
  int32_t E, H1, H2, H3;
  int32_t act, loss, dropout;
  int32_t tensor_cores;   /* 0: fp32 on the CUDA cores; 1: MLP products on tcgen05 with TF32 operands, fp32 accumulation */
  /* ABI 2 -- the He et al. NeuMF variant BASELINE.json configs[0] names ("GMF + MLP, 8-dim"): all zero = the
   * reference class spec above.
   *   EMF           width of the two MF tables (0 = E);
   *   mf_mode       0: predMF = Dot(axes=1) scalar (NeuMFModel.py:79); 1: the Hadamard vector uMF[u]*iMF[i] [EMF] is
   *                 concatenated to h3, so W4 has H3 + EMF rows (GMF of He et al.);
   *   no_batch_norm 1: the two BatchNormalization layers are absent (gamma/beta slots stay in the block, unused). */
  int32_t EMF, mf_mode, no_batch_norm, _pad;
} brk_neumf_model;
typedef struct brk_neumf_workspace {
  float *h1, *h2, *dy1, *dy2;
  double* acc;
} brk_neumf_workspace;
int64_t brk_neumf_dense_floats(int32_t E, int32_t H1, int32_t H2, int32_t H3);
/* length of the dense block when the head takes head_mf MF inputs (1 for the scalar Dot, EMF for the Hadamard vector) */
int64_t brk_neumf_dense_floats_ex(int32_t E, int32_t H1, int32_t H2, int32_t H3, int32_t head_mf);
int64_t brk_neumf_acc_doubles(int32_t H1, int32_t H2);
int brk_neumf_step(brk_ctx* ctx, const brk_neumf_model* m, const int32_t* u, const int32_t* i,
                   const float* y, int64_t batch, int64_t global_batch, int64_t first_index, int32_t training,
                   uint32_t dropout_seed, uint32_t dropout_epoch, const brk_neumf_workspace* ws,
                   float* out, float* loss_out, void* stream);
/* brk_neumf_train_step: one training step of model.fit (src/models/RModel.py:130-137) = brk_neumf_step (training) on the
 * batch u / i / y [batch] + the optimizer: lazy_adam == 0 exact Keras Adam over the four tables and the dense block,
 * != 0 dense block + touched rows only.  When the model is one the one-launch tensor-core kernel covers
 * (csrc/neumf_fused.cu: tensor_cores = 1 with numFactor 32 or 64, or the He et al. variant), Adam is the stock Keras
 * one and the batch fits on chip (148 x 128 samples, twice that at numFactor 32), the WHOLE step -- gather, forward,
 * loss, backward, gradient scatter, Adam over every parameter -- is ONE cooperative kernel launch. */
int brk_neumf_train_step(brk_ctx* ctx, const brk_neumf_model* m, const int32_t* u, const int32_t* i,
                         const float* y, int64_t batch, int64_t first_index, uint32_t dropout_seed,
                         uint32_t dropout_epoch, brk_adam_hyper h, int64_t* adam_state, int32_t lazy_adam,
                         const brk_neumf_workspace* ws, float* out, float* loss_out, void* stream);
/* brk_neumf_train_steps: the inner loop of model.fit (src/models/RModel.py:130-137) over batches of a resident
 * training frame u / i / y [n_rows] (what bootstrapDataset builds, NeuMFModel.py:102-123): for s < n_steps, batch
 * b = batch_index_host[s] = rows [b * batch, min(n_rows, (b + 1) * batch)) goes through brk_neumf_step (training,
 * first_index = b * batch: the dropout stream is a function of the row's position in the frame) and then the
 * optimizer: lazy_adam == 0 exact Keras Adam over the four tables and the dense block (brk_adam_dense_keras),
 * != 0 dense block + touched rows only (brk_adam_rows).  losses [n_steps] (device, may be NULL) receives the step
 * losses, out [batch] the predictions of the last step.  One brk_neumf_train_step per listed batch; enqueues and returns, no sync. */
int brk_neumf_train_steps(brk_ctx* ctx, const brk_neumf_model* m, const int32_t* u, const int32_t* i,
                          const float* y, int64_t n_rows, int64_t batch, const int64_t* batch_index_host,
                          int32_t n_steps, uint32_t dropout_seed, uint32_t dropout_epoch, brk_adam_hyper h,
                          int64_t* adam_state, int32_t lazy_adam, const brk_neumf_workspace* ws, float* out,
                          float* losses, void* stream);

/* Host-fed variant of brk_neumf_train_steps (the tf.data iterator -> device boundary of model.fit, RModel.py:130): the
 * frame stays in page-locked HOST memory, batch-major packed_host [n_batches][3][batch] int32 words (user ids, item
 * ids, labels as float bits).  Per step one cudaMemcpyAsync of the batch (12 * batch bytes) on the context's copy
 * stream into one of four staging slots (d_stage: brk_neumf_host_stage_ints(batch) int32), then brk_neumf_train_step;
 * copies run ahead of the compute.  d_losses [n_steps] device; losses_host [n_steps] pinned (may be NULL), filled by
 * one D2H copy, valid after the stream is synchronised.  Full batches only. */
int64_t brk_neumf_host_stage_ints(int64_t batch);
int brk_neumf_train_steps_host(brk_ctx* ctx, const brk_neumf_model* m, const int32_t* packed_host, int64_t n_batches,
                               int64_t batch, const int64_t* batch_index_host, int32_t n_steps, uint32_t dropout_seed,
                               uint32_t dropout_epoch, brk_adam_hyper h, int64_t* adam_state, int32_t lazy_adam,
                               const brk_neumf_workspace* ws, int32_t* d_stage, float* out, float* d_losses,
                               float* losses_host, void* stream);

/* Test hook for the tcgen05 building blocks of the NeuMF tensor-core path (csrc/neumf_tc.cu): stages A
 * [a_rows, a_cols] and B [b_rows, b_cols] (row-major fp32; cols multiples of 32, rows multiples of 8) as
 * 128-byte-swizzled tiles and computes D = A B^T (mode bit0/bit1 = 0: K-major operand, rows = M / N) or
 * with the operand read transposed (bit set: rows = K); out [128, N] receives TMEM lanes 0..127. */
int brk_tc_selftest(brk_ctx* ctx, int32_t M, int32_t N, int32_t K, int32_t mode, const float* A, int32_t a_rows,
                    int32_t a_cols, const float* B, int32_t b_rows, int32_t b_cols, float* out, void* stream);

/* ---- row-sharded tables over NVLink peer memory ----------------------------------------------------
 * Stands in for the embedding lookups and their IndexedSlices gradients (NeuMFModel.py:58-63) when the
 * tables are too large to mirror on every worker as MultiWorkerMirroredStrategy does (RModel.py:119-121):
 * row r of a table lives on rank r % world at local row r / world.  w / g / touched hold every rank's
 * shard pointer (this rank's own and the NVLink peer mappings of the others).  The fused kernels read
 * peer rows with ordinary loads and send row gradients as REDs into the owner's accumulator (touched
 * bits likewise), i.e. the all-to-all of looked-up rows and of their gradients is carried by the gather
 * and scatter instructions themselves.  brk_neumf_step_sharded: as brk_neumf_step; m's tables describe
 * THIS rank's shards.  After it, every rank must pass brk_peer_barrier before an owner applies its
 * optimizer to its shard, and again (or through brk_dp_adam_peer's own barriers) before the next step
 * reads the updated rows. */
#define BRK_MAX_PEERS 8
typedef struct brk_shards {
  float*    w[BRK_MAX_PEERS];
  float*    g[BRK_MAX_PEERS];
  uint32_t* touched[BRK_MAX_PEERS];
  int32_t   world, rank;
} brk_shards;
typedef struct brk_neumf_shards { brk_shards uMLP, iMLP, uMF, iMF; } brk_neumf_shards;
int brk_neumf_step_sharded(brk_ctx* ctx, const brk_neumf_model* m, const brk_neumf_shards* sh,
                           const int32_t* u, const int32_t* i, const float* y, int64_t batch,
                           int64_t global_batch, int64_t first_index, int32_t training, uint32_t dropout_seed,
                           uint32_t dropout_epoch, const brk_neumf_workspace* ws, float* out, float* loss_out,
                           void* stream);
/* The all-to-all of looked-up rows and of row gradients as stand-alone ops (SURVEY.md section 8b "a2a_rows"): gather
 * out[b,:] = row ids[b] of the sharded table (peer loads), scatter-add values[b,:] into the OWNER's accumulator
 * (16-byte REDs over NVLink, owner's touched bit set).  d % 4 == 0.  The same barriers as after brk_neumf_step_sharded
 * apply before an owner consumes its accumulator. */
int brk_gather_rows_sharded(brk_ctx* ctx, const brk_shards* sh, int32_t d, const int32_t* ids, int64_t n, float* out,
                            void* stream);
int brk_scatter_add_rows_sharded(brk_ctx* ctx, const brk_shards* sh, int32_t d, const int32_t* ids, int64_t n,
                                 const float* values, void* stream);
/* The fused BPR triplet forward/backward (brk_bpr_fwd_bwd) on row-sharded tables of width d. */
int brk_bpr_fwd_bwd_sharded(brk_ctx* ctx, const brk_shards* user, const brk_shards* item, int32_t d,
                            const int32_t* u, const int32_t* p, const int32_t* n, int64_t batch,
                            int64_t global_batch, float* loss_out, void* stream);
/* Cross-GPU barrier on `stream`: returns (in stream order) once every rank's earlier work on its stream
 * has completed.  peer_flags: DEVICE array of `world` pointers to each rank's flag block (world uint32,
 * zero-initialised, peer-mapped); local_sync: 4 uint32 zero-initialised ([0] epoch, [1] error: a peer did
 * not arrive within ~3 s). */
int brk_peer_barrier(brk_ctx* ctx, uint32_t* const* peer_flags, uint32_t* local_sync, int32_t rank,
                     int32_t world, void* stream);

/* ---- data-parallel optimizer over NVLink peer memory ----------------------------------------------
 * Stands in for the per-step gradient all-reduce of MultiWorkerMirroredStrategy
 * (src/models/RModel.py:119-121) + Adam (NeuMFModel.py:89, BPRModel.py:70) when one process drives
 * each GPU: reduce-scatter of the gradient arena, Adam on the owned slice, all-gather of the new
 * weights, fused in one cooperative kernel with its own cross-GPU barriers (no NCCL on this path).
 * peer_w / peer_g / peer_flags are DEVICE arrays of `world` pointers into each rank's symmetric
 * (peer-mapped) weight arena, gradient arena (n floats each, n % 4 == 0) and flag block
 * (2*world uint32, zero-initialised before the first call on every rank).  m, v: local Adam moments of
 * the OWNED slice only (float4 range [rank*n/4/world, (rank+1)*n/4/world)).  local_sync: 8 uint32,
 * zero-initialised; local_sync[4] != 0 afterwards means a barrier timed out (a peer never arrived).
 * All ranks must call it once per step; on return (stream order) every rank's w is updated and
 * bit-identical, and this rank's g is zero. */
typedef struct brk_dp_peer {
  float* const* peer_w;
  float* const* peer_g;
  uint32_t* const* peer_flags;
  float* m;
  float* v;
  uint32_t* local_sync;
  int64_t n;
  int32_t rank, world;
} brk_dp_peer;
int brk_dp_adam_peer(brk_ctx* ctx, const brk_dp_peer* d, brk_adam_hyper h, int64_t* state, void* stream);
/* In-place all-reduce (sum) of a flat fp32 arena over NVLink peer memory (SURVEY.md section 8b "allreduce_dense"): the
 * gradient all-reduce of MultiWorkerMirroredStrategy (src/models/RModel.py:119-121) for steps whose optimizer is not
 * the fused Adam above (Keras Adagrad of trainers/twoTower.py:278-279, lazy Adam).  peer_buf / peer_flags: DEVICE
 * arrays of `world` pointers to each rank's symmetric arena (n floats, n % 4 == 0) and flag block (2*world uint32,
 * zero before the first call); local_sync: 8 uint32, zero-initialised ([4] != 0 afterwards: a peer never arrived, the
 * call was aborted and the arena left as it was).  Every rank sums its float4 slice over all peers in a fixed order
 * and stores it to every peer: the result is bit-identical on all ranks.  No NCCL. */
int brk_allreduce_dense_peer(brk_ctx* ctx, float* const* peer_buf, uint32_t* const* peer_flags, uint32_t* local_sync,
                             int64_t n, int32_t rank, int32_t world, void* stream);
/* The whole mirrored data-parallel BPR loop in ONE cooperative launch per rank: n_steps x (this rank's fused
 * fwd/bwd on batch batch_index_host[k] of its own u/p/n arrays, cross-GPU barrier, reduce-scatter + Adam +
 * all-gather over peer memory, cross-GPU barrier).  user / item must be adjacent views into this rank's arenas
 * of `dp` (user first), all ranks call with the same n_steps and batch (full batches only); gradients are
 * scaled by 1 / (world * batch); losses[k] = this rank's local-batch mean. */
int brk_bpr_train_steps_dp(brk_ctx* ctx, const brk_table* user, const brk_table* item, const int32_t* u,
                           const int32_t* p, const int32_t* n, int64_t total, int64_t batch,
                           const int64_t* batch_index_host, int32_t n_steps, brk_adam_hyper h,
                           const brk_dp_peer* dp, int64_t* step_dev, float* losses, void* stream);

/* ---- two-tower: towers + in-batch softmax / rdZero loss + backward -------------------------------
 * Stands in for TwoTowerModel.computeEmb / computeLossTfrs / computeLossRdZero / train_step
 * (trainers/twoTower.py:77-102) and tfrs.tasks.Retrieval (:47,83).  A tower is an embedding table
 * [rows, E] plus ONE flat dense block: the Keras Dense kernel W [E, S] row-major followed by the bias
 * [S] (twoTower.py:40-41: linear, no activation).
 *   brk_tower_forward : out[n,S] = table[ids] W + b (emb_out [n,E] receives the gathered rows)
 *   brk_twotower_step : mode 0 -- scores = Q C^T [B,B]; off-diagonal entries whose candidate id
 *     (cand_ids, may be NULL) equals the row's positive id get finfo(float32).min/100 added;
 *     loss = sum_b -log softmax_b[b] (reduction SUM, as TFRS).  mode 1 (rdZero) --
 *     sigmoid(<q_b, c_b>) against labels[b], mean binary cross-entropy.
 *     training != 0 additionally accumulates every gradient (emb.g rows, dense.g) for the optimizer.
 * Workspace (caller-owned, floats): eu [B,Eu], ei [B,Ei], q, c, dq, dc [B,S], scores [B,B] (mode 0),
 * ones [B] filled with 1.0, acc 1 double zero-initialised, deu [B,Eu] / dei [B,Ei] (training).
 * Inside the call the item-tower chain and the two Dense-gradient chains run on streams owned by the context,
 * forked from and joined back into `stream` (under stream capture they become branches of the graph).
 *   brk_sgemm : C (+)= alpha opA(A) opB(B) (+ bias); trans_a: A stored [K,M]; trans_b: B stored [N,K]; fp32 FMA.
 *     lda >= (trans_a ? M : K), ldb >= (trans_b ? K : N) and ldc >= N, else BRK_E_ARG before any launch; only
 *     C[0:M, 0:N] is written, for any M and N up to 2^31 - 1.  accumulate = 0 never splits K: row r of C is the same
 *     bits whatever M is and whichever other rows share the call (the item-range top-K indexes are bit-equal to the
 *     whole-catalog index only so).  accumulate != 0 may split K over CTAs that add into C with REDs, the bias once.
 *   brk_gemm_tf32 : the same product on tcgen05 with TF32 operands and fp32 accumulation in TMEM (gemm_tc.cu);
 *     needs 16-byte aligned operands with leading dimensions that are multiples of 4 (else BRK_E_ALIGN).  The same
 *     leading-dimension minimums and the same row guarantee: the tile width it picks from M, N and the SM count does
 *     not change a row's bits (tests/test_gpu_dense_products.py).
 *   brk_twotower_step mode bit 0x100 routes every Dense / in-batch product through brk_gemm_tf32 (falling back to
 *     the fp32 product where the alignment rule fails); results then agree with the fp32 path to TF32 rounding. */
typedef struct brk_tower {
  brk_table emb, dense;
  int32_t E, S;
} brk_tower;
typedef struct brk_twotower_workspace {
  float *eu, *ei, *q, *c, *dq, *dc, *scores, *ones;
  double* acc;
  float *deu, *dei;   /* [B,Eu], [B,Ei]: embedding-row gradients (training only) */
} brk_twotower_workspace;
int brk_sgemm(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int32_t M,
              int32_t N, int32_t K, int32_t lda, int32_t ldb, int32_t ldc, int32_t trans_a, int32_t trans_b,
              float alpha, int32_t accumulate, void* stream);
int brk_gemm_tf32(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int32_t M,
                  int32_t N, int32_t K, int32_t lda, int32_t ldb, int32_t ldc, int32_t trans_a, int32_t trans_b,
                  float alpha, int32_t accumulate, void* stream);
/* Diagnostics: brk_gemm_tf32 with CTA (0,0,0) writing %globaltimer (ns) into trace[0..6] (device uint64 [8]) at kernel
 * entry, TMEM allocated, first K chunk staged, all MMAs complete, accumulators in shared memory, stores issued, TMEM
 * freed (profiles/gemm_trace.py). */
int brk_gemm_tf32_trace(brk_ctx* ctx, const float* A, const float* B, float* C, const float* bias, int32_t M,
                        int32_t N, int32_t K, int32_t lda, int32_t ldb, int32_t ldc, int32_t trans_a,
                        int32_t trans_b, float alpha, int32_t accumulate, uint64_t* trace, void* stream);
int brk_tower_forward(brk_ctx* ctx, const brk_tower* t, const int32_t* ids, int64_t n, float* emb_out,
                      float* out, void* stream);
int brk_twotower_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                      const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                      int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out,
                      void* stream);
/* One training step INCLUDING the optimizer: TwoTowerModel.train_step (trainers/twoTower.py:89-102) with
 * tf.keras.optimizers.Adagrad(lr) (trainers/twoTower.py:278-279; accumulators in the tables' `m`).  mode as above.
 * In-batch-softmax steps with mode bit 0x100 whose batch fits on chip (ceil(batch/128)^2 <= SM count, widths <= 128)
 * run as ONE cooperative launch (csrc/twotower_fused.cu): towers, score tiles that never leave the SM, loss, all
 * gradients and Adagrad on the touched rows + Dense blocks.  Everything else = brk_twotower_step + brk_adagrad_dense /
 * brk_adagrad_rows (row-sparse for tables above rows_threshold_bytes that carry a touched bitmask).  Same results
 * either way up to the summation order of the REDs. */
int brk_twotower_train_step(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                            const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                            int32_t mode, const brk_twotower_workspace* ws, float lr, float eps,
                            int64_t rows_threshold_bytes, float* loss_out, void* stream);
/* Sampling-bias-corrected in-batch softmax (tfrs.tasks.Retrieval(temperature) called with candidate_sampling_probability
 * and sample_weight; Yi et al., RecSys 2019).  For query row b and in-batch candidate column j, in TFRS's order:
 *   s_bj = (q_b . c_j) * inv_temperature;  s_bj -= log(clip(p_j, 1e-6, 1)) (every column, the label column included);
 *   accidental hits masked as in brk_twotower_step;  loss = sum_b w_b (logsumexp_j s_bj - s_bb);
 *   gradient of the logits w_b (softmax_bj - [b == j]) * inv_temperature.
 * p_j: cand_prob[j] (caller-supplied, [batch]), or the streaming frequency estimate of candidate row i[j] (Yi et al.,
 * Algorithm 2, one exact slot per item-table row instead of a hash): state last[rows] (int64, initially 0), gap[rows]
 * (fp32, initially 0) and a device step counter *step (initially 0).  A training step sets t = *step + 1 and, once per
 * distinct item row y of the batch, gap[y] = (1 - alpha) gap[y] + alpha (t - last[y]) (each product and the sum rounded
 * to fp32), last[y] = t; it then stores t in *step and uses p_y = 1 / gap[y] (1 where gap[y] < 1).  training == 0 uses
 * the state as it is and changes nothing.  Neither cand_prob nor last: no correction.  row_weight NULL: w = 1.
 *   brk_twotower_step_retrieval / brk_twotower_train_step_retrieval: brk_twotower_step / brk_twotower_train_step with
 *     these options; rt == NULL is exactly the call without them.  BRK_E_ARG for inv_temperature not finite or <= 0,
 *     cand_prob together with the estimator, alpha outside (0, 1], gap or step NULL with last given, rows below the item
 *     table's rows, and rdZero mode. */
typedef struct brk_tt_retrieval {
  const float* cand_prob;     /* [batch] or NULL */
  const float* row_weight;    /* [batch] or NULL */
  int64_t*     last;          /* [rows] or NULL (no estimator) */
  float*       gap;           /* [rows] */
  int64_t*     step;          /* device counter of training steps */
  int64_t      rows;
  float        inv_temperature;
  float        alpha;
} brk_tt_retrieval;
int brk_twotower_step_retrieval(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                int32_t mode, int32_t training, const brk_twotower_workspace* ws, float* loss_out,
                                void* stream, const brk_tt_retrieval* rt);
int brk_twotower_train_step_retrieval(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                      const int32_t* i, const int32_t* cand_ids, const float* labels, int64_t batch,
                                      int32_t mode, const brk_twotower_workspace* ws, float lr, float eps,
                                      int64_t rows_threshold_bytes, float* loss_out, void* stream,
                                      const brk_tt_retrieval* rt);
/* Two-tower training on row-sharded embedding tables (sharded.ShardedTwoTowerNet): row r of a table lives on
 * rank r % world at local row r / world (brk_shards above); the Dense blocks are mirrored.
 *   brk_twotower_step_sharded: brk_twotower_step with training = 1 on THIS rank's slice of the global batch (its
 *     own items are the in-batch negatives); user / item carry this rank's Dense blocks (w, g), E and S, their emb
 *     tables are not read.  Rows are gathered from the owners' shards (peer loads), row gradients go as 16-byte REDs
 *     into the owner's g and set the owner's touched bits; Dense gradients are added into user / item dense.g.  Mode
 *     bits as brk_twotower_step: with 0x100 and a batch that fits on chip the step is one cooperative launch, else the
 *     multi-kernel step.  No optimizer runs.  batch == 0 does nothing (a rank with an empty slice still joins the
 *     exchanges that follow).  Ordering: after it, every rank must pass brk_peer_barrier before an owner applies
 *     brk_adagrad_rows to its shards, the Dense gradients are summed over ranks (brk_allreduce_dense_peer) before
 *     brk_adagrad_dense, and every rank must pass a cross-GPU barrier after its row pass before the next step
 *     gathers rows (the all-reduce's entry barrier does it when it is issued after the row pass).
 *   brk_tower_forward_sharded: brk_tower_forward with the rows gathered from the shards (inference, evaluation). */
typedef struct brk_twotower_shards { brk_shards user, item; } brk_twotower_shards;
int brk_twotower_step_sharded(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const brk_twotower_shards* sh,
                              const int32_t* u, const int32_t* i, const int32_t* cand_ids, const float* labels,
                              int64_t batch, int32_t mode, const brk_twotower_workspace* ws, float* loss_out,
                              void* stream);
int brk_tower_forward_sharded(brk_ctx* ctx, const brk_tower* t, const brk_shards* sh, const int32_t* ids, int64_t n,
                              float* emb_out, float* out, void* stream);
/* Sampling-bias-corrected softmax on row-sharded tables (sharded.ShardedTwoTowerNet(temperature=, streamingFrequency=)):
 * brk_tt_retrieval's semantics on each rank's slice, with the streaming estimator's state sharded like the item table.
 * last / gap of item row y live on rank y % world at local row y / world (rows per shard each, every rank's shard
 * pointer given: NVLink peer mappings, or local buffers when one process drives every rank); step is this rank's counter.
 *   brk_tt_estimator_update_sharded: the training-step update of the estimator for this rank's slice ids[0..n) of the
 *     global batch.  t = *step + 1; for every distinct row y of the GLOBAL batch exactly one thread on any GPU -- the one
 *     whose system-scope exchange of last[y] returned another step -- sets gap[y] = (1 - alpha) gap[y] + alpha (t -
 *     last[y]) (products and sum rounded to fp32); then *step = t.  So after every rank's update the state equals the
 *     single-process estimator run on the global batch, bit for bit.  n == 0 still advances the counter.  A grid-wide
 *     launch that waits on no other GPU; its launches on one context are stream-ordered (the context's last-block ticket
 *     writes the counter back).  BRK_E_ARG for null est / step / ids (n > 0), n < 0, alpha outside (0, 1], world outside
 *     1..BRK_MAX_PEERS, rank outside [0, world), rows < 1, and a null last / gap shard.
 *   brk_twotower_step_sharded_retrieval: brk_twotower_step_sharded with the options of brk_tt_retrieval on this rank's
 *     slice: logits (q_b . c_j) * inv_temperature - log(clip(p_j, 1e-6, 1)), accidental hits masked, loss = sum_b w_b
 *     (logsumexp_j s_bj - s_bb), logit gradient w_b (softmax_bj - [b == j]) * inv_temperature.  p_j: cand_prob[j]
 *     ([batch], caller-supplied), or with est != NULL 1 / gap of column j's item row read from its owner (1 where gap < 1);
 *     the estimator's state is only read.  row_weight NULL: w = 1.  rt == NULL is exactly brk_twotower_step_sharded.
 *     BRK_E_ARG as brk_twotower_step_sharded, and for inv_temperature not finite or <= 0, cand_prob together with est,
 *     rdZero mode, and an est whose world or rank differ from the shards', with rows < 1 or a null gap shard.
 * Ordering of one training step with the estimator: every rank (an empty slice included) calls
 * brk_tt_estimator_update_sharded, then passes brk_peer_barrier, then calls brk_twotower_step_sharded_retrieval; after it
 * the barriers of brk_twotower_step_sharded.  The next step's update comes after those barriers, so no rank updates the
 * state while another still reads it.  When one process drives every rank (or world == 1) the updates and the step are
 * ordered by the stream and no barrier is needed. */
typedef struct brk_tt_estimator_sharded {
  int64_t* last[BRK_MAX_PEERS];
  float*   gap[BRK_MAX_PEERS];
  int64_t  rows;              /* rows per shard */
  int32_t  world, rank;
} brk_tt_estimator_sharded;
typedef struct brk_tt_retrieval_sharded {
  const float* cand_prob;     /* [batch] or NULL */
  const float* row_weight;    /* [batch] or NULL */
  const brk_tt_estimator_sharded* est;   /* NULL: no estimator */
  float        inv_temperature;
} brk_tt_retrieval_sharded;
int brk_tt_estimator_update_sharded(brk_ctx* ctx, const brk_tt_estimator_sharded* est, const int32_t* ids, int64_t n,
                                    float alpha, int64_t* step, void* stream);
/* Mixed negative sampling (Yang et al., WWW 2020): each training step draws M item-table rows uniformly, with
 * replacement, from [lo, hi) and adds them as candidate columns shared by every query row (TFRS Retrieval called with
 * more candidates than queries).  The models draw from [2, numItem + 2): StringLookup's mask row 0 and OOV row 1 never.
 *   Draw k (0 <= k < M) of step t for replica r: lo + ((w.x * (hi - lo)) >> 32) with w = Philox4x32-10 of counter
 *     (k, uint32(t), uint32(t >> 32), 0x7E) and key (seed, r) (oracle/twotower_sampled.py).  t = *step + 1; the call
 *     writes t back to *step on the device, so CUDA-graph replays draw fresh rows.  The draws go to ids[0..M).
 *   Scores: c_all = item tower of concat(i, ids) (n = batch + M rows); logits Q c_all^T [batch, n] times inv_temperature;
 *     the label of row b is column b; column j != b gets finfo(float32).min/100 added where its item row equals i[b]
 *     (a sampled copy of the row's own positive is masked too); loss = sum_b w_b (logsumexp_j s_bj - s_bb) (SUM).
 *   Gradients: dq = (P - Y) c_all, dc = (P - Y)^T Q over all n rows; the Dense gradient of the item tower covers the
 *     sampled rows, and a sampled row gets its embedding gradient and touched bit like a batch row.
 *   brk_twotower_step_sampled / brk_twotower_train_step_sampled: brk_twotower_step (training = 1) /
 *     brk_twotower_train_step with sampled negatives; rt (optional) gives inv_temperature and row_weight only.
 *   brk_twotower_step_sharded_sampled: brk_twotower_step_sharded with sampled negatives on this rank's slice (rows
 *     gathered from and row gradients sent to their owners); rt (optional) gives inv_temperature and row_weight only.
 *     Each replica passes its own counter and replica number (its rank), so each replica draws its own rows.
 * With mode bit 0x100, widths <= 128 and max(T Tc, 2 (T + Tc)) <= SM count (T = ceil(batch / 128), Tc =
 * ceil((batch + M) / 128)) the step (and for the train step Adagrad) is ONE cooperative launch (csrc/twotower_fused.cu),
 * else the multi-kernel step; same results up to summation order and TF32 rounding.  Workspace as brk_twotower_step
 * except the item side: ei / dei [batch + M, Ei], c / dc [batch + M, S], scores [batch, batch + M].  batch == 0 draws (the counter advances), writes 0 to
 * loss_out and does nothing else.  Evaluation draws nothing: use brk_twotower_step(_retrieval) with training = 0.
 * BRK_E_ARG as the calls they extend, and for: count < 1; [lo, hi) empty, lo < 0 or hi above rows (for the unsharded
 * calls rows must also equal the item table's rows); a null step or ids; cand_prob, an estimator (last / est) or a
 * non-finite or non-positive inv_temperature in rt; rdZero mode; batch * (batch + M) >= 2^31. */
typedef struct brk_tt_sampled {
  int32_t* ids;               /* [count] output: this step's draws */
  int64_t* step;              /* device counter of training steps (initially 0) */
  int64_t  count;             /* M >= 1 */
  int64_t  lo, hi;            /* drawn from item-table rows [lo, hi) */
  int64_t  rows;              /* rows of the (global) item table */
  uint32_t seed, replica;
} brk_tt_sampled;
int brk_twotower_step_sampled(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                              const int32_t* i, int64_t batch, int32_t mode, const brk_twotower_workspace* ws,
                              float* loss_out, void* stream, const brk_tt_sampled* smp, const brk_tt_retrieval* rt);
int brk_twotower_train_step_sampled(brk_ctx* ctx, const brk_tower* user, const brk_tower* item, const int32_t* u,
                                    const int32_t* i, int64_t batch, int32_t mode, const brk_twotower_workspace* ws,
                                    float lr, float eps, int64_t rows_threshold_bytes, float* loss_out, void* stream,
                                    const brk_tt_sampled* smp, const brk_tt_retrieval* rt);
int brk_twotower_step_sharded_sampled(brk_ctx* ctx, const brk_tower* user, const brk_tower* item,
                                      const brk_twotower_shards* sh, const int32_t* u, const int32_t* i, int64_t batch,
                                      int32_t mode, const brk_twotower_workspace* ws, float* loss_out, void* stream,
                                      const brk_tt_sampled* smp, const brk_tt_retrieval_sharded* rt);
int brk_twotower_step_sharded_retrieval(brk_ctx* ctx, const brk_tower* user, const brk_tower* item,
                                        const brk_twotower_shards* sh, const int32_t* u, const int32_t* i,
                                        const int32_t* cand_ids, const float* labels, int64_t batch, int32_t mode,
                                        const brk_twotower_workspace* ws, float* loss_out, void* stream,
                                        const brk_tt_retrieval_sharded* rt);
/* Two-tower training with GLOBAL in-batch negatives (csrc/twotower_global.cu): every rank's queries are scored against
 * the candidates of the whole global batch of n rows.  Rank p holds rows [offset[p], offset[p] + count[p]) (the
 * offsets tile [0, n); slices may be empty).  For rank r's row i (global row o = offset[r] + i) the logits are
 * q_i . c_j over all n candidates, the label column is o, and a candidate j != o whose id equals the row's positive id
 * gets finfo(float32).min/100 added (accidental hits masked across slices); loss_out = the SUM of -log softmax over
 * this rank's rows.  dq stays local; dc_j sums (P - Y)_ij q_i over the queries of every rank: each rank writes its
 * partial for all n candidates into its slot buffer, and the owner of row j adds the world partials in rank order
 * (reproducible run to run).  Then the backward chain of brk_twotower_step / brk_twotower_step_sharded: Dense
 * gradients added into user / item dense.g, row gradients scattered into emb.g (sh == NULL, mirrored tables; touched
 * bits set) or sent as REDs into the owners' shards (sh != NULL).  No optimizer runs.
 * The step is three calls on `stream`, each one phase; every rank calls every phase, an empty slice included:
 *   phase 0: towers; this rank's candidate vectors go to cand[rank], its header {count, S} and ids to ids[rank].
 *   -- cross-GPU barrier (brk_peer_barrier) --
 *   phase 1: gathers the world candidate blocks into c_all [n, S] / ids_all [n] (16-byte peer loads; a header that
 *            disagrees with count[p] or S sets *err = 1 + p), scores = Q C_all^T [count[rank], n] in ws->scores,
 *            masked row softmax, loss, dq = (P - Y) C_all, and this rank's partial (P - Y)^T Q [n, S] in slot[rank].
 *   -- cross-GPU barrier --
 *   phase 2: dc = the rows [offset[rank], offset[rank] + count[rank]) of every slot, summed in rank order; Dense and
 *            row gradients of both towers.
 * Ordering: the phase-0 barrier of the next step comes after every rank's phase 2 in stream order, so no rank
 * overwrites its candidate block or slot buffer while a peer may still read them; the barriers after the step are
 * those of brk_twotower_step_sharded (row-sharded tables) or the Dense all-reduce (mirrored tables).
 * Pointers: cand / ids / slot are every rank's symmetric (peer-mapped) buffers -- cand [cap, S], ids [4 + cap] int32,
 * slot [n_cap, S] -- or G local buffers when one process drives every rank; c_all, ids_all and err are local.
 * Workspace as brk_twotower_step with B = count[rank], except ws->scores [B, n] and ws->c unused.  mode: 0, or 0x100
 * for the tensor-core products; rdZero (mode & 0xFF != 0) has no in-batch negatives and is rejected.  BRK_E_ARG for
 * world outside 1..BRK_MAX_PEERS, rank outside [0, world), offsets that do not tile [0, n), a count above cap or n above
 * n_cap, user and item S that differ, S not a multiple of 4, and null pointers a non-empty slice needs. */
typedef struct brk_twotower_global {
  float*   cand[BRK_MAX_PEERS];
  int32_t* ids[BRK_MAX_PEERS];
  float*   slot[BRK_MAX_PEERS];
  int64_t  offset[BRK_MAX_PEERS], count[BRK_MAX_PEERS];
  int64_t  cap, n_cap;
  float*   c_all;
  int32_t* ids_all;
  int32_t* err;
  int32_t  world, rank;
} brk_twotower_global;
int brk_twotower_step_global(brk_ctx* ctx, int32_t phase, const brk_tower* user, const brk_tower* item,
                             const brk_twotower_shards* sh, const brk_twotower_global* g, const int32_t* u,
                             const int32_t* i, int32_t mode, const brk_twotower_workspace* ws, float* loss_out,
                             void* stream);

/* ---- K7/K8: full-catalog scoring + top-K ------------------------------------------------------
 * Stands in for tfrs.layers.factorized_top_k.BruteForce(k).index(candidates) + call(queries)
 * (trainers/twoTower.py:64-69,60-62,229-230; src/origin_models/svd/SVD.py:424-432), for
 * bpr_predict (src/models/bpr.py:122-133) and for the streaming __topk of
 * trainers/topKmetrics.py:51-72.  scores = Q C^T (bf16 operands, fp32 accumulation on tcgen05);
 * per query row the k best (score, item id) come back sorted by descending score, ties -> lower
 * item id (tf.math.top_k's rule, and __topk's).  Scores are never written to HBM.
 *   brk_bf16_padded_dim(d)      row width of the bf16 operand copies (d rounded up to 64)
 *   brk_rows_to_bf16            fp32 [rows,d] -> bf16 [rows,dpad], zero padded (the "index" step)
 *   brk_score_topk_bf16         out_vals/out_ids [U,k]; id_offset is added to every item id (item-
 *                               range shards); workspace: brk_score_topk_workspace_bytes(...) bytes.
 *                               1 <= k <= 128 for dpad <= 128, k <= 64 for dpad 192 and 256 (BRK_E_ARG
 *                               beyond).  k <= 32 keeps each row's list in registers, longer lists a
 *                               heap per row in shared memory (one CTA per SM); the scores, the order
 *                               and the tie rule are the same, so a longer list's first entries equal
 *                               a shorter call's bit for bit
 *   brk_topk_merge              merges n_parts partial lists [n_parts,U,k] (score desc, id asc) --
 *                               the result is identical to an unsharded scan. */
int32_t brk_bf16_padded_dim(int32_t d);
int brk_rows_to_bf16(brk_ctx* ctx, const float* src, int64_t rows, int32_t d, uint16_t* dst,
                     int32_t dpad, void* stream);
int64_t brk_score_topk_workspace_bytes(brk_ctx* ctx, int64_t U, int64_t I, int32_t k);
int brk_score_topk_bf16(brk_ctx* ctx, const uint16_t* q_bf16, int64_t U, const uint16_t* c_bf16,
                        int64_t I, int32_t dpad, int32_t k, int32_t id_offset, float* out_vals,
                        int32_t* out_ids, void* workspace, int64_t workspace_bytes, void* stream);
/* Per-row exclusions (TFRS TopK.query_with_exclusions): the same top-k with row r's listed global ids left out.
 * A global id is the local candidate index plus id_offset, the id space of the results, so one list serves every
 * item-range shard.  Per row: the first k candidates that are not listed and score > -inf, by descending score, ties
 * -> lower id; (-inf, -1) pads a row with fewer.  Listed ids outside [id_offset, id_offset + I) are ignored, and so
 * are duplicates; with every list empty the result equals brk_score_topk_bf16's bit for bit.
 *   excl_indptr  int64 [U+1], absolute offsets into excl_ids: row r lists excl_ids[excl_indptr[r] .. excl_indptr[r+1]).
 *                It may be a view into a longer indptr (a chunk of rows passes indptr + s0, no rebasing).
 *   excl_ids     int32, ascending within each row (a precondition the caller guarantees).
 * Both are required (BRK_E_ARG if NULL); id_offset + I rounded up to 128 must stay below INT32_MAX.  The workspace
 * size is brk_score_topk_workspace_bytes(...).  Listed ids are tested only for items that beat the row's running
 * k-th best, so lists cost little unless they hold the row's best items. */
int brk_score_topk_bf16_excl(brk_ctx* ctx, const uint16_t* q_bf16, int64_t U, const uint16_t* c_bf16, int64_t I,
                             int32_t dpad, int32_t k, int32_t id_offset, const int64_t* excl_indptr,
                             const int32_t* excl_ids, float* out_vals, int32_t* out_ids, void* workspace,
                             int64_t workspace_bytes, void* stream);
/* The same exclusions on a materialised score matrix [R, I] (row-major): scores[r, id - col_offset] = -inf for every
 * listed id of row r inside [col_offset, col_offset + I), CSR as above.  brk_topk_rows afterwards gives the
 * exclusion semantics (it never selects -inf and pads with -1). */
int brk_mask_excluded(brk_ctx* ctx, float* scores, int64_t R, int64_t I, int32_t col_offset,
                      const int64_t* excl_indptr, const int32_t* excl_ids, void* stream);
/* Top-k per row of a materialised score matrix [R, I] (models without a factorised scorer: NeuMF,
 * trainers/topKmetrics.py:29-33 + __topk :51-72); same ordering rule; ids are column indices,
 * -1 pads rows with fewer than k columns. */
int brk_topk_rows(brk_ctx* ctx, const float* scores, int64_t R, int64_t I, int32_t k, float* out_vals,
                  int32_t* out_ids, void* stream);
int brk_topk_merge(brk_ctx* ctx, const float* part_vals, const int32_t* part_ids, int32_t n_parts,
                   int64_t U, int32_t k, float* out_vals, int32_t* out_ids, void* stream);
/* The merge of brk_topk_merge over lists held in other GPUs' memory: the exchange step of a full-catalog top-k over
 * item-range shards (sharded.ShardedTopKIndex).  part_vals / part_ids / part_hdr are DEVICE arrays of n_parts pointers
 * (1 <= n_parts <= BRK_MAX_PEERS), typically NVLink peer mappings of every rank's symmetric buffer: part s is one
 * rank's list [U, k] (score desc, id asc, (-inf, -1) padded) and its header, 3 int32 {seq, U, k} that the rank wrote
 * before a cross-GPU barrier (brk_peer_barrier) that precedes this call.  Every CTA copies its block of users from all
 * parts into shared memory with 16-byte loads and merges on chip; out_vals / out_ids [U, k] equal brk_topk_merge over
 * the same parts stacked, bit for bit.  If any header differs from {part 0's seq, U, k} -- a rank skipped a call, or
 * the ranks passed different users or a different k -- *err (device int32, left untouched otherwise) receives
 * 1 + the first such part and no result is written.  BRK_E_ARG for null pointers, n_parts outside 1..BRK_MAX_PEERS,
 * k outside 1..128 and U < 0; U = 0 does nothing. */
int brk_topk_merge_peer(brk_ctx* ctx, const float* const* part_vals, const int32_t* const* part_ids,
                        const int32_t* const* part_hdr, int32_t n_parts, int64_t U, int32_t k, float* out_vals,
                        int32_t* out_ids, int32_t* err, void* stream);
/* Full-catalog NeuMF top-k in one tcgen05 launch (csrc/neumf_topk.cu): per user, the k best items by the model's
 * inference prediction, scores never written to HBM.  The first layer factors, x0 W1 + b1 = A_u + B_i, and the caller
 * supplies both halves:
 *   user_side  A [U, H1]  = uMLP[users] W1[0:E]             (TF32 operands, fp32 accumulation: brk_gemm_tf32)
 *   item_side  B [I, H1]  = iMLP[items] W1[E:2E] + b1       (the same)
 *   item_mf    [I, EMF]   = iMF[items], the indexed items' MF rows;  users [U]: rows of m->uMF.
 * Per pair the kernel computes y1 = BN1(relu(A_u + B_i)) with the moving statistics (no BN in the He et al. variant),
 * y2 = BN2(relu(y1 W2 + b2)), h3 = relu(y2 W3 + b3) -- both products tcgen05.mma kind::tf32, fp32 accumulation --
 * then logit = h3 W4[0:H3] + gmf + b4 in fp32 (gmf = <uMF[u], iMF[i]> W4[H3] for the scalar Dot, sum of
 * uMF[u] * W4[H3:H3+EMF] * iMF[i] for the Hadamard GMF) and out = 1 / (1 + expf(-logit)), the value brk_neumf_step
 * returns for the pair (to TF32 rounding).  Selection on out: score desc, ties -> lower item id; ids are local
 * positions plus id_offset; rows with fewer than k candidates are padded with (-inf, -1).  A pair's score does not
 * depend on which other users or items share the call.  k <= 32.  Built instances (relu): the class graph
 * (32;32,16,8) and (64;64,32,16) with tensor_cores = 1, and the He et al. variant E 32, EMF 8, (32,16,8), Hadamard,
 * no BatchNorm; any other model is BRK_E_ARG.  Operands 16-byte aligned.  Workspace: brk_neumf_topk_workspace_bytes.
 * _excl: per-row exclusions with the contract of brk_score_topk_bf16_excl (global ids, ascending per row; ids outside
 * [id_offset, id_offset + I) ignored; empty lists give brk_neumf_score_topk's result bit for bit). */
int64_t brk_neumf_topk_workspace_bytes(brk_ctx* ctx, int64_t U, int64_t I, int32_t k);
int brk_neumf_score_topk(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side, const int32_t* users,
                         int64_t U, const float* item_side, const float* item_mf, int64_t I, int32_t k,
                         int32_t id_offset, float* out_vals, int32_t* out_ids, void* workspace,
                         int64_t workspace_bytes, void* stream);
int brk_neumf_score_topk_excl(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side, const int32_t* users,
                              int64_t U, const float* item_side, const float* item_mf, int64_t I, int32_t k,
                              int32_t id_offset, const int64_t* excl_indptr, const int32_t* excl_ids,
                              float* out_vals, int32_t* out_ids, void* workspace, int64_t workspace_bytes,
                              void* stream);
/* Full-catalog NeuMF top-k for the fp32 models (tensor_cores = 0) in one launch on the CUDA cores
 * (csrc/neumf_topk_fp32.cu).  Arguments and outputs as brk_neumf_score_topk / _excl; both halves of the first layer
 * are fp32 products here:
 *   user_side  A [U, H1]  = uMLP[users] W1[0:E]             (brk_sgemm)
 *   item_side  B [I, H1]  = iMLP[items] W1[E:2E] + b1       (brk_sgemm with bias)
 *   item_mf    [I, EMF]   = iMF[items];  users [U]: rows of m->uMF.
 * Per pair, in fp32 with the sums in the order of the any-width forward: y1 = BN1(act(A_u + B_i)),
 * y2 = BN2(act(y1 W2 + b2)), h3 = act(y2 W3 + b3), logit = h3 W4[0:H3] + gmf + b4 (gmf = W4[H3] <uMF[u], iMF[i]> for
 * the Dot head, sum_f (uMF[u][f] iMF[i][f]) W4[H3 + f] for the Hadamard head), out = 1 / (1 + expf(-logit)); act is
 * m->act (relu or sigmoid), BatchNorm uses the moving statistics (eps 1e-3) and is skipped with no_batch_norm.  out
 * agrees with brk_neumf_step's prediction for the pair to fp32 rounding.  Selection on out: score desc, ties -> lower
 * item id; ids are local positions plus id_offset; rows with fewer than k candidates are padded with (-inf, -1).  A
 * pair's score does not depend on which other users or items share the call.  Any width up to H1 <= 128, H2 <= 64,
 * H3 <= 32, EMF <= 128 (E free), 1 <= k <= 32, U >= 0 (U = 0 does nothing), I >= 1.  BRK_E_ARG for tensor_cores != 0
 * (those models rank through brk_neumf_score_topk), widths beyond the caps, k out of range, null operands and a
 * workspace smaller than brk_neumf_topk_fp32_workspace_bytes (which depends on the model's widths, U and k).
 * _excl: per-row exclusions with the contract of brk_neumf_score_topk_excl. */
int64_t brk_neumf_topk_fp32_workspace_bytes(brk_ctx* ctx, const brk_neumf_model* m, int64_t U, int64_t I, int32_t k);
int brk_neumf_score_topk_fp32(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side, const int32_t* users,
                              int64_t U, const float* item_side, const float* item_mf, int64_t I, int32_t k,
                              int32_t id_offset, float* out_vals, int32_t* out_ids, void* workspace,
                              int64_t workspace_bytes, void* stream);
int brk_neumf_score_topk_fp32_excl(brk_ctx* ctx, const brk_neumf_model* m, const float* user_side,
                                   const int32_t* users, int64_t U, const float* item_side, const float* item_mf,
                                   int64_t I, int32_t k, int32_t id_offset, const int64_t* excl_indptr,
                                   const int32_t* excl_ids, float* out_vals, int32_t* out_ids, void* workspace,
                                   int64_t workspace_bytes, void* stream);

/* ---- K9: ranking metrics ----------------------------------------------------------------------
 * Stands in for topKMetrics (trainers/topKmetrics.py:74-99): ids [U,k] are the recommended item ids
 * of users user_ids[r] (NULL: user r); positives are a CSR over csr_users users with sorted item
 * lists (distinct pairs).  counts_out[0] = tp, counts_out[1] = hits (users with >= 1 tp);
 * fp = U*k - tp, fn = |positives| - tp, tn = U*I - tp - fp - fn, precision, recall and
 * hitRate = hits / U follow on the host.  ndcg_sum_out = sum over users of DCG@k / IDCG@k (NDCG is
 * not in the reference; binary relevance, IDCG over min(|pos_u|, k)).  Negative ids (short lists)
 * count as misses. */
int brk_topk_metrics(brk_ctx* ctx, const int32_t* ids, int64_t U, int32_t k, const int32_t* user_ids,
                     const int64_t* pos_indptr, const int32_t* pos_items, int64_t csr_users,
                     int64_t* counts_out, double* ndcg_sum_out, void* stream);

/* brk_rank_eval_rows: per-user AUC and average precision at k of src/models/bpr.py:230-289 (full_auc ->
 * sklearn roc_auc_score per user; mean_average_precision_k -> Python sort of the whole catalog per user) from ONE
 * counting pass: for every positive p of row r of scores [R, I] (fp32, one row per user, one column per catalog
 * item) its 0-based rank = #{j: s_j > s_p} + #{j < p: s_j == s_p} (stable descending order, the earlier item first
 * among equals) and the number of negatives below / equal to it.
 *   out[2r]   = AUC of row r, ties counted half (NaN when the row has no positive or no negative);
 *   out[2r+1] = sum over positives with rank < k of (positives ranked at or above it) / (rank + 1), divided by
 *               min(actual_len[r], k)  (actual_len NULL: the number of positives; NaN when that is 0).
 * Positives: CSR over rows, pos_indptr int64 [R+1], pos_cols int32 column positions (distinct per row).
 * rank_ws int32 / part_ws double: device scratch, one entry per positive (pos_indptr[R] entries). */
int brk_rank_eval_rows(brk_ctx* ctx, const float* scores, int64_t R, int64_t I, const int64_t* pos_indptr,
                       const int32_t* pos_cols, const int32_t* actual_len, int32_t k, int32_t* rank_ws,
                       double* part_ws, double* out, void* stream);

/* ---- input pipeline (SURVEY.md section 8 rows f1 / f2: the caller's side of the training step) ------
 * brk_epoch_permutation: out[j] = perm(first + j), j < count, where perm is the keyed bijection of [0, n)
 *   "brk perm v1" (oracle/pipeline.py: six-round Feistel network over max(2, ceil(log2 n)) bits, round keys =
 *   Philox4x32-10(counter (round, 0, salt, 0x5E), key (seed, epoch)) words 0/1, two-multiply 32-bit round mixer,
 *   cycle walking).  Stands in for the unseeded shuffles of src/models/NeuMFModel.py:109 (rows, salt 0) and
 *   :117-121 (`.batch().shuffle()`: batches, salt 1) and trainers/twoTower.py:197 -- no sort, no memory.
 *   brk_epoch_permutation_host is the same function evaluated on the host (batch orders of host-driven
 *   loops: batch_index_host of the brk_bpr_train_steps* calls); it needs no device and no context.
 * brk_neumf_epoch_build: rows [first, first+count) of the shuffled training frame of one epoch in ONE launch --
 *   what bootstrapDataset (src/models/NeuMFModel.py:102-109) builds with pandas: row j is source row
 *   s = perm(j) of concat(positives, negatives); s < num_pos: the positive pair s, label 1; otherwise negative
 *   number s - num_pos of the "brk sampler v2" NeuMF stream (brk_philox_neumf_negatives), label 0.
 *   reject != 0 adds what the reference does not do (row f1): a draw that is a known positive (binary search in
 *   the per-user sorted lists csr_indptr int64 [U+1] / csr_items) is re-drawn with Philox counter word 2 =
 *   attempt 1..7; the eighth draw is kept whatever it is. */
int brk_epoch_permutation(brk_ctx* ctx, int64_t n, int64_t first, int64_t count, uint32_t seed,
                          uint32_t epoch, uint32_t salt, int64_t* out, void* stream);
int brk_epoch_permutation_host(int64_t n, int64_t first, int64_t count, uint32_t seed, uint32_t epoch,
                               uint32_t salt, int64_t* out_host);
int brk_neumf_epoch_build(brk_ctx* ctx, const int32_t* pos_users, const int32_t* pos_items,
                          int64_t num_pos, int64_t n_neg, int64_t first, int64_t count, uint32_t seed,
                          uint32_t epoch, int32_t reject, const int64_t* csr_indptr,
                          const int32_t* csr_items, int32_t* users, int32_t* items, float* labels,
                          void* stream);
/* Id factorisation: dense ids in order of first appearance -- `pd.unique` + positional lookup
 * (trainers/loadBinaryMovieLens.py:16-19,58-61) and StringLookup(vocabulary=...) (trainers/twoTower.py:33-36;
 * offset 2: index 0 = mask, 1 = OOV).  Keys are 64-bit (integer ids, or byte strings of <= 8 bytes packed
 * exactly); the key 0xFFFFFFFFFFFFFFFF is reserved.  An open-addressing table (capacity = a power of two
 * >= 2n, brk_vocab_capacity) records every distinct key with the smallest position it occurs at; a prefix sum
 * over the first-occurrence flags turns positions into ranks.
 *   ids[j] = offset + rank of keys[j];  vocab[r] = the r-th distinct key (may be NULL);  *n_unique (device)
 *   = number of distinct keys.  Afterwards (table_keys, table_vals) map key -> id for brk_vocab_lookup_u64,
 *   which writes `oov` for keys that are not in the table.
 * workspace: brk_vocab_workspace_bytes(n) bytes of device scratch.  n < 2^31 - 2^24. */
int64_t brk_vocab_capacity(int64_t n);
int64_t brk_vocab_workspace_bytes(int64_t n);
int brk_vocab_build_u64(brk_ctx* ctx, const uint64_t* keys, int64_t n, int32_t offset,
                        uint64_t* table_keys, int32_t* table_vals, int64_t capacity, int32_t* ids,
                        uint64_t* vocab, int64_t* n_unique, void* workspace, void* stream);
int brk_vocab_lookup_u64(brk_ctx* ctx, const uint64_t* keys, int64_t n, const uint64_t* table_keys,
                         const int32_t* table_vals, int64_t capacity, int32_t oov, int32_t* ids,
                         void* stream);

/* ---- biased-SVD SGD (SURVEY.md section 8 row f4): src/origin_models/svd/SVD.py ---------------------------
 * float64 throughout, like the NumPy original (np.random.random / np.zeros, SVD.py:446-449).
 * brk_svd_schedule: the dependency tickets of a rating file.  sched is int32 [n, 4] = (user, item, tu, ti) with
 *   tu[k] / ti[k] = number of earlier ratings (file order) of the same user / item; built by a stable radix sort
 *   per key column.  *bad_id (device int32) becomes 1 if an id is outside [0, num_users) / [0, num_items): such a
 *   schedule must not be used.  workspace: brk_svd_schedule_workspace_bytes(n, num_users, num_items) bytes.
 * brk_svd_fit_epoch: ONE pass of fit_model (SVD.py:187-221) with the sequential semantics kept exactly: rating by
 *   rating in file order,  e = r - (bu + bi + mu + <q, p>);  q' = q + lr (e p - emb_reg q);
 *   p' = p + lr (e q' - emb_reg p)  (the UPDATED item vector);  b' = b + lr (e b - bias_reg b)  for both biases
 *   (error times the bias itself, as the reference has it).  One warp per rating; a rating starts when both of
 *   its rows carry the version its tickets name and leaves them one version higher -- ratings that share no row
 *   run concurrently, ratings that share one run in file order.  Result = the sequential pass up to the summation
 *   order inside the dot product (element-wise operations are not contracted into FMAs).  During the epoch the
 *   tables live in a self-validating form inside the workspace (every 8-byte word carries its version); P, Q, bu,
 *   bi are read at the start and written back at the end of the call.
 *   workspace: brk_svd_fit_workspace_bytes(num_users, num_items, d) bytes of device scratch; its first uint32 is
 *   an abort flag that is non-zero afterwards only if a wait exceeded its bound (sched does not belong to these
 *   sizes).  warps_per_sm: resident warps per SM (0 = as many as fit).  d <= 512.  Cooperative launch.
 * brk_svd_predict: out[k] = bu[u] + bi[i] + mu + <Q[i], P[u]>  (predict, SVD.py:179-185).
 * brk_svd_errors: out[0] = mean squared error, out[1] = mean absolute error of rating - prediction over n >= 1
 *   ratings (mean_generic_error, SVD.py:223-253); partial sums are combined in a fixed order.
 *   workspace: brk_svd_reduce_workspace_bytes(ctx) bytes.
 * brk_svd_mean: out[0] = mean of x (the global bias, calculate_average SVD.py:139-161), out[1] = 0.
 * brk_svd_quintile_ratings: get_rating without a rating column (SVD.py:255-270):
 *   out = tc_scale * quintile(transaction_count, tc_quintiles) + qs_scale * quintile(quantity_sum, qs_quintiles),
 *   quintile(v, (q1, median, q3)) = 4 if v > q3, 3 if v > median, 2 if v > q1, else 1.  Quintiles: HOST double[3].
 * brk_svd_recommend: recommend (SVD.py:286-299) for a list of users: scores [n_users, num_items] (device scratch)
 *   = <P[users[j]], Q[i]>, then the k best per user, score descending, ties -> lower item index (the reference's
 *   strict '>' replacement keeps the earlier item); ids -1 / -inf pad when k > num_items. */
int64_t brk_svd_schedule_workspace_bytes(int64_t n, int64_t num_users, int64_t num_items);
int brk_svd_schedule(brk_ctx* ctx, const int32_t* users, const int32_t* items, int64_t n, int64_t num_users,
                     int64_t num_items, int32_t* sched, int32_t* bad_id, void* workspace,
                     int64_t workspace_bytes, void* stream);
int brk_svd_fit_epoch(brk_ctx* ctx, const int32_t* sched, const double* ratings, int64_t n, double* P,
                      double* Q, double* bu, double* bi, int64_t num_users, int64_t num_items, int32_t d,
                      double mu, double lr, double emb_reg, double bias_reg, void* workspace,
                      int64_t workspace_bytes, int32_t warps_per_sm, void* stream);
int64_t brk_svd_fit_workspace_bytes(int64_t num_users, int64_t num_items, int32_t d);
int brk_svd_predict(brk_ctx* ctx, const int32_t* users, const int32_t* items, int64_t n, const double* P,
                    const double* Q, const double* bu, const double* bi, int32_t d, double mu, double* out,
                    void* stream);
int64_t brk_svd_reduce_workspace_bytes(const brk_ctx* ctx);
int brk_svd_errors(brk_ctx* ctx, const int32_t* users, const int32_t* items, const double* ratings, int64_t n,
                   const double* P, const double* Q, const double* bu, const double* bi, int32_t d, double mu,
                   double* out_mse_mae, void* workspace, void* stream);
int brk_svd_mean(brk_ctx* ctx, const double* x, int64_t n, double* out2, void* workspace, void* stream);
int brk_svd_quintile_ratings(brk_ctx* ctx, const double* transaction_count, const double* quantity_sum,
                             int64_t n, double tc_scale, double qs_scale, const double* tc_quintiles_host,
                             const double* qs_quintiles_host, double* out, void* stream);
int brk_svd_recommend(brk_ctx* ctx, const double* P, const int32_t* users, int32_t n_users, const double* Q,
                      int64_t num_items, int32_t d, int32_t k, double* scores, double* out_vals,
                      int32_t* out_ids, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BRK_B200_H */
