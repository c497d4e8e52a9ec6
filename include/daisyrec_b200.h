/*
 * daisyrec_b200.h -- C ABI of the B200-native BPR hot path (libdaisyrec_b200.so).
 *
 * The reference (AmazingDD/daisyRec v2.3.0) is pure Python: it has no FFI, so the
 * "boundary" it offers is the duck-typed model / sampler contract consumed by
 * run_examples/test.py:87-95,118-120 and run_examples/tune.py:180-188,210-212
 * (SURVEY.md section 8(b)).  Each entry point below names the reference interface it
 * stands behind (file:line, relative to the reference root); the Python host in
 * daisyrec_b200/ (same class / method names as the reference) binds them with ctypes,
 * and INTEGRATION.md shows the stub a daisyRec maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary.
 *   - "d_" = device pointer, "h_" = host pointer.  Device buffers are allocated by the
 *     caller (any allocator: cudaMalloc, torch) on the current device.
 *   - stream: a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - every function returns DRB_OK (0) or a DRB_ERR_* code; drb_last_error() returns a
 *     thread-local message for the last failure.  Nothing aborts the process.
 *   - tables are row-major fp32: P[user_num, factors], Q[item_num, factors]
 *     (== MF.embed_user.weight / MF.embed_item.weight, daisy/model/MFRecommender.py:53-54).
 *   - index arrays are int32 for batches (the sampler's dtype, daisy/utils/sampler.py:101)
 *     and int64 for rank inputs (torch.tensor of python ints, daisy/utils/dataset.py:37-38).
 */
#ifndef DAISYREC_B200_H
#define DAISYREC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRB_OK 0
#define DRB_ERR_INVALID 1     /* bad argument (null pointer, unsupported factors, ...)            */
#define DRB_ERR_CUDA 2        /* a CUDA runtime call failed; see drb_last_error()                 */
#define DRB_ERR_NAN_LOSS 3    /* loss became NaN: ValueError of AbstractRecommender.py:122-123    */
#define DRB_ERR_EMPTY_SET 4   /* a user has no un-interacted item: numpy "a cannot be empty"      */
#define DRB_ERR_NO_DEVICE 5   /* no sm_100 device / kernel image not loadable on this device     */
#define DRB_ERR_PEER 6        /* multi-GPU peer exchange: a rank did not reach the rendezvous in time */

#define DRB_OPT_SGD 0         /* optim.SGD(lr)   AbstractRecommender.py:55-56                     */
#define DRB_OPT_ADAM 1        /* optim.Adam(lr)  AbstractRecommender.py:53-54 (dense, torch defaults) */
#define DRB_OPT_ADAGRAD 2     /* optim.Adagrad(lr) :57-58 (torch defaults; MF step only)          */
#define DRB_OPT_RMSPROP 3     /* optim.RMSprop(lr) :59-60 (torch defaults, dense; MF step only)   */

#define DRB_LOSS_BPR 0        /* BPRLoss   daisy/utils/loss.py:5-13   -log(1e-10 + sigmoid(pos - neg))           */
#define DRB_LOSS_HL 1         /* HingeLoss daisy/utils/loss.py:16-23  clamp(1 - (pos - neg), min=0)    (MF only)  */
#define DRB_LOSS_TL 2         /* TOP1Loss  daisy/utils/loss.py:26-33  sigmoid(neg - pos) + sigmoid(neg^2) (MF only) */
/* point-wise branch of MF.calc_loss (MFRecommender.py:75-81): the third index plane (d_bj) holds the int label
 * (sampler.py:93-98), only P_u and Q_i are scored and regularised; MF only, single GPU, no fused sampler */
#define DRB_LOSS_CL 3         /* nn.BCEWithLogitsLoss(reduction='sum')  AbstractRecommender.py:79-80 */
#define DRB_LOSS_SL 4         /* nn.MSELoss(reduction='sum')            AbstractRecommender.py:81-82 */

typedef struct drb_hyper {
    float lr;                 /* config['lr']                                                      */
    float reg_1;              /* config['reg_1']  L1 coefficient  (MFRecommender.py:88,94)        */
    float reg_2;              /* config['reg_2']  Frobenius coefficient (MFRecommender.py:89,95)  */
    int32_t opt;              /* DRB_OPT_*                                                         */
    float beta1, beta2, eps;  /* Adam (torch defaults 0.9, 0.999, 1e-8)                           */
    int32_t loss;             /* DRB_LOSS_*: config['loss_type'] of the pair-wise family              */
} drb_hyper;


/* ---- library / device ----------------------------------------------------------- */
int drb_version(void);
const char *drb_last_error(void);
/* sm_count, compute capability, L2 bytes of the current device */
int drb_device_query(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor, int64_t *l2_bytes);
/* Range check of an index array [n_rows, n_cols] (elem_bytes 4 = int32, 8 = int64; n_cols <= 4) resident on the device:
 * h_bad[c] = number of ids in column c outside [0, h_hi[c]).  The kernels index raw tables where the reference's
 * nn.Embedding raises IndexError (torch/nn/functional.py: embedding), so fit() / rank() call this once per uploaded
 * array and raise the same exception.  Synchronises the stream. */
int drb_index_range_check(const void *d_ids, int32_t elem_bytes, int64_t n_rows, int32_t n_cols, const int64_t *h_hi,
                          int64_t *h_bad, void *stream);
/* Which instantiation of the BPR step kernel trains `factors`-wide tables with BPR + SGD / Adam (the path behind
 * GeneralRecommender.fit, daisy/model/AbstractRecommender.py:112-128, for MF): returns 1 for a lean MF instantiation (its own
 * lane geometry; selected once per process on the device: every candidate geometry must reproduce the general instantiation's
 * losses and tables on a small seeded problem, the fastest one on an L2-regime timing problem is used if it beats the general
 * instantiation), 0 for the general one.  table_rows = user_num + item_num selects the regime the choice was made in: tables and
 * accumulators inside the L2 cache (also table_rows = 0) or streamed from HBM.  lanes / chunks (optional) receive the lanes per row and chunks of 4 floats per lane. */
int drb_mf_step_variant(int32_t factors, int64_t table_rows, int32_t *lanes, int32_t *chunks);
/* The timing half of that selection: milliseconds the general instantiation and the best lean candidate took for the same 3
 * steps of 524 288 triples, and the index-tile cap (512 or 1 024 triples) the chosen one runs with. */
int drb_mf_step_selfcheck_ms(int32_t factors, int64_t table_rows, float *ms_general, float *ms_lean, int32_t *tile_cap);
/* Host-only companion (no device): lane geometry of the lean (lean != 0) or canonical instantiation, and the tile size the
 * launcher picks for `per_cta` triples per CTA and step.  DRB_ERR_INVALID when no instantiation exists for `factors`. */
int drb_mf_step_geometry(int32_t factors, int32_t lean, int32_t *lanes, int32_t *chunks, int64_t per_cta, int32_t *tile);

/* ---- pair-wise sampler: BasicNegtiveSampler.sampling(), uniform + BPR branch ------
 * daisy/utils/sampler.py:55-103 (js table :63,84-89; explode :91,99-101).
 * CSR = config['train_ur'] as sorted, duplicate-free user->item rows.
 * Parity mode replays numpy's legacy MT19937 stream (np.random.seed, daisy/utils/config.py:34):
 * the word stream is inherently sequential, so the O(U*G) bounded draws run on the host
 * (drb_sampler_draw_mt19937) and everything proportional to nnz runs on the device. */
int drb_mt19937_seed(uint32_t *h_state625, uint32_t seed); /* numpy RandomState.seed(int) */
/* h_draws[u*G+g] = randint(0, item_num - deg(u)); advances the state exactly like the
 * reference's np.random.choice calls.  *bad_user receives the offending user on DRB_ERR_EMPTY_SET. */
int drb_sampler_draw_mt19937(uint32_t *h_state625, const int64_t *h_row_ptr, int32_t user_num, int32_t item_num,
                             int32_t num_ng, int32_t *h_draws, int32_t *bad_user);
/* counter-based (Philox4x32-10) draws on the device: throughput mode, NOT the reference stream */
int drb_sampler_draw_philox(uint64_t seed, uint64_t offset, const int64_t *d_row_ptr, int32_t user_num,
                            int32_t item_num, int32_t num_ng, int32_t *d_draws, int32_t *d_bad_user, void *stream);
/* js[u,g] = the draws[u,g]-th smallest item NOT in row u  (== setdiff1d(arange(I), past)[k]) */
int drb_sampler_kth_complement(const int64_t *d_row_ptr, const int32_t *d_col, const int32_t *d_draws,
                               int32_t user_num, int32_t item_num, int32_t num_ng, int32_t *d_js, void *stream);
/* triples[(r*G+g), :] = (coo_u[r], coo_i[r], js[coo_u[r], g])  -- int32 [nnz*G, 3] */
int drb_sampler_explode(const int32_t *d_coo_u, const int32_t *d_coo_i, int64_t nnz, const int32_t *d_js,
                        int32_t num_ng, int32_t *d_triples, void *stream);
/* host-buffer convenience: CSR + COO in, triples out (H2D / D2H inside) */
int drb_sample_triples_host(uint32_t *h_state625, const int64_t *h_row_ptr, const int32_t *h_col,
                            const int32_t *h_coo_u, const int32_t *h_coo_i, int64_t nnz, int32_t user_num,
                            int32_t item_num, int32_t num_ng, int32_t *h_js, int32_t *h_triples, int32_t *bad_user);

/* popularity-mixed branch, sample_method 'low-pop' / 'high-pop' (sampler.py:43-53,64-81): per user first
 * uniform_num = num_ng - int(sample_ratio*num_ng) uniform ranks as above, then other_num weighted draws
 * np.random.choice(arange(item_num), p=pop_prob) = searchsorted(cdf, random_sample(), 'right') with
 * cdf = pop_prob.cumsum() / cdf[-1] (RandomState.choice).  The host call replays the word stream (ranks +
 * 53-bit doubles, two words each); the device call turns both into the js table [user_num, uniform_num+other_num]. */
int drb_sampler_draw_mt19937_mixed(uint32_t *h_state625, const int64_t *h_row_ptr, int32_t user_num, int32_t item_num,
                                   int32_t uniform_num, int32_t other_num, int32_t *h_draws, double *h_u01,
                                   int32_t *bad_user);
int drb_sampler_assemble_mixed(const int64_t *d_row_ptr, const int32_t *d_col, const int32_t *d_draws,
                               const double *d_cdf, const double *d_u01, int32_t user_num, int32_t item_num,
                               int32_t uniform_num, int32_t other_num, int32_t *d_js, void *stream);
/* point-wise explode, loss_type CL / SL (sampler.py:93-98): int32 [nnz*(1+G), 3] = the nnz positive rows
 * (u, i, label) followed by the nnz*G negative rows (u, js[u,g], 0). */
int drb_sampler_explode_pointwise(const int32_t *d_coo_u, const int32_t *d_coo_i, const int32_t *d_label, int64_t nnz,
                                  const int32_t *d_js, int32_t num_ng, int32_t *d_rows, void *stream);

/* ---- candidate sets for ranking: build_candidates_set ------------------------------------
 * daisy/utils/utils.py:53-85.  Per test user the reference draws cand_num-|gt| ids from the
 * complement of gt + train positives (or, when |gt| >= cand_num, cand_num ids from gt itself).
 * Generic form: row m draws offsets[m+1]-offsets[m] values uniformly from [0, n[m]) off numpy's
 * MT19937 stream (host, sequential); the complement lookup runs on the device over the CSR of
 * each row's excluded ids (one warp per row). */
int drb_bounded_draws_mt19937(uint32_t *h_state625, const int64_t *h_n, const int64_t *h_offsets, int64_t rows,
                              int32_t *h_draws, int64_t *bad_row);
int drb_kth_complement_var(const int64_t *d_row_ptr, const int32_t *d_col, const int64_t *d_offsets,
                           const int32_t *d_draws, int64_t rows, int32_t *d_out, void *stream);

/* ---- pair-wise train feed: BasicDataset + DataLoader(shuffle=True) ------------------
 * daisy/utils/dataset.py:5-27.  Gathers the epoch's permuted triples into the SoA batch
 * arrays the step kernel streams with TMA: b?[k] = triples[perm[k], ?] (perm NULL = identity). */
int drb_gather_triples(const int32_t *d_triples, const int64_t *d_perm, int64_t n, int32_t *d_bu, int32_t *d_bi,
                       int32_t *d_bj, void *stream);

/* ---- BPR-MF training: GeneralRecommender.fit step loop ------------------------------
 * daisy/model/AbstractRecommender.py:112-128 with MF.calc_loss (MFRecommender.py:70-97),
 * BPRLoss (daisy/utils/loss.py:11), autograd backward (:125) and optimizer.step (:126).
 * One persistent cooperative kernel runs n_steps synchronous steps: every gradient of a
 * step is taken at the pre-step weights, exactly like the reference. */
size_t drb_mf_workspace_bytes(int32_t user_num, int32_t item_num, int32_t factors, int32_t opt);
int drb_mf_workspace_init(void *d_ws, int32_t user_num, int32_t item_num, int32_t factors, int32_t opt,
                          void *stream);
/* Steps first_step .. first_step+n_steps-1 over the SoA batch arrays (n triples total, step s
 * covers [s*batch, min((s+1)*batch, n)); the last batch may be partial, drop_last=False).
 * d_step_loss[n_steps]: fp32-assembled loss of each step (what loss.item() returns, :128).
 * adam_step0: number of optimizer steps already taken (Adam bias correction).
 * Returns DRB_ERR_NAN_LOSS after synchronising if a step produced NaN (tables keep their
 * pre-step values from that step on); *nan_step receives the step index. */
int drb_mf_bpr_train_steps(float *d_P, float *d_Q, void *d_ws, int32_t user_num, int32_t item_num, int32_t factors,
                           const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch,
                           int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                           double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream);
/* Throughput mode with the sampler FUSED into the step (north_star): no negative plane; the negative of every triple is
 * drawn inside phase 1 -- Philox word -> rank k in [0, item_num - deg(u)) -> k-th item missing from the user's sorted CSR
 * row -- i.e. the reference's complement distribution (sampler.py:86) but fresh for every triple and step instead of
 * once per user.  NOT reference semantics (opt-in).  d_neg_out (optional, n int32) receives the drawn negatives. */
int drb_mf_bpr_train_steps_fused_neg(float *d_P, float *d_Q, void *d_ws, int32_t user_num, int32_t item_num,
                                     int32_t factors, const int32_t *d_bu, const int32_t *d_bi, const int64_t *d_row_ptr,
                                     const int32_t *d_col, uint64_t seed, int32_t *d_neg_out, int64_t n, int64_t batch,
                                     int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                                     double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream);
/* MF.calc_loss(batch) only (no update): MFRecommender.py:70-97 */
int drb_mf_bpr_loss(const float *d_P, const float *d_Q, void *d_ws, int32_t user_num, int32_t item_num,
                    int32_t factors, const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t batch,
                    const drb_hyper *hyper, double *d_loss, void *stream);
/* End-to-end step with HOST batch arrays (what calc_loss receives from the DataLoader,
 * MFRecommender.py:71-72,83): H2D of 3*batch int32, one step, D2H of the loss. */
int drb_mf_bpr_train_step_host(float *d_P, float *d_Q, void *d_ws, int32_t user_num, int32_t item_num,
                               int32_t factors, const int32_t *h_bu, const int32_t *h_bi, const int32_t *h_bj,
                               int64_t batch, const drb_hyper *hyper, int64_t adam_step0, int32_t *d_stage,
                               double *h_loss, void *stream);

/* Pipelined end-to-end steps from HOST index planes (pinned): n_steps steps of `batch` triples; the
 * H2D copy of step s+1 overlaps the kernel of step s, every step's loss is read back asynchronously into
 * h_loss[s].  d_stage: 2 * 3 * round_up(batch, 4) int32 (double-buffered staging), d_loss: [n_steps]. */
int drb_mf_bpr_train_steps_host(float *d_P, float *d_Q, void *d_ws, int32_t user_num, int32_t item_num,
                                int32_t factors, const int32_t *h_bu, const int32_t *h_bi, const int32_t *h_bj,
                                int64_t n, int64_t batch, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                                int32_t *d_stage, double *d_loss, double *h_loss, int64_t *nan_step, void *stream);

/* ---- the DataLoader's epoch order on the device (daisy/utils/dataset.py:5-8 get_dataloader(shuffle=True)) ----------
 * torch's RandomSampler yields torch.randperm(n, generator=G) of a private CPU generator G seeded per epoch; ATen's
 * randperm_cpu is a Fisher-Yates walk over MT19937 words.  drb_randperm_torch returns THAT permutation (bit-exact, int64)
 * computed on the device: a one-CTA MT19937 stream + a parallel Fisher-Yates with deterministic reservations (one
 * cooperative launch).  n < 2^32/20 (ATen's branch).  d_ws: drb_randperm_workspace_bytes(n) bytes of scratch.
 * drb_mt19937_stream: the first n tempered 32-bit outputs of at::mt19937(seed) (= numpy's legacy stream for the same seed). */
size_t drb_randperm_workspace_bytes(int64_t n);
int drb_mt19937_stream(uint64_t seed, int64_t n, uint32_t *d_out, void *stream);
/* 1: drb_mt19937_stream runs the segmented kernel for n words (many CTAs generate disjoint segments of the ONE stream after
 * jumping ahead with precomputed polynomials, csrc/mt_jump_table.inc; used only after a one-off device check against the
 * sequential kernel), 0: the one-CTA kernel. */
int drb_mt19937_stream_variant(int64_t n);
int drb_randperm_torch(uint64_t seed, int64_t n, int64_t *d_perm, void *d_ws, void *stream);

/* Deterministic accumulation (opt-in, SURVEY 7 hard part 3): drb_mf_bpr_train_steps with every cross-thread sum (gradient
 * rows, loss, norms) accumulated as fixed-point int64 -- integer addition is associative, so tables and losses are bitwise
 * identical from run to run and independent of the order in which the atomics land.  4 scalar atomics instead of one
 * RED.128 per row chunk and one extra grid barrier per step: a reproducibility / parity mode, not the throughput path.
 * The workspace (drb_mf_workspace_bytes_det, initialised with drb_mf_workspace_init on that size) appends the int64 images. */
size_t drb_mf_workspace_bytes_det(int32_t user_num, int32_t item_num, int32_t factors, int32_t opt);
int drb_mf_bpr_train_steps_det(float *d_P, float *d_Q, void *d_ws, int32_t user_num, int32_t item_num, int32_t factors,
                               const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch,
                               int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                               double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream);

/* ---- FM (daisy/model/FMRecommender.py:16-131; SURVEY 8(f) rank 3) -----------------------------
 * FM.forward :61-68 = MF's factor product + (u_bias[u] + i_bias[i]) + bias_ (the three first-order terms are summed first,
 * fp32); FM.calc_loss :70-97 regularises the factor rows only, exactly as MF does; backward + optimizer.step as for MF,
 * the biases take the plain loss gradient.  d_bias = packed fp32 [u_bias (user_num), i_bias (item_num), bias_ (1)]
 * (== FM.u_bias.weight, FM.i_bias.weight, FM.bias_).  The workspace is the MF workspace plus the bias accumulator and
 * optimiser state.  All DRB_LOSS_* / DRB_OPT_* kinds; apply=0 evaluates the loss of one batch (n_steps must be 1). */
size_t drb_fm_workspace_bytes(int32_t user_num, int32_t item_num, int32_t factors, int32_t opt);
int drb_fm_workspace_init(void *d_ws, int32_t user_num, int32_t item_num, int32_t factors, int32_t opt, void *stream);
int drb_fm_train_steps(float *d_P, float *d_Q, float *d_bias, void *d_ws, int32_t user_num, int32_t item_num,
                       int32_t factors, const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n,
                       int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                       int32_t apply, double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream);
/* FM.rank :103-121 / FM.full_rank :123-131 / FM.predict :97-101: the MF kernels with the first-order terms added to
 * every score before the sort key is built. */
int drb_fm_rank(const float *d_P, const float *d_Q, const float *d_bias, int32_t user_num, int32_t item_num,
                int32_t factors, const int64_t *d_users, int64_t n_users, const int64_t *d_cands, int32_t cand_num,
                int32_t topk, float *d_out, void *stream);
int drb_fm_full_rank(const float *d_P, const float *d_Q, const float *d_bias, int32_t user_num, int32_t item_num,
                     int32_t factors, const int64_t *d_users, int64_t n_users, int32_t topk, int64_t *d_out, void *stream);
int drb_fm_predict(const float *d_P, const float *d_Q, const float *d_bias, int32_t user_num, int32_t item_num,
                   int32_t factors, const int32_t *d_u, const int32_t *d_i, int64_t n, float *d_out, void *stream);

/* ---- Item2Vec (daisy/model/Item2VecRecommender.py; skip-gram sampler daisy/utils/sampler.py:105-160) --------------------
 * SkipGramNegativeSampler.sampling(): the df rows grouped stably by user (groupby(uid)[iid].agg(list), :158-159) are the
 * positions; d_su / d_si [n] = their users (ascending) and items.  drb_sgns_positions writes, per position, the number c of
 * context items of the window (:136-146, = its number of negatives) and the size I - deg(user) of the complement of
 * config['train_ur'][user] (:132-133) its negatives come from.  The negatives are numpy's np.random.choice(cands, size=c)
 * (:148): drb_bounded_draws_mt19937 with one row per position replays them on the host.  drb_sgns_explode then writes the
 * int32 [2 * sum c, 3] rows in the reference's order: per position its c positives [target, seq[j], 1] in ascending j, then
 * its c negatives [target, k-th item outside the user's sorted CSR row, 0].  d_offsets [n+1] = exclusive scan of the counts
 * (row block of position p starts at 2 * d_offsets[p]; its draws at d_offsets[p]). */
int drb_sgns_positions(const int32_t *d_su, int64_t n, const int64_t *d_row_ptr, int32_t item_num, int32_t window,
                       int64_t *d_count, int64_t *d_bound, void *stream);
int drb_sgns_explode(const int32_t *d_su, const int32_t *d_si, int64_t n, int32_t window, const int64_t *d_offsets,
                     const int64_t *d_row_ptr, const int32_t *d_col, const int32_t *d_draws, int32_t *d_rows, void *stream);
/* Item2Vec.fit's step loop (AbstractRecommender.py:112-128 with Item2Vec.calc_loss :62-69): BCEWithLogitsLoss(sum) of
 * <shared[target], shared[context]> against the label, both rows read from and both gradients applied to ONE table d_Q
 * [item_num, factors] (== shared_embedding.weight, dense: every DRB_OPT_* kind moves every row).  The MF step kernel (GEN
 * instantiation) in shared-table mode: one persistent launch for n_steps steps; a triple whose target equals its context
 * contributes both gradients to that row.  hyper->loss must be DRB_LOSS_CL and reg_1 = reg_2 = 0; apply=0 evaluates the loss
 * of one batch (n_steps must be 1).  The workspace covers the item rows only. */
size_t drb_item2vec_workspace_bytes(int32_t item_num, int32_t factors, int32_t opt);
int drb_item2vec_workspace_init(void *d_ws, int32_t item_num, int32_t factors, int32_t opt, void *stream);
int drb_item2vec_train_steps(float *d_Q, void *d_ws, int32_t item_num, int32_t factors, const int32_t *d_bt,
                             const int32_t *d_bc, const int32_t *d_blabel, int64_t n, int64_t batch, int64_t first_step,
                             int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0, int32_t apply, double *d_step_loss,
                             int32_t sync_and_check, int64_t *nan_step, void *stream);
/* The user rows after training (Item2VecRecommender.py:56-60): d_P[u] = sum of d_Q[i] over the user's sorted train CSR row
 * (= config['train_ur'][u]); users with an empty row keep their values.  rank / full_rank / predict are drb_mf_* on
 * (d_P, d_Q). */
int drb_item2vec_user_embed(const int64_t *d_row_ptr, const int32_t *d_col, const float *d_Q, int32_t user_num,
                            int32_t factors, float *d_P, void *stream);

/* ---- NGCF + BPR (daisy/model/NGCFRecommender.py:38-252; SURVEY 8(f) rank 4; node_dropout = 0) -------------------------
 * E0: the ego table cat(embed_user, embed_item) [(U+I), dims[0]];  dims[0..L]: embedding size then hidden_size_list;
 * W: flat fp32 block, per BiGNN layer W1 [out,in], b1 [out], W2 [out,in], b2 [out] (linear, interact_transform; :46-47);
 * adjacency: the normalised CSR + segment list of drb_lgcn_* (get_norm_adj_mat :125-146 is LightGCN's).
 * drb_ngcf_forward      NGCF.forward :157-172 -> [(U+I), sum(dims)] = cat(E_0 .. E_L) (what rank / full_rank / predict score
 *                       with: feed its user / item halves to drb_mf_rank, drb_mf_full_rank, drb_mf_predict)
 * drb_ngcf_bpr_train_steps  calc_loss :174-205 + backward + optimizer.step for n_steps batches (apply = 0: loss of one batch).
 * Both with nn.Dropout(mess_dropout) of :164 active when d_keep != NULL (reference default 0.1; the reference builds the module
 *    inside forward(), so it drops at rank() time too): d_keep = the masks torch draws, one per layer over its [(U+I), width]
 *    output, as bytes, layers concatenated (train_steps: steps concatenated).  d_keep = NULL: no dropout.
 * Layer widths: 1..256.  tower_dtype as for NeuMF (0 fp32, 1 bf16 tcgen05 GEMMs). */
int64_t drb_ngcf_param_count(const int32_t *h_dims, int32_t num_layers);
size_t drb_ngcf_workspace_bytes(int32_t user_num, int32_t item_num, const int32_t *h_dims, int32_t num_layers, int32_t opt);
int drb_ngcf_workspace_init(void *d_ws, int32_t user_num, int32_t item_num, const int32_t *h_dims, int32_t num_layers,
                            int32_t opt, void *stream);
int drb_ngcf_forward(const float *d_E0, const float *d_W, void *d_ws, int32_t user_num, int32_t item_num, const int32_t *h_dims,
                     int32_t num_layers, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                     const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, int32_t tower_dtype,
                     const uint8_t *d_keep, float mess_dropout, float *d_out, void *stream);
int drb_ngcf_bpr_train_steps(float *d_E0, float *d_W, void *d_ws, int32_t user_num, int32_t item_num, const int32_t *h_dims,
                             int32_t num_layers, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                             const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, const int32_t *d_bu,
                             const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch, int64_t first_step,
                             int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0, int32_t apply, int32_t tower_dtype,
                             const uint8_t *d_keep, float mess_dropout, double *d_step_loss, int32_t sync_and_check,
                             int64_t *nan_step, void *stream);

/* ---- NFM + BPR (daisy/model/NFMRecommender.py:14-209; SURVEY 8(f) rank 4) ------------------------------------------
 * P [U,F], Q [I,F] factor tables; d_bias = packed [u_bias (U), i_bias (I), bias_];
 * N: flat fp32 block in module-registration order (:64-90): [gamma0, beta0] of FM_layers' BatchNorm1d (if batch_norm), per
 *    hidden layer W [F,F] (out,in), b [F], [gamma, beta], then prediction.weight [F];
 * Rs: BatchNorm running statistics, per BatchNorm mean [F] then var [F] (NULL without batch_norm).  act: 0 relu, 1 sigmoid, 2 tanh.
 * drb_nfm_bpr_train_steps  calc_loss :125-151 + backward + optimizer.step: the pos and the neg forward are separate calls in the
 *    reference, so every BatchNorm takes the statistics of ITS half of the 2*batch rows and moves its running statistics
 *    twice per step (pos first); apply = 0 evaluates the loss of one batch (the running statistics still move, as under train()).
 *    With d_keep != NULL the Dropout modules of :67,:88 are active (the reference default, assets/nfm.yaml: dropout 0.5):
 *    d_keep holds the masks torch's modules draw, as bytes, per step [forward call: pos, neg][site: FM_layers' Dropout, then
 *    the one behind each activation][batch][factors]; the host draws them on torch's CPU generator in that order
 *    (model/NFMRecommender.py), so a step equals the reference's.  d_keep = NULL: no dropout.
 * drb_nfm_scores  forward() under model.eval() (running statistics) for (d_u[k], d_i[k]) pairs: rank / full_rank / predict
 *    (:153-209); feed the scores to drb_topk_from_scores.  max_rows: rows of activation scratch (>= 2 * batch). */
int64_t drb_nfm_param_count(int32_t factors, int32_t num_layers, int32_t batch_norm);
size_t drb_nfm_workspace_bytes(int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers, int32_t batch_norm,
                               int32_t opt, int64_t max_rows);
int drb_nfm_workspace_init(void *d_ws, int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers,
                           int32_t batch_norm, int32_t opt, int64_t max_rows, void *stream);
int drb_nfm_bpr_train_steps(float *d_P, float *d_Q, float *d_bias, float *d_N, float *d_Rs, void *d_ws, int32_t user_num,
                            int32_t item_num, int32_t factors, int32_t num_layers, int32_t batch_norm, int32_t act,
                            int64_t max_rows, const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n,
                            int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                            int32_t apply, int32_t tower_dtype, const uint8_t *d_keep, float dropout, double *d_step_loss,
                            int32_t sync_and_check, int64_t *nan_step, void *stream);
int drb_nfm_scores(const float *d_P, const float *d_Q, const float *d_bias, const float *d_N, const float *d_Rs, void *d_ws,
                   int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers, int32_t batch_norm, int32_t act,
                   int32_t opt, int64_t max_rows, const int32_t *d_u, const int32_t *d_i, int64_t n, int32_t tower_dtype,
                   float *d_scores, void *stream);

/* ---- Multi-VAE (daisy/model/VAECFRecommender.py) ------------------------------------------------------------------
 * Dims: item_num, hidden[L] (mlp_hidden_size, L <= 8), latent_dim (>= 2).  Encoder item_num -> hidden[0..L-1] -> latent_dim,
 * decoder latent_dim/2 -> hidden[L-1..0] -> item_num, Tanh between the Linears of each side.
 * d_N: flat fp32 block in module-registration order: encoder.0 weight stored TRANSPOSED [item_num, hidden[0]], its bias, then
 *    every other Linear as torch lays it out (weight [out, in], bias [out]); each weight and bias is zero-padded to a multiple
 *    of 4 floats, so all of them start 16-byte aligned (drb_vae_param_count includes the padding).
 * Ratings: CSR over users (d_row_ptr i64[U+1], d_col i32, d_val f32), duplicate-free, zeros dropped.
 * drb_vae_train_steps  calc_loss + backward + optimizer.step (SGD / Adam over the whole block) for n_steps batches of d_users
 *    (a ragged last batch takes the rest); apply = 0 evaluates the loss of one batch.  training != 0: dropout on the normalised
 *    input and z = eps * exp(0.5 logvar) + mu.  Keep bits: d_keep = torch's keep-mask of each step ([batch, item_num] row-major,
 *    bit-packed little-endian into 32-bit words, ceil(batch * item_num / 32) words per step), NULL = Philox4x32-10(seed).
 *    eps: d_eps [n_steps][batch][latent_dim/2], NULL = Philox + Box-Muller.  Step s is update number update0 + s + 1 of the
 *    KL anneal, min(anneal_cap, update / total_anneal_steps) (anneal_cap when total_anneal_steps <= 0).
 *    tower_dtype 1 runs the GEMMs with bf16 operands on tcgen05 where their N fits one MMA.
 * drb_vae_forward  eval mode (no dropout, z = mu) for d_users[0, n): what 0 -> decoder output rows [n, item_num],
 *    1 -> last decoder hidden rows [n, hidden[0]] (latent_dim/2 when L = 0), 2 -> encoder output rows [n, latent_dim].
 * drb_vae_candidate_scores  decoder output at candidate ids only: scores[r, c] = <hidden rows[r], W_out[cands[r, c]]> + b_out. */
int64_t drb_vae_param_count(int32_t item_num, const int32_t *hidden, int32_t num_hidden, int32_t latent_dim);
size_t drb_vae_workspace_bytes(int32_t item_num, const int32_t *hidden, int32_t num_hidden, int32_t latent_dim, int32_t opt,
                               int64_t max_rows);
int drb_vae_workspace_init(void *d_ws, int32_t item_num, const int32_t *hidden, int32_t num_hidden, int32_t latent_dim, int32_t opt,
                           int64_t max_rows, void *stream);
int drb_vae_train_steps(float *d_N, void *d_ws, int32_t item_num, const int32_t *hidden, int32_t num_hidden, int32_t latent_dim,
                        int64_t max_rows, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val, int32_t user_num,
                        const int32_t *d_users, int64_t n, int64_t batch, int64_t first_step, int64_t n_steps, const drb_hyper *h,
                        int64_t adam_step0, int32_t apply, int32_t training, int32_t tower_dtype, float dropout,
                        const uint32_t *d_keep, const float *d_eps, uint64_t seed, double anneal_cap, int64_t total_anneal_steps,
                        int64_t update0, double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream);
int drb_vae_forward(const float *d_N, void *d_ws, int32_t item_num, const int32_t *hidden, int32_t num_hidden, int32_t latent_dim,
                    int32_t opt, int64_t max_rows, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                    int32_t user_num, const int32_t *d_users, int64_t n, int32_t what, int32_t tower_dtype, float *d_out,
                    void *stream);
int drb_vae_candidate_scores(const float *d_N, int32_t item_num, const int32_t *hidden, int32_t num_hidden, int32_t latent_dim,
                             const float *d_hidden, int64_t n, const int64_t *d_cands, int32_t num_cands, float *d_scores,
                             void *stream);

/* ---- multi-GPU (one process per GPU; user-sharded P, replicated Q; SURVEY 8(e)) ---------------
 * There is no multi-device path in the reference (single process, AbstractRecommender.py:99-100);
 * these entry points split the synchronous step where the exchange has to happen:
 *   phase 1 (accumulate on local triples) -> host all-reduces gQ / cntI / acc over NCCL ->
 *   phase 2 (apply: local P rows + the full replicated Q, identically on every rank).
 * drb_mf_workspace_layout: byte offset/size pairs inside the workspace of
 *   [0,1] acc (8 doubles)  [2,3] gQ (fp32 I*F)  [4,5] cntI (u64 I)  [6] gP offset  [7] cntU offset. */
int drb_mf_workspace_layout(int32_t user_num, int32_t item_num, int32_t factors, int32_t opt, int64_t *out8);
int drb_mf_bpr_phase(float *d_P, float *d_Q, void *d_ws, int32_t user_num, int32_t item_num, int32_t factors,
                     const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t begin, int64_t count,
                     int32_t phase, const drb_hyper *hyper, int64_t adam_step0, double *d_loss, void *stream);
/* Sharded train feed: keep the triples of users [user_lo, user_hi) from the GLOBAL epoch permutation,
 * renumber users locally, and report where each global step's local batch starts
 * (d_step_offsets[ceil(n/batch)+1]); d_scratch_counts needs ceil(n/batch) u64. */
int drb_shard_gather_triples(const int32_t *d_triples, const int64_t *d_perm, int64_t n, int32_t user_lo,
                             int32_t user_hi, int64_t batch, unsigned long long *d_scratch_counts,
                             int64_t *d_step_offsets, int32_t *d_bu, int32_t *d_bi, int32_t *d_bj, void *stream);

/* ---- LightGCN + BPR (daisy/model/LightGCNRecommender.py) --------------------------------------
 * E0 = cat(embed_user.weight, embed_item.weight): ONE contiguous fp32 [(U+I), F] table.
 * Adjacency: the symmetric normalised A_hat of get_norm_adj_mat (:73-107) as CSR over the U+I nodes
 * (row_ptr i64, col i32 ascending, val f32), plus its segment list (rows cut into <=256-edge pieces;
 * drb_lgcn_segment_count / drb_lgcn_segments, host).
 * drb_lgcn_propagate       forward() :117-129 -> E_mean (what rank / full_rank / predict score with, :171-211;
 *                          feed its halves to drb_mf_rank / drb_mf_full_rank / drb_mf_predict).
 * drb_lgcn_bpr_train_steps calc_loss :131-169 + backward + optimizer.step for n_steps batches
 *                          (apply = 0: calc_loss of one batch only).  2L sparse products per step. */
int64_t drb_lgcn_segment_count(const int64_t *h_row_ptr, int64_t n_nodes);
int drb_lgcn_segments(const int64_t *h_row_ptr, int64_t n_nodes, int32_t *h_seg_row, int64_t *h_seg_ptr);
size_t drb_lgcn_workspace_bytes(int32_t user_num, int32_t item_num, int32_t factors, int32_t opt);
int drb_lgcn_workspace_init(void *d_ws, int32_t user_num, int32_t item_num, int32_t factors, int32_t opt, void *stream);
int drb_lgcn_propagate(const float *d_E0, void *d_ws, int32_t user_num, int32_t item_num, int32_t factors,
                       int32_t num_layers, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                       const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, float *d_Em, void *stream);
int drb_lgcn_bpr_train_steps(float *d_E0, void *d_ws, int32_t user_num, int32_t item_num, int32_t factors,
                             int32_t num_layers, const int64_t *d_row_ptr, const int32_t *d_col, const float *d_val,
                             const int32_t *d_seg_row, const int64_t *d_seg_ptr, int64_t nseg, const int32_t *d_bu,
                             const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch, int64_t first_step,
                             int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0, int32_t apply,
                             double *d_step_loss, int32_t sync_and_check, int64_t *nan_step, void *stream);

/* ---- NeuMF + BPR (daisy/model/NeuMFRecommender.py) -------------------------------------------------
 * Tables: UG [U,F], IG [I,F] (embed_*_GMF), UM [U,D], IM [I,D] (embed_*_MLP), D = F * 2^(L-1);
 * W: the tower as ONE flat fp32 block in module-registration order -- per layer weight [out,in] then bias [out]
 * (in = 2D / 2^l), then predict_layer weight and bias [1]  (NeuMFRecommender.py:58-71).
 * mode = config['model_name'] (:48-50, :118-137): 0 'NeuMF' / 'NeuMF-pre' (predict over cat(GMF, tower), weight [2F]),
 *        1 'GMF' (predict over the GMF product, weight [F]; the tower is never run and takes no gradient),
 *        2 'MLP' (predict over the tower output, weight [F]).  All four tables are regularised in every mode (:154-167).
 * max_rows: rows of activation scratch (>= 2 * batch for training; any size for scoring).
 * drb_neumf_bpr_train_steps  calc_loss :139-169 (regulariser quirk of :158/:160 included) + backward +
 *                            optimizer.step for n_steps batches; apply = 0: calc_loss of one batch.
 *                            dropout (config['dropout'], :61), two engines:
 *                            d_drop_masks == NULL: counter-based Philox masks keyed by dropout_seed and the global step
 *                              (same distribution as nn.Dropout, not torch's RNG stream);
 *                            d_drop_masks != NULL (parity): the keep-masks nn.Dropout itself would draw, generated on the
 *                              host by torch in the reference's order and bit-packed -- per step drb_neumf_mask_words()
 *                              uint32 words: for layer l = 0..L-1 the [2*batch, n_l] row-major mask (rows [0,batch) = the pos
 *                              forward's mask, [batch, 2*batch) = the neg forward's), padded to a word.
 * drb_neumf_scores           forward :118-137 for (users[r / per_user], items[r]) pairs (items NULL: all item ids):
 *                            what rank / full_rank / predict score with (:171-232); feed to drb_topk_from_scores. */
int64_t drb_neumf_param_count(int32_t factors, int32_t num_layers, int32_t mode);
int64_t drb_neumf_mask_words(int32_t factors, int32_t num_layers, int64_t batch);
size_t drb_neumf_workspace_bytes(int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers, int32_t opt,
                                 int64_t max_rows);
int drb_neumf_workspace_init(void *d_ws, int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers,
                             int32_t opt, int64_t max_rows, void *stream);
int drb_neumf_bpr_train_steps(float *d_UG, float *d_IG, float *d_UM, float *d_IM, float *d_W, void *d_ws,
                              int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers, int64_t max_rows,
                              const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj, int64_t n, int64_t batch,
                              int64_t first_step, int64_t n_steps, const drb_hyper *hyper, int64_t adam_step0,
                              int32_t apply, int32_t tower_dtype, float dropout, uint64_t dropout_seed,
                              const uint32_t *d_drop_masks, int32_t mode, double *d_step_loss, int32_t sync_and_check,
                              int64_t *nan_step, void *stream);
int drb_neumf_scores(const float *d_UG, const float *d_IG, const float *d_UM, const float *d_IM, const float *d_W,
                     void *d_ws, int32_t user_num, int32_t item_num, int32_t factors, int32_t num_layers, int32_t opt,
                     int64_t max_rows, const int64_t *d_users, int64_t n_users, const int64_t *d_items, int32_t per_user,
                     int32_t tower_dtype, int32_t mode, float *d_scores, void *stream);
/* tower_dtype: 0 = fp32 on CUDA cores (parity path), 1 = bf16 operands on tcgen05 tensor cores with the fp32
 * accumulator in tensor memory (BASELINE config 3).  drb_gemm_test exposes the tower's GEMM dispatcher to the tests:
 * variant 0 NT+bias+ReLU (forward), 1 NN+ReLU-mask (input gradient), 2 NN, 3 TN split-K accumulate (weight gradient). */
int drb_gemm_test(int32_t variant, int32_t dtype, int64_t M, int32_t N, int32_t K, const float *d_A, int64_t lda,
                  const float *d_B, int64_t ldb, float *d_C, int64_t ldc, const float *d_bias, const float *d_ref,
                  int64_t ldref, void *stream);
/* top-K of pre-computed scores [n_rows, count]: ids from d_cands (float32 out, rank) or positions (int64 out, full_rank);
 * descending score, ties by lower position. */
int drb_topk_from_scores(const float *d_scores, const int64_t *d_cands, int64_t n_rows, int32_t count, int32_t topk,
                         float *d_out_f, int64_t *d_out_i, void *stream);

/* Native NCCL path of the sharded step: the library enqueues phase 1 -> ONE grouped all-reduce of {gQ, cntI, acc} ->
 * phase 2 for n_steps global steps on `stream` with no host round trip per step.  The communicator is created from a
 * 128-byte ncclUniqueId that rank 0 obtains (drb_comm_unique_id) and the host broadcasts to every rank. */
int drb_comm_unique_id(uint8_t *h_out128);
int drb_comm_init(const uint8_t *h_id128, int32_t rank, int32_t world);
int drb_comm_destroy(void);
int drb_mf_bpr_train_steps_sharded(float *d_P_local, float *d_Q, void *d_ws, int32_t user_num_local, int32_t item_num,
                                   int32_t factors, const int32_t *d_bu, const int32_t *d_bi, const int32_t *d_bj,
                                   const int64_t *h_step_offsets, int64_t first_step, int64_t n_steps,
                                   const drb_hyper *hyper, int64_t adam_step0, double *d_step_loss, void *stream);
/* The same global steps from HOST (pinned) planes holding this rank's share of every global batch (the N > 1 form of
 * drb_mf_bpr_train_steps_host; the reference's per-step `.to(device)` + `loss.item()`, AbstractRecommender.py:116-128):
 * the H2D copy of step s+1 overlaps step s; h_step_loss[s] receives the GLOBAL loss of step s.  d_stage: 2 x 3 x
 * stage_stride int32 (stage_stride = largest local share rounded up to a multiple of 4).  Synchronises the stream. */
int drb_mf_bpr_train_steps_sharded_host(float *d_P_local, float *d_Q, void *d_ws, int32_t user_num_local, int32_t item_num,
                                        int32_t factors, const int32_t *h_bu, const int32_t *h_bi, const int32_t *h_bj,
                                        const int64_t *h_step_offsets, int64_t first_step, int64_t n_steps,
                                        const drb_hyper *hyper, int64_t adam_step0, int32_t *d_stage, int64_t stage_stride,
                                        double *d_step_loss, double *h_step_loss, void *stream);

/* Peer-exchange form of the sharded step (csrc/p2p.cu): ONE persistent cooperative launch per rank runs n_steps global steps;
 * between phase 1 and phase 2 the ranks rendezvous through flags in peer-mapped memory, every rank reduces, updates and
 * broadcasts ITS slice of the item table over NVLink (peer loads / stores), no NCCL call and no relaunch per step.
 *   drb_p2p_buffer_bytes / drb_p2p_q_offset : size of a rank's exchange buffer, offset of its item-table replica inside it
 *   drb_p2p_alloc  : cudaMalloc + zero + 64-byte CUDA IPC handle (the host all-gathers the handles)
 *   drb_p2p_open / _close : map / unmap a peer's buffer;  drb_p2p_free : release the own buffer
 *   drb_mf_bpr_train_steps_p2p : h_peer_bufs[q] = rank q's buffer as mapped here (own buffer at [rank]); step s trains local
 *     triples [d_step_offsets[s], d_step_offsets[s+1]) (DEVICE array from drb_shard_gather_triples); steps_done = global steps
 *     already run on these buffers (rendezvous flags carry absolute step numbers; also Adam's step count).  BPR, SGD / Adam,
 *     factors a multiple of 4 up to 128.  A rank that does not reach a rendezvous within peer_timeout_s (<= 0: 20 s) ends
 *     the launch with DRB_ERR_PEER on every rank instead of hanging the GPUs. */
size_t drb_p2p_buffer_bytes(int32_t item_num, int32_t factors);
size_t drb_p2p_q_offset(int32_t item_num, int32_t factors);
int drb_p2p_alloc(size_t bytes, void **d_ptr, uint8_t *h_handle64);
int drb_p2p_open(const uint8_t *h_handle64, void **d_ptr);
int drb_p2p_close(void *d_ptr);
int drb_p2p_free(void *d_ptr);
int drb_mf_bpr_train_steps_p2p(float *d_P_local, void *d_ws, int32_t user_num_local, int32_t item_num, int32_t factors,
                               void *const *h_peer_bufs, int32_t rank, int32_t world, const int32_t *d_bu,
                               const int32_t *d_bi, const int32_t *d_bj, const int64_t *d_step_offsets, int64_t n_local,
                               int64_t batch_per_rank, int64_t first_step, int64_t n_steps, const drb_hyper *hyper,
                               int64_t steps_done, double *d_step_loss, double peer_timeout_s, int32_t sync_and_check,
                               int64_t *bad_step, void *stream);

/* ---- inference ------------------------------------------------------------------------
 * MF.rank  daisy/model/MFRecommender.py:106-123: per user, score cand_num candidates,
 *   descending sort, first topk ids as float32 (the reference's dtype quirk, :107).
 * MF.full_rank :126-133: all items, first topk ids as int64, no train-item masking.
 * MF.predict :99-104 / MF.forward :63-68.
 * Scores use the canonical fp32 summation order documented in DESIGN.md; equal scores
 * order by lower candidate position (rank) / lower item id (full_rank). */
int drb_mf_rank(const float *d_P, const float *d_Q, int32_t factors, const int64_t *d_users, int64_t n_users,
                const int64_t *d_cands, int32_t cand_num, int32_t topk, float *d_out, void *stream);
int drb_mf_full_rank(const float *d_P, const float *d_Q, int32_t factors, int32_t item_num, const int64_t *d_users,
                     int64_t n_users, int32_t topk, int64_t *d_out, void *stream);
int drb_mf_predict(const float *d_P, const float *d_Q, int32_t factors, const int32_t *d_u, const int32_t *d_i,
                   int64_t n, float *d_out, void *stream);
int drb_mf_rank_host(const float *d_P, const float *d_Q, int32_t factors, const int64_t *h_users, int64_t n_users,
                     const int64_t *h_cands, int32_t cand_num, int32_t topk, float *h_out);

/* ---- producers of the hot path's inputs, on the device -----------------------------------------
 * One sorted, duplicate-free CSR of the train interactions replaces get_ur (daisy/utils/utils.py:19-34), the
 * per-user setdiff1d input of the sampler (daisy/utils/sampler.py:84-89) and get_inter_matrix (utils.py:125-144);
 * with its transpose it yields LightGCN's normalised adjacency (daisy/model/LightGCNRecommender.py:73-107).
 * drb_csr_build: COO pairs (any order, duplicates allowed, int32) -> row_ptr i64[n_rows+1] + ascending unique columns
 *   (d_col_out needs room for nnz entries; *h_nnz_unique receives the number kept).  n_cols <= 2^20.  Synchronises.
 * drb_lgcn_build_adj: user->item CSR + item->user CSR (same nnz) -> A_hat as CSR over U+I nodes (adj_ptr i64[U+I+1],
 *   adj_col i32[2 nnz] ascending, adj_val f32[2 nnz] = float32((deg_r+1e-7)^-1/2 * (deg_c+1e-7)^-1/2), fp64 inside). */
size_t drb_csr_workspace_bytes(int32_t n_rows, int64_t nnz);
int drb_csr_build(const int32_t *d_row, const int32_t *d_col, int64_t nnz, int32_t n_rows, int32_t n_cols, void *d_ws,
                  int64_t *d_row_ptr, int32_t *d_col_out, int64_t *h_nnz_unique, void *stream);
int drb_lgcn_build_adj(const int64_t *d_ui_ptr, const int32_t *d_ui_col, const int64_t *d_iu_ptr, const int32_t *d_iu_col,
                       int32_t user_num, int32_t item_num, int64_t nnz, int64_t *d_adj_ptr, int32_t *d_adj_col,
                       float *d_adj_val, void *stream);

/* ---- evaluation: calc_ranking_results / Metric.run ------------------------------------------------
 * daisy/utils/metrics.py:18-57 (cut-off loop), :59-96 (dispatch), :98-251 (the KPIs).
 * d_preds: rank()'s float32 [n_users, ld] output; ground truth as CSR aligned with its rows
 * (gt_ptr i64[n_users+1], gt_idx i32 ascending inside a row = sorted(test_ur[test_u[row]])).
 * h_ks[nk]: the cut-offs (common_ks of :41-43), each in [1, min(ld, 256)], nk <= 8.
 * d_out: double [nk, DRB_KPI_COUNT], the np.mean over users of each KPI at each cut-off (fp64 like the
 * reference; in1d semantics: duplicate ids in a list each count).  Coverage counts distinct ids in
 * [0, item_num); Popularity needs d_item_pop (double [item_num], loader.py:191-194), NULL leaves it 0. */
#define DRB_KPI_RECALL 0      /* metrics.py:170-180 */
#define DRB_KPI_MRR 1         /* :182-196 */
#define DRB_KPI_NDCG 2        /* :215-238 */
#define DRB_KPI_HIT 3         /* :240-251 */
#define DRB_KPI_PRECISION 4   /* :158-168 */
#define DRB_KPI_MAP 5         /* :198-213 */
#define DRB_KPI_COVERAGE 6    /* :98-102  */
#define DRB_KPI_POPULARITY 7  /* :104-122 */
#define DRB_KPI_COUNT 8
size_t drb_rank_metrics_workspace_bytes(int32_t item_num, int32_t nk);
int drb_rank_metrics(const float *d_preds, int64_t n_users, int32_t ld, const int64_t *d_gt_ptr,
                     const int32_t *d_gt_idx, const int32_t *h_ks, int32_t nk, int32_t item_num,
                     const double *d_item_pop, void *d_ws, double *d_out, void *stream);
/* host-buffer form (numpy in, numpy out: the signature calc_ranking_results is called with) */
int drb_rank_metrics_host(const float *h_preds, int64_t n_users, int32_t ld, const int64_t *h_gt_ptr,
                          const int32_t *h_gt_idx, const int32_t *h_ks, int32_t nk, int32_t item_num,
                          const double *h_item_pop, double *h_out);

#ifdef __cplusplus
}
#endif
#endif /* DAISYREC_B200_H */
