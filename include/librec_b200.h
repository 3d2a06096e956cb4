/* =====================================================================================
 * librec_b200.h -- C ABI of the B200-native LibRec matrix-factorisation hot path.
 *
 * The reference (szkb/librec, LibRec 3.0.0) is pure Java and has NO FFI of its own
 * (SURVEY.md 2.1), so these entry points are what a JNI / Panama shim for this path binds
 * (INTEGRATION.md shows that shim).  Each function names the reference interface it
 * replaces; paths are relative to core/src/main/java/net/librec/ in the reference.
 *
 * Conventions
 *   - plain pointers and sizes only; every buffer is caller-allocated and caller-freed,
 *     row-major, 0-based LibRec inner ids (math/structure/DataFrame.java:370-379).
 *   - every call returns LRK_OK (0) or a negative lrk_status; the text of the last error is
 *     available from lrk_last_error().  Nothing throws or aborts across the ABI; the Java
 *     shim maps a non-zero status to LibrecException (common/LibrecException.java).
 *   - a handle is NOT thread-safe: one handle per recommender instance, caller serialises
 *     (the reference calls train/recommend from one thread: job/RecommenderJob.java:121-143).
 *   - there is no CPU fallback: without a CUDA device every compute call fails with
 *     LRK_ERR_CUDA.
 * ===================================================================================== */
#ifndef LIBREC_B200_H
#define LIBREC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRK_ABI_VERSION 1

#if defined(__GNUC__)
#define LRK_API __attribute__((visibility("default")))
#else
#define LRK_API
#endif

typedef struct lrk_handle_s* lrk_handle_t;

typedef enum {
    LRK_OK = 0,
    LRK_ERR_INVALID = -1,   /* bad argument / call order                       */
    LRK_ERR_CUDA = -2,      /* CUDA runtime error (incl. no device)            */
    LRK_ERR_NCCL = -3,      /* NCCL error                                      */
    LRK_ERR_NOMEM = -4,     /* host or device allocation failed                */
    LRK_ERR_DIVERGED = -5   /* loss is NaN/Inf: AbstractRecommender.java:259-262 */
} lrk_status;

/* rec.recommender.class values served by this path (resources/driver.classes.props):
 * biasedmf -> recommender/cf/rating/BiasedMFRecommender.java
 * pmf      -> vanilla PMF loop, recommender/cf/rating/PMFSimilarityRecommender.java:59-90
 * bpr      -> recommender/cf/ranking/BPRRecommender.java */
typedef enum {
    LRK_MODEL_BIASEDMF = 0,
    LRK_MODEL_PMF = 1,
    LRK_MODEL_BPR = 2,
    /* ranksgd -> recommender/cf/ranking/RankSGDRecommender.java:62-108 (SURVEY.md 8f row N3): one update per train entry
     * against a negative drawn by item popularity; single GPU; lrk_sgd_epoch ignores the regularisation arguments */
    LRK_MODEL_RANKSGD = 3,
    /* gbpr -> recommender/cf/ranking/GBPRRecommender.java:82-172 (SURVEY.md 8f row N3): group-preference BPR.  Item biases only
     * (lrk_set_factors: bi is required; it ignores bu and global_mean and keeps zero user biases and a zero mean, so every
     * prediction and top-N score is predict() = b_i + p_u.q_i, GBPRRecommender.java:194-196; training reads no global mean);
     * rec.gpbr.rho / rec.gpbr.gsize through lrk_set_param; single GPU; lrk_sgd_epoch's reg_b is rec.bias.regularization */
    LRK_MODEL_GBPR = 4,
    /* svdpp -> recommender/cf/rating/SVDPlusPlusRecommender.java:62-123 (SURVEY.md 8f row N3): BiasedMF plus the implicit-feedback
     * factors impItemFactors (I x k) -- handed over / read back with lrk_set_matrix / lrk_get_matrix("svdpp.y"),
     * rec.impItem.regularization through lrk_set_param("svdpp.reg_imp").  Training only, single GPU: its predict() needs the
     * per-user sum of the implicit factors, so the scoring entry points return LRK_ERR_INVALID for this model (the shim keeps
     * the reference's predict() on the matrices it reads back). */
    LRK_MODEL_SVDPP = 5,
    /* aobpr -> recommender/cf/ranking/AoBPRRecommender.java:60-200 (SURVEY.md 8f row N3): BPR with adaptive oversampling of the
     * negative item; rec.item.distribution.parameter through lrk_set_param("aobpr.lambda") (required, as in the reference);
     * single GPU; scoring and lrk_bpr_peek_samples as for BPR */
    LRK_MODEL_AOBPR = 6,
    /* wrmf -> recommender/cf/ranking/WRMFRecommender.java:74-166 (SURVEY.md 8f row N3): alternating least squares with the
     * reference's Gauss-Jordan inverse (math/structure/DenseMatrix.java:362-437).  lrk_set_train_csr takes the WEIGHTED values
     * (weightMatrix() stays in the shim's setup()); lrk_sgd_epoch = one iteration (lr and reg_b ignored, loss 0 -- the class
     * never assigns it); fp64 in the reference's operation order: factors BIT-identical to the reference's; rec.factor.number <= 112;
     * several GPUs through lrk_create_multi (bit-identical to one GPU), not as a DSGD rank (lrk_comm_init); scoring as for PMF */
    LRK_MODEL_WRMF = 7,
    /* eals -> recommender/cf/ranking/EALSRecommender.java:114-214 (SURVEY.md 8f row N3): element-wise ALS.  Weighted values as
     * for WRMF; the item confidences (:65-83, computed in the shim's setup()) through lrk_set_matrix("eals.confidences");
     * the caller hands over zero user factors (:125 replaces them).  Bit-identical like WRMF; single GPU */
    LRK_MODEL_EALS = 8
} lrk_model;

/* how concurrent updates to one factor row are combined */
typedef enum {
    LRK_UPDATE_ATOMIC = 0,  /* red.global.add.v4.f32: no lost updates (default; needed for RMSE parity) */
    LRK_UPDATE_HOGWILD = 1, /* plain racy read-modify-write stores                                      */
    /* parity mode: the reference's sequential CSR-order walk executed as a dependency wavefront in
     * fp64 with Java's operation order -- learned factors are bit-identical to the reference
     * arithmetic; throughput is bounded by the longest dependency chain.  BiasedMF, PMF and BPR.
     * BPR: each epoch draws numRates samples from the reference's java.util.Random state (Randoms.r, see
     * "jdk.random.state" under lrk_set_matrix) exactly as BPRRecommender.java:54-67 does, and applies them in
     * sample order; Maths.logistic is evaluated with StrictMath.exp (fdlibm), so the factors and the generator state
     * after the epoch equal a JVM's whose Math.exp is StrictMath.exp.  Single GPU, fp64 masters as the working set,
     * no rollback safeguard; the reported loss may differ from the sequential sum in its last bits. */
    LRK_UPDATE_REFERENCE_ORDER = 2
} lrk_update_mode;

typedef struct {
    int32_t device;        /* CUDA device ordinal                                               */
    int32_t model;         /* lrk_model                                                         */
    int32_t num_factors;   /* rec.factor.number  (MatrixFactorizationRecommender.java:75), 1..256 */
    int32_t update_mode;   /* lrk_update_mode                                                   */
    uint64_t seed;         /* shuffle / BPR-sampling seed (rec.cuda.seed)                       */
    int32_t topn_path;     /* 0 auto, 1 exact fp64 kernel only, 2 force tensor-core candidates  */
    int32_t reserved[7];   /* must be zero                                                      */
} lrk_config_t;

/* ---- lifecycle ---------------------------------------------------------------------- */
LRK_API const char* lrk_version(void);
LRK_API int32_t lrk_abi_version(void);
/* number of visible CUDA devices (0 when none / driver missing); never fails */
LRK_API int32_t lrk_device_count(void);
/* replaces: the no-arg constructor + setup() allocation of DenseMatrix factors
 * (recommender/MatrixFactorizationRecommender.java:67-94). */
LRK_API int lrk_create(const lrk_config_t* cfg, lrk_handle_t* out);
/* replaces the same constructor for rec.cuda.devices=d0,d1,... (1 to 8 devices of one box): ONE handle, driven from the one thread
 * job/RecommenderJob.java:121-143 runs, that trains on all listed GPUs.  It takes and returns the FULL matrices exactly like a
 * single-device handle; inside, users are cut into contiguous blocks, one per device, each device runs a DSGD rank on its own host
 * thread (NCCL communicator created inside this process; item blocks rotate over NVLink), and lrk_topn shards the queried users over
 * the devices with the full item matrix on each (no collective).  BiasedMF, PMF, BPR and WRMF; the other models take one device.
 * WRMF needs no communicator: every device stages the full train matrix and holds full copies of both factor matrices, solves its
 * own range of users and of items (contiguous ranges of about equal solve cost), and the devices exchange the new rows after each
 * half-iteration (peer copies); the factors are bit-identical to a single device's, and lrk_last_epoch_ms is the wall time of the
 * whole iteration.  With one device a multi handle is a plain handle.  cfg->device is ignored.  Supported on a multi handle:
 * lrk_set_train_csr, lrk_set_factors, lrk_sgd_epoch(s), lrk_get_factors, lrk_topn, lrk_topn_stats, lrk_stage_stats, lrk_last_epoch_ms,
 * lrk_sgd_safeguard_state, lrk_launch_count, lrk_synchronize, lrk_probe_l2, lrk_last_error, lrk_destroy; the remaining entry points
 * return LRK_ERR_INVALID (gather the factors with lrk_get_factors and use a single-device handle for them). */
LRK_API int lrk_create_multi(const lrk_config_t* cfg, const int32_t* devices, int32_t n_devices, lrk_handle_t* out);
LRK_API int lrk_destroy(lrk_handle_t h);
/* h may be NULL: returns the last error of the calling thread for calls that had no handle */
LRK_API const char* lrk_last_error(lrk_handle_t h);
/* run all work of this handle on an externally owned cudaStream_t (NULL = handle's own stream) */
LRK_API int lrk_set_stream(lrk_handle_t h, void* cuda_stream);
LRK_API int lrk_synchronize(lrk_handle_t h);

/* pinned host staging buffers for the shim's flatten step (direct ByteBuffers on the Java side) */
LRK_API int lrk_host_alloc(void** out, uint64_t bytes);
LRK_API int lrk_host_free(void* p);

/* ---- staging ------------------------------------------------------------------------ */
/* replaces: trainMatrix = (SequentialAccessSparseMatrix) getDataModel().getTrainDataSet()
 * (recommender/MatrixRecommender.java:90) -- the per-row int[]/double[] pieces
 * (math/structure/RowSequentialAccessSparseMatrix.java:19, OrderedIntDoubleMapping) flattened to
 * rowptr[U+1], col[nnz] (ascending inside a row), val[nnz].  Builds the device CSR and a
 * device-shuffled COO stream for the SGD epoch.  nnz < 2^31 per handle (under DSGD / a multi handle: per rank; a WRMF multi handle
 * stages the whole matrix on every device, so there the limit is on the full matrix). */
LRK_API int lrk_set_train_csr(lrk_handle_t h, int32_t num_users, int32_t num_items,
                      const int64_t* rowptr, const int32_t* col, const double* val);
/* replaces: DenseMatrix userFactors/itemFactors (double[][], math/structure/DenseMatrix.java:20),
 * VectorBasedDenseVector userBiases/itemBiases (BiasedMFRecommender.java:40-45), globalMean
 * (MatrixRecommender.java:109).  P is U x k, Q is I x k; bu/bi may be NULL unless model is BIASEDMF (GBPR: bi is required). */
LRK_API int lrk_set_factors(lrk_handle_t h, const double* P, const double* Q, const double* bu, const double* bi,
                    double global_mean);
/* copies the current factors back (any pointer may be NULL to skip it) so the inherited Java
 * predict()/recommendRating()/evaluators keep working on DenseMatrix. */
LRK_API int lrk_get_factors(lrk_handle_t h, double* P, double* Q, double* bu, double* bi);

/* model hyper-parameters that are not arguments of lrk_sgd_epoch (read by the reference in setup()):
 *   "gbpr.rho"   rec.gpbr.rho   (float, default 1.5; GBPRRecommender.java:71)
 *   "gbpr.gsize" rec.gpbr.gsize (int 1..8, default 2; GBPRRecommender.java:72)
 *   "svdpp.reg_imp" rec.impItem.regularization (default 0.015; SVDPlusPlusRecommender.java:52)
 *   "aobpr.lambda" rec.item.distribution.parameter (no default; AoBPRRecommender.java:63)
 * Unknown names fail with LRK_ERR_INVALID. */
LRK_API int lrk_set_param(lrk_handle_t h, const char* name, double value);

/* model matrices beyond P / Q / biases, row-major doubles like lrk_set_factors (call after it):
 *   "svdpp.y"  impItemFactors, numItems x numFactors (SVDPlusPlusRecommender.java:55-56)
 *   "eals.confidences"  confidences, numItems doubles (EALSRecommender.java:50,65-83); needs only lrk_set_train_csr before it
 *   "jdk.random.state"  BPR in LRK_UPDATE_REFERENCE_ORDER only: 1 double, the 48-bit state of Randoms.r (java.util.Random.seed,
 *                       math/algorithm/Randoms.java:31) as an exact integer in [0, 2^48).  Set it before the first epoch and read it
 *                       after the last, so that the caller's generator continues where the epochs left it.  Defaults to
 *                       new Random(cfg.seed)'s scrambled seed; lrk_set_train_csr and lrk_set_factors leave it alone.  Any time,
 *                       no ordering with the other calls. */
LRK_API int lrk_set_matrix(lrk_handle_t h, const char* name, const double* values);
LRK_API int lrk_get_matrix(lrk_handle_t h, const char* name, double* values);

/* ---- training ----------------------------------------------------------------------- */
/* replaces ONE iteration of trainModel():
 *   BiasedMFRecommender.java:68-100, PMFSimilarityRecommender.java:59-90, BPRRecommender.java:48-93.
 * lr/reg_u/reg_i are the float fields of MatrixFactorizationRecommender.java:16,54,59; reg_b is the
 * double regBias (BiasedMFRecommender.java:36; ignored unless BIASEDMF).  epoch_idx is the 1-based
 * iteration number (selects the BPR sample stream; reference-order BPR continues its java.util.Random state instead).  *loss_out receives the epoch loss with the
 * reference's definition (0.5 * (sum e^2 + reg terms); BPR: sum -ln sigma(x) + reg terms, no 0.5),
 * so isConverged()/updateLRate() stay on the caller's side.  Returns LRK_ERR_DIVERGED (and still
 * writes *loss_out) when the loss is NaN/Inf. */
LRK_API int lrk_sgd_epoch(lrk_handle_t h, float lr, float reg_u, float reg_i, double reg_b,
                  int32_t epoch_idx, double* loss_out);
/* replaces n_epochs iterations of trainModel() in one call, for the configurations in which the Java loop takes no decision between
 * iterations: rec.recommender.earlystop=false and rec.learnrate.bolddriver=false (the shipped *-test.properties).  The learning
 * rate follows updateLRate's decay branch (MatrixFactorizationRecommender.java:131-138): lr *= decay when 0 < decay < 1, clamped to
 * max_lr when max_lr > 0, in float arithmetic.  losses_out[n_epochs] receives every epoch's loss (for the shim's log lines and its
 * NaN check); stops at the first epoch that fails and returns its status. */
LRK_API int lrk_sgd_epochs(lrk_handle_t h, int32_t n_epochs, float lr, float decay, float max_lr, float reg_u, float reg_i, double reg_b,
                   int32_t first_epoch_idx, double* losses_out);
/* staging statistics of the last lrk_set_train_csr: out[0] ratings staged, out[1] ratings staged as item-run tiles (32 ratings of
 * one item, csrc/staging.cuh), out[2] largest item degree, out[3] smallest item degree that forms runs */
LRK_API int lrk_stage_stats(lrk_handle_t h, int64_t out[4]);
/* debug / test aid: the staged COO stream of the SGD epoch (su / si / sr, nnz entries each; any pointer may be NULL) and, when the
 * stream is unit-ordered (csrc/staging_group.cuh), its unit table: units[4 * n] = {stream start, ratings, first user,
 * users | slices << 16} for n = *n_units_out units (0 for the shuffled item-run-tile stream).  Single GPU: item ids are global. */
LRK_API int lrk_debug_stream(lrk_handle_t h, int32_t* su, int32_t* si, float* sr, int32_t* units, int64_t max_units, int64_t* n_units_out);
/* device time of the last lrk_sgd_epoch kernel in milliseconds (CUDA events on its stream) */
LRK_API int lrk_last_epoch_ms(lrk_handle_t h, float* ms_out);
/* Safeguard of the fast (parallel) SGD modes.  The reference applies one rating at a time; here thousands are in
 * flight, which is a larger effective step for popular items.  Every epoch starts from a device snapshot of the
 * factors; a non-finite loss, or one above 10x the last accepted loss, rolls the epoch back and re-runs it with 4x
 * fewer ratings in flight (kept for the following epochs, relaxed by 2x after 8 good ones).  Only if that still
 * diverges does lrk_sgd_epoch return LRK_ERR_DIVERGED (AbstractRecommender.java:259-262).
 * conc_div = current divisor of the grid (1 = full concurrency), rollbacks = epochs re-run since creation. */
LRK_API int lrk_sgd_safeguard_state(lrk_handle_t h, int32_t* conc_div, int64_t* rollbacks);
/* number of kernels this handle has launched since creation */
LRK_API int lrk_launch_count(lrk_handle_t h, uint64_t* out);
/* debug / test aid: the (user, positive item, negative item) triples that BPR epoch `epoch_idx`
 * draws for samples [first, first+n) -- out is int32[3*n]; GBPR: int32[11*n] = {u, i, j, the group's users (8 slots, -1 padded)}.
 * BPR in LRK_UPDATE_REFERENCE_ORDER: samples [first, first+n) of the NEXT epoch, drawn from the current "jdk.random.state",
 * which the call does not advance (first + n may exceed numRates: the stream continues); epoch_idx is ignored. */
LRK_API int lrk_bpr_peek_samples(lrk_handle_t h, int32_t epoch_idx, int64_t first, int64_t n, int32_t* out);

/* ---- prediction --------------------------------------------------------------------- */
/* replaces predict(u,i) without bound: MatrixFactorizationRecommender.java:104-106 /
 * BiasedMFRecommender.java:118-120, fp64, summed f = 0..k-1 left to right like
 * math/structure/DenseVector.java:104-111.  Bit-exact for identical factors. */
LRK_API int lrk_predict_pairs(lrk_handle_t h, const int32_t* users, const int32_t* items, int64_t n, double* out);
/* replaces recommendRating(DataSet) + RMSE/MAE evaluators
 * (MatrixRecommender.java:211-248,272-284; eval/rating/RMSEEvaluator.java:33-69, MAEEvaluator.java:34-70):
 * bounded predictions for every test-CSR entry (pred_out may be NULL) and the two metrics. */
LRK_API int lrk_eval_rating(lrk_handle_t h, int32_t num_users, const int64_t* t_rowptr, const int32_t* t_col,
                    const double* t_val, double min_rate, double max_rate,
                    double* pred_out, double* rmse_out, double* mae_out);

/* ---- top-N ranking ------------------------------------------------------------------ */
/* replaces recommendRank(): MatrixRecommender.java:137-201 + util/Lists.java:416-468
 * (+ recommender/item/RecommendedList.java:85-88).  For each queried user (users == NULL means
 * users 0..nq-1) scores every item not in the user's train row (exclude_train != 0), drops NaN,
 * keeps the top `topn` with java.util.PriorityQueue + stable-sort tie semantics.
 * out_items / out_scores are [nq x topn] (unused slots: item -1, score 0), out_counts[nq]. */
LRK_API int lrk_topn(lrk_handle_t h, const int32_t* users, int32_t nq, int32_t topn, int32_t exclude_train,
             int32_t* out_items, double* out_scores, int32_t* out_counts);
/* replaces RecommenderJob's ranking evaluation (job/RecommenderJob.java:205-271 with rec.recommender.isranking=true):
 * recommendRank() for EVERY user with the train items excluded, then
 * eval/ranking/{AUC,AveragePrecision,NormalizedDCG,Precision,Recall,ReciprocalRank,Novelty,Entropy}Evaluator.java against the test
 * CSR (ground truth = test rows in CSR order, eval/EvalContext.java:75-88; numDropped = numItems - |train row|,
 * recommender/MatrixRecommender.java:110-113) while the lists are still on the device.
 * out_measures[8] = {AUC, AP, NDCG, Precision, Recall, RR, Novelty, Entropy} -- the default ranking measures of
 * eval/Measure.java:71-97; the three list outputs may be NULL.  1 <= topn <= 64. */
LRK_API int lrk_eval_ranking(lrk_handle_t h, int32_t topn, const int64_t* t_rowptr, const int32_t* t_col, const double* t_val,
                     int32_t* out_items, double* out_scores, int32_t* out_counts, double out_measures[8]);
/* statistics of the last lrk_topn call: users served by the tensor-core candidate path, users
 * that failed the exactness certificate and were re-done by the exact fp64 kernel, device ms */
LRK_API int lrk_topn_stats(lrk_handle_t h, int64_t* fast_users, int64_t* fallback_users, float* ms_out);
/* device time of the phases of the last tensor-core lrk_topn call, CUDA events on the handle's stream:
 * out[0] operand build, out[1] tcgen05 score sweep + fused selection (topn_tc_kernel), out[2] exact fp64
 * re-score + certificate (and the second sweep of rows whose margin was too thin), out[3] exact fallback for rows
 * still without a certificate.  out[4] is a self-check of the certificate: the largest observed
 * |fp16 sweep score - exact score| over all re-scored candidates divided by the error bound the certificate
 * assumes (must stay below 1).  out[5] = number of rows that went through the second sweep.
 * Zeros if the exact path ran. */
LRK_API int lrk_topn_phase_ms(lrk_handle_t h, float out[6]);

/* ---- measurement aid ------------------------------------------------------------------ */
/* L2 roofline probe of the SGD epoch kernels (no reference counterpart; bench.py's roofline.bound = "l2"): the epoch kernels gather
 * factor rows through L2 and apply vector reductions (red.global.add.v4.f32) to them on an L2-resident factor set, so what bounds
 * them is the L2's rate for exactly those two operations.  Runs them alone -- same instruction widths, rows of `row_floats` floats
 * (64 or 128), uniformly random rows of a working set of `working_set_bytes` -- and reports GB/s of row bytes through L2:
 * out_gbps[0] gathers only, [1] REDs only, [2] one RED per gather (the epoch kernel's mix). */
LRK_API int lrk_probe_l2(lrk_handle_t h, uint64_t working_set_bytes, int32_t row_floats, double out_gbps[3]);

/* ---- multi-GPU DSGD (one process per GPU; SURVEY.md 8e) ----------------------------- */
/* 128-byte NCCL unique id, created on rank 0 and broadcast by the host (torch.distributed / MPI / JVM) */
LRK_API int lrk_comm_unique_id(uint8_t out[128]);
/* joins the handle to a world of `world` ranks.  After this, lrk_set_train_csr expects the
 * rank's OWN user block (a CSR with the rank's users as rows 0..U_local-1 and GLOBAL item ids; every rank passes the same
 * num_items) and lrk_set_factors the rank's rows of P / userBiases together with the FULL Q / itemBiases (identical on every
 * rank).  lrk_get_factors returns the rank's user rows and the full item side gathered from the ring. */
LRK_API int lrk_comm_init(lrk_handle_t h, int32_t rank, int32_t world, const uint8_t unique_id[128]);

#ifdef __cplusplus
}
#endif
#endif /* LIBREC_B200_H */
