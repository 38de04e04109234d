/* libesac_b200.so -- C ABI of the B200-native ESAC differentiable-RANSAC hot path.
 *
 * Drop-in boundary for the reference's `esac` Python extension
 * (/root/reference/code/esac/esac.cpp:513-516: m.def("forward", &esac_forward), m.def("backward",
 * &esac_backward)).  esacb200_forward / esacb200_backward take exactly the arguments of
 * esac_forward (esac.cpp:64-77) / esac_backward (esac.cpp:213-230) with the at::Tensor arguments
 * flattened to pointer + sizes; everything else in this header is additive (context handling,
 * seeding, a scoring-only entry for measurement, read-back of intermediates for tests).
 *
 * Conventions
 *  - plain C types only, no exceptions across the boundary; every entry returns 0 on success or a
 *    negative esacb200_status, and esacb200_last_error(ctx) holds a message;
 *  - `coords`, `grads`, `assign`, `out_pose`, `gt_pose` may be HOST or DEVICE pointers (detected with
 *    cudaPointerGetAttributes); host buffers are copied on the context's stream (pinned memory gets
 *    full PCIe speed), device buffers are used in place;
 *  - calls are synchronous like the reference's (they return an int / a double), the work is enqueued
 *    on the stream set with esacb200_set_stream (default: a stream owned by the context);
 *  - there is NO CPU fallback: without a CUDA device esacb200_create fails.
 */
#ifndef ESAC_B200_H
#define ESAC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct esacb200_ctx esacb200_ctx;

typedef enum {
    ESACB200_OK = 0,
    ESACB200_ERR_CUDA = -1,       /* a CUDA runtime call failed */
    ESACB200_ERR_ARG = -2,        /* bad size / null pointer / expert index out of range */
    ESACB200_ERR_NO_DEVICE = -3   /* no usable CUDA device */
} esacb200_status;

/* ---- context -------------------------------------------------------------------------------- */
/* Replaces the reference's only persistent state, the static per-thread RNG
 * (thread_rand.cpp:4-5,13-30; default seeds 1305 + thread id). */
int esacb200_create(int device, esacb200_ctx** out);
void esacb200_destroy(esacb200_ctx* ctx);
const char* esacb200_last_error(const esacb200_ctx* ctx);
/* cudaStream_t to enqueue on (0 / NULL = the context's own stream). */
int esacb200_set_stream(esacb200_ctx* ctx, void* cuda_stream);
/* Seed of the minimal-set stream; also resets the call counter (each forward/backward call advances
 * it so successive calls draw fresh samples, as the reference's persistent generators do). */
int esacb200_set_seed(esacb200_ctx* ctx, uint64_t seed);
/* Options: "max_tries" (esac.cpp:44 MAX_SAMPLING_TRIES, default 1000000), "max_ref_steps"
 * (esac.cpp:45 MAX_REF_STEPS, default 100), "fixed_seed" (1: do not advance the call counter),
 * "refine_group" (CTAs per refinement job, 0 = automatic), "refine_jobs_per_group" (jobs a group
 * works through when many hypotheses are refined), "refine_profile", "sample_prefilter" (default 1; 0 sends every sampling
 * try through the exact fp64 path -- the results must not change, only the time), "hyp_offset" (global index of
 * local hypothesis 0 for the minimal-set stream; sharded runs), "score_ppt" / "score_hc" (scoring launch shape). */
int esacb200_set_option(esacb200_ctx* ctx, const char* key, double value);
/* Inject minimal sets instead of drawing them: cells int32 [M][T][4][2] (x, y), host pointer,
 * copied; T candidate sets per hypothesis tried in order.  NULL clears.  Applies to the next call. */
int esacb200_inject_cells(esacb200_ctx* ctx, const int32_t* cells, int M, int T);

/* ---- the reference's two entry points ------------------------------------------------------- */
/* esac_forward (esac.cpp:64-190).  coords float32 [E,3,H,W] contiguous; assign int64 [M] with element
 * stride `assign_stride` (0 for the reference's expert.expand() tensors, test_esac.py:173); out_pose
 * float32 [4,4] camera->world, written in place; *out_expert = winning expert index (the reference's
 * return value). */
int esacb200_forward(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                     int64_t assign_stride, int M, float* out_pose, int shiftX, int shiftY, float focalLength,
                     float ppointX, float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta,
                     float maxReproj, int subSampling, int* out_expert);

/* esac_backward (esac.cpp:213-511).  grads float32 [E,3,H,W] is ACCUMULATED in place (+=, esac.cpp:501-506);
 * gt_pose float32 [4,4] camera->world; *out_loss = expected pose loss (the reference's return value). */
int esacb200_backward(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W,
                      const int64_t* assign, int64_t assign_stride, int M, const float* gt_pose, float wLossRot,
                      float wLossTrans, float lossCut, int shiftX, int shiftY, float focalLength, float ppointX,
                      float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta, float maxReproj,
                      int subSampling, double* out_loss);

/* ---- additive entry points ------------------------------------------------------------------ */
/* esac_backward over hypotheses sharded across processes (one per GPU; experts expert-major, so gradient slices are
 * disjoint).  The path has two exchange steps (SURVEY.md 8e); the library calls `exchange` on the host at each:
 *   phase 1: values = {local max score, local sum exp(score - local max)}  -> replace by the GLOBAL {max, sum exp(score - max)}
 *   phase 2: values = {local sum_h p_h loss_h}                               -> replace by the sum over all ranks
 * (return 0 on success).  The caller implements them with its collective of choice (esac_b200/sharded.py: NCCL
 * all-gather / all-reduce through torch.distributed).  *out_loss = the global expected loss.  Set option "hyp_offset" to
 * the global index of this shard's first hypothesis so that the shards draw the minimal sets of the unsharded problem. */
typedef int (*esacb200_exchange_fn)(void* user, int phase, double* values, int n);
int esacb200_backward_sharded(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W,
                              const int64_t* assign, int64_t assign_stride, int M, const float* gt_pose, float wLossRot,
                              float wLossTrans, float lossCut, int shiftX, int shiftY, float focalLength, float ppointX,
                              float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta, float maxReproj,
                              int subSampling, esacb200_exchange_fn exchange, void* user, double* out_loss);

/* The local half of a sharded esac_forward, enqueued WITHOUT a host synchronisation: runs sample -> score -> select ->
 * refine on this shard's experts / hypotheses and writes the record the shards exchange,
 *   pack_out[0..M_pad)      soft-inlier scores (esac.cpp:147-150); entries >= M are -inf (shards may hold different numbers
 *                           of hypotheses, the records of a collective must have one size: M_pad = the largest M),
 *   pack_out[M_pad..+16)    camera pose of the local winner,
 *   pack_out[M_pad+16]      expert_offset + its expert (or -1 if hypAssignment held an index outside [0,E)),
 *   pack_out[M_pad+17]      its local hypothesis index,        pack_out[M_pad+18]  M,
 *   pack_out[M_pad+19/20]   options "hyp_offset" / "hyp_stride": local hypothesis k is hypothesis offset + k * stride of the
 *                           unsharded problem (its minimal-set stream and its place in draw()'s first-maximum order),
 * as doubles into DEVICE memory, stream-ordered on the context's stream.  coords / assign must be device pointers (a host
 * buffer would force the synchronisation this entry exists to avoid).  M may be 0 (coords / assign are then ignored).
 * The record has M_pad + 21 doubles. */
int esacb200_forward_pack(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                          int64_t assign_stride, int M, int M_pad, int shiftX, int shiftY, float focalLength, float ppointX,
                          float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta, float maxReproj,
                          int subSampling, int expert_offset, double* pack_out);

/* ---- sharded entry points over NCCL (one process per GPU) ------------------------------------------------------------
 * The path has ONE exchange in forward (scores -> softMax / draw, esac.cpp:153-155) and TWO in backward (softmax
 * normalisation; the expectation sum_h p_h loss_h, esac.cpp:357-362, esac_derivative.h:372-374); SURVEY.md 8e.  The library
 * issues them itself as NCCL collectives on the context's stream.  NCCL is resolved at run time (dlopen of libnccl.so.2, the
 * copy the process already holds if any), so the library still loads where NCCL is absent.
 * esacb200_nccl_unique_id: 128-byte ncclUniqueId (rank 0 creates it, the caller distributes it by any means).
 * esacb200_comm_init:     ncclCommInitRank on the context's device; collective over all ranks. */
int esacb200_nccl_unique_id(void* out128);
int esacb200_comm_init(esacb200_ctx* ctx, int world, int rank, const void* id128);
int esacb200_comm_destroy(esacb200_ctx* ctx);
/* esac_forward over all shards: local pipeline -> record -> one ncclAllGather -> softMax / draw over the records on the device
 * (first strict maximum in rank-major order) -> one 80-byte read-back.  Every rank receives the global winner's camera pose
 * and (global) expert index.  coords / assign host or device pointers; M may be 0; M_pad = max M over the ranks. */
int esacb200_forward_sharded(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                             int64_t assign_stride, int M, int M_pad, float* out_pose, int shiftX, int shiftY, float focalLength,
                             float ppointX, float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta,
                             float maxReproj, int subSampling, int expert_offset, int* out_expert);
/* esac_backward over all shards (gradient slices are disjoint when experts are dealt expert-major: no gradient collective):
 * all-gather of (max score, sum exp) -> global probabilities; all-reduce of the partial expectations -> *out_loss = the
 * global expected loss on every rank.  Option "hyp_offset" as for esacb200_backward_sharded.  M may be 0.
 * reduce_grads != 0: HYPOTHESIS-major sharding -- every rank holds all E planes and a slice of the hypotheses (the refinement
 * of the contributing hypotheses then shards too, which expert-major dealing cannot do when the gating concentrates them on
 * one expert); gradient slices overlap, so the local gradients are summed over the ranks with one ncclAllReduce of E*3*H*W
 * floats and the sum is added to `grads` on every rank (grads stays "+=", esac.cpp:501-506). */
int esacb200_backward_sharded_nccl(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W,
                                   const int64_t* assign, int64_t assign_stride, int M, const float* gt_pose, float wLossRot,
                                   float wLossTrans, float lossCut, int shiftX, int shiftY, float focalLength, float ppointX,
                                   float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta, float maxReproj,
                                   int subSampling, int reduce_grads, double* out_loss);

/* esac_forward over B images of one shape (the reference's callers loop with batch_size=1, test_esac.py:137):
 * coords float32 [B,E,3,H,W], assign int64 [B,M] (rows contiguous, element stride assign_stride; 0 = one expert for all),
 * out_poses float32 [B,4,4], out_experts int [B] (host).  One host synchronisation for the whole batch; host maps are
 * double-buffered and copied on a second stream, overlapping the previous image's kernels. */
int esacb200_forward_batch(esacb200_ctx* ctx, int B, const float* coords, int E, int H, int W, const int64_t* assign,
                           int64_t assign_stride, int M, float* out_poses, int shiftX, int shiftY, float focalLength,
                           float ppointX, float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta,
                           float maxReproj, int subSampling, int* out_experts);

/* esac_backward over B images of one shape (the reference trains with batch_size=1, train_esac.py:96-100, one
 * esac.backward per image): coords / grads float32 [B,E,3,H,W] (grads accumulated in place, as esac.cpp:490-508),
 * assign int64 [B,M] (as in esacb200_forward_batch), gt_poses float32 [B,4,4] (camera->world), shiftX / shiftY int [B]
 * on the host or NULL (= 0: the per-image random shift of train_esac.py:125), out_losses host double [B].
 * Image b draws the minimal sets that the b-th of B consecutive esacb200_backward calls on this context would draw, so
 * the batch returns exactly what that loop returns; images are spread over option "batch_workers" (default 8) internal
 * streams, each with its own workspace and host thread, so their kernels and the per-image host synchronisations overlap. */
int esacb200_backward_batch(esacb200_ctx* ctx, int B, const float* coords, float* grads, int E, int H, int W,
                            const int64_t* assign, int64_t assign_stride, int M, const float* gt_poses, float wLossRot,
                            float wLossTrans, float lossCut, const int* shiftX, const int* shiftY, float focalLength,
                            float ppointX, float ppointY, float inlierThreshold, float inlierAlpha, float inlierBeta,
                            float maxReproj, int subSampling, double* out_losses);

/* Hypothesis assignment on the device, the three host steps the reference's callers run before esac.forward/backward:
 * util.clamp_probs (util.py:38-48; keep_top < 0 = off), torch.multinomial(probs, M, replacement=True)
 * (train_esac.py:133-137, test_esac.py:169-174; single_expert != 0 = one draw expanded to M, the "expertselection" mode)
 * and torch.histc over the experts (train_esac.py:140).  weights float32 [B,E] >= 0 (host or device, not necessarily
 * normalised), out_assign int64 [B,M], out_hist float32 [B,E] or NULL (both host or device).  The draws are a pure
 * function of (seed, image, hypothesis).  Negative / non-finite weights or an all-zero row are an error, as in torch. */
int esacb200_assign_hypotheses(esacb200_ctx* ctx, int B, int E, int M, const float* weights, int keep_top,
                               int single_expert, uint64_t seed, int64_t* out_assign, float* out_hist);

/* Robust reprojection loss of the expert refinement stage and its gradient, one fused pass (ref_expert.py:103-146, where
 * it is six elementwise torch ops + autograd): coords float32 [B,3,H,W] (one expert's prediction per image; the reference
 * has B = 1), grads float32 [B,3,H,W] or NULL = d loss_b / d coords (overwritten, not accumulated), gt_poses float32
 * [B,4,4] camera->world (inverted here, ref_expert.py:127), shiftX / shiftY host int [B] or NULL (padX / padY, :110-111),
 * target pixel of cell (x,y) = (x*sub + sub/2 - padX, y*sub + sub/2 - padY) with real-valued sub/2 (:84-89),
 * depth clamped from below at minDepth (0.1, :136), error clamped to [0, maxReproj] (100, :142), square-root loss above
 * cutLoss (:144-146), mean over the H*W cells (:148).  out_losses host double [B].  fp32 arithmetic like the original. */
int esacb200_reproj_loss(esacb200_ctx* ctx, int B, const float* coords, float* grads, int H, int W, const float* gt_poses,
                         const int* shiftX, const int* shiftY, float focalLength, float ppointX, float ppointY,
                         int subSampling, float cutLoss, float maxReproj, float minDepth, double* out_losses);

/* Scene-coordinate loss of the expert initialisation stage and its gradient, one fused pass (init_expert.py:112-132,
 * where it is about ten torch ops, two of them boolean-mask gathers, + autograd): pred float32 [B,3,pred_H,pred_W] and gt
 * float32 [B,3,gt_H,gt_W], each contiguous at its own size; like util.assert_size both are cropped top-left to
 * (min H, min W) (strides, no copy) and sizes that differ by more than 1 in either direction are an error.  A cell is valid
 * where any gt component is nonzero (NaN included); d = ||pred - gt||; per image
 *   out_sums[b]   = sum over valid cells of (d <= cutLoss ? d : sqrt(cutLoss * d))   (NaN d in neither branch)
 *   out_counts[b] = number of valid cells (NaN d included)
 * so init_expert.py's loss is out_sums[b] / out_counts[b] (NaN for an image without valid cells, as 0/0.0 in the reference).
 * grads float32 [B,3,pred_H,pred_W] or NULL = d out_sums[b] / d pred -- the gradient of the SUM, not of the mean: scale by
 * 1/out_counts[b] (overwritten, not accumulated; 0 for invalid and cropped-away cells and where d == 0, NaN where d is
 * NaN).  out_sums host double [B], out_counts host int64 [B].  fp32 cell arithmetic like the original, fp64 sums in a
 * fixed order: repeated calls are bit-identical. */
int esacb200_init_loss(esacb200_ctx* ctx, int B, const float* pred, int pred_H, int pred_W, const float* gt, int gt_H,
                       int gt_W, float* grads, float cutLoss, double* out_sums, int64_t* out_counts);

/* Soft-inlier scores of given poses (getReproErrs + getHypScores, esac_util.h:235-363) without
 * sampling/selection/refinement: poses6 = host double [M][6] (rvec, tvec); out_scores host double [M]. */
int esacb200_score_poses(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                         int64_t assign_stride, int M, const double* poses6, int shiftX, int shiftY,
                         float focalLength, float ppointX, float ppointY, float inlierThreshold, float inlierAlpha,
                         float inlierBeta, float maxReproj, int subSampling, double* out_scores);

/* Refine given poses (refineHyp, esac_util.h:378-454): poses6 in/out host double [M][6]; out_rounds
 * host int [M] accepted rounds; out_inliers host int [M] size of the final inlier set (may be NULL). */
int esacb200_refine_poses(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                          int64_t assign_stride, int M, double* poses6, int shiftX, int shiftY, float focalLength,
                          float ppointX, float ppointY, float inlierThreshold, float maxReproj, int subSampling,
                          int* out_rounds, int* out_inliers);

typedef struct {
    int M;
    int winner;            /* hypothesis index selected by draw() */
    int n_contrib;         /* hypotheses with p >= PROB_THRESH */
    int refine_rounds;     /* accepted refinement rounds of the winner (forward) */
    double entropy;        /* esac_util.h:489-497 */
    double expected_loss;  /* backward only */
    /* device time of the last call's stages in milliseconds (CUDA events on the launching stream) */
    float ms_h2d, ms_prep, ms_sample, ms_score, ms_select, ms_refine, ms_backward, ms_total;
    int score_launches;    /* launches of the scoring kernel in the last call */
    int kernel_launches;   /* all kernel launches of the last call */
    int score_ppt, score_grid, refine_group;
} esacb200_stats;
int esacb200_get_stats(esacb200_ctx* ctx, esacb200_stats* out);

/* Diagnostics: with option "refine_profile" = 1 block 0 of the refinement kernel accumulates clock64() cycles per phase of
 * an LM evaluation of the root block: [0] produce + receive the command (Rodrigues of the new parameters), [1] pass over
 * the cells, [2] block reduction + slot write + change of variables, [3] wait for the group's epoch flags, [4] slot
 * summation, [5] map the sums to (rvec, tvec), [6] accept / reject + LM step; [8] = number of evaluations.
 * out16: host long long [16]. */
int esacb200_get_refine_profile(esacb200_ctx* ctx, long long* out16);

/* Diagnostics of the last call's sampling stage (summed over its lanes): [0] tries that went through the float prefilter,
 * [1] survivors the fp64 path judged, [2] waves that had work (max over lanes), [3] hypotheses left to the tail kernel,
 * [4] accepted tries staged, [5] lanes.  out8: host long long [8]. */
int esacb200_get_sample_profile(esacb200_ctx* ctx, long long* out8);
/* With option "sample_trace" = 1 the prefilter / exact kernels of the sampling waves stamp %globaltimer: out512 (host uint64
 * [4 lanes][32 waves][2 kernels: prefilter, exact][2: first CTA start, last CTA end], ns; start = ~0 where nothing ran). */
int esacb200_get_sample_trace(esacb200_ctx* ctx, unsigned long long* out512);

/* Read back intermediates of the last forward/backward call (any pointer may be NULL):
 * poses6 double [M][6] initial hypotheses, cells int32 [M][4][2], tries int32 [M], scores / probs double [M],
 * refined6 double [M][6] (backward: refined poses; forward: only the winner's row is meaningful),
 * losses double [M] (backward). */
int esacb200_get_hypotheses(esacb200_ctx* ctx, double* poses6, int32_t* cells, int32_t* tries, double* scores,
                            double* probs, double* refined6, double* losses);

/* Copies the last call's scores (double [M]) to `dst` (host or device pointer), stream-ordered on the
 * context's stream; used by the multi-GPU path to feed its all-gather without a host round trip. */
int esacb200_copy_last_scores(esacb200_ctx* ctx, double* dst, int M);

/* Device properties the bench needs without importing a CUDA binding: SM count and name. */
int esacb200_device_info(esacb200_ctx* ctx, int* sm_count, char* name, int name_len);

#ifdef __cplusplus
}
#endif
#endif /* ESAC_B200_H */
