// Internal declarations shared by the translation units of libesac_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "esac_geom.cuh"

namespace esacb200 {

#ifdef __CUDACC__
// Warp reduce-scatter of NV <= 32 doubles per lane: lane L returns the warp total of value L (0 for L >= NV).
// A transposing butterfly: 31 double shuffles instead of 5*NV.
template <int NV>
__device__ __forceinline__ double warp_reduce_scatter(const double (&v)[NV]) {
    static_assert(NV <= 32, "at most 32 values");
    const int lane = threadIdx.x & 31;
    double w[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) w[i] = i < NV ? v[i] : 0.0;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const bool up = (lane & o) != 0;
#pragma unroll
        for (int i = 0; i < o; ++i) {
            const double keep = up ? w[i + o] : w[i];
            const double send = up ? w[i] : w[i + o];
            w[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
    }
    return w[0];
}
#endif

// Per-call problem description (esac.cpp:64-77 arguments + tensor sizes).
struct Problem {
    int E, H, W, N, M;
    int shiftX, shiftY, sub;
    float f, ppx, ppy;
    float tau, alpha, beta, max_reproj;
};

// Hypotheses of one expert are contiguous in "sorted slot" order (stable by hypothesis index);
// a chunk is <= kMaxChunk consecutive slots of one expert: the unit the scoring kernel pairs with a
// pixel tile.
constexpr int kMaxChunk = 64;
struct ChunkDesc {
    int expert;
    int slot0;
    int count;
    int pad;
};

// Folded fp32 pose for the scoring kernel: rows [A_r0 A_r1 A_r2 | b_r] of diag(f,f,1)*R and
// diag(f,f,1)*(R*c + t); FFMA2 broadcasts a scalar register operand to both f32x2 lanes.
struct PosePk {
    float4 v[3];
};

struct ScoreArgs {
    const float* coords;     // [E,3,N]
    const float* centres;    // [E,3]
    const PosePk* poses;     // [M] sorted slots
    const ChunkDesc* chunks;
    const int* n_chunks;     // device scalar
    int* work_counter;       // device scalar, zeroed by the prep kernel
    float* part;             // [M, T] partial soft-inlier sums (slot-major)
    Problem P;
    int T;                   // pixel tiles per plane
    int hc;                  // hypotheses per chunk used when building the chunk table
    float k1, k0;            // beta*log2(e), -beta*tau*log2(e)
    int vec_ok;              // planes are 16-byte aligned and N % 4 == 0
};

// --- score.cu -----------------------------------------------------------------------------
// prep: int64 strided assignment -> int32, per-expert histogram / offsets / stable permutation,
// chunk table, work counter reset, plane centres.  flags[0] != 0 on a bad expert index.
void launch_prep(const float* coords, const long long* assign, long long assign_stride, const Problem& P, int hc,
                 int* assign32, int* counts, int* offsets, int* perm, int* slot_of, ChunkDesc* chunks, int* n_chunks,
                 int* work_counter, float* centres, int* flags, int roles, cudaStream_t st);
void launch_fold(const Pose* poses, const int* perm, const int* assign32, const float* centres, const Problem& P,
                 PosePk* out, cudaStream_t st);
int score_tile_pixels(int ppt);
void launch_score(const ScoreArgs& a, int ppt, int grid, cudaStream_t st);
// scores[h] = (alpha/W/H) * sum_tiles part ; softmax ; entropy ; argmax ; contributing list
void launch_select(const float* part, const int* slot_of, const Problem& P, int T, double* scores, double* probs,
                   double* stats /* [0]=entropy [1]=winner [2]=n_contrib */, int* winner, int* contrib,
                   int* n_contrib, cudaStream_t st);

void launch_rescale_probs(const double* scores, const Problem& P, double gmax, double gsum, double* probs, int* contrib,
                          int* n_contrib, cudaStream_t st);
void launch_rescale_probs_gathered(const double* scores, const Problem& P, const double* pairs, int world, double* norm_out,
                                   double* probs, int* contrib, int* n_contrib, cudaStream_t st);

// --- hyp.cu -------------------------------------------------------------------------------
// Work state of the sampling waves (all device memory, M = hypotheses).
struct Accepted {
    Pose pose;
    int cells[8];
};
struct SampleState {
    unsigned long long* best;  // [M] (lowest accepted try << 32) | staging slot; ~0 = none yet
    Accepted* stage;           // [cap_acc] poses of accepted tries
    int cap_acc;
    int* base;      // [M] first try not judged yet
    int* ovf;       // [M] lowest survivor that did not fit the list in the current wave
    int* list;      // [2M] unresolved hypotheses (second half: scratch for rebuilding)
    int2* surv;     // [cap] (hypothesis, try) pairs that passed the float prefilter
    int cap;
    int* counters;  // [0] unresolved, [1] survivors, [2] staged accepts, [3] span of the current wave, [4] ticket,
                    // diagnostics: [5] tries prefiltered, [6] survivors judged, [7] waves that had work
    int M;
};
// Returns the number of kernel launches it enqueued.
int launch_sample(const float* coords, float4* coords4, const int* assign32, const Problem& P, uint64_t seed, int max_tries,
                  const int* injected, int inj_T, const SampleState* st, int n_lanes, int sm_count, int use_prefilter,
                  int hyp_offset, int hyp_stride, Pose* poses, int* cells, int* tries, const cudaStream_t* lanes,
                  cudaEvent_t ev_fork, const cudaEvent_t* ev_join, int split_e, const int* perm, const int* offsets,
                  const cudaEvent_t* ev_half, int span0, float window, int n_waves,
                  unsigned long long* trace, float tail_boost);
void launch_trace_init(unsigned long long* trace, int slots, cudaStream_t st);

// --- refine.cu ----------------------------------------------------------------------------
// Refines poses_in[jobs[j]] -> poses_out[jobs[j]] for j < *n_jobs (device scalar) or n_jobs_host.
// masks: [job][ceil(N/32)] final inlier bit masks (may be null), rounds: [job] accepted rounds.
struct RefineArgs {
    const float* coords;
    const float* centres;    // [E,3] plane centres (prep kernel)
    const int* assign32;
    const Pose* poses_in;
    Pose* poses_out;
    const int* jobs;
    const int* n_jobs;       // device scalar (null -> n_jobs_host)
    int n_jobs_host;
    uint32_t* masks;
    int mask_words;          // words per job
    int* rounds;
    double* scratch;         // cross-CTA reduction slots
    unsigned int* barrier;   // per group: one epoch flag per block + the root's command flag, zeroed before launch
    int* job_counter;        // next job to hand out (dynamic scheduling), zeroed before launch
    int group;               // CTAs cooperating on one job
    int cache;               // 1: every CTA's share of the map fits the shared-memory cell cache
    int compact;             // 1: LM evaluations walk a per-CTA list of the round's inlier cells
    int pretest;             // 1: the inlier selection classifies clear cases in fp32 (error-bounded), exact arithmetic for the rest
    unsigned short* clist;   // [n_groups][words * 32] inlier lists of blocks whose share does not fit shared memory (or null)
    long long* prof;         // diagnostics: 16 cycle counters of block 0 (null = off)
    Problem P;
    int max_ref_steps;
};
void launch_refine(const RefineArgs& a, int n_groups, cudaStream_t st);
int refine_max_coresident_blocks(int sm_count);
int refine_cache_words();
int refine_max_compact_words();
size_t refine_scratch_doubles(int n_groups, int group);
size_t refine_flag_words(int n_groups, int group);
// camera->world 4x4 float of poses[*winner] packed for one D2H copy: out[0..15], out[16] = expert id,
// out[17] = bad-assignment flag, out[18] = winning hypothesis
void launch_finish_forward(const Pose* poses, const int* winner, const int* assign32, const int* flags, float* out20,
                           cudaStream_t st);

void launch_pack_forward(const double* scores, const float* out20, int M, int M_pad, int expert_offset, int hyp_offset, int hyp_stride,
                         double* pack, cudaStream_t st);
constexpr int kPackTail = 21;  // doubles behind the M_pad scores of a shard's record
void launch_select_gathered(const double* gathered, int world, int M_pad, float* out20, cudaStream_t st);

// --- gating.cu ----------------------------------------------------------------------------
int assign_max_experts();
void launch_assign(const float* weights, int B, int E, int M, int keep_top, int single, uint64_t seed, int64_t* out_assign,
                   float* out_hist, int* flags, cudaStream_t stream);

// --- reproj.cu ----------------------------------------------------------------------------
int reproj_blocks_per_image(int N, int B, int sm_count);
// img: per image 16 floats = world->camera 3x4 (row major), padX, padY, 2 unused.  partial: B * blocks_per_image doubles,
// tickets: B zeroed counters (left zeroed), losses: B doubles.  grads may be null (loss only).
void launch_reproj(const float* coords, float* grads, const float* img, int B, int N, int W, float sub, float f, float cx,
                   float cy, float cut, float max_err, float min_depth, int blocks_per_image, double* partial,
                   unsigned* tickets, double* losses, cudaStream_t stream);

// --- initloss.cu --------------------------------------------------------------------------
int init_loss_blocks_per_image(int N);
// pred / grads [B,3,pH,pW], gt [B,3,gH,gW] (|pH-gH|, |pW-gW| <= 1; the common top-left region counts), grads may be null.
// partial_sum / partial_cnt: B * blocks_per_image each, tickets: B zeroed counters (left zeroed), sums / counts: B each.
void launch_init_loss(const float* pred, const float* gt, float* grads, int B, int pH, int pW, int gH, int gW, float cut,
                      int blocks_per_image, double* partial_sum, unsigned* partial_cnt, unsigned* tickets, double* sums,
                      long long* counts, cudaStream_t stream);

// --- bwd.cu -------------------------------------------------------------------------------
struct BwdArgs {
    const float* coords;
    float* grads;            // [E,3,N] accumulated in place
    const int* assign32;
    const int* perm;         // slot -> hyp
    const int* counts;
    const int* offsets;
    const Pose* init;        // [M]
    const Pose* ref;         // [M] (== init for non-contributing)
    const int* cells;        // [M,4,2]
    const double* probs;     // [M]
    const int* contrib;      // contributing hypothesis ids (ascending)
    const int* n_contrib;    // device scalar
    const int* job_of;       // [M] hypothesis -> job index (or -1)
    const uint32_t* masks;
    int mask_words;
    const int* rounds;       // [job]
    double* losses;          // [M]
    double* out_loss;        // device scalar: expected loss
    double* red;             // [job][tiles][kRedVals] partial reductions
    void* hyp_grad;          // [job] HypGrad records
    float gt[16];
    float wRot, wTrans, cut;
    Problem P;
    const double* expected_override;  // device scalar: global expected loss (multi-GPU), or null
};
void launch_backward(const BwdArgs& a, int max_jobs, cudaStream_t st);
// phase split for the multi-GPU path: losses + local expectation only / everything after the loss exchange
void launch_backward_losses(const BwdArgs& a, cudaStream_t st);
void launch_add_inplace(float* dst, const float* src, size_t n, cudaStream_t st);
void launch_expert_flags(const int* contrib, const int* n_contrib, const int* assign32, int E, int* flags, cudaStream_t st);
size_t bwd_hypgrad_bytes();
int bwd_red_vals();
int bwd_tiles(int N);

}  // namespace esacb200
