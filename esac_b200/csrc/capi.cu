// Host side of libesac_b200.so: context, workspace, stage orchestration, the C ABI of include/esac_b200.h.
//
// Orchestration follows esac_forward (esac.cpp:64-190) and esac_backward (esac.cpp:213-511) stage by
// stage; every stage is a CUDA kernel launched on one stream with no host round trip until the final
// 68-byte (forward) / 8-byte (backward) result copy.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <exception>
#include <new>
#include <vector>
#include <thread>
#include <chrono>

#include "../../include/esac_b200.h"
#include "../../include/esac_b200_testhooks.h"
#include "esac_internal.h"
#include "esac_p3p_fast.cuh"
#include "esac_rng.cuh"

using namespace esacb200;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const { return (T*)p; }
};

enum { EV_START = 0, EV_H2D, EV_PREP, EV_SAMPLE, EV_FOLD, EV_SCORE, EV_SELECT, EV_REFINE, EV_BWD, EV_END, EV_COUNT };

}  // namespace

struct esacb200_ctx {
    int device = 0;
    int sm_count = 0;
    char dev_name[128] = {0};
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaStream_t aux_stream = nullptr;   // second lane of the sampling stage
    cudaStream_t aux_more[2] = {nullptr, nullptr};  // third and fourth lane (option sample_groups; no gain measured)
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_join_more[2] = {nullptr, nullptr};
    int sample_groups = 2;
    int upload_split = 1;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
    cudaStream_t stream = nullptr;
    uint64_t seed = 1305;  // thread_rand.h:103
    uint64_t calls = 0;
    int max_tries = 1000000;
    int max_ref_steps = 100;
    int fixed_seed = 0;
    int refine_group_opt = 0;
    int* h_flags = nullptr;    // pinned: per-expert "receives gradient on some rank" flags (hypothesis-major sharding)
    int h_flags_cap = 0;
    int refine_pretest = 1;    // inlier selection: float pretest with a rounding-error bound, exact arithmetic only where in doubt
    int refine_compact = 1;    // LM evaluations over per-CTA inlier lists instead of predicated passes over all cells
    int refine_profile = 0;    // 1: block 0 of the refinement kernel records phase cycle counts (esacb200_get_refine_profile)
    int refine_jobs_per_group = 3;
    int sample_prefilter = 1;
    int sample_span0 = 256;       // tries per hypothesis in the first wave (a multiple of the 256-try pass of a prefilter CTA)
    float sample_window = 1.25f;  // later waves: window / acceptance rate
    int sample_waves = 6;         // launched unconditionally (empty ones cost ~6 us each); what is left after them goes to tail_kernel
    float sample_tail_boost = 1.f;  // window factor once <= 64 hypotheses are left in a lane (x2 more for <= 8)
    int sample_trace = 0;         // 1: prefilter / exact kernels stamp first-CTA-start / last-CTA-end times (esacb200_get_sample_trace)
    int smp_groups_last = 0;      // lanes of the last run_sample (diagnostics read-back)
    int smp_Mg_last = 0;
    int hyp_offset = 0, hyp_stride = 1;
    int score_ppt_opt = 0, score_hc_opt = 0;
    int refine_coresident = 0;
    char err[512] = {0};
    // workspace
    DevBuf coords, grads, assign64, assign32, counts, offsets, perm, slot_of, chunks, scalars, centres, poses, poses_ref,
        cells, tries, posepk, part, scores, probs, stats, contrib, masks, rounds, scratch, barrier, out17, inject,
        losses, red, hypgrad, job_of, gt, smp_int, smp_surv, smp_trace, clist, eflags, coords4, coords_alt, assign64_alt, out_batch, prof;
    float* h_out = nullptr;  // pinned staging: 32 floats
    double* h_dbl = nullptr; // pinned staging: 8 doubles
    int inj_M = 0, inj_T = 0;
    cudaEvent_t ev[EV_COUNT] = {nullptr};
    bool ev_used[EV_COUNT] = {false};
    esacb200_stats st;
    int last_M = 0;
    bool last_backward = false;
    int batch_workers = 8;
    // NCCL communicator of the sharded entry points (esacb200_comm_init); the library is resolved at run time with dlopen
    void* nccl_comm = nullptr;
    int comm_world = 1, comm_rank = 0;
    DevBuf gathered, grads_work;
    std::vector<esacb200_ctx*> workers;  // lazily created contexts of esacb200_backward_batch (own stream + workspace each)
};

namespace {

// Every entry point works on the context's device and leaves the caller's current device as it found it (torch reads the
// current device with cudaGetDevice: a library that silently switches it redirects the caller's later allocations).
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; }
        if (prev != device) cudaSetDevice(device);
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};

// ---- NCCL, resolved at run time ---------------------------------------------------------------------------------
// The library must load on machines without NCCL (the CPU test box) and must share the NCCL instance the host process already
// holds (torch bundles its own libnccl.so.2): no link-time dependency, dlopen of the soname instead -- RTLD_NOLOAD first, so an
// already loaded copy is reused.  Only the five entry points below are needed; their prototypes are NCCL's public ABI.
struct NcclApi {
    typedef struct { char internal[128]; } UniqueId;
    int (*GetUniqueId)(UniqueId*) = nullptr;
    int (*CommInitRank)(void**, int, UniqueId, int) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
};
constexpr int kNcclFloat32 = 7;  // ncclFloat
constexpr int kNcclFloat64 = 8;  // ncclDouble
constexpr int kNcclSum = 0;      // ncclSum
constexpr int kNcclInt32 = 2;    // ncclInt32
constexpr int kNcclMax = 2;      // ncclMax

NcclApi& nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api;
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return api;
    api.GetUniqueId = (int (*)(NcclApi::UniqueId*))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (int (*)(void**, int, NcclApi::UniqueId, int))dlsym(h, "ncclCommInitRank");
    api.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
    api.AllGather = (int (*)(const void*, void*, size_t, int, void*, cudaStream_t))dlsym(h, "ncclAllGather");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
    api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllGather && api.AllReduce;
    return api;
}

int fail(esacb200_ctx* c, int code, const char* fmt, ...);
#define CKN(call)                                                                                              \
    do {                                                                                                       \
        int r__ = (call);                                                                                      \
        if (r__ != 0)                                                                                          \
            return fail(ctx, ESACB200_ERR_CUDA, "%s failed: %s (%s:%d)", #call,                                \
                        nccl_api().GetErrorString ? nccl_api().GetErrorString(r__) : "NCCL error", __FILE__, __LINE__); \
    } while (0)

int fail(esacb200_ctx* c, int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(c->err, sizeof(c->err), fmt, ap);
    va_end(ap);
    return code;
}

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess)                                                                           \
            return fail(ctx, ESACB200_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
                        __FILE__, __LINE__);                                                              \
    } while (0)

bool is_device_ptr(const void* p) {
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

void mark(esacb200_ctx* c, int id) {
    cudaEventRecord(c->ev[id], c->stream);
    c->ev_used[id] = true;
}

float span(esacb200_ctx* c, int a, int b) {
    if (!c->ev_used[a] || !c->ev_used[b]) return 0.f;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev[a], c->ev[b]) != cudaSuccess) {
        cudaGetLastError();
        return 0.f;
    }
    return ms;
}

// scalars buffer layout (ints): [0]=n_chunks [1]=work_counter [2]=flags [3]=winner [4]=n_contrib
enum { S_NCHUNKS = 0, S_WORK, S_FLAGS, S_WINNER, S_NCONTRIB, S_COUNT = 16 };

struct Plan {
    Problem P;
    int T, ppt, hc, grid, vec_ok;
    const float* d_coords;
    const long long* d_assign;
    long long assign_stride;
    int split_e = 0;  // > 0: host maps are uploaded in two halves [0, split_e) / [split_e, E) on the copy stream (ev_copied[0/1])
};

int fill_problem(esacb200_ctx* ctx, Problem& P, int E, int H, int W, int M, int shiftX, int shiftY, float f, float ppx,
                 float ppy, float tau, float alpha, float beta, float maxReproj, int sub) {
    if (E <= 0 || H <= 0 || W <= 0 || M <= 0) return fail(ctx, ESACB200_ERR_ARG, "empty tensor (E=%d H=%d W=%d M=%d)", E, H, W, M);
    if ((long long)H * W > (1ll << 30)) return fail(ctx, ESACB200_ERR_ARG, "coordinate map too large");
    P.E = E; P.H = H; P.W = W; P.N = H * W; P.M = M;
    P.shiftX = shiftX; P.shiftY = shiftY; P.sub = sub;
    P.f = f; P.ppx = ppx; P.ppy = ppy; P.tau = tau; P.alpha = alpha; P.beta = beta; P.max_reproj = maxReproj;
    return 0;
}

// Upload (or alias) the inputs.  Host coordinate maps go to `cbuf` on `copy_stream` (pinned memory: asynchronous).
int upload_inputs(esacb200_ctx* ctx, Plan& pl, const float* coords, const int64_t* assign, int64_t stride, DevBuf& cbuf,
                  DevBuf& abuf, cudaStream_t copy_stream, bool allow_split = false) {
    const Problem& P = pl.P;
    const size_t cbytes = (size_t)P.E * 3 * P.N * sizeof(float);
    pl.split_e = 0;
    if (is_device_ptr(coords)) {
        pl.d_coords = coords;
    } else if (allow_split && P.E >= 2 && cbytes >= (size_t)(4 << 20) && P.M >= 64 && ctx->aux_stream && ctx->sample_groups > 1 &&
               ctx->upload_split) {
        // Large host maps: two halves on the copy stream, so the first half's experts are sampled while the second half is
        // still on the wire (launch_sample deals its two lanes by expert in this case).
        CK(cbuf.ensure(cbytes));
        const int es = (P.E + 1) / 2;
        const size_t first = (size_t)es * 3 * P.N * sizeof(float);
        CK(cudaMemcpyAsync(cbuf.p, coords, first, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(ctx->ev_copied[0], ctx->copy_stream));
        CK(cudaMemcpyAsync((char*)cbuf.p + first, (const char*)coords + first, cbytes - first, cudaMemcpyHostToDevice, ctx->copy_stream));
        CK(cudaEventRecord(ctx->ev_copied[1], ctx->copy_stream));
        pl.d_coords = cbuf.as<float>();
        pl.split_e = es;
    } else {
        CK(cbuf.ensure(cbytes));
        CK(cudaMemcpyAsync(cbuf.p, coords, cbytes, cudaMemcpyHostToDevice, copy_stream));
        pl.d_coords = cbuf.as<float>();
    }
    if (is_device_ptr(assign)) {
        pl.d_assign = (const long long*)assign;
        pl.assign_stride = stride;
    } else {
        std::vector<long long> tmp((size_t)P.M);
        for (int h = 0; h < P.M; ++h) tmp[h] = (long long)assign[(long long)h * stride];
        CK(abuf.ensure((size_t)P.M * 8));
        // pageable source: the copy is staged before cudaMemcpyAsync returns, so tmp may die
        CK(cudaMemcpyAsync(abuf.p, tmp.data(), (size_t)P.M * 8, cudaMemcpyHostToDevice, copy_stream));
        pl.d_assign = abuf.as<long long>();
        pl.assign_stride = 1;
    }
    return 0;
}

// Scoring launch shape, workspace, prep kernel.
int plan_and_prep(esacb200_ctx* ctx, Plan& pl) {
    const Problem& P = pl.P;
    // scoring launch shape
    int ppt = 8, hc = 64;
    const int want = 2 * 2 * ctx->sm_count;
    auto items = [&](int ppt_, int hc_) {
        int T = (P.N + score_tile_pixels(ppt_) - 1) / score_tile_pixels(ppt_);
        int nch = (P.M + hc_ - 1) / hc_ + (P.E > 1 ? P.E / 2 : 0);
        return (long long)T * nch;
    };
    if (items(8, 64) < want) { ppt = 4; hc = 32; }
    if (ppt == 4 && items(4, 32) < want) { ppt = 2; hc = 16; }
    if (ctx->score_ppt_opt == 2 || ctx->score_ppt_opt == 4 || ctx->score_ppt_opt == 8) ppt = ctx->score_ppt_opt;
    if (ctx->score_hc_opt > 0) hc = ctx->score_hc_opt < 64 ? ctx->score_hc_opt : 64;
    pl.ppt = ppt;
    pl.hc = hc;
    pl.T = (P.N + score_tile_pixels(ppt) - 1) / score_tile_pixels(ppt);
    const int max_chunks = (P.M + hc - 1) / hc + P.E;
    long long it = (long long)pl.T * max_chunks;
    pl.grid = (int)(it < 2ll * ctx->sm_count ? it : 2ll * ctx->sm_count);
    const int need_align = ppt >= 4 ? 4 : 2;
    pl.vec_ok = (P.N % need_align == 0) && (((uintptr_t)pl.d_coords) % (need_align * 4) == 0);

    CK(ctx->assign32.ensure((size_t)P.M * 4));
    CK(ctx->counts.ensure((size_t)P.E * 4));
    CK(ctx->offsets.ensure((size_t)(P.E + 1) * 4));
    CK(ctx->perm.ensure((size_t)P.M * 4));
    CK(ctx->slot_of.ensure((size_t)P.M * 4));
    CK(ctx->chunks.ensure((size_t)(P.M + P.E) * sizeof(ChunkDesc)));
    CK(ctx->scalars.ensure(S_COUNT * 4));
    CK(ctx->centres.ensure((size_t)P.E * 3 * 4));
    CK(ctx->poses.ensure((size_t)P.M * sizeof(Pose)));
    CK(ctx->poses_ref.ensure((size_t)P.M * sizeof(Pose)));
    CK(ctx->cells.ensure((size_t)P.M * 8 * 4));
    CK(ctx->tries.ensure((size_t)P.M * 4));
    CK(ctx->posepk.ensure((size_t)P.M * sizeof(PosePk)));
    CK(ctx->part.ensure((size_t)P.M * pl.T * 4));
    CK(ctx->scores.ensure((size_t)P.M * 8));
    CK(ctx->probs.ensure((size_t)P.M * 8));
    CK(ctx->stats.ensure(8 * 8));
    CK(ctx->contrib.ensure((size_t)P.M * 4));
    CK(ctx->out17.ensure(32 * 4));
    int* sc = ctx->scalars.as<int>();
    launch_prep(pl.d_coords, pl.d_assign, pl.assign_stride, P, hc, ctx->assign32.as<int>(), ctx->counts.as<int>(),
                ctx->offsets.as<int>(), ctx->perm.as<int>(), ctx->slot_of.as<int>(), ctx->chunks.as<ChunkDesc>(),
                sc + S_NCHUNKS, sc + S_WORK, ctx->centres.as<float>(), sc + S_FLAGS, pl.split_e ? 1 : 3, ctx->stream);
    ctx->st.kernel_launches += 1;
    mark(ctx, EV_PREP);
    return 0;
}

int stage_inputs(esacb200_ctx* ctx, Plan& pl, const float* coords, const int64_t* assign, int64_t stride, bool allow_split = false) {
    int rc = upload_inputs(ctx, pl, coords, assign, stride, ctx->coords, ctx->assign64, ctx->stream, allow_split);
    if (rc) return rc;
    mark(ctx, EV_H2D);
    return plan_and_prep(ctx, pl);
}

int run_sample(esacb200_ctx* ctx, const Plan& pl, uint64_t seed) {
    const Problem& P = pl.P;
    const int cap = 1 << 19;       // per group
    const int cap_acc = 1 << 15;
    // two lanes pay once a wave's kernels are long enough to overlap (full-resolution maps, or very many hypotheses)
    int G = pl.split_e ? 2 : ((ctx->sample_groups > 1 && ctx->aux_stream && P.M >= 64 && (P.N >= 65536 || P.M >= 1024)) ? ctx->sample_groups : 1);
    if (G > 2 && (!ctx->aux_more[0] || !ctx->aux_more[1] || P.M < 512)) G = 2;
    const int Mg = pl.split_e ? P.M : (P.M + G - 1) / G;  // capacity of a lane's work list
    // ints: [best: 2M] [base: M] [ovf: M] then per group [list: 2*Mg] [counters: 8]
    const size_t per_group_ints = (size_t)2 * Mg + 8;
    CK(ctx->smp_int.ensure(((size_t)P.M * 4 + G * per_group_ints) * 4 + 8));
    const size_t per_group_bytes = (size_t)cap * sizeof(int2) + (size_t)cap_acc * sizeof(Accepted);
    CK(ctx->smp_surv.ensure(G * per_group_bytes));
    SampleState st[4];
    int* b = ctx->smp_int.as<int>() + 2 * (size_t)P.M;
    for (int g = 0; g < G; ++g) {
        st[g].best = ctx->smp_int.as<unsigned long long>();  // 8-byte aligned: first in the buffer
        st[g].base = b;
        st[g].ovf = b + P.M;
        st[g].list = b + 2 * (size_t)P.M + g * per_group_ints;
        st[g].counters = st[g].list + 2 * (size_t)Mg;
        char* sb = (char*)ctx->smp_surv.p + g * per_group_bytes;
        st[g].surv = (int2*)sb;
        st[g].stage = (Accepted*)(sb + (size_t)cap * sizeof(int2));
        st[g].cap = cap;
        st[g].cap_acc = cap_acc;
        st[g].M = Mg;
    }
    CK(ctx->coords4.ensure((size_t)P.E * P.N * sizeof(float4)));
    unsigned long long* trace = nullptr;
    if (ctx->sample_trace) {  // 4 lanes x 32 waves x 2 kernels x (start, end)
        CK(ctx->smp_trace.ensure(512 * 8));
        CK(cudaMemsetAsync(ctx->smp_trace.p, 0, 512 * 8, ctx->stream));
        trace = ctx->smp_trace.as<unsigned long long>();
        launch_trace_init(trace, 256, ctx->stream);
    }
    const cudaStream_t lane_streams[4] = {ctx->stream, ctx->aux_stream, ctx->aux_more[0], ctx->aux_more[1]};
    const cudaEvent_t lane_joins[4] = {nullptr, ctx->ev_join, ctx->ev_join_more[0], ctx->ev_join_more[1]};
    ctx->st.kernel_launches += launch_sample(pl.d_coords, ctx->coords4.as<float4>(), ctx->assign32.as<int>(), P, seed, ctx->max_tries,
                                             ctx->inj_M ? ctx->inject.as<int>() : nullptr, ctx->inj_T, st, G, ctx->sm_count,
                                             ctx->sample_prefilter, ctx->hyp_offset, ctx->hyp_stride, ctx->poses.as<Pose>(), ctx->cells.as<int>(),
                                             ctx->tries.as<int>(), lane_streams, ctx->ev_fork, lane_joins,
                                             pl.split_e, ctx->perm.as<int>(), ctx->offsets.as<int>(), ctx->ev_copied,
                                             ctx->sample_span0, ctx->sample_window, ctx->sample_waves, trace, ctx->sample_tail_boost);
    CK(cudaGetLastError());
    ctx->smp_groups_last = G;
    ctx->smp_Mg_last = Mg;
    if (pl.split_e) {
        // both halves have landed (the join orders this stream after lane 1, which waited for the second half): plane centres
        int* sc = ctx->scalars.as<int>();
        launch_prep(pl.d_coords, pl.d_assign, pl.assign_stride, P, pl.hc, ctx->assign32.as<int>(), ctx->counts.as<int>(),
                    ctx->offsets.as<int>(), ctx->perm.as<int>(), ctx->slot_of.as<int>(), ctx->chunks.as<ChunkDesc>(),
                    sc + S_NCHUNKS, sc + S_WORK, ctx->centres.as<float>(), sc + S_FLAGS, 2, ctx->stream);
        ctx->st.kernel_launches += 1;
    }
    mark(ctx, EV_SAMPLE);
    return 0;
}

int run_score(esacb200_ctx* ctx, const Plan& pl) {
    const Problem& P = pl.P;
    int* sc = ctx->scalars.as<int>();
    launch_fold(ctx->poses.as<Pose>(), ctx->perm.as<int>(), ctx->assign32.as<int>(), ctx->centres.as<float>(), P,
                ctx->posepk.as<PosePk>(), ctx->stream);
    mark(ctx, EV_FOLD);
    ScoreArgs a;
    a.coords = pl.d_coords;
    a.centres = ctx->centres.as<float>();
    a.poses = ctx->posepk.as<PosePk>();
    a.chunks = ctx->chunks.as<ChunkDesc>();
    a.n_chunks = sc + S_NCHUNKS;
    a.work_counter = sc + S_WORK;
    a.part = ctx->part.as<float>();
    a.P = P;
    a.T = pl.T;
    a.hc = pl.hc;
    const float log2e = 1.4426950408889634f;
    a.k1 = P.beta * log2e;
    a.k0 = -P.beta * P.tau * log2e;
    a.vec_ok = pl.vec_ok;
    launch_score(a, pl.ppt, pl.grid, ctx->stream);
    mark(ctx, EV_SCORE);
    launch_select(ctx->part.as<float>(), ctx->slot_of.as<int>(), P, pl.T, ctx->scores.as<double>(), ctx->probs.as<double>(),
                  ctx->stats.as<double>(), sc + S_WINNER, ctx->contrib.as<int>(), sc + S_NCONTRIB, ctx->stream);
    mark(ctx, EV_SELECT);
    ctx->st.kernel_launches += 3;
    ctx->st.score_launches += 1;
    ctx->st.score_ppt = pl.ppt;
    ctx->st.score_grid = pl.grid;
    return 0;
}

int pick_group(esacb200_ctx* ctx, const Problem& P, int jobs_hint) {
    if (ctx->refine_group_opt > 0) return ctx->refine_group_opt < ctx->refine_coresident ? ctx->refine_group_opt : ctx->refine_coresident;
    const int words = (P.N + 31) / 32;
    // ~320 cells per CTA, up to every co-resident CTA: with the warp-parallel slot summation the inter-CTA barrier costs less
    // than the fp64 work it spreads, at every shape measured (profiles/r01m_refine_groups.txt: 60x80 -> 16, 480x640 -> 148)
    int g = words / 10;
    if (g < 1) g = 1;
    // Jobs are handed out dynamically inside the kernel, so a group may work through several jobs: fewer, larger groups even
    // out the differing job lengths (rounds x LM iterations) -- worth it only while a block's share of the map stays large
    // against the cost of a group exchange (480x640: 8.5 vs 11.2 ms for 47 jobs; 60x80: 0.79 vs 0.39 ms, so not there;
    // profiles/r02e_refine_timing.txt)
    int waves = jobs_hint >= 8 ? ctx->refine_jobs_per_group : 1;
    int concurrent = jobs_hint > 0 ? (jobs_hint + waves - 1) / waves : 1;
    int cap = ctx->refine_coresident / concurrent;
    if (waves > 1 && (cap < 1 || P.N / (cap < 1 ? 1 : cap) < 4096)) cap = ctx->refine_coresident / (jobs_hint > 0 ? jobs_hint : 1);
    if (cap < 1) cap = 1;
    if (g > cap) g = cap;
    return g;
}

// Refinement of `n_jobs` (host count, or device scalar when d_njobs != null) hypotheses listed in d_jobs.
int run_refine(esacb200_ctx* ctx, const Plan& pl, const Pose* in, Pose* out, const int* d_jobs, const int* d_njobs,
               int n_jobs_host, int max_jobs, int group) {
    const Problem& P = pl.P;
    const int words = (P.N + 31) / 32;
    int n_groups = ctx->refine_coresident / group;
    if (n_groups > max_jobs) n_groups = max_jobs;
    if (n_groups < 1) n_groups = 1;
    CK(ctx->masks.ensure((size_t)max_jobs * 2 * words * 4));
    CK(ctx->rounds.ensure((size_t)max_jobs * 2 * 4));
    CK(ctx->scratch.ensure(refine_scratch_doubles(n_groups, group) * 8));
    if (group > 1) CK(cudaMemsetAsync(ctx->scratch.p, 0, refine_scratch_doubles(n_groups, group) * 8, ctx->stream));  // LL elements: no stale sequence numbers
    const size_t n_flags = refine_flag_words(n_groups, group);
    CK(ctx->barrier.ensure((n_flags + 4) * 4));
    CK(cudaMemsetAsync(ctx->barrier.p, 0, (n_flags + 4) * 4, ctx->stream));
    RefineArgs a;
    a.coords = pl.d_coords;
    a.centres = ctx->centres.as<float>();
    a.assign32 = ctx->assign32.as<int>();
    a.poses_in = in;
    a.poses_out = out;
    a.jobs = d_jobs;
    a.n_jobs = d_njobs;
    a.n_jobs_host = n_jobs_host;
    a.masks = ctx->masks.as<uint32_t>();
    a.mask_words = words;
    a.rounds = ctx->rounds.as<int>();
    a.scratch = ctx->scratch.as<double>();
    a.barrier = ctx->barrier.as<unsigned int>();
    a.job_counter = (int*)(ctx->barrier.as<unsigned int>() + n_flags);
    a.group = group;
    const int wpc = (words + group - 1) / group;
    a.cache = wpc <= refine_cache_words() ? 1 : 0;
    a.compact = ctx->refine_compact;
    a.pretest = ctx->refine_pretest;
    a.clist = nullptr;
    if (a.compact && !a.cache && wpc <= refine_max_compact_words()) {
        CK(ctx->clist.ensure((size_t)n_groups * words * 32 * sizeof(unsigned short)));
        a.clist = ctx->clist.as<unsigned short>();
    }
    a.prof = nullptr;
    if (ctx->refine_profile) {
        CK(ctx->prof.ensure(16 * 8));
        CK(cudaMemsetAsync(ctx->prof.p, 0, 16 * 8, ctx->stream));
        a.prof = ctx->prof.as<long long>();
    }
    a.P = P;
    a.max_ref_steps = ctx->max_ref_steps;
    launch_refine(a, n_groups, ctx->stream);
    CK(cudaGetLastError());
    ctx->st.kernel_launches += 1;
    ctx->st.refine_group = group;
    return 0;
}

uint64_t call_seed(esacb200_ctx* ctx) {
    uint64_t s = ctx->fixed_seed ? ctx->seed : mix64(ctx->seed + kGold * ctx->calls);
    if (ctx->calls == 0) s = ctx->seed;
    ++ctx->calls;
    return s;
}

// sample -> score -> select -> refine(winner) -> camera pose + expert id into d_out17 (17 floats + flags at [17]); no sync.
int enqueue_forward_core(esacb200_ctx* ctx, const Plan& pl, float* d_out17) {
    const Problem& P = pl.P;
    int* sc = ctx->scalars.as<int>();
    const uint64_t seed = call_seed(ctx);
    int rc = run_sample(ctx, pl, seed);
    if (rc) return rc;
    rc = run_score(ctx, pl);
    if (rc) return rc;
    const int group = pick_group(ctx, P, 1);
    rc = run_refine(ctx, pl, ctx->poses.as<Pose>(), ctx->poses_ref.as<Pose>(), sc + S_WINNER, nullptr, 1, 1, group);
    if (rc) return rc;
    mark(ctx, EV_REFINE);
    launch_finish_forward(ctx->poses_ref.as<Pose>(), sc + S_WINNER, ctx->assign32.as<int>(), sc + S_FLAGS, d_out17, ctx->stream);
    ctx->st.kernel_launches += 1;
    return 0;
}

void begin_call(esacb200_ctx* ctx) {
    memset(&ctx->st, 0, sizeof(ctx->st));
    for (int i = 0; i < EV_COUNT; ++i) ctx->ev_used[i] = false;
    ctx->err[0] = 0;
    mark(ctx, EV_START);
}

void finish_stats(esacb200_ctx* ctx) {
    esacb200_stats& s = ctx->st;
    s.ms_h2d = span(ctx, EV_START, EV_H2D);
    s.ms_prep = span(ctx, EV_H2D, EV_PREP);
    s.ms_sample = span(ctx, EV_PREP, EV_SAMPLE);
    s.ms_score = span(ctx, EV_FOLD, EV_SCORE);
    s.ms_select = span(ctx, EV_SCORE, EV_SELECT);
    s.ms_refine = span(ctx, EV_SELECT, EV_REFINE);
    s.ms_backward = span(ctx, EV_REFINE, EV_BWD);
    s.ms_total = span(ctx, EV_START, EV_END);
}


}  // namespace

// No C++ exception may cross the C ABI (std::vector / std::thread can throw): every entry point that allocates on the host is
// a function-try-block ending in this handler.
#define ESAC_ABI_CATCH(ctx)                                                                                   \
    catch (const std::exception& e) {                                                                         \
        return (ctx) ? fail((ctx), ESACB200_ERR_ARG, "host-side failure: %s", e.what()) : ESACB200_ERR_ARG;   \
    }                                                                                                         \
    catch (...) {                                                                                             \
        return (ctx) ? fail((ctx), ESACB200_ERR_ARG, "host-side failure (unknown exception)") : ESACB200_ERR_ARG; \
    }

// =================================================================================================
extern "C" {

int esacb200_create(int device, esacb200_ctx** out) {
    if (!out) return ESACB200_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return ESACB200_ERR_NO_DEVICE;
    }
    esacb200_ctx* ctx = new (std::nothrow) esacb200_ctx();
    if (!ctx) return ESACB200_ERR_ARG;
    ctx->device = device;
    DeviceGuard device_guard(device);
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return ESACB200_ERR_NO_DEVICE; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return ESACB200_ERR_CUDA; }
    ctx->sm_count = prop.multiProcessorCount;
    snprintf(ctx->dev_name, sizeof(ctx->dev_name), "%s", prop.name);
    if (cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return ESACB200_ERR_CUDA; }
    ctx->stream = ctx->own_stream;
    cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking);
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, hi) != cudaSuccess) { ctx->aux_stream = nullptr; cudaGetLastError(); }
        cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
        for (int i = 0; i < 2; ++i) {
            if (cudaStreamCreateWithPriority(&ctx->aux_more[i], cudaStreamNonBlocking, hi) != cudaSuccess) { ctx->aux_more[i] = nullptr; cudaGetLastError(); }
            cudaEventCreateWithFlags(&ctx->ev_join_more[i], cudaEventDisableTiming);
        }
    }
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ctx->ev_consumed[i], cudaEventDisableTiming);
    }
    for (int i = 0; i < EV_COUNT; ++i) cudaEventCreate(&ctx->ev[i]);
    cudaMallocHost((void**)&ctx->h_out, 32 * sizeof(float));
    cudaMallocHost((void**)&ctx->h_dbl, 8 * sizeof(double));
    ctx->refine_coresident = refine_max_coresident_blocks(ctx->sm_count);
    if (ctx->refine_coresident < 1) ctx->refine_coresident = 1;
    memset(&ctx->st, 0, sizeof(ctx->st));
    *out = ctx;
    return ESACB200_OK;
}

void esacb200_destroy(esacb200_ctx* ctx) {
    if (!ctx) return;
    for (esacb200_ctx* w : ctx->workers) esacb200_destroy(w);
    ctx->workers.clear();
    DeviceGuard device_guard(ctx->device);
    if (ctx->nccl_comm) { cudaStreamSynchronize(ctx->stream); nccl_api().CommDestroy(ctx->nccl_comm); ctx->nccl_comm = nullptr; }
    cudaStreamSynchronize(ctx->stream);
    DevBuf* bufs[] = {&ctx->coords, &ctx->grads, &ctx->assign64, &ctx->assign32, &ctx->counts, &ctx->offsets, &ctx->perm,
                      &ctx->slot_of, &ctx->chunks, &ctx->scalars, &ctx->centres, &ctx->poses, &ctx->poses_ref, &ctx->cells,
                      &ctx->tries, &ctx->posepk, &ctx->part, &ctx->scores, &ctx->probs, &ctx->stats, &ctx->contrib,
                      &ctx->masks, &ctx->rounds, &ctx->scratch, &ctx->barrier, &ctx->out17, &ctx->inject, &ctx->losses,
                      &ctx->red, &ctx->hypgrad, &ctx->job_of, &ctx->gt, &ctx->smp_int, &ctx->smp_surv, &ctx->smp_trace, &ctx->clist, &ctx->eflags, &ctx->coords4, &ctx->coords_alt, &ctx->assign64_alt, &ctx->out_batch, &ctx->prof, &ctx->gathered, &ctx->grads_work};
    for (DevBuf* b : bufs) b->release();
    for (int i = 0; i < EV_COUNT; ++i)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    if (ctx->h_out) cudaFreeHost(ctx->h_out);
    if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
    if (ctx->h_dbl) cudaFreeHost(ctx->h_dbl);
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]);
        if (ctx->ev_consumed[i]) cudaEventDestroy(ctx->ev_consumed[i]);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    for (int i = 0; i < 2; ++i) {
        if (ctx->aux_more[i]) cudaStreamDestroy(ctx->aux_more[i]);
        if (ctx->ev_join_more[i]) cudaEventDestroy(ctx->ev_join_more[i]);
    }
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

const char* esacb200_last_error(const esacb200_ctx* ctx) { return ctx ? ctx->err : "null context"; }

int esacb200_set_stream(esacb200_ctx* ctx, void* s) {
    if (!ctx) return ESACB200_ERR_ARG;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return ESACB200_OK;
}

int esacb200_set_seed(esacb200_ctx* ctx, uint64_t seed) {
    if (!ctx) return ESACB200_ERR_ARG;
    ctx->seed = seed;
    ctx->calls = 0;
    return ESACB200_OK;
}

int esacb200_set_option(esacb200_ctx* ctx, const char* key, double v) {
    if (!ctx || !key) return ESACB200_ERR_ARG;
    if (!strcmp(key, "max_tries")) ctx->max_tries = v < 1 ? 1 : (int)v;
    else if (!strcmp(key, "max_ref_steps")) ctx->max_ref_steps = v < 0 ? 0 : (int)v;
    else if (!strcmp(key, "fixed_seed")) ctx->fixed_seed = v != 0;
    else if (!strcmp(key, "refine_group")) ctx->refine_group_opt = (int)v;
    else if (!strcmp(key, "refine_pretest")) ctx->refine_pretest = v != 0;
    else if (!strcmp(key, "refine_compact")) ctx->refine_compact = v != 0;
    else if (!strcmp(key, "refine_profile")) ctx->refine_profile = v != 0;
    else if (!strcmp(key, "refine_jobs_per_group")) ctx->refine_jobs_per_group = v < 1 ? 1 : (int)v;
    else if (!strcmp(key, "sample_prefilter")) ctx->sample_prefilter = v != 0;
    else if (!strcmp(key, "sample_tail_boost")) ctx->sample_tail_boost = v < 1 ? 1.f : (float)v;
    else if (!strcmp(key, "sample_trace")) ctx->sample_trace = v != 0;
    else if (!strcmp(key, "sample_span0")) ctx->sample_span0 = v < 256 ? 256 : ((int)v + 255) / 256 * 256;
    else if (!strcmp(key, "sample_window")) ctx->sample_window = v < 0.05 ? 0.05f : (float)v;
    else if (!strcmp(key, "sample_waves")) ctx->sample_waves = v < 0 ? 0 : (v > 64 ? 64 : (int)v);
    else if (!strcmp(key, "upload_split")) ctx->upload_split = v != 0;  // host maps in two halves, sampling under the second copy
    else if (!strcmp(key, "sample_groups")) ctx->sample_groups = v >= 4 ? 4 : (v >= 2 ? (int)v : 1);  // interleaved lanes, one stream each
    else if (!strcmp(key, "hyp_offset")) ctx->hyp_offset = (int)v;  // global index of local hypothesis 0 (sharded runs)
    else if (!strcmp(key, "hyp_stride")) ctx->hyp_stride = v < 1 ? 1 : (int)v;  // ... of local hypothesis h: offset + h * stride
    else if (!strcmp(key, "score_ppt")) ctx->score_ppt_opt = (int)v;   // 0 = automatic, else 2 / 4 / 8 cells per thread
    else if (!strcmp(key, "score_hc")) ctx->score_hc_opt = (int)v;     // 0 = automatic, else hypotheses per chunk (<= 64)
    else if (!strcmp(key, "batch_workers")) ctx->batch_workers = v < 1 ? 1 : (v > 16 ? 16 : (int)v);  // streams of backward_batch
    else return fail(ctx, ESACB200_ERR_ARG, "unknown option '%s'", key);
    return ESACB200_OK;
}

int esacb200_inject_cells(esacb200_ctx* ctx, const int32_t* cells, int M, int T) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!cells) { ctx->inj_M = ctx->inj_T = 0; return ESACB200_OK; }
    if (M <= 0 || T <= 0) return fail(ctx, ESACB200_ERR_ARG, "inject_cells: M and T must be positive");
    size_t bytes = (size_t)M * T * 8 * 4;
    CK(ctx->inject.ensure(bytes));
    CK(cudaMemcpy(ctx->inject.p, cells, bytes, cudaMemcpyHostToDevice));
    ctx->inj_M = M;
    ctx->inj_T = T;
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_device_info(esacb200_ctx* ctx, int* sm_count, char* name, int name_len) {
    if (!ctx) return ESACB200_ERR_ARG;
    if (sm_count) *sm_count = ctx->sm_count;
    if (name && name_len > 0) snprintf(name, name_len, "%s", ctx->dev_name);
    return ESACB200_OK;
}

// -------------------------------------------------------------------------------------------------
int esacb200_forward(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                     int64_t assign_stride, int M, float* out_pose, int shiftX, int shiftY, float f, float ppx,
                     float ppy, float tau, float alpha, float beta, float maxReproj, int sub, int* out_expert) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !assign || !out_pose) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    Plan pl;
    int rc = fill_problem(ctx, pl.P, E, H, W, M, shiftX, shiftY, f, ppx, ppy, tau, alpha, beta, maxReproj, sub);
    if (rc) return rc;
    if ((long long)(W - 1) * (H - 1) < 4) return fail(ctx, ESACB200_ERR_ARG, "map %dx%d too small to draw 4 distinct cells from [0,W-2]x[0,H-2]", W, H);
    if (ctx->inj_M && ctx->inj_M != M) return fail(ctx, ESACB200_ERR_ARG, "injected cells are for M=%d, call has M=%d", ctx->inj_M, M);
    begin_call(ctx);
    rc = stage_inputs(ctx, pl, coords, assign, assign_stride, /*allow_split=*/!ctx->inj_M);
    if (rc) return rc;
    const Problem& P = pl.P;
    int* sc = ctx->scalars.as<int>();
    rc = enqueue_forward_core(ctx, pl, ctx->out17.as<float>());
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_out, ctx->out17.p, 17 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_out + 20, sc, 8 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_dbl, ctx->stats.p, 3 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_dbl + 4, ctx->rounds.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (is_device_ptr(out_pose)) CK(cudaMemcpyAsync(out_pose, ctx->out17.p, 16 * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    const int* hs = (const int*)(ctx->h_out + 20);
    if (hs[S_FLAGS]) return fail(ctx, ESACB200_ERR_ARG, "hypAssignment holds an expert index outside [0, %d)", E);
    if (!is_device_ptr(out_pose)) memcpy(out_pose, ctx->h_out, 16 * sizeof(float));
    if (out_expert) *out_expert = (int)ctx->h_out[16];
    ctx->st.M = M;
    ctx->st.winner = hs[S_WINNER];
    ctx->st.n_contrib = hs[S_NCONTRIB];
    ctx->st.entropy = ctx->h_dbl[0];
    ctx->st.refine_rounds = ((const int*)(ctx->h_dbl + 4))[0];
    ctx->last_M = M;
    ctx->last_backward = false;
    finish_stats(ctx);
    ctx->inj_M = ctx->inj_T = 0;
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
// local half of a sharded forward: pipeline + record, no synchronisation (shared by forward_pack and forward_sharded)
static int enqueue_forward_record(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                                  int64_t assign_stride, int M, int M_pad, int shiftX, int shiftY, float f, float ppx, float ppy,
                                  float tau, float alpha, float beta, float maxReproj, int sub, int expert_offset, double* pack_out) {
    if (M_pad < M || M_pad < 1) return fail(ctx, ESACB200_ERR_ARG, "M_pad (%d) must be >= M (%d) and >= 1", M_pad, M);
    begin_call(ctx);
    ctx->inj_M = ctx->inj_T = 0;
    if (M > 0) {
        Plan pl;
        int rc = fill_problem(ctx, pl.P, E, H, W, M, shiftX, shiftY, f, ppx, ppy, tau, alpha, beta, maxReproj, sub);
        if (rc) return rc;
        if ((long long)(W - 1) * (H - 1) < 4) return fail(ctx, ESACB200_ERR_ARG, "map %dx%d too small", W, H);
        rc = stage_inputs(ctx, pl, coords, assign, assign_stride);
        if (rc) return rc;
        rc = enqueue_forward_core(ctx, pl, ctx->out17.as<float>());
        if (rc) return rc;
    } else {
        CK(ctx->scores.ensure(8));
        CK(ctx->out17.ensure(32 * 4));
    }
    launch_pack_forward(ctx->scores.as<double>(), ctx->out17.as<float>(), M, M_pad, expert_offset, ctx->hyp_offset, ctx->hyp_stride,
                        pack_out, ctx->stream);
    CK(cudaGetLastError());
    ctx->st.kernel_launches += 1;
    ctx->st.M = M;
    ctx->last_M = M;
    ctx->last_backward = false;
    return ESACB200_OK;
}

int esacb200_forward_pack(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                          int64_t assign_stride, int M, int M_pad, int shiftX, int shiftY, float f, float ppx, float ppy, float tau,
                          float alpha, float beta, float maxReproj, int sub, int expert_offset, double* pack_out) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!pack_out || (M > 0 && (!coords || !assign))) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    if ((M > 0 && (!is_device_ptr(coords) || !is_device_ptr(assign))) || !is_device_ptr(pack_out))
        return fail(ctx, ESACB200_ERR_ARG, "forward_pack takes device pointers only");
    int rc = enqueue_forward_record(ctx, coords, E, H, W, assign, assign_stride, M, M_pad, shiftX, shiftY, f, ppx, ppy, tau, alpha,
                                    beta, maxReproj, sub, expert_offset, pack_out);
    if (rc) return rc;
    mark(ctx, EV_END);
    return ESACB200_OK;   // stage timers of this call are not collected: that would need the synchronisation
} ESAC_ABI_CATCH(ctx)

// ---- communicator -----------------------------------------------------------------------------------
int esacb200_nccl_unique_id(void* out128) {
    if (!out128) return ESACB200_ERR_ARG;
    NcclApi& n = nccl_api();
    if (!n.ok) return ESACB200_ERR_NO_DEVICE;
    NcclApi::UniqueId id;
    if (n.GetUniqueId(&id) != 0) return ESACB200_ERR_CUDA;
    memcpy(out128, id.internal, 128);
    return ESACB200_OK;
}

int esacb200_comm_init(esacb200_ctx* ctx, int world, int rank, const void* id128) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!id128 || world < 1 || rank < 0 || rank >= world) return fail(ctx, ESACB200_ERR_ARG, "bad communicator arguments");
    NcclApi& n = nccl_api();
    if (!n.ok) return fail(ctx, ESACB200_ERR_NO_DEVICE, "libnccl.so.2 cannot be loaded");
    if (ctx->nccl_comm) { n.CommDestroy(ctx->nccl_comm); ctx->nccl_comm = nullptr; }
    NcclApi::UniqueId id;
    memcpy(id.internal, id128, 128);
    CKN(n.CommInitRank(&ctx->nccl_comm, world, id, rank));
    ctx->comm_world = world;
    ctx->comm_rank = rank;
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_comm_destroy(esacb200_ctx* ctx) {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (ctx->nccl_comm) {
        cudaStreamSynchronize(ctx->stream);
        nccl_api().CommDestroy(ctx->nccl_comm);
        ctx->nccl_comm = nullptr;
    }
    ctx->comm_world = 1;
    ctx->comm_rank = 0;
    return ESACB200_OK;
}

// esac_forward with the experts / hypotheses sharded over the ranks of the communicator (SURVEY 8e): local pipeline ->
// record -> ONE ncclAllGather on the context's stream -> softMax / draw over all records on the device -> one 80-byte
// read-back.  Every rank returns the global winner's pose and expert.  M may be 0 (a shard without hypotheses); M_pad is
// the largest M of any rank (records must have one size).
int esacb200_forward_sharded(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                             int64_t assign_stride, int M, int M_pad, float* out_pose, int shiftX, int shiftY, float f, float ppx,
                             float ppy, float tau, float alpha, float beta, float maxReproj, int sub, int expert_offset,
                             int* out_expert) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!ctx->nccl_comm) return fail(ctx, ESACB200_ERR_ARG, "no communicator: call esacb200_comm_init first");
    if (!out_pose || (M > 0 && (!coords || !assign))) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    const int world = ctx->comm_world;
    const size_t rec = (size_t)M_pad + kPackTail;
    CK(ctx->gathered.ensure((world + 1) * rec * 8));
    double* mine = ctx->gathered.as<double>() + (size_t)world * rec;
    int rc = enqueue_forward_record(ctx, coords, E, H, W, assign, assign_stride, M, M_pad, shiftX, shiftY, f, ppx, ppy, tau, alpha,
                                    beta, maxReproj, sub, expert_offset, mine);
    if (rc) return rc;
    CKN(nccl_api().AllGather(mine, ctx->gathered.p, rec, kNcclFloat64, ctx->nccl_comm, ctx->stream));
    launch_select_gathered(ctx->gathered.as<double>(), world, M_pad, ctx->out17.as<float>(), ctx->stream);
    CK(cudaGetLastError());
    ctx->st.kernel_launches += 2;
    CK(cudaMemcpyAsync(ctx->h_out, ctx->out17.p, 20 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (is_device_ptr(out_pose)) CK(cudaMemcpyAsync(out_pose, ctx->out17.p, 16 * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    if (ctx->h_out[17] != 0.f) return fail(ctx, ESACB200_ERR_ARG, "a shard's hypAssignment holds an expert index outside its experts");
    if (!is_device_ptr(out_pose)) memcpy(out_pose, ctx->h_out, 16 * sizeof(float));
    if (out_expert) *out_expert = (int)ctx->h_out[16];
    ctx->st.winner = (int)ctx->h_out[18];
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
// esac_forward over a batch of B images of one shape (BASELINE configs[2]: "batch 8 images").  The reference has no such
// entry: its callers loop over a DataLoader with batch_size=1 (test_esac.py:137).  Images are processed back to back on
// the compute stream with ONE host synchronisation at the end; host coordinate maps are double-buffered and copied on a
// second stream so the copy of image b+1 overlaps the kernels of image b.
int esacb200_forward_batch(esacb200_ctx* ctx, int B, const float* coords, int E, int H, int W, const int64_t* assign,
                           int64_t assign_stride, int M, float* out_poses, int shiftX, int shiftY, float f, float ppx,
                           float ppy, float tau, float alpha, float beta, float maxReproj, int sub, int* out_experts) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !assign || !out_poses || B <= 0) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument or empty batch");
    Plan pl;
    int rc = fill_problem(ctx, pl.P, E, H, W, M, shiftX, shiftY, f, ppx, ppy, tau, alpha, beta, maxReproj, sub);
    if (rc) return rc;
    if ((long long)(W - 1) * (H - 1) < 4) return fail(ctx, ESACB200_ERR_ARG, "map %dx%d too small", W, H);
    begin_call(ctx);
    ctx->inj_M = ctx->inj_T = 0;
    const size_t cstride = (size_t)E * 3 * H * W;
    const bool host_coords = !is_device_ptr(coords);
    const bool host_assign = !is_device_ptr(assign);
    // element stride between the assignments of consecutive images: rows of a [B, M] tensor
    const int64_t arow = assign_stride == 0 ? 0 : (int64_t)M * assign_stride;
    CK(ctx->out_batch.ensure((size_t)B * 20 * sizeof(float)));
    DevBuf* cb[2] = {&ctx->coords, &ctx->coords_alt};
    DevBuf* ab[2] = {&ctx->assign64, &ctx->assign64_alt};
    for (int b = 0; b < B; ++b) {
        const int buf = b & 1;
        if (host_coords && b >= 2) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_consumed[buf], 0));
        rc = upload_inputs(ctx, pl, coords + (size_t)b * cstride, assign + (size_t)b * arow, assign_stride, *cb[buf], *ab[buf],
                           host_coords ? ctx->copy_stream : ctx->stream);
        if (rc) return rc;
        if (host_coords) {
            CK(cudaEventRecord(ctx->ev_copied[buf], ctx->copy_stream));
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_copied[buf], 0));
        }
        (void)host_assign;
        if (b == 0) mark(ctx, EV_H2D);
        rc = plan_and_prep(ctx, pl);
        if (rc) return rc;
        rc = enqueue_forward_core(ctx, pl, ctx->out_batch.as<float>() + (size_t)b * 20);
        if (rc) return rc;
        if (host_coords) CK(cudaEventRecord(ctx->ev_consumed[buf], ctx->stream));
    }
    std::vector<float> host((size_t)B * 20);
    CK(cudaMemcpyAsync(host.data(), ctx->out_batch.p, host.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    const bool dev_out = is_device_ptr(out_poses);
    if (dev_out)
        CK(cudaMemcpy2DAsync(out_poses, 16 * sizeof(float), ctx->out_batch.p, 20 * sizeof(float), 16 * sizeof(float), B,
                             cudaMemcpyDeviceToDevice, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    for (int b = 0; b < B; ++b) {
        const float* o = host.data() + (size_t)b * 20;
        if (o[17] != 0.f) return fail(ctx, ESACB200_ERR_ARG, "image %d: hypAssignment holds an expert index outside [0, %d)", b, E);
        if (!dev_out) memcpy(out_poses + (size_t)b * 16, o, 16 * sizeof(float));
        if (out_experts) out_experts[b] = (int)o[16];
    }
    ctx->st.M = M;
    ctx->st.winner = (int)host[(size_t)(B - 1) * 20 + 18];
    ctx->last_M = M;
    ctx->last_backward = false;
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
int esacb200_score_poses(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                         int64_t assign_stride, int M, const double* poses6, int shiftX, int shiftY, float f, float ppx,
                         float ppy, float tau, float alpha, float beta, float maxReproj, int sub, double* out_scores) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !assign || !poses6 || !out_scores) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    Plan pl;
    int rc = fill_problem(ctx, pl.P, E, H, W, M, shiftX, shiftY, f, ppx, ppy, tau, alpha, beta, maxReproj, sub);
    if (rc) return rc;
    begin_call(ctx);
    rc = stage_inputs(ctx, pl, coords, assign, assign_stride);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->poses.p, poses6, (size_t)M * sizeof(Pose), cudaMemcpyHostToDevice, ctx->stream));
    mark(ctx, EV_SAMPLE);
    rc = run_score(ctx, pl);
    if (rc) return rc;
    CK(cudaMemcpyAsync(out_scores, ctx->scores.p, (size_t)M * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_out + 20, ctx->scalars.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    const int* hs = (const int*)(ctx->h_out + 20);
    if (hs[S_FLAGS]) return fail(ctx, ESACB200_ERR_ARG, "hypAssignment holds an expert index outside [0, %d)", E);
    ctx->st.M = M;
    ctx->st.winner = hs[S_WINNER];
    ctx->st.n_contrib = hs[S_NCONTRIB];
    ctx->last_M = M;
    ctx->last_backward = false;
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
int esacb200_refine_poses(esacb200_ctx* ctx, const float* coords, int E, int H, int W, const int64_t* assign,
                          int64_t assign_stride, int M, double* poses6, int shiftX, int shiftY, float f, float ppx,
                          float ppy, float tau, float maxReproj, int sub, int* out_rounds, int* out_inliers) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !assign || !poses6) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    Plan pl;
    int rc = fill_problem(ctx, pl.P, E, H, W, M, shiftX, shiftY, f, ppx, ppy, tau, 100.f, 0.5f, maxReproj, sub);
    if (rc) return rc;
    begin_call(ctx);
    rc = stage_inputs(ctx, pl, coords, assign, assign_stride);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->poses.p, poses6, (size_t)M * sizeof(Pose), cudaMemcpyHostToDevice, ctx->stream));
    std::vector<int> jobs((size_t)M);
    for (int i = 0; i < M; ++i) jobs[i] = i;
    CK(cudaMemcpyAsync(ctx->contrib.p, jobs.data(), (size_t)M * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int group = pick_group(ctx, pl.P, M);
    mark(ctx, EV_SELECT);
    rc = run_refine(ctx, pl, ctx->poses.as<Pose>(), ctx->poses_ref.as<Pose>(), ctx->contrib.as<int>(), nullptr, M, M, group);
    if (rc) return rc;
    mark(ctx, EV_REFINE);
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    CK(cudaMemcpy(poses6, ctx->poses_ref.p, (size_t)M * sizeof(Pose), cudaMemcpyDeviceToHost));
    std::vector<int> rr((size_t)M * 2);
    CK(cudaMemcpy(rr.data(), ctx->rounds.p, (size_t)M * 8, cudaMemcpyDeviceToHost));
    const int words = (pl.P.N + 31) / 32;
    std::vector<uint32_t> mk;
    if (out_inliers) {
        mk.resize((size_t)M * 2 * words);
        CK(cudaMemcpy(mk.data(), ctx->masks.p, mk.size() * 4, cudaMemcpyDeviceToHost));
    }
    for (int i = 0; i < M; ++i) {
        if (out_rounds) out_rounds[i] = rr[2 * i];
        if (out_inliers) {
            int c = 0;
            if (rr[2 * i] > 0) {
                const uint32_t* m = mk.data() + ((size_t)i * 2 + rr[2 * i + 1]) * words;
                for (int w = 0; w < words; ++w) c += __builtin_popcount(m[w]);
            }
            out_inliers[i] = c;
        }
    }
    ctx->st.M = M;
    ctx->last_M = M;
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)


// Hypothesis-major sharding: the planes that receive gradient on SOME rank (flags after the max-all-reduce, host copy in
// ctx->h_flags) are the only ones whose slices have to be summed over the ranks -- with a peaked gating that is one plane of
// twenty (3.7 of 74 MB at 480x640).  phase 0: zero those slices of the work buffer; phase 1: all-reduce them and add them to dst.
static int ensure_host_flags(esacb200_ctx* ctx, int E) {
    if (ctx->h_flags_cap >= E + 1) return 0;
    if (ctx->h_flags) cudaFreeHost(ctx->h_flags);
    ctx->h_flags = nullptr; ctx->h_flags_cap = 0;
    CK(cudaMallocHost((void**)&ctx->h_flags, (size_t)(E + 1) * sizeof(int)));
    ctx->h_flags_cap = E + 1;
    return 0;
}
static int for_flagged_planes(esacb200_ctx* ctx, int E, size_t plane, float* work, float* dst, int phase) {
    for (int e = 0; e < E;) {
        if (!ctx->h_flags[e]) { ++e; continue; }
        int e1 = e;
        while (e1 < E && ctx->h_flags[e1]) ++e1;
        float* w = work + (size_t)e * plane;
        const size_t n = (size_t)(e1 - e) * plane;
        if (phase == 0) {
            CK(cudaMemsetAsync(w, 0, n * sizeof(float), ctx->stream));
        } else {
            CKN(nccl_api().AllReduce(w, w, n, kNcclFloat32, kNcclSum, ctx->nccl_comm, ctx->stream));
            launch_add_inplace(dst + (size_t)e * plane, w, n, ctx->stream);
            ctx->st.kernel_launches += 2;
        }
        e = e1;
    }
    return 0;
}

// -------------------------------------------------------------------------------------------------
static int backward_impl(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W, const int64_t* assign,
                         int64_t assign_stride, int M, const float* gt_pose, float wRot, float wTrans, float cut, int shiftX,
                         int shiftY, float f, float ppx, float ppy, float tau, float alpha, float beta, float maxReproj, int sub,
                         esacb200_exchange_fn exchange, void* user, double* out_loss, bool use_nccl = false,
                         bool reduce_grads = false) {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !assign || !grads || !gt_pose) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    Plan pl;
    int rc = fill_problem(ctx, pl.P, E, H, W, M, shiftX, shiftY, f, ppx, ppy, tau, alpha, beta, maxReproj, sub);
    if (rc) return rc;
    if ((long long)(W - 1) * (H - 1) < 4) return fail(ctx, ESACB200_ERR_ARG, "map %dx%d too small to draw 4 distinct cells from [0,W-2]x[0,H-2]", W, H);
    if (ctx->inj_M && ctx->inj_M != M) return fail(ctx, ESACB200_ERR_ARG, "injected cells are for M=%d, call has M=%d", ctx->inj_M, M);
    begin_call(ctx);
    const Problem& P = pl.P;
    const size_t cbytes = (size_t)P.E * 3 * P.N * sizeof(float);
    float* d_grads = grads;
    const bool grads_on_host = !is_device_ptr(grads);
    if (grads_on_host) {
        CK(ctx->grads.ensure(cbytes));
        CK(cudaMemcpyAsync(ctx->grads.p, grads, cbytes, cudaMemcpyHostToDevice, ctx->stream));
        d_grads = ctx->grads.as<float>();
    }
    // hypothesis-major sharding: every rank holds all planes and a slice of the hypotheses, so the gradient slices overlap:
    // the local gradient goes to a zeroed work buffer, is summed over the ranks and only then added to the caller's tensor
    float* d_dst = d_grads;
    if (reduce_grads) {
        CK(ctx->grads_work.ensure(cbytes));
        d_grads = ctx->grads_work.as<float>();  // (the slices that will be used are zeroed once they are known, below)
        rc = ensure_host_flags(ctx, E);
        if (rc) return rc;
    }
    rc = stage_inputs(ctx, pl, coords, assign, assign_stride);
    if (rc) return rc;
    int* sc = ctx->scalars.as<int>();
    const uint64_t seed = call_seed(ctx);
    rc = run_sample(ctx, pl, seed);
    if (rc) return rc;
    rc = run_score(ctx, pl);
    if (rc) return rc;
    if (exchange) {
        // exchange 1 (SURVEY 8e): softmax normalisation over the hypotheses of ALL ranks
        CK(cudaMemcpyAsync(ctx->h_dbl, ctx->stats.as<double>() + 5, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        double v[2] = {ctx->h_dbl[0], ctx->h_dbl[1]};
        if (exchange(user, 1, v, 2) != 0) return fail(ctx, ESACB200_ERR_ARG, "exchange callback failed (phase 1)");
        launch_rescale_probs(ctx->scores.as<double>(), P, v[0], v[1], ctx->probs.as<double>(), ctx->contrib.as<int>(),
                             sc + S_NCONTRIB, ctx->stream);
        ctx->st.kernel_launches += 1;
    } else if (use_nccl) {
        // exchange 1 on the device: all-gather of the (max, sum exp) pairs, merged by the kernel that rebuilds the probabilities
        CK(ctx->gathered.ensure((size_t)ctx->comm_world * 2 * 8));
        CKN(nccl_api().AllGather(ctx->stats.as<double>() + 5, ctx->gathered.p, 2, kNcclFloat64, ctx->nccl_comm, ctx->stream));
        launch_rescale_probs_gathered(ctx->scores.as<double>(), P, ctx->gathered.as<double>(), ctx->comm_world, nullptr,
                                      ctx->probs.as<double>(), ctx->contrib.as<int>(), sc + S_NCONTRIB, ctx->stream);
        ctx->st.kernel_launches += 2;
    }
    // refHyps = initHyps for everything below PROB_THRESH (esac.cpp:331-334)
    CK(cudaMemcpyAsync(ctx->poses_ref.p, ctx->poses.p, (size_t)M * sizeof(Pose), cudaMemcpyDeviceToDevice, ctx->stream));
    // Refining many hypotheses is fp64-throughput bound, so every SM should be busy and no CTA should wait at an inter-CTA
    // barrier longer than needed: one 4-byte read-back of the number of contributing hypotheses (a ~20 us stall on a
    // multi-millisecond call) lets the group size be coresident / jobs.
    CK(cudaMemcpyAsync(ctx->h_out + 28, sc + S_NCONTRIB, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    if (reduce_grads) {  // which planes receive gradient on some rank: rides on the same host synchronisation
        CK(ctx->eflags.ensure((size_t)E * sizeof(int)));
        launch_expert_flags(ctx->contrib.as<int>(), sc + S_NCONTRIB, ctx->assign32.as<int>(), E, ctx->eflags.as<int>(), ctx->stream);
        CKN(nccl_api().AllReduce(ctx->eflags.p, ctx->eflags.p, (size_t)E, kNcclInt32, kNcclMax, ctx->nccl_comm, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_flags, ctx->eflags.p, (size_t)E * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        ctx->st.kernel_launches += 2;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    if (reduce_grads) {
        rc = for_flagged_planes(ctx, E, (size_t)3 * P.N, d_grads, d_dst, 0);
        if (rc) return rc;
    }
    int n_jobs_now = *(const int*)(ctx->h_out + 28);
    if (n_jobs_now < 1) n_jobs_now = 1;
    int group = pick_group(ctx, P, n_jobs_now);
    rc = run_refine(ctx, pl, ctx->poses.as<Pose>(), ctx->poses_ref.as<Pose>(), ctx->contrib.as<int>(), sc + S_NCONTRIB, 0, M, group);
    if (rc) return rc;
    mark(ctx, EV_REFINE);
    const int tiles = bwd_tiles(P.N);
    CK(ctx->losses.ensure((size_t)M * 8));
    CK(ctx->red.ensure((size_t)M * tiles * bwd_red_vals() * 8));
    CK(ctx->hypgrad.ensure((size_t)M * bwd_hypgrad_bytes()));
    CK(ctx->job_of.ensure((size_t)(M > E ? M : E) * 4));
    BwdArgs b;
    b.coords = pl.d_coords;
    b.grads = d_grads;
    b.assign32 = ctx->assign32.as<int>();
    b.perm = ctx->perm.as<int>();
    b.counts = ctx->counts.as<int>();
    b.offsets = ctx->offsets.as<int>();
    b.init = ctx->poses.as<Pose>();
    b.ref = ctx->poses_ref.as<Pose>();
    b.cells = ctx->cells.as<int>();
    b.probs = ctx->probs.as<double>();
    b.contrib = ctx->contrib.as<int>();
    b.n_contrib = sc + S_NCONTRIB;
    b.job_of = ctx->job_of.as<int>();
    b.masks = ctx->masks.as<uint32_t>();
    b.mask_words = (P.N + 31) / 32;
    b.rounds = ctx->rounds.as<int>();
    b.losses = ctx->losses.as<double>();
    b.out_loss = ctx->stats.as<double>() + 4;
    b.red = ctx->red.as<double>();
    b.hyp_grad = ctx->hypgrad.p;
    if (is_device_ptr(gt_pose)) {
        CK(cudaMemcpyAsync(ctx->h_out, gt_pose, 16 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        memcpy(b.gt, ctx->h_out, 16 * sizeof(float));
    } else {
        memcpy(b.gt, gt_pose, 16 * sizeof(float));
    }
    b.wRot = wRot; b.wTrans = wTrans; b.cut = cut;
    b.P = P;
    b.expected_override = nullptr;
    double global_loss = 0;
    if (exchange) {
        // exchange 2: the expectation sum_h p_h loss_h runs over the hypotheses of all ranks (esac.cpp:357-362, esac_derivative.h:372-374)
        launch_backward_losses(b, ctx->stream);
        CK(cudaMemcpyAsync(ctx->h_dbl, ctx->stats.as<double>() + 4, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        double v[1] = {ctx->h_dbl[0]};
        if (exchange(user, 2, v, 1) != 0) return fail(ctx, ESACB200_ERR_ARG, "exchange callback failed (phase 2)");
        global_loss = v[0];
        ctx->h_dbl[6] = v[0];
        CK(cudaMemcpyAsync(ctx->stats.as<double>() + 7, ctx->h_dbl + 6, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        b.expected_override = ctx->stats.as<double>() + 7;
        ctx->st.kernel_launches += 1;
    } else if (use_nccl) {
        // exchange 2 on the device: all-reduce of the partial expectations, no host round trip
        launch_backward_losses(b, ctx->stream);
        CKN(nccl_api().AllReduce(ctx->stats.as<double>() + 4, ctx->stats.as<double>() + 7, 1, kNcclFloat64, kNcclSum, ctx->nccl_comm,
                                 ctx->stream));
        b.expected_override = ctx->stats.as<double>() + 7;
        ctx->st.kernel_launches += 2;
    }
    launch_backward(b, M, ctx->stream);
    CK(cudaGetLastError());
    ctx->st.kernel_launches += 5;
    if (reduce_grads) {
        rc = for_flagged_planes(ctx, E, (size_t)3 * P.N, d_grads, d_dst, 1);
        if (rc) return rc;
        CK(cudaGetLastError());
        d_grads = d_dst;
    }
    mark(ctx, EV_BWD);
    if (grads_on_host) CK(cudaMemcpyAsync(grads, d_grads, cbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_out + 20, sc, 8 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_dbl, ctx->stats.p, 8 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    const int* hs = (const int*)(ctx->h_out + 20);
    if (hs[S_FLAGS]) return fail(ctx, ESACB200_ERR_ARG, "hypAssignment holds an expert index outside [0, %d)", E);
    if (use_nccl) global_loss = ctx->h_dbl[7];
    if (out_loss) *out_loss = (exchange || use_nccl) ? global_loss : ctx->h_dbl[4];
    ctx->st.M = M;
    ctx->st.winner = hs[S_WINNER];
    ctx->st.n_contrib = hs[S_NCONTRIB];
    ctx->st.entropy = ctx->h_dbl[0];
    ctx->st.expected_loss = (exchange || use_nccl) ? global_loss : ctx->h_dbl[4];
    ctx->last_M = M;
    ctx->last_backward = true;
    finish_stats(ctx);
    ctx->inj_M = ctx->inj_T = 0;
    return ESACB200_OK;
}

int esacb200_backward(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W, const int64_t* assign,
                      int64_t assign_stride, int M, const float* gt_pose, float wRot, float wTrans, float cut, int shiftX,
                      int shiftY, float f, float ppx, float ppy, float tau, float alpha, float beta, float maxReproj, int sub,
                      double* out_loss) try {
    return backward_impl(ctx, coords, grads, E, H, W, assign, assign_stride, M, gt_pose, wRot, wTrans, cut, shiftX, shiftY, f, ppx,
                         ppy, tau, alpha, beta, maxReproj, sub, nullptr, nullptr, out_loss);
} ESAC_ABI_CATCH(ctx)

int esacb200_backward_sharded(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W, const int64_t* assign,
                              int64_t assign_stride, int M, const float* gt_pose, float wRot, float wTrans, float cut,
                              int shiftX, int shiftY, float f, float ppx, float ppy, float tau, float alpha, float beta,
                              float maxReproj, int sub, esacb200_exchange_fn exchange, void* user, double* out_loss) try {
    if (!exchange) return ctx ? fail(ctx, ESACB200_ERR_ARG, "exchange callback is null") : ESACB200_ERR_ARG;
    return backward_impl(ctx, coords, grads, E, H, W, assign, assign_stride, M, gt_pose, wRot, wTrans, cut, shiftX, shiftY, f, ppx,
                         ppy, tau, alpha, beta, maxReproj, sub, exchange, user, out_loss);
} ESAC_ABI_CATCH(ctx)

// esac_backward with the experts / hypotheses sharded over the ranks of the communicator: the two exchanges of the path
// (SURVEY 8e) run as NCCL collectives on the context's stream -- an all-gather of two doubles per rank and an all-reduce of
// one -- with no host callback.  M may be 0: the rank then only takes part in the collectives.
int esacb200_backward_sharded_nccl(esacb200_ctx* ctx, const float* coords, float* grads, int E, int H, int W,
                                   const int64_t* assign, int64_t assign_stride, int M, const float* gt_pose, float wRot,
                                   float wTrans, float cut, int shiftX, int shiftY, float f, float ppx, float ppy, float tau,
                                   float alpha, float beta, float maxReproj, int sub, int reduce_grads, double* out_loss) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!ctx->nccl_comm) return fail(ctx, ESACB200_ERR_ARG, "no communicator: call esacb200_comm_init first");
    if (M > 0)
        return backward_impl(ctx, coords, grads, E, H, W, assign, assign_stride, M, gt_pose, wRot, wTrans, cut, shiftX, shiftY, f, ppx,
                             ppy, tau, alpha, beta, maxReproj, sub, nullptr, nullptr, out_loss, /*use_nccl=*/true, reduce_grads != 0);
    // no hypotheses here: neutral contributions to both collectives
    begin_call(ctx);
    CK(ctx->stats.ensure(8 * 8));
    CK(ctx->gathered.ensure((size_t)ctx->comm_world * 2 * 8));
    ctx->h_dbl[0] = 0.; ctx->h_dbl[1] = -1e300; ctx->h_dbl[2] = 0.;  // stats[4] partial expectation, [5] max score, [6] sum exp
    CK(cudaMemcpyAsync(ctx->stats.as<double>() + 4, ctx->h_dbl, 3 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    // the collectives below come in the order backward_impl issues them on the ranks that do hold hypotheses
    CKN(nccl_api().AllGather(ctx->stats.as<double>() + 5, ctx->gathered.p, 2, kNcclFloat64, ctx->nccl_comm, ctx->stream));
    const size_t n = reduce_grads ? (size_t)E * 3 * H * W : 0;
    float* d_dst = grads;
    if (reduce_grads) {  // zero contribution to the gradient sum, then the sum is added to this rank's tensor like everywhere
        if (!grads || E <= 0 || H <= 0 || W <= 0) return fail(ctx, ESACB200_ERR_ARG, "reduce_grads needs the gradient tensor and its shape on every rank");
        CK(ctx->grads_work.ensure(n * 4));
        int rc = ensure_host_flags(ctx, E);
        if (rc) return rc;
        CK(ctx->eflags.ensure((size_t)E * sizeof(int)));
        CK(cudaMemsetAsync(ctx->eflags.p, 0, (size_t)E * sizeof(int), ctx->stream));
        CKN(nccl_api().AllReduce(ctx->eflags.p, ctx->eflags.p, (size_t)E, kNcclInt32, kNcclMax, ctx->nccl_comm, ctx->stream));
        CK(cudaMemcpyAsync(ctx->h_flags, ctx->eflags.p, (size_t)E * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (!is_device_ptr(grads)) {
            CK(ctx->grads.ensure(n * 4));
            CK(cudaMemcpyAsync(ctx->grads.p, grads, n * 4, cudaMemcpyHostToDevice, ctx->stream));
            d_dst = ctx->grads.as<float>();
        }
        rc = for_flagged_planes(ctx, E, (size_t)3 * H * W, ctx->grads_work.as<float>(), d_dst, 0);
        if (rc) return rc;
    }
    CKN(nccl_api().AllReduce(ctx->stats.as<double>() + 4, ctx->stats.as<double>() + 7, 1, kNcclFloat64, kNcclSum, ctx->nccl_comm,
                             ctx->stream));
    if (reduce_grads) {
        int rc = for_flagged_planes(ctx, E, (size_t)3 * H * W, ctx->grads_work.as<float>(), d_dst, 1);
        if (rc) return rc;
        if (!is_device_ptr(grads)) CK(cudaMemcpyAsync(grads, ctx->grads.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(ctx->h_dbl + 4, ctx->stats.as<double>() + 7, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    if (out_loss) *out_loss = ctx->h_dbl[4];
    ctx->st.expected_loss = ctx->h_dbl[4];
    ctx->last_M = 0;
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
// esac_backward over a batch.  Every image is an independent problem (SURVEY 8e: "images in a batch are fully
// independent"), so the images are dealt round-robin to a few worker contexts, each driven by its own host thread on its
// own stream: the small kernels of one image fill the gaps the host synchronisations of another leave.
int esacb200_backward_batch(esacb200_ctx* ctx, int B, const float* coords, float* grads, int E, int H, int W,
                            const int64_t* assign, int64_t assign_stride, int M, const float* gt_poses, float wRot,
                            float wTrans, float cut, const int* shiftX, const int* shiftY, float f, float ppx, float ppy,
                            float tau, float alpha, float beta, float maxReproj, int sub, double* out_losses) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !grads || !assign || !gt_poses || B <= 0) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument or empty batch");
    if (ctx->inj_M) return fail(ctx, ESACB200_ERR_ARG, "injected cells are a single-image test hook");
    if (E <= 0 || H <= 0 || W <= 0 || M <= 0) return fail(ctx, ESACB200_ERR_ARG, "bad sizes E=%d H=%d W=%d M=%d", E, H, W, M);
    const size_t cstride = (size_t)E * 3 * H * W;
    const int64_t arow = assign_stride == 0 ? 0 : (int64_t)M * assign_stride;
    std::vector<float> gt_host;
    const float* gt = gt_poses;
    if (is_device_ptr(gt_poses)) {
        gt_host.resize((size_t)B * 16);
        CK(cudaMemcpyAsync(gt_host.data(), gt_poses, gt_host.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        gt = gt_host.data();
    }
    // everything the caller queued on its stream (the experts' outputs) is visible to the workers after this
    CK(cudaStreamSynchronize(ctx->stream));
    std::vector<uint64_t> seeds((size_t)B);
    for (int b = 0; b < B; ++b) seeds[b] = call_seed(ctx);
    const int nw = ctx->batch_workers < B ? ctx->batch_workers : B;
    while ((int)ctx->workers.size() < nw) {
        esacb200_ctx* w = nullptr;
        int rc = esacb200_create(ctx->device, &w);
        if (rc) return fail(ctx, rc, "cannot create batch worker context");
        ctx->workers.push_back(w);
    }
    std::vector<int> rcs((size_t)nw, 0), failed_at((size_t)nw, -1);
    std::vector<esacb200_stats> last((size_t)nw);
    std::vector<unsigned long long> launches((size_t)nw, 0);
    auto work = [&](int wi) {
        try {
        esacb200_ctx* w = ctx->workers[wi];
        cudaSetDevice(ctx->device);
        w->max_tries = ctx->max_tries;
        w->max_ref_steps = ctx->max_ref_steps;
        w->refine_group_opt = ctx->refine_group_opt;
        w->refine_jobs_per_group = ctx->refine_jobs_per_group;
        w->refine_compact = ctx->refine_compact;
        w->refine_pretest = ctx->refine_pretest;
        w->sample_prefilter = ctx->sample_prefilter;
        w->sample_tail_boost = ctx->sample_tail_boost;
        w->hyp_offset = ctx->hyp_offset;
        w->hyp_stride = ctx->hyp_stride;
        w->score_ppt_opt = ctx->score_ppt_opt;
        w->score_hc_opt = ctx->score_hc_opt;
        w->fixed_seed = 1;
        for (int b = wi; b < B; b += nw) {
            w->seed = seeds[b];
            double loss = 0;
            int rc = backward_impl(w, coords + (size_t)b * cstride, grads + (size_t)b * cstride, E, H, W, assign + (size_t)b * arow,
                                   assign_stride, M, gt + (size_t)b * 16, wRot, wTrans, cut, shiftX ? shiftX[b] : 0,
                                   shiftY ? shiftY[b] : 0, f, ppx, ppy, tau, alpha, beta, maxReproj, sub, nullptr, nullptr, &loss);
            if (rc) { rcs[wi] = rc; failed_at[wi] = b; return; }
            if (out_losses) out_losses[b] = loss;
            launches[wi] += w->st.kernel_launches;
        }
        last[wi] = w->st;
        } catch (...) {  // an exception escaping a std::thread would terminate the process
            rcs[wi] = ESACB200_ERR_ARG;
            failed_at[wi] = -1;
            snprintf(ctx->workers[wi]->err, sizeof(ctx->workers[wi]->err), "host-side failure in a batch worker");
        }
    };
    const auto t0 = std::chrono::steady_clock::now();
    if (nw == 1) {
        work(0);
    } else {
        std::vector<std::thread> th;
        for (int wi = 0; wi < nw; ++wi) th.emplace_back(work, wi);
        for (auto& t : th) t.join();
    }
    const double wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    for (int wi = 0; wi < nw; ++wi)
        if (rcs[wi]) return fail(ctx, rcs[wi], "image %d: %s", failed_at[wi], ctx->workers[wi]->err);
    // statistics of the call: those of the worker that handled the last image, wall time and launches of the whole batch
    ctx->st = last[(B - 1) % nw];
    unsigned long long total = 0;
    for (int wi = 0; wi < nw; ++wi) total += launches[wi];
    ctx->st.kernel_launches = total;
    ctx->st.ms_total = (float)wall_ms;
    ctx->last_M = 0;  // the per-hypothesis buffers live in the workers
    ctx->last_backward = true;
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
int esacb200_assign_hypotheses(esacb200_ctx* ctx, int B, int E, int M, const float* weights, int keep_top, int single_expert,
                               uint64_t seed, int64_t* out_assign, float* out_hist) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!weights || !out_assign) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    if (B <= 0 || E <= 0 || M <= 0) return fail(ctx, ESACB200_ERR_ARG, "bad sizes B=%d E=%d M=%d", B, E, M);
    if (E > assign_max_experts()) return fail(ctx, ESACB200_ERR_ARG, "E=%d exceeds the %d experts one CTA holds", E, assign_max_experts());
    const bool w_host = !is_device_ptr(weights), a_host = !is_device_ptr(out_assign), h_host = out_hist && !is_device_ptr(out_hist);
    const size_t wb = (size_t)B * E * sizeof(float), ab = (size_t)B * M * sizeof(int64_t);
    // staging layout in `scratch`: [flags int (16 B)] [weights] [hist] [assign]
    const size_t off_w = 16, off_h = off_w + ((wb + 15) & ~(size_t)15), off_a = off_h + ((wb + 15) & ~(size_t)15);
    CK(ctx->scratch.ensure(off_a + ab));
    char* base = (char*)ctx->scratch.p;
    const float* d_w = weights;
    if (w_host) {
        CK(cudaMemcpyAsync(base + off_w, weights, wb, cudaMemcpyHostToDevice, ctx->stream));
        d_w = (const float*)(base + off_w);
    }
    int64_t* d_a = a_host ? (int64_t*)(base + off_a) : out_assign;
    float* d_h = !out_hist ? nullptr : (h_host ? (float*)(base + off_h) : out_hist);
    CK(cudaMemsetAsync(base, 0, 16, ctx->stream));
    launch_assign(d_w, B, E, M, keep_top, single_expert, seed, d_a, d_h, (int*)base, ctx->stream);
    CK(cudaGetLastError());
    if (a_host) CK(cudaMemcpyAsync(out_assign, d_a, ab, cudaMemcpyDeviceToHost, ctx->stream));
    if (h_host) CK(cudaMemcpyAsync(out_hist, d_h, wb, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_out + 30, base, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int flags = *(const int*)(ctx->h_out + 30);
    if (flags & 1) return fail(ctx, ESACB200_ERR_ARG, "probability tensor contains either inf, nan or element < 0");
    if (flags & 2) return fail(ctx, ESACB200_ERR_ARG, "invalid multinomial distribution (sum of probabilities <= 0)");
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// -------------------------------------------------------------------------------------------------
int esacb200_reproj_loss(esacb200_ctx* ctx, int B, const float* coords, float* grads, int H, int W, const float* gt_poses,
                         const int* shiftX, const int* shiftY, float f, float ppx, float ppy, int sub, float cut,
                         float maxReproj, float minDepth, double* out_losses) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!coords || !gt_poses || !out_losses) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    if (B <= 0 || H <= 0 || W <= 0 || sub <= 0) return fail(ctx, ESACB200_ERR_ARG, "bad sizes B=%d H=%d W=%d sub=%d", B, H, W, sub);
    if ((long long)H * W > (1ll << 30)) return fail(ctx, ESACB200_ERR_ARG, "map %dx%d too large", W, H);
    begin_call(ctx);
    const int N = H * W;
    const size_t cbytes = (size_t)B * 3 * N * sizeof(float);
    const bool c_host = !is_device_ptr(coords), g_host = grads && !is_device_ptr(grads);
    const float* d_coords = coords;
    float* d_grads = grads;
    if (c_host) {
        CK(ctx->coords.ensure(cbytes));
        CK(cudaMemcpyAsync(ctx->coords.p, coords, cbytes, cudaMemcpyHostToDevice, ctx->stream));
        d_coords = ctx->coords.as<float>();
    }
    if (g_host) {
        CK(ctx->grads.ensure(cbytes));
        d_grads = ctx->grads.as<float>();
    }
    std::vector<float> gt((size_t)B * 16);
    if (is_device_ptr(gt_poses)) {
        CK(cudaMemcpyAsync(gt.data(), gt_poses, gt.size() * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    } else {
        memcpy(gt.data(), gt_poses, gt.size() * sizeof(float));
    }
    // world->camera rows: inverse of the affine camera->world matrix (torch's .inverse()[0:3,:], ref_expert.py:127)
    std::vector<float> img((size_t)B * 16, 0.f);
    for (int b = 0; b < B; ++b) {
        const float* T = gt.data() + (size_t)b * 16;
        double A[9], inv[9];
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) A[r * 3 + c] = T[r * 4 + c];
        const double det = A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) + A[2] * (A[3] * A[7] - A[4] * A[6]);
        if (det == 0. || !(det == det)) return fail(ctx, ESACB200_ERR_ARG, "image %d: ground-truth pose is singular", b);
        inv[0] = (A[4] * A[8] - A[5] * A[7]) / det; inv[1] = (A[2] * A[7] - A[1] * A[8]) / det; inv[2] = (A[1] * A[5] - A[2] * A[4]) / det;
        inv[3] = (A[5] * A[6] - A[3] * A[8]) / det; inv[4] = (A[0] * A[8] - A[2] * A[6]) / det; inv[5] = (A[2] * A[3] - A[0] * A[5]) / det;
        inv[6] = (A[3] * A[7] - A[4] * A[6]) / det; inv[7] = (A[1] * A[6] - A[0] * A[7]) / det; inv[8] = (A[0] * A[4] - A[1] * A[3]) / det;
        float* o = img.data() + (size_t)b * 16;
        for (int r = 0; r < 3; ++r) {
            for (int c = 0; c < 3; ++c) o[r * 4 + c] = (float)inv[r * 3 + c];
            o[r * 4 + 3] = (float)-(inv[r * 3] * T[3] + inv[r * 3 + 1] * T[7] + inv[r * 3 + 2] * T[11]);
        }
        o[12] = shiftX ? (float)shiftX[b] : 0.f;
        o[13] = shiftY ? (float)shiftY[b] : 0.f;
    }
    const int bpi = reproj_blocks_per_image(N, B, ctx->sm_count);
    // scratch layout: [tickets B u32, padded] [img B*16 f32] [losses B f64] [partials B*bpi f64]
    const size_t off_img = ((size_t)B * 4 + 63) & ~(size_t)63, off_loss = off_img + (size_t)B * 64,
                 off_part = off_loss + (((size_t)B * 8 + 63) & ~(size_t)63);
    CK(ctx->scratch.ensure(off_part + (size_t)B * bpi * 8));
    char* base = (char*)ctx->scratch.p;
    CK(cudaMemsetAsync(base, 0, off_img, ctx->stream));
    CK(cudaMemcpyAsync(base + off_img, img.data(), img.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    mark(ctx, EV_H2D);
    mark(ctx, EV_FOLD);  // ms_score = the kernel alone
    launch_reproj(d_coords, d_grads, (const float*)(base + off_img), B, N, W, (float)sub, f, ppx, ppy, cut, maxReproj, minDepth, bpi,
                  (double*)(base + off_part), (unsigned*)base, (double*)(base + off_loss), ctx->stream);
    CK(cudaGetLastError());
    ctx->st.kernel_launches += 1;
    mark(ctx, EV_SCORE);
    if (g_host) CK(cudaMemcpyAsync(grads, d_grads, cbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_losses, base + off_loss, (size_t)B * 8, cudaMemcpyDeviceToHost, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    ctx->last_M = 0;
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_init_loss(esacb200_ctx* ctx, int B, const float* pred, int pred_H, int pred_W, const float* gt, int gt_H,
                       int gt_W, float* grads, float cutLoss, double* out_sums, int64_t* out_counts) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!pred || !gt || !out_sums || !out_counts) return fail(ctx, ESACB200_ERR_ARG, "null pointer argument");
    if (B <= 0 || B > 65535 || pred_H <= 0 || pred_W <= 0 || gt_H <= 0 || gt_W <= 0)
        return fail(ctx, ESACB200_ERR_ARG, "bad sizes B=%d pred %dx%d gt %dx%d", B, pred_H, pred_W, gt_H, gt_W);
    if (abs(pred_H - gt_H) > 1 || abs(pred_W - gt_W) > 1)   // util.assert_size
        return fail(ctx, ESACB200_ERR_ARG, "Tensor size mismatch: prediction %dx%d, ground truth %dx%d (tolerance 1 px)",
                    pred_H, pred_W, gt_H, gt_W);
    if ((long long)pred_H * pred_W > (1ll << 30) || (long long)gt_H * gt_W > (1ll << 30))
        return fail(ctx, ESACB200_ERR_ARG, "map too large");
    begin_call(ctx);
    const size_t pbytes = (size_t)B * 3 * pred_H * pred_W * sizeof(float), gbytes = (size_t)B * 3 * gt_H * gt_W * sizeof(float);
    const bool p_host = !is_device_ptr(pred), t_host = !is_device_ptr(gt), g_host = grads && !is_device_ptr(grads);
    const float* d_pred = pred;
    const float* d_gt = gt;
    float* d_grads = grads;
    if (p_host) {
        CK(ctx->coords.ensure(pbytes));
        CK(cudaMemcpyAsync(ctx->coords.p, pred, pbytes, cudaMemcpyHostToDevice, ctx->stream));
        d_pred = ctx->coords.as<float>();
    }
    if (t_host) {
        CK(ctx->coords_alt.ensure(gbytes));
        CK(cudaMemcpyAsync(ctx->coords_alt.p, gt, gbytes, cudaMemcpyHostToDevice, ctx->stream));
        d_gt = ctx->coords_alt.as<float>();
    }
    if (g_host) {
        CK(ctx->grads.ensure(pbytes));
        d_grads = ctx->grads.as<float>();
    }
    const int bpi = init_loss_blocks_per_image(pred_H * pred_W);
    // scratch layout: [tickets B u32, padded] [sums B f64] [counts B i64] [partial sums B*bpi f64] [partial counts B*bpi u32]
    const size_t pad = 63, off_sum = ((size_t)B * 4 + pad) & ~pad, off_cnt = off_sum + (((size_t)B * 8 + pad) & ~pad),
                 off_psum = off_cnt + (((size_t)B * 8 + pad) & ~pad), off_pcnt = off_psum + (((size_t)B * bpi * 8 + pad) & ~pad);
    CK(ctx->scratch.ensure(off_pcnt + (size_t)B * bpi * 4));
    char* base = (char*)ctx->scratch.p;
    CK(cudaMemsetAsync(base, 0, off_sum, ctx->stream));
    mark(ctx, EV_H2D);
    mark(ctx, EV_FOLD);  // ms_score = the kernel alone
    launch_init_loss(d_pred, d_gt, d_grads, B, pred_H, pred_W, gt_H, gt_W, cutLoss, bpi, (double*)(base + off_psum),
                     (unsigned*)(base + off_pcnt), (unsigned*)base, (double*)(base + off_sum), (long long*)(base + off_cnt),
                     ctx->stream);
    CK(cudaGetLastError());
    ctx->st.kernel_launches += 1;
    mark(ctx, EV_SCORE);
    if (g_host) CK(cudaMemcpyAsync(grads, d_grads, pbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_sums, base + off_sum, (size_t)B * 8, cudaMemcpyDefault, ctx->stream));
    CK(cudaMemcpyAsync(out_counts, base + off_cnt, (size_t)B * 8, cudaMemcpyDefault, ctx->stream));
    mark(ctx, EV_END);
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    ctx->last_M = 0;
    finish_stats(ctx);
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_copy_last_scores(esacb200_ctx* ctx, double* dst, int M) try {
    if (!ctx || !dst) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (M != ctx->last_M) return fail(ctx, ESACB200_ERR_ARG, "last call had M=%d, asked for %d", ctx->last_M, M);
    CK(cudaMemcpyAsync(dst, ctx->scores.p, (size_t)M * 8, cudaMemcpyDefault, ctx->stream));
    if (!is_device_ptr(dst)) CK(cudaStreamSynchronize(ctx->stream));
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_get_refine_profile(esacb200_ctx* ctx, long long* out16) try {
    if (!ctx || !out16) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!ctx->prof.p) return fail(ctx, ESACB200_ERR_ARG, "no refinement ran with option refine_profile = 1");
    CK(cudaMemcpy(out16, ctx->prof.p, 16 * 8, cudaMemcpyDeviceToHost));
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_get_stats(esacb200_ctx* ctx, esacb200_stats* out) {
    if (!ctx || !out) return ESACB200_ERR_ARG;
    *out = ctx->st;
    return ESACB200_OK;
}

int esacb200_get_sample_trace(esacb200_ctx* ctx, unsigned long long* out512) try {
    if (!ctx || !out512) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    if (!ctx->smp_trace.p) return fail(ctx, ESACB200_ERR_ARG, "no sampling ran with option sample_trace = 1");
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(out512, ctx->smp_trace.p, 512 * 8, cudaMemcpyDeviceToHost));
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_get_sample_profile(esacb200_ctx* ctx, long long* out8) try {
    if (!ctx || !out8) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    for (int i = 0; i < 8; ++i) out8[i] = 0;
    const int G = ctx->smp_groups_last, M = ctx->last_M, Mg = ctx->smp_Mg_last;
    if (G <= 0 || M <= 0) return fail(ctx, ESACB200_ERR_ARG, "no previous call");
    CK(cudaStreamSynchronize(ctx->stream));
    const size_t per_group_ints = (size_t)2 * Mg + 8;
    for (int g = 0; g < G; ++g) {
        int c[8];
        const int* src = ctx->smp_int.as<int>() + 4 * (size_t)M + g * per_group_ints + 2 * (size_t)Mg;
        CK(cudaMemcpy(c, src, sizeof(c), cudaMemcpyDeviceToHost));
        out8[0] += (unsigned)c[5];
        out8[1] += (unsigned)c[6];
        out8[2] = out8[2] > c[7] ? out8[2] : c[7];
        out8[3] += c[0];
        out8[4] += c[2];
    }
    out8[5] = G;
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

int esacb200_get_hypotheses(esacb200_ctx* ctx, double* poses6, int32_t* cells, int32_t* tries, double* scores,
                            double* probs, double* refined6, double* losses) try {
    if (!ctx) return ESACB200_ERR_ARG;
    DeviceGuard device_guard(ctx->device);
    const int M = ctx->last_M;
    if (M <= 0) return fail(ctx, ESACB200_ERR_ARG, "no previous call");
    if (poses6) CK(cudaMemcpy(poses6, ctx->poses.p, (size_t)M * sizeof(Pose), cudaMemcpyDeviceToHost));
    if (cells) CK(cudaMemcpy(cells, ctx->cells.p, (size_t)M * 32, cudaMemcpyDeviceToHost));
    if (tries) CK(cudaMemcpy(tries, ctx->tries.p, (size_t)M * 4, cudaMemcpyDeviceToHost));
    if (scores) CK(cudaMemcpy(scores, ctx->scores.p, (size_t)M * 8, cudaMemcpyDeviceToHost));
    if (probs) CK(cudaMemcpy(probs, ctx->probs.p, (size_t)M * 8, cudaMemcpyDeviceToHost));
    if (refined6) CK(cudaMemcpy(refined6, ctx->poses_ref.p, (size_t)M * sizeof(Pose), cudaMemcpyDeviceToHost));
    if (losses) {
        if (!ctx->last_backward) return fail(ctx, ESACB200_ERR_ARG, "losses exist only after backward");
        CK(cudaMemcpy(losses, ctx->losses.p, (size_t)M * 8, cudaMemcpyDeviceToHost));
    }
    return ESACB200_OK;
} ESAC_ABI_CATCH(ctx)

// ------------------------------------------------------------------------------------------------
// host test hooks (esac_b200_testhooks.h)
// ------------------------------------------------------------------------------------------------
void esacb200_host_rodrigues(const double r[3], double R[9], double J[27]) { rodrigues_v2m(r, R, J); }
void esacb200_host_rodrigues_inv(const double R[9], double r[3]) { rodrigues_m2v(R, r); }

int esacb200_host_p3p_all(const double* y9, const double* x9, double* Rs36, double* ts12) {
    double y[3][3], x[3][3], Rs[4][9], ts[4][3];
    for (int i = 0; i < 3; ++i)
        for (int c = 0; c < 3; ++c) { y[i][c] = y9[i * 3 + c]; x[i][c] = x9[i * 3 + c]; }
    int n = p3p_solve(y, x, Rs, ts);
    for (int s = 0; s < n; ++s) {
        for (int c = 0; c < 9; ++c) Rs36[s * 9 + c] = Rs[s][c];
        for (int c = 0; c < 3; ++c) ts12[s * 3 + c] = ts[s][c];
    }
    return n;
}

int esacb200_host_p3p_pose(const float* obj12, const float* img8, float f, float ppx, float ppy, float tau, double* pose6,
                           int* gate) {
    float obj[4][3], img[4][2];
    for (int i = 0; i < 4; ++i) {
        for (int c = 0; c < 3; ++c) obj[i][c] = obj12[i * 3 + c];
        for (int c = 0; c < 2; ++c) img[i][c] = img8[i * 2 + c];
    }
    Pose p;
    bool ok = p3p_pose(obj, img, (double)f, (double)ppx, (double)ppy, p);
    if (gate) *gate = 0;
    if (!ok) { for (int i = 0; i < 6; ++i) pose6[i] = 0; return 0; }
    for (int i = 0; i < 3; ++i) { pose6[i] = p.r[i]; pose6[3 + i] = p.t[i]; }
    if (gate) *gate = minimal_set_gate(obj, img, p, (double)f, (double)ppx, (double)ppy, tau) ? 1 : 0;
    return 1;
}

void esacb200_host_try(const float* obj12, const float* img8, float f, float ppx, float ppy, float tau, float margin,
                       int* may_pass, int* accept) {
    float obj[4][3], img[4][2];
    for (int i = 0; i < 4; ++i) {
        for (int c = 0; c < 3; ++c) obj[i][c] = obj12[i * 3 + c];
        for (int c = 0; c < 2; ++c) img[i][c] = img8[i * 2 + c];
    }
    *may_pass = p3p_may_pass_fast(obj, img, f, ppx, ppy, tau, margin) ? 1 : 0;
    Pose p;
    bool ok = p3p_pose(obj, img, (double)f, (double)ppx, (double)ppy, p);
    *accept = (ok && minimal_set_gate(obj, img, p, (double)f, (double)ppx, (double)ppy, tau)) ? 1 : 0;
}

void esacb200_host_try_verdict(const float* obj12, const float* img8, float f, float ppx, float ppy, float tau, int* accept,
                               double* pose6) {
    float obj[4][3], img[4][2];
    for (int i = 0; i < 4; ++i) {
        for (int c = 0; c < 3; ++c) obj[i][c] = obj12[i * 3 + c];
        for (int c = 0; c < 2; ++c) img[i][c] = img8[i * 2 + c];
    }
    Pose p;
    const bool ok = p3p_pose(obj, img, (double)f, (double)ppx, (double)ppy, p, 1.25 * (double)tau + 1.);  // as hyp.cu exact_try(verdict_only)
    *accept = (ok && minimal_set_gate(obj, img, p, (double)f, (double)ppx, (double)ppy, tau)) ? 1 : 0;
    if (pose6 && ok)
        for (int i = 0; i < 3; ++i) { pose6[i] = p.r[i]; pose6[3 + i] = p.t[i]; }
}

void esacb200_host_project(const double pose6[6], float f, float ppx, float ppy, const float X[3], float uv_f[2],
                           double uv[2], double J12[12]) {
    double R[9], dRdr[27];
    rodrigues_v2m(pose6, R, dRdr);
    project_point_f(R, pose6 + 3, (double)f, (double)ppx, (double)ppy, X[0], X[1], X[2], uv_f[0], uv_f[1]);
    double Ju[6], Jv[6];
    project_point_jac(R, pose6 + 3, dRdr, (double)f, (double)ppx, (double)ppy, (double)X[0], (double)X[1], (double)X[2], uv[0],
                      uv[1], Ju, Jv);
    for (int i = 0; i < 6; ++i) { J12[i] = Ju[i]; J12[6 + i] = Jv[i]; }
}

double esacb200_host_loss(const double* T1, const double* T2, double wRot, double wTrans, double cut) {
    return pose_loss(T1, T2, wRot, wTrans, cut);
}

void esacb200_host_dloss(const double est6[6], const double gt6[6], double wRot, double wTrans, double cut, double out6[6]) {
    Pose a, b;
    for (int i = 0; i < 3; ++i) { a.r[i] = est6[i]; a.t[i] = est6[3 + i]; b.r[i] = gt6[i]; b.t[i] = gt6[3 + i]; }
    pose_dloss(a, b, wRot, wTrans, cut, out6);
}

void esacb200_host_pose2trans(const double pose6[6], double T16[16]) {
    Pose a;
    for (int i = 0; i < 3; ++i) { a.r[i] = pose6[i]; a.t[i] = pose6[3 + i]; }
    pose2trans(a, T16);
}

void esacb200_host_trans2pose(const double T16[16], double pose6[6]) {
    Pose a;
    trans2pose(T16, a);
    for (int i = 0; i < 3; ++i) { pose6[i] = a.r[i]; pose6[3 + i] = a.t[i]; }
}

void esacb200_host_dprojectdobj(const float pt[2], const float obj[3], const double pose6[6], float f, float ppx, float ppy,
                                float maxReproj, double out3[3]) {
    double R[9];
    rodrigues_v2m(pose6, R, nullptr);
    d_project_d_obj(pt[0], pt[1], obj[0], obj[1], obj[2], R, pose6 + 3, (double)f, (double)ppx, (double)ppy, (double)maxReproj, out3);
}

void esacb200_host_pinv6(const double A[36], double out[36]) { pinv_sym6(A, out); }

void esacb200_host_draw_cells(uint64_t seed, uint32_t h, uint32_t t, int W, int H, int32_t* cells8) {
    int cx[4], cy[4];
    draw_minimal_set(seed, h, t, W, H, cx, cy);
    for (int j = 0; j < 4; ++j) { cells8[2 * j] = cx[j]; cells8[2 * j + 1] = cy[j]; }
}

}  // extern "C"
