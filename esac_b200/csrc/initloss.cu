// Scene-coordinate loss of the expert initialisation stage, forward and gradient in one pass.
//
// init_expert.py:112-132 crops prediction and target to a common size (util.assert_size), masks out target cells that are
// all zero, takes the Euclidean distance of every remaining cell and applies the same L1 / square-root robust loss as the
// refinement stage, then lets autograd walk back through two boolean-mask gathers (each a device->host synchronisation).
// Here that is one launch over a batch of maps: 24 B read + 12 B written per cell, each thread 4 consecutive cells with
// 128-bit streaming loads/stores where the layout allows.  The crop is a pair of strides, not a copy.
//
//   valid = |gt|.sum(0) != 0            (any nonzero component; NaN counts as valid, +-0 does not)    init_expert.py:119
//   d     = ||pred - gt||                                                                                   :123
//   sum   = sum_{d<=cut} d + sum_{d>cut} sqrt(cut*d),   count = number of valid cells (NaN d included)      :126-130
//
// The kernel returns the per-image (sum, count) and writes d sum / d pred: the 1/count of the mean is only known once the
// whole image has been read, and the caller folds it into the one multiply its backward does anyway (autograd.InitLoss).
// Sum (fp64) and count are reduced in a fixed order -- block partials, then the last block of the image -- so repeated
// calls return bit-identical results.
#include "esac_internal.h"

namespace esacb200 {

namespace {

constexpr int kThreads = 256;
constexpr int kCellsPerThread = 4;

// One cell in IEEE fp32 (the kernel is far below its issue budget, so correctly rounded sqrt / division cost nothing).
// Gradient of the per-image sum, as torch's autograd gives it: 0 for invalid cells and where d == 0 (norm backward is
// masked there), (p - g)/d on the L1 branch (d == cut included), 0.5*sqrt(cut/d)*(p - g)/d above, NaN where d is NaN.
__device__ __forceinline__ float init_cell(float px, float py, float pz, float gx, float gy, float gz, float cut,
                                           float half_cut, bool live, float* o, int& valid) {
    valid = live && !(gx == 0.f && gy == 0.f && gz == 0.f);
    const float dx = px - gx, dy = py - gy, dz = pz - gz;
    const float d = sqrtf(fmaf(dx, dx, fmaf(dy, dy, dz * dz)));
    const bool l1 = d <= cut;
    const float sq = sqrtf(cut * d);
    const float gd = l1 ? 1.f : __fdiv_rn(half_cut, sq);   // d loss / d d (sqrt backward: cut / (2 sqrt(cut d)))
    float f = __fdiv_rn(gd, d);
    f = d == 0.f ? 0.f : f;                                 // NaN d keeps f = NaN
    o[0] = valid ? dx * f : 0.f;                            // exact zero even where the prediction is not finite
    o[1] = valid ? dy * f : 0.f;
    o[2] = valid ? dz * f : 0.f;
    const float loss = l1 ? d : (d > cut ? sq : 0.f);       // NaN d: in neither sum
    return valid ? loss : 0.f;
}

// grid = (blocks_per_image, B).  Cells are enumerated over the prediction's pH x pW map; cells outside the common
// h x w region get a zero gradient and are not counted.  VEC: pW % 4 == 0 and gW % 4 == 0 (so pW == gW == w: the
// widths differ by at most one) and 16-byte aligned bases -- a group of 4 cells then never straddles a row and is live
// iff its row is below h.
template <bool VEC>
__global__ void __launch_bounds__(kThreads) init_loss_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                                                             float* __restrict__ grads, int pW, int pN, int gW, int gN,
                                                             int h, int w, float cut, double* __restrict__ partial_sum,
                                                             unsigned* __restrict__ partial_cnt, unsigned* __restrict__ tickets,
                                                             double* __restrict__ sums, long long* __restrict__ counts) {
    __shared__ double warp_sum[kThreads / 32];
    __shared__ unsigned warp_cnt[kThreads / 32];
    __shared__ bool last;
    const int b = blockIdx.y;
    const float* pp = pred + (size_t)b * 3 * pN;
    const float* gp = gt + (size_t)b * 3 * gN;
    float* go = grads ? grads + (size_t)b * 3 * pN : nullptr;
    const float half_cut = 0.5f * cut;
    double acc = 0.;
    unsigned cnt = 0;
    const int per_block = kThreads * kCellsPerThread;
    for (int base = blockIdx.x * per_block; base < pN; base += gridDim.x * per_block) {
        const int p0 = base + threadIdx.x * kCellsPerThread;
        if (p0 >= pN) continue;
        float P[3][4], G[3][4], O[3][4];
        bool live[4];
        const int n = min(kCellsPerThread, pN - p0);
        if (VEC) {
            const bool row_live = p0 / pW < h;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float4 a = __ldcs(reinterpret_cast<const float4*>(pp + (size_t)c * pN + p0));
                P[c][0] = a.x; P[c][1] = a.y; P[c][2] = a.z; P[c][3] = a.w;
                float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
                if (row_live) g = __ldcs(reinterpret_cast<const float4*>(gp + (size_t)c * gN + p0));
                G[c][0] = g.x; G[c][1] = g.y; G[c][2] = g.z; G[c][3] = g.w;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) live[i] = row_live;
        } else {
            const int y0 = p0 / pW;
            int y = y0, x = p0 - y0 * pW;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                live[i] = i < n && y < h && x < w;
                const int q = y * gW + x;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    P[c][i] = i < n ? pp[(size_t)c * pN + p0 + i] : 0.f;
                    G[c][i] = live[i] ? gp[(size_t)c * gN + q] : 0.f;
                }
                if (++x == pW) { x = 0; ++y; }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float o[3];
            int v;
            const float l = init_cell(P[0][i], P[1][i], P[2][i], G[0][i], G[1][i], G[2][i], cut, half_cut, live[i], o, v);
            acc += (double)l;
            cnt += (unsigned)v;
            O[0][i] = o[0]; O[1][i] = o[1]; O[2][i] = o[2];
        }
        if (go) {
            if (VEC) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    __stcs(reinterpret_cast<float4*>(go + (size_t)c * pN + p0), make_float4(O[c][0], O[c][1], O[c][2], O[c][3]));
            } else {
                for (int i = 0; i < n; ++i)
                    for (int c = 0; c < 3; ++c) go[(size_t)c * pN + p0 + i] = O[c][i];
            }
        }
    }
    // block sums in a fixed order (result valid in thread 0), then the last block of the image adds the partials
    auto block_sum = [&](double v, unsigned k, unsigned& k_out) -> double {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            v += __shfl_xor_sync(0xffffffffu, v, o);
            k += __shfl_xor_sync(0xffffffffu, k, o);
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) {
            warp_sum[threadIdx.x >> 5] = v;
            warp_cnt[threadIdx.x >> 5] = k;
        }
        __syncthreads();
        double s = 0.;
        unsigned t = 0;
        if (threadIdx.x == 0)
            for (int wi = 0; wi < kThreads / 32; ++wi) {
                s += warp_sum[wi];
                t += warp_cnt[wi];
            }
        k_out = t;
        return s;
    };
    unsigned mine_cnt;
    const double mine = block_sum(acc, cnt, mine_cnt);
    if (threadIdx.x == 0) {
        partial_sum[(size_t)b * gridDim.x + blockIdx.x] = mine;
        partial_cnt[(size_t)b * gridDim.x + blockIdx.x] = mine_cnt;
        __threadfence();
        last = atomicAdd(&tickets[b], 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last) {
        __threadfence();
        double v = 0.;
        unsigned k = 0;
        for (unsigned j = threadIdx.x; j < gridDim.x; j += kThreads) {
            v += __ldcg(&partial_sum[(size_t)b * gridDim.x + j]);
            k += __ldcg(&partial_cnt[(size_t)b * gridDim.x + j]);
        }
        unsigned total;
        const double s = block_sum(v, k, total);
        if (threadIdx.x == 0) {
            sums[b] = s;
            counts[b] = (long long)total;
            tickets[b] = 0;  // ready for the next launch
        }
    }
}

}  // namespace

int init_loss_blocks_per_image(int N) {
    // As reproj_blocks_per_image: many short CTAs, up to four passes each on large maps; a pure function of N, which the
    // fixed summation order depends on.
    const int per_block = kThreads * kCellsPerThread;
    const int need = (N + per_block - 1) / per_block;
    return need < 64 ? need : (need < 256 ? (need + 1) / 2 : (need + 3) / 4);
}

void launch_init_loss(const float* pred, const float* gt, float* grads, int B, int pH, int pW, int gH, int gW, float cut,
                      int blocks_per_image, double* partial_sum, unsigned* partial_cnt, unsigned* tickets, double* sums,
                      long long* counts, cudaStream_t stream) {
    const dim3 grid(blocks_per_image, B);
    const int pN = pH * pW, gN = gH * gW;
    const int h = pH < gH ? pH : gH, w = pW < gW ? pW : gW;
    const bool vec = pW % 4 == 0 && gW % 4 == 0 && (uintptr_t)pred % 16 == 0 && (uintptr_t)gt % 16 == 0 &&
                     (!grads || (uintptr_t)grads % 16 == 0);
    if (vec)
        init_loss_kernel<true><<<grid, kThreads, 0, stream>>>(pred, gt, grads, pW, pN, gW, gN, h, w, cut, partial_sum,
                                                              partial_cnt, tickets, sums, counts);
    else
        init_loss_kernel<false><<<grid, kThreads, 0, stream>>>(pred, gt, grads, pW, pN, gW, gN, h, w, cut, partial_sum,
                                                               partial_cnt, tickets, sums, counts);
}

}  // namespace esacb200
