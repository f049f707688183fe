// K4: TD target + masked loss sums + dL/dq_tot   (learners/q_learner.py:39-44, 86-97, 109-116)
// K6: grad-norm clip + RMSprop + hard target sync  (learners/q_learner.py:102-107, 118-122)
#include "common.cuh"

namespace pmb {

namespace {

// block-wide sum of 5 doubles, result valid in thread 0
__device__ __forceinline__ void block_sum5(double (&v)[5], double (*sh)[5]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 5; ++i) v[i] = warp_sum(v[i]);
    if (lane == 0)
#pragma unroll
        for (int i = 0; i < 5; ++i) sh[w][i] = v[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int ww = 1; ww < (int)(blockDim.x >> 5); ++ww)
#pragma unroll
            for (int i = 0; i < 5; ++i) v[i] += sh[ww][i];
    }
}

// element index i = m*W + w,  m = b*(T-1) + t.  W = 1 (QMIX / VDN) or N (IQL: mask.expand_as(td)).
__global__ void __launch_bounds__(256)
td_loss_kernel(int B, int T, int W, float gamma, const float* __restrict__ q_tot, const float* __restrict__ t_tot,
               const float* __restrict__ reward, int64_t reward_sb, const uint8_t* __restrict__ terminated,
               int64_t term_sb, const int64_t* __restrict__ filled, int64_t filled_sb,
               const int64_t* __restrict__ ep_index, float* __restrict__ g_out, double* __restrict__ stats,
               double* __restrict__ partials) {
    __shared__ double sh[8][5];
    __shared__ int s_last;
    const int64_t total = (int64_t)B * (T - 1) * W;
    double acc[5] = {0, 0, 0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t m = i / W;
        int64_t b = m / (T - 1);
        int t = (int)(m - b * (T - 1));
        const int64_t be = ep_row(ep_index, b);
        float term = (float)__ldg(terminated + be * term_sb + t);
        float mask = (float)__ldg(filled + be * filled_sb + t);
        if (t > 0) mask = mask * (1.f - (float)__ldg(terminated + be * term_sb + (t - 1)));
        float r = __ldg(reward + be * reward_sb + t);
        float q = __ldg(q_tot + i);
        float y = r + (gamma * (1.f - term)) * __ldg(t_tot + i);
        float td = q - y;
        float mtd = td * mask;
        g_out[i] = 2.f * mtd * mask;
        acc[0] += (double)mask;
        acc[1] += (double)(mtd * mtd);
        acc[2] += (double)fabsf(mtd);
        acc[3] += (double)(q * mask);
        acc[4] += (double)(y * mask);
    }
    block_sum5(acc, sh);
    if (!partials) {                       // stand-alone pmb_td_loss: accumulate into the caller's sums
        if (threadIdx.x == 0) {
#pragma unroll
            for (int i = 0; i < 5; ++i) atomicAdd(stats + i, acc[i]);
        }
        return;
    }
    // deterministic: every block stores its sums, the last block to finish adds them in block order (ticket = the last slot
    // of the stats buffer, zeroed with it at the start of the step)
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < 5; ++i) partials[(int64_t)blockIdx.x * 5 + i] = acc[i];
        __threadfence();
        const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(stats + PMB_S_COUNT - 1), 1ULL);
        s_last = t == (unsigned long long)gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x < 5) {
        __threadfence();
        const volatile double* pv = partials;
        double tot = 0.0;
        for (unsigned bb = 0; bb < gridDim.x; ++bb) tot += pv[(int64_t)bb * 5 + threadIdx.x];
        stats[threadIdx.x] = tot;
    }
}

__global__ void stats_reset_kernel(double* stats) {
    if (threadIdx.x < PMB_S_COUNT) stats[threadIdx.x] = 0.0;
}

// Data-parallel exchange: the five double loss sums ride in the tail of the fp32 gradient buffer as (hi, lo) float pairs,
// so ONE all-reduce(sum, fp32) over [grads | 10 floats] carries everything a step exchanges (dp_pack_sum, common.cuh).
// hi + lo reproduces the double to 2^-48; the fp32 sums over W <= 8 ranks add at most (W - 1) 2^-24 of the sum of the
// magnitudes, and mask_sum stays exact up to a global count of 2^36.
__global__ void dp_pack_stats_kernel(const double* __restrict__ stats, float* __restrict__ tail) {
    const int i = threadIdx.x;
    if (i < 5) {
        dp_pack_sum(i, stats[i], tail + 2 * i);
    } else if (i < PMB_DP_TAIL_FLOATS / 2) {
        tail[2 * i] = 0.f;
        tail[2 * i + 1] = 0.f;
    }
}
__global__ void dp_unpack_stats_kernel(const float* __restrict__ tail, double* __restrict__ stats) {
    const int i = threadIdx.x;
    if (i < 5) stats[i] = (double)tail[2 * i] + (double)tail[2 * i + 1];
}

constexpr int OPT_BLOCKS = 256, OPT_THREADS = 256;

// fixed grid-stride assignment -> the partial sums, and their fixed-order total, are deterministic
__global__ void __launch_bounds__(OPT_THREADS)
grad_sumsq_kernel(int64_t n, const float* __restrict__ g, double* __restrict__ partial) {
    __shared__ double sh[OPT_THREADS / 32];
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = (double)g[i];
        s += v * v;
    }
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < OPT_THREADS / 32; ++w) tot += sh[w];
        partial[blockIdx.x] = tot;
    }
}

__global__ void __launch_bounds__(OPT_THREADS)
rmsprop_apply_kernel(int64_t n, float* __restrict__ p, float* __restrict__ g, float* __restrict__ sq,
                     float* __restrict__ target, int do_sync, const double* __restrict__ partial,
                     double* __restrict__ stats, float lr, float alpha, float eps, float clip, int skip_if_empty) {
    __shared__ float s_scale, s_coef;
    // skip_if_empty (COMA critic, coma_learner.py:120-121 `if mask_t.sum() == 0: continue`): no step when nothing is unmasked
    if (skip_if_empty && stats[PMB_S_MASK_SUM] <= 0.0) return;
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int b = 0; b < OPT_BLOCKS; ++b) tot += partial[b];
        double mask_sum = stats[PMB_S_MASK_SUM];
        float scale = (float)(1.0 / mask_sum);
        float norm = (float)(sqrt(tot) / mask_sum);                 // norm of the normalised gradient
        float coef = clip / (norm + 1e-6f);
        coef = coef < 1.f ? coef : 1.f;
        s_scale = scale;
        s_coef = coef;
        if (blockIdx.x == 0) {
            stats[PMB_S_GRAD_NORM] = (double)norm;
            stats[PMB_S_CLIP_COEF] = (double)coef;
            stats[PMB_S_LOSS] = stats[PMB_S_TD2_SUM] / mask_sum;
        }
    }
    __syncthreads();
    const float scale = s_scale, coef = s_coef;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float gv = (g[i] * scale) * coef;
        float v = sq[i] * alpha + ((1.f - alpha) * gv) * gv;
        float avg = sqrtf(v) + eps;
        float pv = p[i] + (-lr * gv) / avg;
        g[i] = gv;
        sq[i] = v;
        p[i] = pv;
        if (do_sync && target) target[i] = pv;
    }
}

}  // namespace

int launch_td_loss(const pmb_dims* d, const pmb_batch* b, const float* q_tot, const float* t_tot, float gamma,
                   float* g_out, double* stats, cudaStream_t s, double* partials, int64_t partial_bytes) {
    const int W = d->mixer == PMB_MIXER_NONE ? d->N : 1;
    const int64_t total = (int64_t)d->B * (d->T - 1) * W;
    if (total <= 0) return PMB_OK;
    int64_t grid = ceil_div(total, 256);
    int64_t cap = 8 * (int64_t)sm_count();
    if (grid > cap) grid = cap;
    if (partials && partial_bytes < grid * 5 * (int64_t)sizeof(double)) partials = nullptr;
    td_loss_kernel<<<(unsigned)grid, 256, 0, s>>>(d->B, d->T, W, gamma, q_tot, t_tot, b->reward, b->reward_sb,
                                                  b->terminated, b->terminated_sb, b->filled, b->filled_sb, b->ep_index, g_out,
                                                  stats, partials);
    PMB_LAUNCH_CHECK("td_loss_kernel");
    return PMB_OK;
}

int launch_stats_reset(double* stats, cudaStream_t s) {
    stats_reset_kernel<<<1, 32, 0, s>>>(stats);
    PMB_LAUNCH_CHECK("stats_reset_kernel");
    return PMB_OK;
}

int launch_dp_pack(const double* stats, float* tail, cudaStream_t s) {
    dp_pack_stats_kernel<<<1, 32, 0, s>>>(stats, tail);
    PMB_LAUNCH_CHECK("dp_pack_stats_kernel");
    return PMB_OK;
}

int launch_dp_unpack(const float* tail, double* stats, cudaStream_t s) {
    dp_unpack_stats_kernel<<<1, 32, 0, s>>>(tail, stats);
    PMB_LAUNCH_CHECK("dp_unpack_stats_kernel");
    return PMB_OK;
}

int launch_clip_rmsprop(int64_t n, float* p, float* g, float* sq, float* target, int do_sync, double* stats, float lr,
                        float alpha, float eps, float clip, float* scratch, cudaStream_t s, int skip_if_empty) {
    if (n <= 0) return PMB_OK;
    double* partial = reinterpret_cast<double*>(scratch);          // OPT_BLOCKS doubles (<= 4096 floats)
    grad_sumsq_kernel<<<OPT_BLOCKS, OPT_THREADS, 0, s>>>(n, g, partial);
    PMB_LAUNCH_CHECK("grad_sumsq_kernel");
    rmsprop_apply_kernel<<<OPT_BLOCKS, OPT_THREADS, 0, s>>>(n, p, g, sq, target, do_sync, partial, stats, lr, alpha,
                                                           eps, clip, skip_if_empty);
    PMB_LAUNCH_CHECK("rmsprop_apply_kernel");
    return PMB_OK;
}

}  // namespace pmb
