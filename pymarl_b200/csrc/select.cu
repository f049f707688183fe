// K2: chosen-action gather + avail masking + double-Q target  (learners/q_learner.py:55-78)
// K7: epsilon-greedy action selection                          (components/action_selectors.py:44-62)
// Both are pure bandwidth kernels: 8-lane groups walk the action axis with coalesced loads
// and resolve arg-max ties to the lowest index with a shuffle reduction.
#include <math.h>
#include "common.cuh"

namespace pmb {

namespace {

constexpr int GL = 8;            // lanes per row group

// (value, index) arg-max with lowest index on ties, across the GL lanes of a group
__device__ __forceinline__ void group_argmax(float& v, int& idx) {
#pragma unroll
    for (int o = GL / 2; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, v, o);
        int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
}

__global__ void __launch_bounds__(256)
target_select_kernel(int B, int T, int N, int A, int double_q, const float* __restrict__ q_on,
                     const float* __restrict__ q_tg, const int32_t* __restrict__ avail, int64_t avail_sb,
                     const int64_t* __restrict__ actions, int64_t actions_sb, float* __restrict__ chosen,
                     float* __restrict__ tmax, int32_t* __restrict__ cur_max) {
    const int64_t n_rows = (int64_t)B * (T - 1) * N;
    const int64_t R = (int64_t)B * N;
    int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / GL;
    const int lane = threadIdx.x % GL;
    const bool active = gid < n_rows;
    int64_t m = active ? gid : 0;           // m = (b*(T-1) + t)*N + n
    int64_t bt = m / N;
    int n = (int)(m - bt * N);
    int64_t b = bt / (T - 1);
    int t = (int)(bt - b * (T - 1));
    int64_t p = b * N + n;
    const float* qo1 = q_on + ((int64_t)(t + 1) * R + p) * A;
    const float* qt1 = q_tg + ((int64_t)(t + 1) * R + p) * A;
    const int32_t* av1 = avail + b * avail_sb + ((int64_t)(t + 1) * N + n) * A;

    float best = -INFINITY;
    int bidx = 0x7fffffff;
    for (int a = lane; a < A; a += GL) {
        bool ok = __ldg(av1 + a) != 0;
        float v = double_q ? __ldg(qo1 + a) : __ldg(qt1 + a);
        v = ok ? v : kMaskValue;
        if (v > best) { best = v; bidx = a; }      // ascending a: strict > keeps the lowest index
    }
    if (bidx == 0x7fffffff) { bidx = lane < A ? lane : 0; best = -INFINITY; }   // all-NaN row: pick lowest
    group_argmax(best, bidx);
    if (active && lane == 0) {
        float tv;
        if (double_q) {
            bool ok = __ldg(av1 + bidx) != 0;
            tv = ok ? __ldg(qt1 + bidx) : kMaskValue;
        } else {
            tv = best;
        }
        int a_taken = (int)__ldg(actions + b * actions_sb + (int64_t)t * N + n);
        chosen[m] = __ldg(q_on + ((int64_t)t * R + p) * A + a_taken);
        tmax[m] = tv;
        if (cur_max) cur_max[m] = bidx;
    }
}

// ---- Philox4x32-10 (counter based; same round constants as curand / torch) -----------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0; key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) {          // (0, 1]
    return ((float)(x >> 8) + 1.0f) * (1.0f / 16777216.0f);
}

__global__ void __launch_bounds__(256)
epsilon_greedy_kernel(int64_t rows, int N, int A, const float* __restrict__ q, const int32_t* __restrict__ avail,
                      int64_t avail_sb, float epsilon, const float* __restrict__ u, const float* __restrict__ expo,
                      uint64_t seed, uint64_t offset, int64_t* __restrict__ actions_out) {
    int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / GL;
    const int lane = threadIdx.x % GL;
    const bool active = gid < rows;
    int64_t row = active ? gid : 0;
    int64_t b = row / N;
    int n = (int)(row - b * N);
    const float* qr = q + row * A;
    const int32_t* av = avail + b * avail_sb + (int64_t)n * A;

    // greedy arg-max over q with unavailable actions at -inf; count of available actions
    float best = -INFINITY;
    int bidx = 0x7fffffff;
    int cnt = 0;
    for (int a = lane; a < A; a += GL) {
        bool ok = __ldg(av + a) != 0;
        cnt += ok ? 1 : 0;
        float v = ok ? __ldg(qr + a) : -INFINITY;
        if (v > best) { best = v; bidx = a; }
    }
    if (bidx == 0x7fffffff) bidx = lane < A ? lane : 0x7ffffffe;     // all -inf: first index wins
#pragma unroll
    for (int o = GL / 2; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    group_argmax(best, bidx);

    int ridx;
    uint4 r0 = make_uint4(0, 0, 0, 0);
    if (expo) {
        // reference arithmetic with injected draws: Categorical(avail.float()).sample() == argmax_a (avail[a] / cnt) / Exp(1)[a]
        const float prob = __fdiv_rn(1.0f, (float)cnt);
        float rbest = -INFINITY;
        ridx = 0x7fffffff;
        for (int a = lane; a < A; a += GL) {
            bool ok = __ldg(av + a) != 0;
            float ratio = __fdiv_rn(ok ? prob : 0.0f, __ldg(expo + row * A + a));
            if (ratio > rbest) { rbest = ratio; ridx = a; }
        }
        if (ridx == 0x7fffffff) ridx = lane < A ? lane : 0x7ffffffe;
        group_argmax(rbest, ridx);
    } else {
        // Philox mode: the same distribution (uniform over the available actions) from ONE counter block per row:
        // word x -> the epsilon test, word y -> the rank k of the chosen action among the available ones
        r0 = philox4x32_10(make_uint4((uint32_t)offset, (uint32_t)(offset >> 32), (uint32_t)row, ((uint32_t)(row >> 32) << 16)),
                           make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        int k = (int)((1.0f - u01(r0.y)) * (float)cnt);
        if (k >= cnt) k = cnt - 1;
        ridx = 0;
        int seen = 0;
        for (int a = 0; a < A; ++a) {                  // every lane walks the whole row: A is small, the loads hit L1
            const bool ok = __ldg(av + a) != 0;
            if (ok && seen == k) ridx = a;
            seen += ok ? 1 : 0;
        }
    }

    if (active && lane == 0) {
        float uu;
        if (u) {
            uu = __ldg(u + row);
        } else {
            uu = 1.0f - u01(r0.x);                 // [0, 1)
        }
        int pick = (cnt > 0 && uu < epsilon) ? ridx : bidx;
        if (pick >= A) pick = 0;
        actions_out[row] = pick;
    }
}

}  // namespace

int launch_target_select(const pmb_dims* d, const pmb_batch* b, const float* q_on, const float* q_tg, float* chosen,
                         float* tmax, int32_t* cur_max, cudaStream_t s) {
    int64_t n_rows = (int64_t)d->B * (d->T - 1) * d->N;
    if (n_rows <= 0) return PMB_OK;
    unsigned grid = (unsigned)ceil_div(n_rows * GL, 256);
    target_select_kernel<<<grid, 256, 0, s>>>(d->B, d->T, d->N, d->A, d->double_q, q_on, q_tg, static_cast<const int32_t*>(b->avail), b->avail_sb,
                                              b->actions, b->actions_sb, chosen, tmax, cur_max);
    PMB_LAUNCH_CHECK("target_select_kernel");
    return PMB_OK;
}

int launch_epsilon_greedy(int64_t rows, int N, int A, const float* q, const int32_t* avail, int64_t avail_sb,
                          float epsilon, const float* u, const float* expo, uint64_t seed, uint64_t offset,
                          int64_t* actions_out, cudaStream_t s) {
    if (rows <= 0) return PMB_OK;
    unsigned grid = (unsigned)ceil_div(rows * GL, 256);
    epsilon_greedy_kernel<<<grid, 256, 0, s>>>(rows, N, A, q, avail, avail_sb, epsilon, u, expo, seed, offset,
                                               actions_out);
    PMB_LAUNCH_CHECK("epsilon_greedy_kernel");
    return PMB_OK;
}

}  // namespace pmb
