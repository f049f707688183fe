// COMA learner kernels (SURVEY.md section 8f rank 4): learners/coma_learner.py:32-148, modules/critics/coma.py:22-59,
// utils/rl_utils.py:4-15, the policy head of controllers/basic_controller.py:51-73 and
// components/action_selectors.py:9-33.  fp32 (CUDA-core) tier: the critic is trained with one optimiser step per
// timestep on B*N rows, so the step is a long chain of small launches; the GEMMs reuse gemm_simt.cu.
#include "common.cuh"

namespace pmb {
namespace {

// ---- critic inputs (coma.py:29-50), never read from actions_onehot: one-hot blocks are generated from actions / filled ----
// rows (b, tt, n), tt in [0, nt) <-> batch timestep t0 + tt; D = S + O + 2*N*A + N columns:
//   [ state | obs | one-hot actions of all agents at t with the own block zeroed | one-hot actions at t-1 | one-hot(n) ]
__global__ void __launch_bounds__(256)
coma_inputs_kernel(int B, int N, int O, int S, int A, int t0, int nt, const float* __restrict__ state, int64_t state_sb,
                   const float* __restrict__ obs, int64_t obs_sb, const int64_t* __restrict__ actions, int64_t actions_sb,
                   const int64_t* __restrict__ filled, int64_t filled_sb, float* __restrict__ out) {
    const int64_t row = blockIdx.x;
    const int n = (int)(row % N);
    const int tt = (int)((row / N) % nt);
    const int64_t b = row / ((int64_t)N * nt);
    const int t = t0 + tt;
    const int NA = N * A, D = S + O + 2 * NA + N;
    const bool f_t = filled[b * filled_sb + t] != 0;
    const bool f_p = t > 0 && filled[b * filled_sb + (t - 1)] != 0;
    float* o = out + row * D;
    for (int c = threadIdx.x; c < D; c += blockDim.x) {
        float v;
        if (c < S) v = __ldg(state + b * state_sb + (int64_t)t * S + c);
        else if (c < S + O) v = __ldg(obs + b * obs_sb + ((int64_t)t * N + n) * O + (c - S));
        else if (c < S + O + NA) {
            const int k = c - S - O, m = k / A, a = k - m * A;
            v = (f_t && m != n && (int)__ldg(actions + b * actions_sb + (int64_t)t * N + m) == a) ? 1.f : 0.f;
        } else if (c < S + O + 2 * NA) {
            const int k = c - S - O - NA, m = k / A, a = k - m * A;
            v = (f_p && (int)__ldg(actions + b * actions_sb + (int64_t)(t - 1) * N + m) == a) ? 1.f : 0.f;
        } else v = (c - S - O - 2 * NA) == n ? 1.f : 0.f;
        o[c] = v;
    }
}

// targets_taken[b][t][n] = q[(b, tt, n)][actions[b, t0 + tt, n]]  (coma_learner.py:106) for one chunk of timesteps
__global__ void coma_gather_taken_kernel(int64_t rows, int N, int A, int T, int t0, int nt, const float* __restrict__ q,
                                         const int64_t* __restrict__ actions, int64_t actions_sb, float* __restrict__ taken) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    const int n = (int)(row % N);
    const int tt = (int)((row / N) % nt);
    const int64_t b = row / ((int64_t)N * nt);
    const int t = t0 + tt;
    const int a = (int)__ldg(actions + b * actions_sb + (int64_t)t * N + n);
    taken[(b * T + t) * N + n] = q[row * A + a];
}

// build_td_lambda_targets (utils/rl_utils.py:4-15): one thread per (b, n), backward recursion over t
__global__ void coma_td_lambda_kernel(int B, int T, int N, float gamma, float lam, const float* __restrict__ taken,
                                      const float* __restrict__ reward, int64_t reward_sb, const uint8_t* __restrict__ term,
                                      int64_t term_sb, const int64_t* __restrict__ filled, int64_t filled_sb,
                                      float* __restrict__ targets) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * N) return;
    const int64_t b = i / N;
    const int n = (int)(i - b * N);
    float tsum = 0.f;
    for (int t = 0; t < T - 1; ++t) tsum += (float)term[b * term_sb + t];
    float ret = taken[(b * T + (T - 1)) * N + n] * (1.f - tsum);
    for (int t = T - 2; t >= 0; --t) {
        const float tm = (float)term[b * term_sb + t];
        float mask = (float)filled[b * filled_sb + t];
        if (t > 0) mask = mask * (1.f - (float)term[b * term_sb + (t - 1)]);
        const float r = reward[b * reward_sb + t];
        ret = (lam * gamma) * ret + mask * (r + (((1.f - lam) * gamma) * taken[(b * T + (t + 1)) * N + n]) * (1.f - tm));
        targets[(b * (T - 1) + t) * N + n] = ret;
    }
}

// one critic timestep (coma_learner.py:118-146): td error at the taken action, masked L2 loss sums, the (sparse) dq as one
// value per row, q_t copied into q_vals[:, t].  stats row: [mask_sum, td2_sum, tdabs_sum, qtaken_sum, target_sum]
__global__ void __launch_bounds__(256)
coma_critic_td_kernel(int B, int T, int N, int A, int t, const float* __restrict__ q_t, const float* __restrict__ targets,
                      const int64_t* __restrict__ actions, int64_t actions_sb, const uint8_t* __restrict__ term,
                      int64_t term_sb, const int64_t* __restrict__ filled, int64_t filled_sb, float* __restrict__ q_vals,
                      float* __restrict__ dqv, int32_t* __restrict__ dqa, double* __restrict__ stats,
                      double* __restrict__ partials) {
    __shared__ double sh[8][5];
    __shared__ int s_last;
    const int64_t R = (int64_t)B * N;
    double acc[5] = {0, 0, 0, 0, 0};
    for (int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; row < R; row += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = row / N;
        const int n = (int)(row - b * N);
        float mask = (float)filled[b * filled_sb + t];
        if (t > 0) mask = mask * (1.f - (float)term[b * term_sb + (t - 1)]);
        const int a = (int)__ldg(actions + b * actions_sb + (int64_t)t * N + n);
        const float* qr = q_t + row * A;
        float* qv = q_vals + ((b * (T - 1) + t) * N + n) * A;
        for (int k = 0; k < A; ++k) qv[k] = qr[k];
        const float qt = qr[a];
        const float y = targets[(b * (T - 1) + t) * N + n];
        const float mtd = (qt - y) * mask;
        dqv[row] = 2.f * mtd * mask;                 // un-normalised: the update kernel applies 1 / mask_sum
        dqa[row] = a;
        acc[0] += (double)mask; acc[1] += (double)(mtd * mtd); acc[2] += (double)fabsf(mtd);
        acc[3] += (double)(qt * mask); acc[4] += (double)(y * mask);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 5; ++i) acc[i] = warp_sum(acc[i]);
    if (lane == 0)
#pragma unroll
        for (int i = 0; i < 5; ++i) sh[w][i] = acc[i];
    __syncthreads();
    // deterministic cross-block total: per-block sums, the last block (ticket in the row's last slot) adds them in order
    if (threadIdx.x < 5) {
        double s = 0;
        for (int ww = 0; ww < (int)(blockDim.x >> 5); ++ww) s += sh[ww][threadIdx.x];
        partials[(int64_t)blockIdx.x * 5 + threadIdx.x] = s;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
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

// dense dq rows for the fc3 weight gradient GEMM: dq[row][a] = dqv[row] at a = dqa[row], else 0
__global__ void coma_dq_dense_kernel(int64_t R, int A, const float* __restrict__ dqv, const int32_t* __restrict__ dqa,
                                     float* __restrict__ dq) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * A) return;
    const int64_t row = i / A;
    dq[i] = (int)(i - row * A) == dqa[row] ? dqv[row] : 0.f;
}

// dx2[row][k] = dqv[row] * W3[a_row][k] * (x2 > 0)      (fc3 backward through the sparse dq + ReLU mask)
__global__ void coma_dx2_kernel(int64_t R, int Hc, const float* __restrict__ dqv, const int32_t* __restrict__ dqa,
                                const float* __restrict__ w3, const float* __restrict__ x2, float* __restrict__ dx2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R * Hc) return;
    const int64_t row = i / Hc;
    const int k = (int)(i - row * Hc);
    dx2[i] = x2[i] > 0.f ? dqv[row] * w3[(int64_t)dqa[row] * Hc + k] : 0.f;
}

__global__ void relu_mask_kernel(int64_t n, const float* __restrict__ x, float* __restrict__ dx) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !(x[i] > 0.f)) dx[i] = 0.f;
}

__global__ void transpose_kernel(int rows, int cols, const float* __restrict__ in, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols) return;
    const int r = i / cols, c = i - r * cols;
    out[(int64_t)c * rows + r] = in[i];
}

// ---- policy head + COMA loss + d(loss)/d(logits) ------------------------------------------------------------------
// One warp per row (b, t, n), t < T' (= T-1 unrolled steps), logits time major [T'][R][A].
//   BasicMAC.forward (basic_controller.py:55-71): z = logits, -1e10 where unavailable; s = softmax(z);
//       e = (1 - eps) s + eps / n_avail; e = 0 where unavailable
//   learner (coma_learner.py:62-80): p = e (0 where unavailable), pi = p / sum(p), baseline = sum pi q,
//       adv = q_taken - baseline, loss = -sum(adv log pi_taken mask) / sum(mask)
// dlogits (un-normalised by sum(mask)): G = -adv mask; dp_b = G (1[b = u] / p_u - 1 / Z) on available b; ds = (1 - eps) dp;
//       dz = s (ds - sum_b ds_b s_b)
// stats row: [mask_sum, sum(adv log_pi mask), sum(adv mask), sum(pi_max mask)]
__global__ void __launch_bounds__(256)
coma_policy_kernel(int B, int T, int N, int A, float eps, const float* __restrict__ logits, const float* __restrict__ q_vals,
                   const int32_t* __restrict__ avail, int64_t avail_sb, const int64_t* __restrict__ actions, int64_t actions_sb,
                   const uint8_t* __restrict__ term, int64_t term_sb, const int64_t* __restrict__ filled, int64_t filled_sb,
                   float* __restrict__ dlogits, float* __restrict__ pi_out, double* __restrict__ stats,
                   double* __restrict__ partials) {
    __shared__ double sh[8][4];
    __shared__ int s_last;
    const int Tp = T - 1;
    const int64_t R = (int64_t)B * N, total = (int64_t)Tp * R;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    double acc[4] = {0, 0, 0, 0};
    for (int64_t item = (int64_t)blockIdx.x * wpb + w; item < total; item += (int64_t)gridDim.x * wpb) {
        const int t = (int)(item / R);
        const int64_t row = item - (int64_t)t * R;
        const int64_t b = row / N;
        const int n = (int)(row - b * N);
        float mask = (float)filled[b * filled_sb + t];
        if (t > 0) mask = mask * (1.f - (float)term[b * term_sb + (t - 1)]);
        const int u = (int)__ldg(actions + b * actions_sb + (int64_t)t * N + n);
        const float* lg = logits + item * A;
        const int32_t* av = avail + b * avail_sb + ((int64_t)t * N + n) * A;
        const float* qv = q_vals + ((b * Tp + t) * N + n) * A;
        // up to 64 actions: two per lane
        float z[2], s[2], q[2];
        bool ok[2];
        float zmax = -3.0e38f;
        int nav = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int a = lane + 32 * h;
            ok[h] = a < A && av[a] != 0;
            z[h] = a < A ? (ok[h] ? lg[a] : -1e10f) : -3.0e38f;
            q[h] = a < A ? qv[a] : 0.f;
            zmax = fmaxf(zmax, z[h]);
            nav += ok[h] ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            zmax = fmaxf(zmax, __shfl_xor_sync(0xffffffffu, zmax, o));
            nav += __shfl_xor_sync(0xffffffffu, nav, o);
        }
        float esum = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            s[h] = (lane + 32 * h) < A ? expf(z[h] - zmax) : 0.f;
            esum += s[h];
        }
        esum = warp_sum(esum);
        float p[2], Z = 0.f, base = 0.f, pmax = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            s[h] = s[h] / esum;
            p[h] = ok[h] ? (1.f - eps) * s[h] + eps / (float)nav : 0.f;
            Z += p[h];
        }
        Z = warp_sum(Z);
        float pi[2], pu = 0.f, qu = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            pi[h] = ok[h] ? p[h] / Z : 0.f;
            base += pi[h] * q[h];
            pmax = fmaxf(pmax, pi[h]);
            if (lane + 32 * h == u) { pu = pi[h]; qu = q[h]; }
            if (pi_out && lane + 32 * h < A) pi_out[item * A + lane + 32 * h] = pi[h];
        }
        base = warp_sum(base);
        pu = warp_sum(pu);                            // only the owner lane holds a non-zero value
        qu = warp_sum(qu);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) pmax = fmaxf(pmax, __shfl_xor_sync(0xffffffffu, pmax, o));
        const float adv = qu - base;
        const float logp = mask == 0.f ? 0.f : logf(pu);
        const float G = mask == 0.f ? 0.f : -adv * mask;
        // ds_b = (1 - eps) G (1[b = u] / p_u - 1 / Z) on available b, with p_u = pi_u Z
        float ds[2], dot = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            ds[h] = 0.f;
            if (ok[h] && G != 0.f) ds[h] = (1.f - eps) * G * (((lane + 32 * h == u) ? 1.f / (pu * Z) : 0.f) - 1.f / Z);
            dot += ds[h] * s[h];
        }
        dot = warp_sum(dot);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int a = lane + 32 * h;
            if (a < A) dlogits[item * A + a] = ok[h] ? s[h] * (ds[h] - dot) : 0.f;
        }
        if (lane == 0) {
            acc[0] += (double)mask; acc[1] += (double)(adv * logp * mask); acc[2] += (double)(adv * mask);
            acc[3] += (double)(pmax * mask);
        }
    }
    if (lane == 0)
#pragma unroll
        for (int i = 0; i < 4; ++i) sh[w][i] = acc[i];
    __syncthreads();
    if (threadIdx.x < 4) {
        double s2 = 0;
        for (int ww = 0; ww < wpb; ++ww) s2 += sh[ww][threadIdx.x];
        partials[(int64_t)blockIdx.x * 4 + threadIdx.x] = s2;
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long t = atomicAdd(reinterpret_cast<unsigned long long*>(stats + PMB_S_COUNT - 1), 1ULL);
        s_last = t == (unsigned long long)gridDim.x - 1;
    }
    __syncthreads();
    if (s_last && threadIdx.x < 4) {
        __threadfence();
        const volatile double* pv = partials;
        double tot = 0.0;
        for (unsigned bb = 0; bb < gridDim.x; ++bb) tot += pv[(int64_t)bb * 4 + threadIdx.x];
        stats[threadIdx.x] = tot;
    }
}

// BasicMAC.forward's policy head alone (rollout): probs [rows][A] from logits [rows][A]; test_mode = plain softmax
__global__ void __launch_bounds__(256)
policy_head_kernel(int64_t rows, int A, float eps, int test_mode, const float* __restrict__ logits,
                   const int32_t* __restrict__ avail, float* __restrict__ probs) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    for (int64_t row = (int64_t)blockIdx.x * wpb + w; row < rows; row += (int64_t)gridDim.x * wpb) {
        float z[2], s[2];
        bool ok[2];
        float zmax = -3.0e38f;
        int nav = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int a = lane + 32 * h;
            ok[h] = a < A && avail[row * A + a] != 0;
            z[h] = a < A ? (ok[h] ? logits[row * A + a] : -1e10f) : -3.0e38f;
            zmax = fmaxf(zmax, z[h]);
            nav += ok[h] ? 1 : 0;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            zmax = fmaxf(zmax, __shfl_xor_sync(0xffffffffu, zmax, o));
            nav += __shfl_xor_sync(0xffffffffu, nav, o);
        }
        float esum = 0.f;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            s[h] = (lane + 32 * h) < A ? expf(z[h] - zmax) : 0.f;
            esum += s[h];
        }
        esum = warp_sum(esum);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int a = lane + 32 * h;
            if (a >= A) continue;
            float v = s[h] / esum;
            if (!test_mode) v = ok[h] ? (1.f - eps) * v + eps / (float)nav : 0.f;
            probs[row * A + a] = v;
        }
    }
}

// MultinomialActionSelector (action_selectors.py:19-31): Categorical(masked probs).sample() == arg-max(p / Exp(1)) with the
// probabilities renormalised over the available actions; greedy arg-max in test mode.  expo != null: injected draws.
__device__ __forceinline__ uint32_t mix32(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return (uint32_t)x;
}
__global__ void multinomial_kernel(int64_t rows, int A, const float* __restrict__ probs, const int32_t* __restrict__ avail,
                                   const float* __restrict__ expo, int greedy, uint64_t seed, uint64_t offset,
                                   int64_t* __restrict__ out) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float sum = 0.f;
    for (int a = 0; a < A; ++a) sum += avail[row * A + a] != 0 ? probs[row * A + a] : 0.f;
    float best = -1.f;
    int arg = 0;
    for (int a = 0; a < A; ++a) {
        float p = avail[row * A + a] != 0 ? probs[row * A + a] : 0.f;
        float key;
        if (greedy) key = p;
        else {
            float e;
            if (expo) e = expo[row * A + a];
            else {
                const uint32_t r = mix32(seed ^ (offset * 0x9e3779b97f4a7c15ull) ^ ((uint64_t)row * 131 + a) * 0xd6e8feb86659fd93ull);
                e = -logf(((float)r + 1.f) * 2.3283064e-10f);         // Exp(1) from a uniform in (0, 1]
            }
            key = (p / sum) / e;
        }
        if (key > best) { best = key; arg = a; }
    }
    out[row] = arg;
}

}  // namespace

int coma_launch_inputs(const pmb_dims* d, const pmb_batch* b, int t0, int nt, float* out, cudaStream_t s) {
    const int64_t rows = (int64_t)d->B * nt * d->N;
    if (rows <= 0) return PMB_OK;
    coma_inputs_kernel<<<(unsigned)rows, 256, 0, s>>>(d->B, d->N, d->O, d->S, d->A, t0, nt, static_cast<const float*>(b->state), b->state_sb, static_cast<const float*>(b->obs), b->obs_sb,
                                                      b->actions, b->actions_sb, b->filled, b->filled_sb, out);
    PMB_LAUNCH_CHECK("coma_inputs_kernel");
    return PMB_OK;
}

int coma_launch_gather_taken(const pmb_dims* d, const pmb_batch* b, int t0, int nt, const float* q, float* taken, cudaStream_t s) {
    const int64_t rows = (int64_t)d->B * nt * d->N;
    coma_gather_taken_kernel<<<(unsigned)ceil_div(rows, 256), 256, 0, s>>>(rows, d->N, d->A, d->T, t0, nt, q, b->actions,
                                                                          b->actions_sb, taken);
    PMB_LAUNCH_CHECK("coma_gather_taken_kernel");
    return PMB_OK;
}

int coma_launch_td_lambda(const pmb_dims* d, const pmb_batch* b, float gamma, float lam, const float* taken, float* targets,
                          cudaStream_t s) {
    const int64_t n = (int64_t)d->B * d->N;
    coma_td_lambda_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, s>>>(d->B, d->T, d->N, gamma, lam, taken, b->reward, b->reward_sb,
                                                                    b->terminated, b->terminated_sb, b->filled, b->filled_sb,
                                                                    targets);
    PMB_LAUNCH_CHECK("coma_td_lambda_kernel");
    return PMB_OK;
}

int coma_launch_critic_td(const pmb_dims* d, const pmb_batch* b, int t, const float* q_t, const float* targets, float* q_vals,
                          float* dqv, int32_t* dqa, double* stats_row, double* partials, cudaStream_t s) {
    const int64_t R = (int64_t)d->B * d->N;
    int64_t grid = ceil_div(R, 256);
    if (grid > 4 * sm_count()) grid = 4 * sm_count();
    coma_critic_td_kernel<<<(unsigned)grid, 256, 0, s>>>(d->B, d->T, d->N, d->A, t, q_t, targets, b->actions, b->actions_sb,
                                                        b->terminated, b->terminated_sb, b->filled, b->filled_sb, q_vals, dqv,
                                                        dqa, stats_row, partials);
    PMB_LAUNCH_CHECK("coma_critic_td_kernel");
    return PMB_OK;
}

int coma_launch_critic_bwd_pointwise(int64_t R, int A, int Hc, const float* dqv, const int32_t* dqa, const float* w3,
                                     const float* x2, float* dq_dense, float* dx2, cudaStream_t s) {
    coma_dq_dense_kernel<<<(unsigned)ceil_div(R * A, 256), 256, 0, s>>>(R, A, dqv, dqa, dq_dense);
    PMB_LAUNCH_CHECK("coma_dq_dense_kernel");
    coma_dx2_kernel<<<(unsigned)ceil_div(R * Hc, 256), 256, 0, s>>>(R, Hc, dqv, dqa, w3, x2, dx2);
    PMB_LAUNCH_CHECK("coma_dx2_kernel");
    return PMB_OK;
}

int launch_relu_mask(int64_t n, const float* x, float* dx, cudaStream_t s) {
    relu_mask_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(n, x, dx);
    PMB_LAUNCH_CHECK("relu_mask_kernel");
    return PMB_OK;
}

int launch_transpose(int rows, int cols, const float* in, float* out, cudaStream_t s) {
    transpose_kernel<<<(unsigned)ceil_div((int64_t)rows * cols, 256), 256, 0, s>>>(rows, cols, in, out);
    PMB_LAUNCH_CHECK("transpose_kernel");
    return PMB_OK;
}

int coma_launch_policy(const pmb_dims* d, const pmb_batch* b, float eps, const float* logits, const float* q_vals,
                       float* dlogits, float* pi_out, double* stats_row, double* partials, cudaStream_t s) {
    const int64_t total = (int64_t)(d->T - 1) * d->B * d->N;
    if (total <= 0) return PMB_OK;
    int64_t grid = ceil_div(total, 8);
    if (grid > 8 * sm_count()) grid = 8 * sm_count();
    coma_policy_kernel<<<(unsigned)grid, 256, 0, s>>>(d->B, d->T, d->N, d->A, eps, logits, q_vals, static_cast<const int32_t*>(b->avail), b->avail_sb,
                                                     b->actions, b->actions_sb, b->terminated, b->terminated_sb, b->filled,
                                                     b->filled_sb, dlogits, pi_out, stats_row, partials);
    PMB_LAUNCH_CHECK("coma_policy_kernel");
    return PMB_OK;
}

int launch_policy_head(int64_t rows, int A, float eps, int test_mode, const float* logits, const int32_t* avail, float* probs,
                       cudaStream_t s) {
    if (rows <= 0) return PMB_OK;
    int64_t grid = ceil_div(rows, 8);
    if (grid > 8 * sm_count()) grid = 8 * sm_count();
    policy_head_kernel<<<(unsigned)grid, 256, 0, s>>>(rows, A, eps, test_mode, logits, avail, probs);
    PMB_LAUNCH_CHECK("policy_head_kernel");
    return PMB_OK;
}

int launch_multinomial(int64_t rows, int A, const float* probs, const int32_t* avail, const float* expo, int greedy,
                       uint64_t seed, uint64_t offset, int64_t* out, cudaStream_t s) {
    if (rows <= 0) return PMB_OK;
    multinomial_kernel<<<(unsigned)ceil_div(rows, 128), 128, 0, s>>>(rows, A, probs, avail, expo, greedy, seed, offset, out);
    PMB_LAUNCH_CHECK("multinomial_kernel");
    return PMB_OK;
}

}  // namespace pmb
