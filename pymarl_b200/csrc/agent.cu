// RNNAgent kernels, fp32 parity tier.
//
//   gru_unroll_fwd : persistent per row-tile unroll of GRUCell + fc2 over time.  W_ih, W_hh,
//                    fc2 stay resident in shared memory for all T steps, the hidden state tile
//                    never leaves the SM (only the stash the backward needs is written).
//   gru_unroll_bwd : BPTT for the online net; dh lives in registers across the whole unroll,
//                    gate gradients overwrite the stashed gates in place.
//   agent_scatter_grads : deterministic scatter-type gradients (fc2 rows by action, the
//                    last-action and agent-id columns of fc1).
//
// reference: modules/agents/rnn_agent.py:27-36, controllers/basic_controller.py:40-49,100-135,
//            learners/q_learner.py:47-52,58-62 and torch autograd through them (:101).
#include "common.cuh"

namespace pmb {

namespace {

constexpr int NT = 256;

template <int JW>
__device__ __forceinline__ void lds_vec(float (&dst)[JW], const float* src) {
    if constexpr (JW == 4) {
        float4 v = *reinterpret_cast<const float4*>(src);
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    } else if constexpr (JW == 2) {
        float2 v = *reinterpret_cast<const float2*>(src);
        dst[0] = v.x; dst[1] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < JW; ++i) dst[i] = src[i];
    }
}
template <int JW>
__device__ __forceinline__ void ldg_vec(float (&dst)[JW], const float* src) {
    if constexpr (JW == 4) {
        float4 v = __ldg(reinterpret_cast<const float4*>(src));
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
    } else if constexpr (JW == 2) {
        float2 v = __ldg(reinterpret_cast<const float2*>(src));
        dst[0] = v.x; dst[1] = v.y;
    } else {
#pragma unroll
        for (int i = 0; i < JW; ++i) dst[i] = __ldg(src + i);
    }
}
template <int JW>
__device__ __forceinline__ void stg_vec(float* dst, const float (&src)[JW]) {
    if constexpr (JW == 4) {
        *reinterpret_cast<float4*>(dst) = make_float4(src[0], src[1], src[2], src[3]);
    } else if constexpr (JW == 2) {
        *reinterpret_cast<float2*>(dst) = make_float2(src[0], src[1]);
    } else {
#pragma unroll
        for (int i = 0; i < JW; ++i) dst[i] = src[i];
    }
}

// ------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------
template <int H, int RW>
struct FwdSmem {
    static constexpr int RT = 16 * RW;
    static constexpr int LD = H + 1;
    static size_t floats(int A) {
        return (size_t)2 * H * 3 * H + (size_t)H * A + 6 * H + A + (size_t)2 * RT * LD + (size_t)RT * A;
    }
};

template <int H, int RW>
__global__ void __launch_bounds__(NT, 1)
gru_unroll_fwd_kernel(AgentParams p, int A, int64_t R, int nt, const float* __restrict__ x,
                      const float* h0, float* __restrict__ h_stash, float* __restrict__ gates,
                      float* __restrict__ q, float* h_last) {       // h0 and h_last may alias (rollout step)
    constexpr int RT = 16 * RW, JW = H / 16, LD = H + 1, H3 = 3 * H;
    extern __shared__ __align__(16) float smem[];
    float* WihT = smem;                       // [H][3H]   WihT[k][c] = w_ih[c][k]
    float* WhhT = WihT + H * H3;              // [H][3H]
    float* W2T = WhhT + H * H3;               // [H][A]
    float* bih = W2T + H * A;                 // [3H]
    float* bhh = bih + H3;                    // [3H]
    float* b2 = bhh + H3;                     // [A]
    float* xs = b2 + A;                       // [RT][LD]
    float* hs = xs + RT * LD;                 // [RT][LD]
    float* qs = hs + RT * LD;                 // [RT][A]

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int j0 = tx * JW, r0 = ty * RW;
    const int64_t row0 = (int64_t)blockIdx.x * RT;

    for (int i = tid; i < H3 * H; i += NT) {
        int c = i / H, k = i - c * H;
        WihT[k * H3 + c] = p.w_ih[i];
        WhhT[k * H3 + c] = p.w_hh[i];
    }
    for (int i = tid; i < A * H; i += NT) {
        int a = i / H, k = i - a * H;
        W2T[k * A + a] = p.fc2_w[i];
    }
    for (int i = tid; i < H3; i += NT) { bih[i] = p.b_ih[i]; bhh[i] = p.b_hh[i]; }
    for (int i = tid; i < A; i += NT) b2[i] = p.fc2_b[i];

    // own (row, j) elements: x and h tiles are filled by their owners
    float xr[RW][JW];
    bool rok[RW];
#pragma unroll
    for (int i = 0; i < RW; ++i) {
        int64_t row = row0 + r0 + i;
        rok[i] = row < R;
        float hv[JW];
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) { hv[jj] = 0.f; xr[i][jj] = 0.f; }
        if (rok[i]) {
            if (h0) {
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) hv[jj] = h0[row * H + j0 + jj];
            }
            ldg_vec<JW>(xr[i], x + row * H + j0);
            if (h_stash) stg_vec<JW>(h_stash + row * H + j0, hv);
        }
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) {
            hs[(r0 + i) * LD + j0 + jj] = hv[jj];
            xs[(r0 + i) * LD + j0 + jj] = xr[i][jj];
        }
    }
    __syncthreads();

    for (int t = 0; t < nt; ++t) {
        // prefetch next x tile into registers
        if (t + 1 < nt) {
#pragma unroll
            for (int i = 0; i < RW; ++i)
                if (rok[i]) ldg_vec<JW>(xr[i], x + ((int64_t)(t + 1) * R + row0 + r0 + i) * H + j0);
        }
        float ar[RW][JW], az[RW][JW], ain[RW][JW], ahn[RW][JW];
#pragma unroll
        for (int i = 0; i < RW; ++i)
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) { ar[i][jj] = 0.f; az[i][jj] = 0.f; ain[i][jj] = 0.f; ahn[i][jj] = 0.f; }

#pragma unroll 4
        for (int k = 0; k < H; ++k) {
            float xv[RW], hv[RW];
#pragma unroll
            for (int i = 0; i < RW; ++i) { xv[i] = xs[(r0 + i) * LD + k]; hv[i] = hs[(r0 + i) * LD + k]; }
            float wir[JW], wiz[JW], win[JW], whr[JW], whz[JW], whn[JW];
            lds_vec<JW>(wir, WihT + k * H3 + j0);
            lds_vec<JW>(wiz, WihT + k * H3 + H + j0);
            lds_vec<JW>(win, WihT + k * H3 + 2 * H + j0);
            lds_vec<JW>(whr, WhhT + k * H3 + j0);
            lds_vec<JW>(whz, WhhT + k * H3 + H + j0);
            lds_vec<JW>(whn, WhhT + k * H3 + 2 * H + j0);
#pragma unroll
            for (int i = 0; i < RW; ++i)
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) {
                    ar[i][jj] = fmaf(xv[i], wir[jj], ar[i][jj]);
                    ar[i][jj] = fmaf(hv[i], whr[jj], ar[i][jj]);
                    az[i][jj] = fmaf(xv[i], wiz[jj], az[i][jj]);
                    az[i][jj] = fmaf(hv[i], whz[jj], az[i][jj]);
                    ain[i][jj] = fmaf(xv[i], win[jj], ain[i][jj]);
                    ahn[i][jj] = fmaf(hv[i], whn[jj], ahn[i][jj]);
                }
        }
        // gates (torch GRUCell: r, z, n; h' = n + z (h - n))
        float hnew[RW][JW], gr[RW][JW], gz[RW][JW], gn[RW][JW], ghn[RW][JW];
#pragma unroll
        for (int i = 0; i < RW; ++i)
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                int j = j0 + jj;
                float r = sigmoidf_acc(ar[i][jj] + bih[j] + bhh[j]);
                float z = sigmoidf_acc(az[i][jj] + bih[H + j] + bhh[H + j]);
                float hn = ahn[i][jj] + bhh[2 * H + j];
                float n = tanhf(ain[i][jj] + bih[2 * H + j] + r * hn);
                float hold = hs[(r0 + i) * LD + j];
                hnew[i][jj] = n + z * (hold - n);
                gr[i][jj] = r; gz[i][jj] = z; gn[i][jj] = n; ghn[i][jj] = hn;
            }
        __syncthreads();                       // every thread is done reading xs / hs
#pragma unroll
        for (int i = 0; i < RW; ++i) {
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                hs[(r0 + i) * LD + j0 + jj] = hnew[i][jj];
                xs[(r0 + i) * LD + j0 + jj] = xr[i][jj];
            }
            if (rok[i]) {
                int64_t row = row0 + r0 + i;
                if (h_stash) stg_vec<JW>(h_stash + ((int64_t)(t + 1) * R + row) * H + j0, hnew[i]);
                if (gates) {
                    float* g = gates + ((int64_t)t * R + row) * 4 * H + j0;
                    stg_vec<JW>(g, gr[i]);
                    stg_vec<JW>(g + H, gz[i]);
                    stg_vec<JW>(g + 2 * H, gn[i]);
                    stg_vec<JW>(g + 3 * H, ghn[i]);
                }
                if (h_last && t == nt - 1) stg_vec<JW>(h_last + row * H + j0, hnew[i]);
            }
        }
        __syncthreads();
        // fc2 on the new hidden state
        {
            const int row = tid % RT;
            constexpr int AG = NT / RT;
            for (int a = tid / RT; a < A; a += AG) {
                float s = b2[a];
#pragma unroll 8
                for (int k = 0; k < H; ++k) s = fmaf(hs[row * LD + k], W2T[k * A + a], s);
                qs[row * A + a] = s;
            }
        }
        __syncthreads();
        {
            int64_t valid = R - row0 < RT ? R - row0 : RT;
            float* qo = q + ((int64_t)t * R + row0) * A;
            for (int i = tid; i < valid * A; i += NT) qo[i] = qs[i];
        }
        // the next sync (after the next step's GEMM) orders these reads before qs is rewritten
    }
}

// ------------------------------------------------------------------------------------------
// backward
// ------------------------------------------------------------------------------------------
template <int H, int RW>
struct BwdSmem {
    static constexpr int RT = 16 * RW;
    static constexpr int LDG_ = 4 * H + 1;
    static size_t floats(int A) { return (size_t)2 * 3 * H * H + (size_t)A * H + (size_t)RT * LDG_; }
};

template <int H, int RW>
__global__ void __launch_bounds__(NT, 1)
gru_unroll_bwd_kernel(AgentParams p, int A, int N, int T, int64_t R, const float* __restrict__ x,
                      const float* __restrict__ h_stash, float* __restrict__ gates,
                      const float* __restrict__ d_chosen, const int64_t* __restrict__ actions, int64_t actions_sb,
                      float* __restrict__ dpre1, const float* __restrict__ dq_full) {
    // dq_full != null (COMA policy gradient): dense dL/dq [T][R][A] for EVERY unrolled step instead of the Q-learner's
    // gradient at the taken action of steps t < T-1
    constexpr int RT = 16 * RW, JW = H / 16, H3 = 3 * H, LDD = 4 * H + 1;
    extern __shared__ __align__(16) float smem[];
    float* Wih = smem;                        // [3H][H]
    float* Whh = Wih + H3 * H;                // [3H][H]
    float* W2 = Whh + H3 * H;                 // [A][H]
    float* dgs = W2 + A * H;                  // [RT][4H+1]  da_r | da_z | da_n | da_n*r

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int j0 = tx * JW, r0 = ty * RW;
    const int64_t row0 = (int64_t)blockIdx.x * RT;

    for (int i = tid; i < H3 * H; i += NT) { Wih[i] = p.w_ih[i]; Whh[i] = p.w_hh[i]; }
    for (int i = tid; i < A * H; i += NT) W2[i] = p.fc2_w[i];

    bool rok[RW];
    int64_t bidx[RW];
    int nidx[RW];
    float dh[RW][JW];
#pragma unroll
    for (int i = 0; i < RW; ++i) {
        int64_t row = row0 + r0 + i;
        rok[i] = row < R;
        bidx[i] = rok[i] ? row / N : 0;
        nidx[i] = rok[i] ? (int)(row - bidx[i] * N) : 0;
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) dh[i][jj] = 0.f;
    }
    __syncthreads();

    for (int t = T - 1; t >= 0; --t) {
        float zk[RW][JW], xk[RW][JW];
#pragma unroll
        for (int i = 0; i < RW; ++i) {
            float dr_[JW], dz_[JW], dn_[JW], dnr_[JW];
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) { dr_[jj] = dz_[jj] = dn_[jj] = dnr_[jj] = 0.f; zk[i][jj] = 0.f; xk[i][jj] = 0.f; }
            if (rok[i]) {
                int64_t row = row0 + r0 + i;
                float* g = gates + ((int64_t)t * R + row) * 4 * H + j0;
                float r[JW], z[JW], n[JW], ghn[JW], hp[JW];
                ldg_vec<JW>(r, g);
                ldg_vec<JW>(z, g + H);
                ldg_vec<JW>(n, g + 2 * H);
                ldg_vec<JW>(ghn, g + 3 * H);
                ldg_vec<JW>(hp, h_stash + ((int64_t)t * R + row) * H + j0);
                ldg_vec<JW>(xk[i], x + ((int64_t)t * R + row) * H + j0);
                if (dq_full) {
                    const float* dqr = dq_full + ((int64_t)t * R + row) * A;
                    for (int a = 0; a < A; ++a) {
                        const float dq = __ldg(dqr + a);
#pragma unroll
                        for (int jj = 0; jj < JW; ++jj) dh[i][jj] = fmaf(dq, W2[a * H + j0 + jj], dh[i][jj]);
                    }
                } else if (t < T - 1) {
                    float dq = __ldg(d_chosen + (bidx[i] * (T - 1) + t) * N + nidx[i]);
                    int a = (int)__ldg(actions + bidx[i] * actions_sb + (int64_t)t * N + nidx[i]);
#pragma unroll
                    for (int jj = 0; jj < JW; ++jj) dh[i][jj] = fmaf(dq, W2[a * H + j0 + jj], dh[i][jj]);
                }
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) {
                    float d = dh[i][jj];
                    float dn = d * (1.f - z[jj]);
                    float dz = d * (hp[jj] - n[jj]);
                    float da_n = dn * (1.f - n[jj] * n[jj]);
                    float da_r = (da_n * ghn[jj]) * r[jj] * (1.f - r[jj]);
                    float da_z = dz * z[jj] * (1.f - z[jj]);
                    dr_[jj] = da_r; dz_[jj] = da_z; dn_[jj] = da_n; dnr_[jj] = da_n * r[jj];
                    zk[i][jj] = z[jj];
                }
                stg_vec<JW>(g, dr_);
                stg_vec<JW>(g + H, dz_);
                stg_vec<JW>(g + 2 * H, dn_);
                stg_vec<JW>(g + 3 * H, dnr_);
            }
            float* ds = dgs + (r0 + i) * LDD + j0;
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                ds[jj] = dr_[jj]; ds[H + jj] = dz_[jj]; ds[2 * H + jj] = dn_[jj]; ds[3 * H + jj] = dnr_[jj];
            }
        }
        __syncthreads();
        float dx[RW][JW], dhp[RW][JW];
#pragma unroll
        for (int i = 0; i < RW; ++i)
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) { dx[i][jj] = 0.f; dhp[i][jj] = 0.f; }
#pragma unroll 4
        for (int c = 0; c < 2 * H; ++c) {
            float wi[JW], wh[JW], d[RW];
            lds_vec<JW>(wi, Wih + c * H + j0);
            lds_vec<JW>(wh, Whh + c * H + j0);
#pragma unroll
            for (int i = 0; i < RW; ++i) d[i] = dgs[(r0 + i) * LDD + c];
#pragma unroll
            for (int i = 0; i < RW; ++i)
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) {
                    dx[i][jj] = fmaf(d[i], wi[jj], dx[i][jj]);
                    dhp[i][jj] = fmaf(d[i], wh[jj], dhp[i][jj]);
                }
        }
#pragma unroll 4
        for (int c = 2 * H; c < H3; ++c) {
            float wi[JW], wh[JW], d1[RW], d2[RW];
            lds_vec<JW>(wi, Wih + c * H + j0);
            lds_vec<JW>(wh, Whh + c * H + j0);
#pragma unroll
            for (int i = 0; i < RW; ++i) { d1[i] = dgs[(r0 + i) * LDD + c]; d2[i] = dgs[(r0 + i) * LDD + c + H]; }
#pragma unroll
            for (int i = 0; i < RW; ++i)
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) {
                    dx[i][jj] = fmaf(d1[i], wi[jj], dx[i][jj]);
                    dhp[i][jj] = fmaf(d2[i], wh[jj], dhp[i][jj]);
                }
        }
#pragma unroll
        for (int i = 0; i < RW; ++i) {
            float dp[JW];
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                dp[jj] = xk[i][jj] > 0.f ? dx[i][jj] : 0.f;
                dh[i][jj] = dh[i][jj] * zk[i][jj] + dhp[i][jj];
            }
            if (rok[i]) stg_vec<JW>(dpre1 + ((int64_t)t * R + row0 + r0 + i) * H + j0, dp);
        }
        __syncthreads();                       // dgs is rewritten by the next step
    }
}

// ------------------------------------------------------------------------------------------
// scatter-type gradients: fc2.weight/bias (rows selected by the taken action), fc1.weight
// columns of the last-action one-hot and of the agent id.  Each CTA owns a contiguous range of
// (t, row) items; inside a CTA NT/H lanes-groups walk the range with a fixed stride and every
// thread owns one hidden column j, so all additions happen in a fixed order.
// ------------------------------------------------------------------------------------------
template <int H>
__global__ void __launch_bounds__(NT)
agent_scatter_grads_kernel(int A, int N, int T, int64_t R, const float* __restrict__ h_stash,
                           const float* __restrict__ dpre1, const float* __restrict__ d_chosen,
                           const int64_t* __restrict__ actions, int64_t actions_sb,
                           const int64_t* __restrict__ filled, int64_t filled_sb, int use_act, int use_id,
                           int64_t items_per_cta, float* __restrict__ partial, int ti_tiles) {
    // ti_tiles > 0: h_stash and dpre1 are bf16 tile images [t][ti_tiles][16 KB] (bf16 tier)
    auto ti_fetch = [&](const float* base, int64_t t, int64_t row, int jj) -> float {
        const uint8_t* tile = reinterpret_cast<const uint8_t*>(base) + (t * ti_tiles + (row >> 7)) * 16384;
        const uint32_t rr = (uint32_t)(row & 127);
        const uint16_t w = *reinterpret_cast<const uint16_t*>(tile + rr * 128u + ((((uint32_t)jj >> 3) ^ (rr & 7u)) << 4) +
                                                              ((uint32_t)jj & 7u) * 2u);
        return __uint_as_float((uint32_t)w << 16);
    };
    constexpr int G = NT / H;
    extern __shared__ __align__(16) float smem[];
    // per group: w2 [A][H], b2 [A], act [A][H], id [N][H]
    const int per_group = A * H + A + A * H + N * H;
    const int tid = threadIdx.x, g = tid / H, j = tid - g * H;
    float* acc_w2 = smem + (size_t)g * per_group;
    float* acc_b2 = acc_w2 + A * H;
    float* acc_act = acc_b2 + A;
    float* acc_id = acc_act + A * H;
    for (int i = tid; i < G * per_group; i += NT) smem[i] = 0.f;
    __syncthreads();

    const int64_t total = (int64_t)T * R;
    const int64_t beg = (int64_t)blockIdx.x * items_per_cta;
    const int64_t end = beg + items_per_cta < total ? beg + items_per_cta : total;
    // batches of U items: all loads of a batch are issued before the first accumulation (the loop is
    // latency bound otherwise); accumulation order stays item order -> deterministic
    constexpr int U = 8;
    for (int64_t it0 = beg + g; it0 < end; it0 += (int64_t)G * U) {
        float dp[U], dq[U], hv[U];
        int nn[U], ap[U], aa[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t it = it0 + (int64_t)u * G;
            dp[u] = 0.f; dq[u] = 0.f; hv[u] = 0.f; nn[u] = -1; ap[u] = -1; aa[u] = -1;
            if (it < end) {
                int t = (int)(it / R);
                int64_t row = it - (int64_t)t * R;
                int64_t b = row / N;
                int n = (int)(row - b * N);
                nn[u] = n;
                dp[u] = ti_tiles > 0 ? ti_fetch(dpre1, t, row, j) : __ldg(dpre1 + it * H + j);
                if (use_act && t > 0 && __ldg(filled + b * filled_sb + (t - 1)) != 0)
                    ap[u] = (int)__ldg(actions + b * actions_sb + (int64_t)(t - 1) * N + n);
                if (d_chosen && t < T - 1) {           // d_chosen == null: the caller computes the fc2 gradients itself (dense dq)
                    dq[u] = __ldg(d_chosen + (b * (T - 1) + t) * N + n);
                    aa[u] = (int)__ldg(actions + b * actions_sb + (int64_t)t * N + n);
                    hv[u] = ti_tiles > 0 ? ti_fetch(h_stash, t + 1, row, j)
                                         : __ldg(h_stash + ((int64_t)(t + 1) * R + row) * H + j);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (nn[u] < 0) continue;
            if (use_id) acc_id[nn[u] * H + j] += dp[u];
            if (ap[u] >= 0) acc_act[ap[u] * H + j] += dp[u];
            if (aa[u] >= 0) {
                acc_w2[aa[u] * H + j] = fmaf(dq[u], hv[u], acc_w2[aa[u] * H + j]);
                if (j == 0) acc_b2[aa[u]] += dq[u];
            }
        }
    }
    __syncthreads();
    float* out = partial + (size_t)blockIdx.x * per_group;
    for (int i = tid; i < per_group; i += NT) {
        float s = 0.f;
#pragma unroll
        for (int gg = 0; gg < G; ++gg) s += smem[(size_t)gg * per_group + i];
        out[i] = s;
    }
}

__global__ void agent_scatter_reduce_kernel(const float* __restrict__ partial, int n_cta, int A, int N, int H, int O,
                                            int D_in, int use_act, int use_id, AgentGrads gr) {
    const int per_group = A * H + A + A * H + N * H;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= per_group) return;
    float s = 0.f;
    for (int c = 0; c < n_cta; ++c) s += partial[(size_t)c * per_group + i];
    if (i < A * H) {
        gr.fc2_w[i] = s;
    } else if (i < A * H + A) {
        gr.fc2_b[i - A * H] = s;
    } else if (i < 2 * A * H + A) {
        int k = i - (A * H + A);
        int a = k / H, j = k - a * H;
        if (use_act) gr.fc1_w[(int64_t)j * D_in + O + a] = s;
    } else {
        int k = i - (2 * A * H + A);
        int n = k / H, j = k - n * H;
        if (use_id) gr.fc1_w[(int64_t)j * D_in + O + (use_act ? A : 0) + n] = s;
    }
}

template <int H, int RW>
int launch_fwd(const AgentParams& p, int A, int64_t R, int nt, const float* x, const float* h0, float* h_stash,
               float* gates, float* q, float* h_last, cudaStream_t s) {
    size_t bytes = FwdSmem<H, RW>::floats(A) * sizeof(float);
    auto kern = gru_unroll_fwd_kernel<H, RW>;
    PMB_SMEM_ATTR(kern, (int)bytes);
    unsigned grid = (unsigned)ceil_div(R, 16 * RW);
    kern<<<grid, NT, bytes, s>>>(p, A, R, nt, x, h0, h_stash, gates, q, h_last);
    PMB_LAUNCH_CHECK("gru_unroll_fwd_kernel");
    return PMB_OK;
}

template <int H, int RW>
int launch_bwd(const AgentParams& p, int A, int N, int T, int64_t R, const float* x, const float* h_stash,
               float* gates, const float* d_chosen, const int64_t* actions, int64_t actions_sb, float* dpre1,
               cudaStream_t s, const float* dq_full) {
    size_t bytes = BwdSmem<H, RW>::floats(A) * sizeof(float);
    auto kern = gru_unroll_bwd_kernel<H, RW>;
    PMB_SMEM_ATTR(kern, (int)bytes);
    unsigned grid = (unsigned)ceil_div(R, 16 * RW);
    kern<<<grid, NT, bytes, s>>>(p, A, N, T, R, x, h_stash, gates, d_chosen, actions, actions_sb, dpre1, dq_full);
    PMB_LAUNCH_CHECK("gru_unroll_bwd_kernel");
    return PMB_OK;
}

// rows per thread: 4 (64-row tiles) once there are enough tiles to fill the machine twice
inline int pick_rw(int64_t R) { return ceil_div(R, 64) >= 2 * (int64_t)sm_count() ? 4 : 1; }

int scatter_ctas(int64_t items) {
    int64_t c = 4 * (int64_t)sm_count();
    int64_t mx = ceil_div(items, 64);
    if (c > mx) c = mx;
    return (int)(c < 1 ? 1 : c);
}

}  // namespace

// gru_h128.cu: rnn_hidden_dim 128 (W_ih and W_hh do not both fit in shared memory there)
int h128_fwd(const pmb_dims* d, int prec, const AgentParams& p, int64_t R, int nt, const float* x, const float* h0,
             float* h_seq, float* gates, int64_t ldg, int keep_gates, float* q, float* h_last, void* scratch,
             int64_t scratch_bytes, cudaStream_t s);
int h128_bwd(const pmb_dims* d, const pmb_batch* b, const AgentParams& p, const float* h_stash, float* gates,
             const float* d_chosen, cudaStream_t s, const float* dq_full);

int gru_fwd_dispatch(const pmb_dims* d, const AgentParams& p, int64_t R, int nt, const float* x, const float* h0,
                     float* h_stash, float* gates, float* q, float* h_last, cudaStream_t s) {
    int rw = pick_rw(R);
#define PMB_FWD(HH)                                                                                         \
    return rw == 4 ? launch_fwd<HH, 4>(p, d->A, R, nt, x, h0, h_stash, gates, q, h_last, s)                 \
                   : launch_fwd<HH, 1>(p, d->A, R, nt, x, h0, h_stash, gates, q, h_last, s)
    switch (d->H) {
        case 16: PMB_FWD(16);
        case 32: PMB_FWD(32);
        case 64: PMB_FWD(64);
        // input gates in `gates`, q from `h_stash`: both buffers are required (CUDA-core GEMMs on every tier, as the
        // unroll kernels above are fp32 on every tier)
        case 128: return h128_fwd(d, PMB_PREC_FP32, p, R, nt, x, h0, h_stash, gates, 4 * d->H, 1, q, h_last, nullptr, 0, s);
    }
#undef PMB_FWD
    set_error("rnn_hidden_dim %d unsupported (16, 32, 64, 128)", d->H);
    return PMB_ERR_INVALID;
}

int gru_bwd_dispatch(const pmb_dims* d, const pmb_batch* b, const AgentParams& p, const float* x,
                     const float* h_stash, float* gates, const float* d_chosen, float* dpre1, cudaStream_t s,
                     const float* dq_full) {
    int64_t R = (int64_t)d->B * d->N;
    int rw = pick_rw(R);
#define PMB_BWD(HH)                                                                                              \
    return rw == 4 ? launch_bwd<HH, 4>(p, d->A, d->N, d->T, R, x, h_stash, gates, d_chosen, b->actions,           \
                                       b->actions_sb, dpre1, s, dq_full)                                          \
                   : launch_bwd<HH, 1>(p, d->A, d->N, d->T, R, x, h_stash, gates, d_chosen, b->actions,           \
                                       b->actions_sb, dpre1, s, dq_full)
    switch (d->H) {
        case 16: PMB_BWD(16);
        case 32: PMB_BWD(32);
        case 64: PMB_BWD(64);
        case 128: return h128_bwd(d, b, p, h_stash, gates, d_chosen, s, dq_full);     // dpre1: agent_bwd, after it
    }
#undef PMB_BWD
    set_error("rnn_hidden_dim %d unsupported (16, 32, 64, 128)", d->H);
    return PMB_ERR_INVALID;
}

int64_t scatter_scratch_bytes(const pmb_dims* d) {
    int64_t items = (int64_t)d->T * d->B * d->N;
    int64_t per_group = (int64_t)2 * d->A * d->H + d->A + (int64_t)d->N * d->H;
    return align_up((int64_t)scatter_ctas(items) * per_group * 4, 256);
}

int scatter_grads_dispatch(const pmb_dims* d, const pmb_batch* b, const float* h_stash, const float* dpre1,
                           const float* d_chosen, AgentGrads gr, void* scratch, int64_t scratch_bytes,
                           cudaStream_t s, int ti_tiles) {
    int64_t R = (int64_t)d->B * d->N, items = (int64_t)d->T * R;
    int n_cta = scatter_ctas(items);
    if (scatter_scratch_bytes(d) > scratch_bytes) {
        set_error("agent scatter grads: scratch too small");
        return PMB_ERR_WORKSPACE;
    }
    int per_group = 2 * d->A * d->H + d->A + d->N * d->H;
    int64_t items_per_cta = ceil_div(items, n_cta);
    float* partial = static_cast<float*>(scratch);
    size_t smem = (size_t)(NT / d->H) * per_group * sizeof(float);
#define PMB_SC(HH)                                                                                                \
    {                                                                                                             \
        auto kern = agent_scatter_grads_kernel<HH>;                                                               \
        PMB_SMEM_ATTR(kern, (int)smem);             \
        kern<<<n_cta, NT, smem, s>>>(d->A, d->N, d->T, R, h_stash, dpre1, d_chosen, b->actions, b->actions_sb,    \
                                     b->filled, b->filled_sb, d->obs_last_action, d->obs_agent_id, items_per_cta, \
                                     partial, ti_tiles);                                                          \
    }                                                                                                             \
    break
    switch (d->H) {
        case 16: PMB_SC(16);
        case 32: PMB_SC(32);
        case 64: PMB_SC(64);
        case 128: PMB_SC(128);
        default: set_error("rnn_hidden_dim %d unsupported (16, 32, 64, 128)", d->H); return PMB_ERR_INVALID;
    }
#undef PMB_SC
    PMB_LAUNCH_CHECK("agent_scatter_grads_kernel");
    agent_scatter_reduce_kernel<<<(unsigned)ceil_div(per_group, 256), 256, 0, s>>>(
        partial, n_cta, d->A, d->N, d->H, d->O, d_in_of(d), d->obs_last_action, d->obs_agent_id, gr);
    PMB_LAUNCH_CHECK("agent_scatter_reduce_kernel");
    return PMB_OK;
}

}  // namespace pmb
