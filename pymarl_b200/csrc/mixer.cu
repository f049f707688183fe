// K3 / K4b: QMIX and VDN mixers, forward and backward (modules/mixers/qmix.py:28-47, vdn.py:9-10).
//
// QMIX forward = one GEMM  raw[M, (N+3)E] = state[M, S] . W_cat^T + b_cat  (the four hypernets
// share the state operand: hyper_w_1 | hyper_w_final | hyper_b_1 | V.0) followed by a warp-per-row
// mixing kernel:  hidden = ELU(q . |w1| + b1),  q_tot = hidden . |w_final| + V.2(ReLU(v0)).
// Backward: the mixing kernel is differentiated by hand (d|x| = sign, dELU = 1 or exp(pre),
// dReLU = x > 0), d_raw overwrites raw in place, and the hypernet weight gradients are
// d_raw^T . state (deterministic split-M GEMM); no gradient flows to the state.
#include "common.cuh"

namespace pmb {

namespace {

__device__ __forceinline__ float sgn(float x) { return (float)((x > 0.f) - (x < 0.f)); }

// raw row layout: [ w1 (N*E) | w_final (E) | b1 (E) | v0 (E) ]
__global__ void __launch_bounds__(256)
qmix_mix_fwd_kernel(int64_t M, int N, int E, const float* __restrict__ raw, const float* __restrict__ agent_qs,
                    const float* __restrict__ v2_w, const float* __restrict__ v2_b, float* __restrict__ q_tot) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= M) return;
    const int C = (N + 3) * E;
    const float* r = raw + warp * C;
    const float* qs = agent_qs + warp * N;
    float part = 0.f;
    for (int e = lane; e < E; e += 32) {
        float pre = 0.f;
        for (int n = 0; n < N; ++n) pre = fmaf(__ldg(qs + n), fabsf(__ldg(r + n * E + e)), pre);
        pre += __ldg(r + (N + 1) * E + e);
        float hidden = pre > 0.f ? pre : expm1f(pre);
        float wf = fabsf(__ldg(r + N * E + e));
        float v0 = fmaxf(__ldg(r + (N + 2) * E + e), 0.f);
        part = fmaf(hidden, wf, part);
        part = fmaf(v0, __ldg(v2_w + e), part);
    }
    part = warp_sum(part);
    if (lane == 0) q_tot[warp] = part + __ldg(v2_b);
}

__global__ void __launch_bounds__(256)
vdn_fwd_kernel(int64_t M, int N, const float* __restrict__ agent_qs, float* __restrict__ q_tot) {
    int64_t m = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= M) return;
    float s = 0.f;
    for (int n = 0; n < N; ++n) s += __ldg(agent_qs + m * N + n);
    q_tot[m] = s;
}

__global__ void __launch_bounds__(256)
vdn_bwd_kernel(int64_t M, int N, const float* __restrict__ g, float* __restrict__ d_qs) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= M * N) return;
    d_qs[i] = __ldg(g + i / N);
}

// One warp per row, grid-stride; V.2 gradients are accumulated per lane in registers and
// written as per-block partials (fixed assignment -> deterministic).
constexpr int MIXB_BLOCK = 256;
__global__ void __launch_bounds__(MIXB_BLOCK)
qmix_mix_bwd_kernel(int64_t M, int N, int E, float* __restrict__ raw, const float* __restrict__ agent_qs,
                    const float* __restrict__ v2_w, const float* __restrict__ g, float* __restrict__ d_qs,
                    float* __restrict__ v2_partial /* [grid][E+1] */) {
    __shared__ float red[MIXB_BLOCK / 32][65];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warps_total = (int64_t)gridDim.x * (MIXB_BLOCK / 32);
    const int C = (N + 3) * E;
    float dv2w[2] = {0.f, 0.f};        // e = lane, lane + 32  (E <= 64)
    float dv2b = 0.f;
    for (int64_t m = (int64_t)blockIdx.x * (MIXB_BLOCK / 32) + wib; m < M; m += warps_total) {
        float* r = raw + m * C;
        const float* qs = agent_qs + m * N;
        const float gm = __ldg(g + m);
        if (lane == 0) dv2b += gm;
        float dpre[2] = {0.f, 0.f};
        int ei = 0;
        for (int e = lane; e < E; e += 32, ++ei) {
            float pre = 0.f;
            for (int n = 0; n < N; ++n) pre = fmaf(__ldg(qs + n), fabsf(r[n * E + e]), pre);
            pre += r[(N + 1) * E + e];
            float hidden = pre > 0.f ? pre : expm1f(pre);
            float wf_raw = r[N * E + e];
            float v0_raw = r[(N + 2) * E + e];
            float dhid = gm * fabsf(wf_raw);
            float dp = dhid * (pre > 0.f ? 1.f : expf(pre));
            dpre[ei] = dp;
            dv2w[ei] = fmaf(gm, fmaxf(v0_raw, 0.f), dv2w[ei]);
            r[N * E + e] = sgn(wf_raw) * (gm * hidden);
            r[(N + 1) * E + e] = dp;
            r[(N + 2) * E + e] = v0_raw > 0.f ? gm * __ldg(v2_w + e) : 0.f;
        }
        for (int n = 0; n < N; ++n) {
            float qn = __ldg(qs + n);
            float acc = 0.f;
            ei = 0;
            for (int e = lane; e < E; e += 32, ++ei) {
                float w = r[n * E + e];
                acc = fmaf(fabsf(w), dpre[ei], acc);
                r[n * E + e] = sgn(w) * qn * dpre[ei];
            }
            acc = warp_sum(acc);
            if (lane == 0) d_qs[m * N + n] = acc;
        }
    }
    // block reduction of the V.2 partials in warp order
    red[wib][lane] = dv2w[0];
    red[wib][32 + lane] = dv2w[1];
    if (lane == 0) red[wib][64] = dv2b;
    __syncthreads();
    if (threadIdx.x < 65) {
        float s = 0.f;
        for (int w = 0; w < MIXB_BLOCK / 32; ++w) s += red[w][threadIdx.x];
        if (threadIdx.x < E) v2_partial[(int64_t)blockIdx.x * (E + 1) + threadIdx.x] = s;
        if (threadIdx.x == 64) v2_partial[(int64_t)blockIdx.x * (E + 1) + E] = s;
    }
}

__global__ void v2_reduce_kernel(const float* __restrict__ partial, int n_blocks, int E, float* __restrict__ dv2_w,
                                 float* __restrict__ dv2_b) {
    int i = threadIdx.x;
    if (i > E) return;
    float s = 0.f;
    for (int b = 0; b < n_blocks; ++b) s += partial[(int64_t)b * (E + 1) + i];
    if (i < E) dv2_w[i] = s; else dv2_b[0] = s;
}

int mixb_grid(int64_t M) {
    int64_t g = 8 * (int64_t)sm_count();
    int64_t mx = ceil_div(M, MIXB_BLOCK / 32);
    if (g > mx) g = mx;
    return (int)(g < 1 ? 1 : g);
}

}  // namespace

int launch_mixer_fwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs,
                     int t_off, float* raw, float* q_tot, cudaStream_t s) {
    const int64_t M = (int64_t)d->B * (d->T - 1);
    if (M <= 0) return PMB_OK;
    if (d->mixer == PMB_MIXER_VDN) {
        vdn_fwd_kernel<<<(unsigned)ceil_div(M, 256), 256, 0, s>>>(M, d->N, agent_qs, q_tot);
        PMB_LAUNCH_CHECK("vdn_fwd_kernel");
        return PMB_OK;
    }
    PMB_REQUIRE(d->mixer == PMB_MIXER_QMIX, "mixer_fwd: no mixer configured (IQL)");
    PMB_REQUIRE(b->state != nullptr && raw != nullptr, "mixer_fwd: state and raw are required for QMIX");
    MixerParams mp = mixer_params(d, flat_mixer);
    const int C = (d->N + 3) * d->E;
    RowMap smap{b->state_sb, (int64_t)d->S, 0, d->T - 1, 1};
    int rc = launch_gemm_tn(static_cast<const float*>(b->state) + (int64_t)t_off * d->S, smap, M, d->S, mp.w_cat, d->S, C, mp.b_cat, raw, C, 0, s);
    if (rc) return rc;
    qmix_mix_fwd_kernel<<<(unsigned)ceil_div(M * 32, 256), 256, 0, s>>>(M, d->N, d->E, raw, agent_qs, mp.v2_w, mp.v2_b,
                                                                       q_tot);
    PMB_LAUNCH_CHECK("qmix_mix_fwd_kernel");
    return PMB_OK;
}

int64_t mixer_bwd_scratch_bytes(const pmb_dims* d) {
    if (d->mixer != PMB_MIXER_QMIX) return 256;
    const int64_t M = (int64_t)d->B * (d->T - 1);
    const int C = (d->N + 3) * d->E;
    return atb_scratch_bytes(d->precision, C, d->S, M) + align_up((int64_t)mixb_grid(M) * (d->E + 1) * 4, 256);
}

int launch_mixer_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs, float* raw,
                     const float* g, float* d_agent_qs, float* flat_grad_mixer, void* scratch, int64_t scratch_bytes,
                     cudaStream_t s) {
    const int64_t M = (int64_t)d->B * (d->T - 1);
    if (M <= 0) return PMB_OK;
    if (d->mixer == PMB_MIXER_VDN) {
        vdn_bwd_kernel<<<(unsigned)ceil_div(M * d->N, 256), 256, 0, s>>>(M, d->N, g, d_agent_qs);
        PMB_LAUNCH_CHECK("vdn_bwd_kernel");
        return PMB_OK;
    }
    PMB_REQUIRE(d->mixer == PMB_MIXER_QMIX, "mixer_bwd: no mixer configured (IQL)");
    if (mixer_bwd_scratch_bytes(d) > scratch_bytes) {
        set_error("mixer_bwd: scratch too small");
        return PMB_ERR_WORKSPACE;
    }
    pmb_layout L;
    compute_layout(d, &L);
    MixerParams mp = mixer_params(d, flat_mixer);
    float* gbase = flat_grad_mixer - L.n_agent;        // index with absolute layout offsets
    const int C = (d->N + 3) * d->E;
    const int grid = mixb_grid(M);
    float* v2_partial = static_cast<float*>(scratch);
    char* atb_scratch = static_cast<char*>(scratch) + align_up((int64_t)grid * (d->E + 1) * 4, 256);
    int64_t atb_bytes = scratch_bytes - align_up((int64_t)grid * (d->E + 1) * 4, 256);
    qmix_mix_bwd_kernel<<<grid, MIXB_BLOCK, 0, s>>>(M, d->N, d->E, raw, agent_qs, mp.v2_w, g, d_agent_qs, v2_partial);
    PMB_LAUNCH_CHECK("qmix_mix_bwd_kernel");
    v2_reduce_kernel<<<1, 128, 0, s>>>(v2_partial, grid, d->E, gbase + L.offset[PMB_P_V2_W], gbase + L.offset[PMB_P_V2_B]);
    PMB_LAUNCH_CHECK("v2_reduce_kernel");
    // hypernet weights and biases:  dW_cat = d_raw^T . state[:, :-1],  db_cat = column sums
    RowMap smap{b->state_sb, (int64_t)d->S, 0, d->T - 1, 1};
    return gemm_atb_any(d->precision, raw, dense_map(C), C, static_cast<const float*>(b->state), smap, d->S, M, gbase + L.offset[PMB_P_HW1_W],
                        d->S, gbase + L.offset[PMB_P_HW1_B], atb_scratch, atb_bytes, s);
}

}  // namespace pmb
