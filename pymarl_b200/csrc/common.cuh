// Shared device/host helpers for libpymarl_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include "../../include/pymarl_b200.h"

namespace pmb {

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define PMB_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t _e = (call);                                                    \
        if (_e != cudaSuccess) return ::pmb::cuda_fail(_e, #call, __FILE__, __LINE__); \
    } while (0)
extern std::atomic<long long> g_launch_count;     // kernels launched by this library (pmb_launch_count)
cudaError_t set_smem_attr(const void* func, int bytes);     // MaxDynamicSharedMemorySize, once per (kernel, device)
#define PMB_SMEM_ATTR(kern, bytes) PMB_CUDA(::pmb::set_smem_attr(reinterpret_cast<const void*>(kern), (int)(bytes)))
#define PMB_LAUNCH_CHECK(name)                                                      \
    do {                                                                            \
        ++::pmb::g_launch_count;                                                    \
        cudaError_t _e = cudaGetLastError();                                        \
        if (_e != cudaSuccess) return ::pmb::cuda_fail(_e, name, __FILE__, __LINE__); \
    } while (0)
#define PMB_REQUIRE(cond, ...)                                                      \
    do {                                                                            \
        if (!(cond)) { ::pmb::set_error(__VA_ARGS__); return PMB_ERR_INVALID; }     \
    } while (0)

int  sm_count();

// Launch with programmatic stream serialization (programmatic dependent launch): the kernel may start while its
// predecessor in the stream is still running - once every CTA of the predecessor has executed
// griddepcontrol.launch_dependents or exited - and must execute griddepcontrol.wait before it touches anything the
// predecessor reads or writes.  A predecessor that never triggers gives the ordinary stream order.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
bool rollout_pdl_enabled();                       // PMB_ROLLOUT_PDL=0 turns the dependent launches of the rollout step off
int  validate_dims(const pmb_dims* d);

inline __host__ __device__ int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline __host__ __device__ int64_t align_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

constexpr float kMaskValue = -9999999.0f;       // learners/q_learner.py:68,74

// batch row -> episode of the underlying buffer (pmb_batch.ep_index; NULL = identity)
__device__ __forceinline__ int64_t ep_row(const int64_t* ep_index, int64_t b) { return ep_index ? __ldg(ep_index + b) : b; }

// ---- row maps ---------------------------------------------------------------------------
// A logical row index m = (b*T + t)*N + n is mapped to  base + b*sb + t*st + n*sn  (element
// offsets).  Dense [M, ld] matrices use T = N = 1, sb = ld.
struct RowMap {
    int64_t sb, st, sn;
    int32_t T, N;
    __host__ __device__ inline int64_t offset(int64_t m) const {
        if (T == 1 && N == 1) return m * sb;                       // dense matrix
        const int64_t tn = (int64_t)T * N;
        if (((uint64_t)m | (uint64_t)tn) >> 31 == 0) {             // 32-bit divisions (the common case)
            const uint32_t mm = (uint32_t)m, tnn = (uint32_t)tn;
            const uint32_t b = mm / tnn, r = mm - b * tnn;
            const uint32_t t = r / (uint32_t)N, n = r - t * (uint32_t)N;
            return (int64_t)b * sb + (int64_t)t * st + (int64_t)n * sn;
        }
        int64_t b = m / tn;
        int32_t r = (int32_t)(m - b * tn);
        int32_t t = r / N;
        int32_t n = r - t * N;
        return b * sb + (int64_t)t * st + (int64_t)n * sn;
    }
};
inline RowMap dense_map(int64_t ld) { return RowMap{ld, 0, 0, 1, 1}; }

// ---- warp helpers -----------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- data-parallel exchange: loss sum i as a (hi, lo) float pair (pmb_dp_pack, dp_peer.cu) ----
// hi + lo reproduces the double to 2^-48.  mask_sum, an integer count, is split at a multiple of 2^12 instead: hi =
// floor(v / 2^12) * 2^12, lo = v - hi < 2^12.  Then every partial fp32 sum over up to 8 ranks of the hi parts (multiples of
// 2^12) and of the lo parts (integers < 2^15) is exact, so the exchanged count stays exact up to 2^36 in all; with the
// plain split an odd global count above 2^24 would round.
__device__ __forceinline__ void dp_pack_sum(int i, double v, float* pair) {
    const double hi = i == PMB_S_MASK_SUM ? floor(v * (1.0 / 4096.0)) * 4096.0 : (double)(float)v;
    pair[0] = (float)hi;
    pair[1] = (float)(v - hi);
}

__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }

// flat parameter views -----------------------------------------------------------------------
struct AgentParams {
    const float *fc1_w, *fc1_b, *w_ih, *w_hh, *b_ih, *b_hh, *fc2_w, *fc2_b;
};
struct AgentGrads {
    float *fc1_w, *fc1_b, *w_ih, *w_hh, *b_ih, *b_hh, *fc2_w, *fc2_b;
};
struct MixerParams {
    const float *w_cat;      // [(N+3)E, S]  hyper_w_1 | hyper_w_final | hyper_b_1 | V.0
    const float *b_cat;      // [(N+3)E]
    const float *v2_w;       // [E]
    const float *v2_b;       // [1]
};

void compute_layout(const pmb_dims* d, pmb_layout* L);
inline int d_in_of(const pmb_dims* d) {
    return d->O + (d->obs_last_action ? d->A : 0) + (d->obs_agent_id ? d->N : 0);
}
inline AgentParams agent_params(const pmb_dims* d, const float* flat) {
    pmb_layout L; compute_layout(d, &L);
    return AgentParams{flat + L.offset[PMB_P_FC1_W], flat + L.offset[PMB_P_FC1_B], flat + L.offset[PMB_P_W_IH],
                       flat + L.offset[PMB_P_W_HH], flat + L.offset[PMB_P_B_IH], flat + L.offset[PMB_P_B_HH],
                       flat + L.offset[PMB_P_FC2_W], flat + L.offset[PMB_P_FC2_B]};
}
inline AgentGrads agent_grads(const pmb_dims* d, float* flat) {
    pmb_layout L; compute_layout(d, &L);
    return AgentGrads{flat + L.offset[PMB_P_FC1_W], flat + L.offset[PMB_P_FC1_B], flat + L.offset[PMB_P_W_IH],
                      flat + L.offset[PMB_P_W_HH], flat + L.offset[PMB_P_B_IH], flat + L.offset[PMB_P_B_HH],
                      flat + L.offset[PMB_P_FC2_W], flat + L.offset[PMB_P_FC2_B]};
}
// flat_mixer points at the start of the mixer block (= flat + L.n_agent)
inline MixerParams mixer_params(const pmb_dims* d, const float* flat_mixer) {
    pmb_layout L; compute_layout(d, &L);
    int64_t base = L.n_agent;
    return MixerParams{flat_mixer + (L.offset[PMB_P_HW1_W] - base), flat_mixer + (L.offset[PMB_P_HW1_B] - base),
                       flat_mixer + (L.offset[PMB_P_V2_W] - base), flat_mixer + (L.offset[PMB_P_V2_B] - base)};
}

// COMA critic, flat layout in state_dict order: fc1.weight [Hc][D] | fc1.bias | fc2.weight [Hc][Hc] | fc2.bias |
// fc3.weight [A][Hc] | fc3.bias
struct CriticParams { const float *w1, *b1, *w2, *b2, *w3, *b3; };
struct CriticGrads { float *w1, *b1, *w2, *b2, *w3, *b3; };
template <class P, class F>
P critic_views(F* flat, int64_t D, int64_t Hc, int64_t A) {
    F* w1 = flat; F* b1 = w1 + Hc * D; F* w2 = b1 + Hc; F* b2 = w2 + Hc * Hc; F* w3 = b2 + Hc; F* b3 = w3 + A * Hc;
    return P{w1, b1, w2, b2, w3, b3};
}

// ---- kernels implemented in other translation units (host launchers) ---------------------
// gemm_simt.cu
//   C[m, n] (+ epilogue) = sum_k A[rowmap(m) + k] * W[n*ldw + k]
struct Fc1Epilogue {          // x = relu(acc + b1 + W_id[:, n] + W_act[:, a_prev]) -> x_out time major
    const float* fc1_w;       // [H, D_in]
    const float* fc1_b;
    const int64_t* actions; int64_t actions_sb;
    const int64_t* filled;  int64_t filled_sb;
    float* x_out;             // [nt][R][H]
    int32_t T_batch, t0, nt, N, O, A, H, D_in, use_act, use_id;
    int64_t R;
};
int launch_fc1_gemm(const float* obs, RowMap map, int64_t M, int32_t K, const float* W, int32_t ldw, int32_t Ncols,
                    const Fc1Epilogue& ep, cudaStream_t s);
//   plain:  C[m*ldc + n] = acc + bias[n]   (bias may be null), optional relu
int launch_gemm_tn(const float* A, RowMap map, int64_t M, int32_t K, const float* W, int32_t ldw, int32_t Ncols,
                   const float* bias, float* C, int64_t ldc, int relu, cudaStream_t s);
//   out[c*ldo + k] = sum_m D[dmap(m) + c] * A[amap(m) + k]  for c < C, k < K ; bias_out[c] = sum_m D[dmap(m)+c]
//   deterministic split over m: scratch holds the per-slice partials.
int64_t gemm_atb_scratch_bytes(int32_t C, int32_t K, int64_t M);
int launch_gemm_atb(const float* D, RowMap dmap, int32_t C, const float* A, RowMap amap, int32_t K, int64_t M,
                    float* out, int64_t ldo, float* bias_out, void* scratch, int64_t scratch_bytes, cudaStream_t s);

// tc_atb.cu: same contract on tcgen05 (bf16 operands, fp32 accumulate)
int64_t tc_atb_scratch_bytes(int C, int K, int64_t M);
int tc_gemm_atb(const float* D, RowMap dmap, int C, const float* A, RowMap amap, int K, int64_t M, float* out,
                int64_t ldo, float* bias_out, void* scratch, int64_t scratch_bytes, cudaStream_t s);
// dispatch on the precision tier
inline int64_t atb_scratch_bytes(int prec, int C, int K, int64_t M) {
    return prec == PMB_PREC_BF16 ? tc_atb_scratch_bytes(C, K, M) : gemm_atb_scratch_bytes(C, K, M);
}
inline int gemm_atb_any(int prec, const float* D, RowMap dmap, int C, const float* A, RowMap amap, int K, int64_t M,
                        float* out, int64_t ldo, float* bias_out, void* scratch, int64_t scratch_bytes, cudaStream_t s) {
    return prec == PMB_PREC_BF16 ? tc_gemm_atb(D, dmap, C, A, amap, K, M, out, ldo, bias_out, scratch, scratch_bytes, s)
                                 : launch_gemm_atb(D, dmap, C, A, amap, K, M, out, ldo, bias_out, scratch, scratch_bytes, s);
}

}  // namespace pmb
