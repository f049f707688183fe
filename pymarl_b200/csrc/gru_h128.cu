// RNNAgent at rnn_hidden_dim 128, both precision tiers.
//
// The unroll kernels of agent.cu keep W_ih and W_hh in shared memory: 2 x 3H x H fp32 = 384 KB at H = 128, beyond the
// 227 KB a block can have.  Here the GRU is split so that only the sequential part holds weights on chip:
//   forward  : gi = x W_ih^T + b_ih for all nt x R rows as ONE time-parallel GEMM into the first 3H columns of `gates`;
//              gru_h128_fwd_kernel runs the recurrence with W_hh^T (192 KB) resident and writes h_t to a [nt+1][R][H]
//              sequence; q = h_t W_2^T + b_2 is one GEMM over that sequence afterwards (W_2, up to 32 KB, does not fit
//              beside W_hh^T and the h tile).
//   backward : gru_h128_bwd_kernel carries dh through the chain with W_hh (192 KB) resident and overwrites `gates` with
//              the gate pre-activation gradients (the layout agent.cu's backward leaves); it computes no dx.
//              dpre1 = relu'(x) * ([da_r | da_z | da_n] W_ih) is one GEMM plus the ReLU mask.
// The GEMMs run on tcgen05 (bf16 operands, fp32 accumulate) on the bf16 tier and on the CUDA-core gemm_tn on the fp32
// tier; the two recurrence kernels are fp32 on both tiers.
//
// Both kernels: 256 threads own a 64-row tile, thread = 8 rows x 4 hidden columns (of each gate).  A warp covers 4
// column groups x all 64 rows, so per k it reads 64 B of weights and 256 B of the transposed h (or dgate) tile, both
// without bank conflicts: the loops are FFMA bound.  Shared memory: 192 KB weights + a 32 KB [H][64] tile = 224 KB.
//
// reference: modules/agents/rnn_agent.py:27-36 and torch autograd through GRUCell.
#include <cuda_bf16.h>
#include "common.cuh"
#include "mixer_tc.cuh"

namespace pmb {

int tc_gemm_plain(const float* A, RowMap amap, int64_t M, int K, const __nv_bfloat16* Wp, int Ncols_padded, int Nreal,
                  const float* bias, float* C, int64_t ldc, cudaStream_t s);
int launch_relu_mask(int64_t n, const float* x, float* dx, cudaStream_t s);
int launch_transpose(int rows, int cols, const float* in, float* out, cudaStream_t s);
void phase_mark(cudaStream_t s, const char* name);

namespace {

constexpr int H = 128, H3 = 3 * H, NT = 256, RT = 64, RW = 8, JW = 4;
constexpr size_t kSmemBytes = (size_t)(H3 * H + H * RT) * sizeof(float);     // 229376 B
static_assert(kSmemBytes <= 232448, "W_hh + the row tile must fit the 227 KB opt-in");

// tile row of the thread's i-th row: rows rg*4 .. rg*4+3 and 32 + rg*4 .. 32 + rg*4+3, so the two float4 reads of a
// [k][64] tile row by one warp cover 128 contiguous bytes each
__device__ __forceinline__ int tile_row(int rg, int i) { return (i & 4) * 8 + rg * 4 + (i & 3); }

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float a, float b, float c, float d) {
    *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// ------------------------------------------------------------------------------------------
// forward recurrence: gates[t][row][0, 3H) holds gi = x_t W_ih^T + b_ih (row stride ldg).
//   h_seq (may be null): [nt+1][R][H], slot 0 = h0, slot t+1 = h_t
//   keep_gates: gates[t][row] is overwritten with (r, z, n, W_hn h + b_hn) for the backward (ldg = 4H)
//   h_last (may alias h0): h_{nt}
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
gru_h128_fwd_kernel(const float* __restrict__ w_hh, const float* __restrict__ b_hh, int64_t R, int nt, float* gates,
                    int64_t ldg, int keep_gates, const float* h0, float* __restrict__ h_seq, float* h_last) {
    extern __shared__ __align__(16) float smem[];
    float* WhhT = smem;                       // [H][3H]  WhhT[k][c] = w_hh[c][k]
    float* hsT = WhhT + H * H3;               // [H][RT]  hsT[k][r] = h_{t-1}[row0 + r][k]
    const int tid = threadIdx.x, lane = tid & 31;
    const int j0 = ((tid >> 5) * 4 + (lane & 3)) * JW, rg = lane >> 2;
    const int64_t row0 = (int64_t)blockIdx.x * RT;

    for (int i = tid; i < H3 * H; i += NT) {
        const int c = i / H, k = i - c * H;
        WhhT[k * H3 + c] = w_hh[i];
    }
    float bh[3][JW];
#pragma unroll
    for (int g = 0; g < 3; ++g)
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) bh[g][jj] = b_hh[g * H + j0 + jj];

    float h[RW][JW];
#pragma unroll
    for (int i = 0; i < RW; ++i) {
        const int64_t row = row0 + tile_row(rg, i);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < R) {
            if (h0) v = *reinterpret_cast<const float4*>(h0 + row * H + j0);
            if (h_seq) st4(h_seq + row * H + j0, v.x, v.y, v.z, v.w);
        }
        h[i][0] = v.x; h[i][1] = v.y; h[i][2] = v.z; h[i][3] = v.w;
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) hsT[(j0 + jj) * RT + tile_row(rg, i)] = h[i][jj];
    }
    __syncthreads();

    for (int t = 0; t < nt; ++t) {
        if (t + 1 < nt) {                     // the next step's input gates: HBM -> L2 under this step's FFMA loop
#pragma unroll
            for (int i = 0; i < RW; ++i) {
                const int64_t row = row0 + tile_row(rg, i);
                if (row < R) {
                    const float* g = gates + ((int64_t)(t + 1) * R + row) * ldg + j0;
                    prefetch_l2(g); prefetch_l2(g + H); prefetch_l2(g + 2 * H);
                }
            }
        }
        float acc[3][RW][JW];
#pragma unroll
        for (int g = 0; g < 3; ++g)
#pragma unroll
            for (int i = 0; i < RW; ++i)
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) acc[g][i][jj] = 0.f;
#pragma unroll 2
        for (int k = 0; k < H; ++k) {
            const float4 ha = ld4(hsT + k * RT + rg * 4), hb = ld4(hsT + k * RT + 32 + rg * 4);
            const float hv[RW] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
#pragma unroll
            for (int g = 0; g < 3; ++g) {
                const float4 w = ld4(WhhT + k * H3 + g * H + j0);
                const float wv[JW] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int i = 0; i < RW; ++i)
#pragma unroll
                    for (int jj = 0; jj < JW; ++jj) acc[g][i][jj] = fmaf(hv[i], wv[jj], acc[g][i][jj]);
            }
        }
        __syncthreads();                      // every thread is done reading hsT
#pragma unroll
        for (int i = 0; i < RW; ++i) {
            const int64_t row = row0 + tile_row(rg, i);
            const bool ok = row < R;
            float* g = gates + ((int64_t)t * R + row) * ldg + j0;
            float4 gr = make_float4(0.f, 0.f, 0.f, 0.f), gz = gr, gn = gr;
            if (ok) { gr = ldg4(g); gz = ldg4(g + H); gn = ldg4(g + 2 * H); }
            const float gir[JW] = {gr.x, gr.y, gr.z, gr.w}, giz[JW] = {gz.x, gz.y, gz.z, gz.w};
            const float gin[JW] = {gn.x, gn.y, gn.z, gn.w};
            // torch GRUCell: r, z, n; h' = n + z (h - n)
            float r[JW], z[JW], n[JW], hn[JW];
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                r[jj] = sigmoidf_acc(gir[jj] + acc[0][i][jj] + bh[0][jj]);
                z[jj] = sigmoidf_acc(giz[jj] + acc[1][i][jj] + bh[1][jj]);
                hn[jj] = acc[2][i][jj] + bh[2][jj];
                n[jj] = tanhf(gin[jj] + r[jj] * hn[jj]);
                h[i][jj] = n[jj] + z[jj] * (h[i][jj] - n[jj]);
                hsT[(j0 + jj) * RT + tile_row(rg, i)] = h[i][jj];
            }
            if (ok) {
                if (keep_gates) {
                    st4(g, r[0], r[1], r[2], r[3]);
                    st4(g + H, z[0], z[1], z[2], z[3]);
                    st4(g + 2 * H, n[0], n[1], n[2], n[3]);
                    st4(g + 3 * H, hn[0], hn[1], hn[2], hn[3]);
                }
                if (h_seq) st4(h_seq + ((int64_t)(t + 1) * R + row) * H + j0, h[i][0], h[i][1], h[i][2], h[i][3]);
                if (h_last && t == nt - 1) st4(h_last + row * H + j0, h[i][0], h[i][1], h[i][2], h[i][3]);
            }
        }
        __syncthreads();                      // hsT holds h_t
    }
}

// ------------------------------------------------------------------------------------------
// BPTT.  dh lives in registers across the unroll; per step the gate gradients overwrite gates[t] in place
// (da_r | da_z | da_n | da_n * r) and dh_{t-1} = dh_t z + [da_r | da_z | da_n r] W_hh, one gate block at a time
// through the [H][64] tile.  dq_full != null (COMA): dense dL/dq [T][R][A] for every step; else the Q-learner's
// gradient at the taken action of the steps t < T-1.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(NT, 1)
gru_h128_bwd_kernel(const float* __restrict__ w_hh, const float* __restrict__ w2, int A, int N, int T, int64_t R,
                    const float* __restrict__ h_stash, float* __restrict__ gates, const float* __restrict__ d_chosen,
                    const int64_t* __restrict__ actions, int64_t actions_sb, const float* __restrict__ dq_full) {
    extern __shared__ __align__(16) float smem[];
    float* Whh = smem;                        // [3H][H] as stored
    float* dsT = Whh + H3 * H;                // [H][RT]  one gate block of the pre-activation gradients, transposed
    const int tid = threadIdx.x, lane = tid & 31;
    const int j0 = ((tid >> 5) * 4 + (lane & 3)) * JW, rg = lane >> 2;
    const int64_t row0 = (int64_t)blockIdx.x * RT;

    for (int i = tid; i < H3 * H / 4; i += NT)
        reinterpret_cast<float4*>(Whh)[i] = __ldg(reinterpret_cast<const float4*>(w_hh) + i);

    float dh[RW][JW];
#pragma unroll
    for (int i = 0; i < RW; ++i)
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) dh[i][jj] = 0.f;

    for (int t = T - 1; t >= 0; --t) {
        float dr[RW][JW], dz[RW][JW], dnr[RW][JW];
#pragma unroll
        for (int i = 0; i < RW; ++i) {
            const int64_t row = row0 + tile_row(rg, i);
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) dr[i][jj] = dz[i][jj] = dnr[i][jj] = 0.f;
            if (row < R) {
                const int64_t b = row / N;
                const int n_ = (int)(row - b * N);
                if (dq_full) {
                    const float* dqr = dq_full + ((int64_t)t * R + row) * A;
                    for (int a = 0; a < A; ++a) {
                        const float dq = __ldg(dqr + a);
                        const float4 w = ldg4(w2 + (int64_t)a * H + j0);
                        dh[i][0] = fmaf(dq, w.x, dh[i][0]); dh[i][1] = fmaf(dq, w.y, dh[i][1]);
                        dh[i][2] = fmaf(dq, w.z, dh[i][2]); dh[i][3] = fmaf(dq, w.w, dh[i][3]);
                    }
                } else if (t < T - 1) {
                    const float dq = __ldg(d_chosen + (b * (T - 1) + t) * N + n_);
                    const int a = (int)__ldg(actions + b * actions_sb + (int64_t)t * N + n_);
                    const float4 w = ldg4(w2 + (int64_t)a * H + j0);
                    dh[i][0] = fmaf(dq, w.x, dh[i][0]); dh[i][1] = fmaf(dq, w.y, dh[i][1]);
                    dh[i][2] = fmaf(dq, w.z, dh[i][2]); dh[i][3] = fmaf(dq, w.w, dh[i][3]);
                }
                float* g = gates + ((int64_t)t * R + row) * 4 * H + j0;
                const float4 r4 = ldg4(g), z4 = ldg4(g + H), n4 = ldg4(g + 2 * H), hn4 = ldg4(g + 3 * H);
                const float4 hp4 = ldg4(h_stash + ((int64_t)t * R + row) * H + j0);
                const float r[JW] = {r4.x, r4.y, r4.z, r4.w}, z[JW] = {z4.x, z4.y, z4.z, z4.w};
                const float n[JW] = {n4.x, n4.y, n4.z, n4.w}, ghn[JW] = {hn4.x, hn4.y, hn4.z, hn4.w};
                const float hp[JW] = {hp4.x, hp4.y, hp4.z, hp4.w};
                float dn_[JW];
#pragma unroll
                for (int jj = 0; jj < JW; ++jj) {
                    const float d = dh[i][jj];
                    const float dn = d * (1.f - z[jj]);
                    const float dzz = d * (hp[jj] - n[jj]);
                    const float da_n = dn * (1.f - n[jj] * n[jj]);
                    dr[i][jj] = (da_n * ghn[jj]) * r[jj] * (1.f - r[jj]);
                    dz[i][jj] = dzz * z[jj] * (1.f - z[jj]);
                    dn_[jj] = da_n;
                    dnr[i][jj] = da_n * r[jj];
                    dh[i][jj] = d * z[jj];
                }
                st4(g, dr[i][0], dr[i][1], dr[i][2], dr[i][3]);
                st4(g + H, dz[i][0], dz[i][1], dz[i][2], dz[i][3]);
                st4(g + 2 * H, dn_[0], dn_[1], dn_[2], dn_[3]);
                st4(g + 3 * H, dnr[i][0], dnr[i][1], dnr[i][2], dnr[i][3]);
            }
        }
#pragma unroll
        for (int gb = 0; gb < 3; ++gb) {
            __syncthreads();                  // the previous block's (or step's) reads of dsT are done
#pragma unroll
            for (int i = 0; i < RW; ++i)
#pragma unroll
                for (int jj = 0; jj < JW; ++jj)
                    dsT[(j0 + jj) * RT + tile_row(rg, i)] = gb == 0 ? dr[i][jj] : gb == 1 ? dz[i][jj] : dnr[i][jj];
            __syncthreads();
            const float* W = Whh + (int64_t)gb * H * H;
#pragma unroll 4
            for (int c = 0; c < H; ++c) {
                const float4 da = ld4(dsT + c * RT + rg * 4), db = ld4(dsT + c * RT + 32 + rg * 4);
                const float dv[RW] = {da.x, da.y, da.z, da.w, db.x, db.y, db.z, db.w};
                const float4 w = ld4(W + c * H + j0);
                const float wv[JW] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int i = 0; i < RW; ++i)
#pragma unroll
                    for (int jj = 0; jj < JW; ++jj) dh[i][jj] = fmaf(dv[i], wv[jj], dh[i][jj]);
            }
        }
    }
}

// C[m][n] = A[m][:K] . W[n][:K] + bias[n] on the precision tier's GEMM; W is packed into `scratch` on the bf16 tier
int gemm_tn_tier(int prec, const float* A, int64_t lda, int64_t M, int K, const float* W, int Ncols, const float* bias,
                 float* C, int64_t ldc, char*& scratch, cudaStream_t s) {
    if (prec != PMB_PREC_BF16) return launch_gemm_tn(A, dense_map(lda), M, K, W, K, Ncols, bias, C, ldc, 0, s);
    __nv_bfloat16* wp = reinterpret_cast<__nv_bfloat16*>(scratch);
    scratch += align_up(tc_packed_elems((int)align_up(Ncols, 32), K) * 2, 256);
    const float* ptrs[1] = {W};
    int rows[1] = {Ncols}, lds[1] = {K};
    int rc = tc_pack_w(ptrs, rows, lds, 1, K, wp, s);
    if (rc) return rc;
    return tc_gemm_plain(A, dense_map(lda), M, K, wp, (int)align_up(Ncols, 32), Ncols, bias, C, ldc, s);
}

int64_t packed_bytes(int Ncols, int K) { return align_up(tc_packed_elems((int)align_up(Ncols, 32), K) * 2, 256); }

}  // namespace

int64_t h128_fwd_scratch_bytes(const pmb_dims* d, int prec) {
    return prec == PMB_PREC_BF16 ? packed_bytes(H3, H) + packed_bytes(d->A, H) : 0;
}

int64_t h128_dpre1_scratch_bytes(int prec) {
    return align_up((int64_t)H3 * H * 4, 256) + (prec == PMB_PREC_BF16 ? packed_bytes(H, H3) : 0);
}

// gi GEMM -> recurrence -> fc2 GEMM over nt steps of R rows.  gates [nt][R][ldg] (ldg >= 3H, 4H with keep_gates);
// h_seq [nt+1][R][H] or null when nt == 1 (fc2 then reads h_last).
int h128_fwd(const pmb_dims* d, int prec, const AgentParams& p, int64_t R, int nt, const float* x, const float* h0,
             float* h_seq, float* gates, int64_t ldg, int keep_gates, float* q, float* h_last, void* scratch,
             int64_t scratch_bytes, cudaStream_t s) {
    PMB_REQUIRE(d->H == H, "h128_fwd: rnn_hidden_dim %d", d->H);
    PMB_REQUIRE(gates && ldg >= (keep_gates ? 4 * H : H3) && ldg % 4 == 0, "rnn_hidden_dim 128 needs the gates buffer");
    PMB_REQUIRE(h_seq || (nt == 1 && h_last), "rnn_hidden_dim 128 needs h_stash (or nt = 1 and h_last)");
    PMB_REQUIRE(scratch_bytes >= h128_fwd_scratch_bytes(d, prec), "h128_fwd: scratch too small");
    char* sp = static_cast<char*>(scratch);
    const int64_t M = (int64_t)nt * R;
    phase_mark(s, "h128_gi_gemm");
    int rc = gemm_tn_tier(prec, x, H, M, H, p.w_ih, H3, p.b_ih, gates, ldg, sp, s);
    if (rc) return rc;
    phase_mark(s, "h128_recurrence");
    PMB_SMEM_ATTR(gru_h128_fwd_kernel, kSmemBytes);
    gru_h128_fwd_kernel<<<(unsigned)ceil_div(R, RT), NT, kSmemBytes, s>>>(p.w_hh, p.b_hh, R, nt, gates, ldg, keep_gates, h0,
                                                                          h_seq, h_last);
    PMB_LAUNCH_CHECK("gru_h128_fwd_kernel");
    if (!q) return PMB_OK;
    phase_mark(s, "h128_fc2_gemm");
    return gemm_tn_tier(prec, h_seq ? h_seq + R * H : h_last, H, M, H, p.fc2_w, d->A, p.fc2_b, q, d->A, sp, s);
}

int h128_bwd(const pmb_dims* d, const pmb_batch* b, const AgentParams& p, const float* h_stash, float* gates,
             const float* d_chosen, cudaStream_t s, const float* dq_full) {
    const int64_t R = (int64_t)d->B * d->N;
    PMB_SMEM_ATTR(gru_h128_bwd_kernel, kSmemBytes);
    gru_h128_bwd_kernel<<<(unsigned)ceil_div(R, RT), NT, kSmemBytes, s>>>(p.w_hh, p.fc2_w, d->A, d->N, d->T, R, h_stash,
                                                                          gates, d_chosen, b->actions, b->actions_sb,
                                                                          dq_full);
    PMB_LAUNCH_CHECK("gru_h128_bwd_kernel");
    return PMB_OK;
}

// dpre1[t][row] = relu'(x[t][row]) * ([da_r | da_z | da_n] W_ih): the input-path gradient the BPTT kernel leaves out
int h128_dpre1(int prec, const AgentParams& p, int64_t rows, const float* gates, const float* x, float* dpre1,
               void* scratch, int64_t scratch_bytes, cudaStream_t s) {
    PMB_REQUIRE(scratch_bytes >= h128_dpre1_scratch_bytes(prec), "h128_dpre1: scratch too small");
    float* wihT = static_cast<float*>(scratch);               // [H][3H]
    char* sp = static_cast<char*>(scratch) + align_up((int64_t)H3 * H * 4, 256);
    int rc = launch_transpose(H3, H, p.w_ih, wihT, s);
    if (rc) return rc;
    if ((rc = gemm_tn_tier(prec, gates, 4 * H, rows, H3, wihT, H, nullptr, dpre1, H, sp, s))) return rc;
    return launch_relu_mask(rows * H, x, dpre1, s);
}

}  // namespace pmb
