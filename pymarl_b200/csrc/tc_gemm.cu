#include <cstdlib>
#include <algorithm>
// bf16 tensor-core tier: C[m, n] = sum_k A[m, k] * W[n, k] on tcgen05 with fp32 accumulation in TMEM.
//
//   A  fp32 in global memory, addressed through RowMap (the EpisodeBatch fields are consumed in
//      place).  Eight producer warps stream it with coalesced loads, convert to bf16 in registers
//      and write the 128-byte-swizzled K-major operand tile into shared memory.
//   W  packed once per step (pack_w_kernel) into bf16 tiles that already are the shared-memory image
//      (K-major, 128B swizzle), so one elected thread brings a tile in with a single bulk async copy
//      (cp.async.bulk, completion on an mbarrier) - no tensor map needed.
//   D  128 x <=256 fp32 accumulator in TMEM, double buffered (2 x 256 columns): the four epilogue warps
//      drain pass p with tcgen05.ld while the MMA thread already accumulates pass p+1.
//
// Warp roles (448 threads): 0-3 epilogue (warp i owns TMEM lanes 32i..32i+31 = tile rows),
// 4 TMEM allocator + single-thread tcgen05.mma issuer, 5 W bulk-copy issuer, 6-13 A producers.
// Pipelines: 4 shared-memory stages (full/empty mbarriers), 2 accumulator buffers (tmem_full/tmem_empty).
// Persistent over 128-row tiles: grid = min(#tiles, #SMs).
#include "common.cuh"
#include "tc_common.cuh"
#include "mixer_tc.cuh"

namespace pmb {
namespace tc {

constexpr int BM = 128;              // rows per tile = UMMA M
constexpr int BK = 64;               // bf16 elements per k-chunk = one 128-byte swizzle row
constexpr int BN_MAX = 256;          // columns per pass = UMMA N
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BM * 128;          // 16 KB
constexpr int W_STAGE_BYTES = BN_MAX * 128;      // 32 KB
constexpr int N_EPI_WARPS = 4, MMA_WARP = 4, WLOAD_WARP = 5, FIRST_PROD_WARP = 6, N_PROD_WARPS = 8;
constexpr int THREADS = 32 * (FIRST_PROD_WARP + N_PROD_WARPS);     // 448
constexpr int SMEM_BYTES = 1024 /*align slack*/ + STAGES * (A_STAGE_BYTES + W_STAGE_BYTES) + 256;

struct GemmParams {
    const float* A;
    RowMap amap;
    int64_t M;
    int K;                 // real reduction length
    int n_chunks;          // ceil(K / 64)
    const __nv_bfloat16* Wp;   // packed tiles: pass-major, then k-chunk; each tile ncols_p rows x 128 B
    int Ncols;             // multiple of 32
    // time-major tiled row order (tm_R > 0): logical row m = t * tm_Rpad + p, p = b*N + n < tm_R is valid and
    // maps to batch row (b*tm_T + t)*tm_N + n of amap; rows p >= tm_R are padding.  A 128-row tile then is
    // exactly one (t, tile) tile image of the bf16 tier.
    int64_t tm_R, tm_Rpad;
    int tm_N, tm_T;
    uint8_t* a_img_out;    // optional: the converted A tiles are also written to global, [tile][k-chunk][16 KB]
    const uint8_t* a_img;  // optional: A is already bf16 tile images [tile][k-chunk][16 KB] -> bulk copied, no producers
};

__host__ __device__ inline int pass_cols(int Ncols, int p) {
    int left = Ncols - p * BN_MAX;
    return left < BN_MAX ? left : BN_MAX;
}
__host__ __device__ inline int64_t packed_tile_offset(int Ncols, int n_chunks, int p, int c) {   // in elements
    return ((int64_t)p * BN_MAX * n_chunks + (int64_t)c * pass_cols(Ncols, p)) * BK;
}

// ------------------------------------------------------------------------------------------
// W packing: up to 4 row segments of fp32 [rows, ld] matrices -> bf16 swizzled tiles
// ------------------------------------------------------------------------------------------
struct PackSegs {
    const float* ptr[4];
    int rows[4];
    int ld[4];
    int nseg;
};

__global__ void __launch_bounds__(256)
pack_w_kernel(PackSegs segs, int K, int n_chunks, int Ncols, __nv_bfloat16* __restrict__ out) {
    // one thread per 16-byte chunk (8 bf16) of the packed image
    const int64_t total = (int64_t)Ncols * n_chunks * 8;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int j = (int)(i & 7);
    int64_t rc = i >> 3;
    int col = (int)(rc % Ncols);
    int c = (int)(rc / Ncols);
    int p = col / BN_MAX, r = col - p * BN_MAX;
    const float* src = nullptr;
    int rr = col;
    for (int s = 0; s < segs.nseg; ++s) {
        if (rr < segs.rows[s]) { src = segs.ptr[s] ? segs.ptr[s] + (int64_t)rr * segs.ld[s] : nullptr; break; }
        rr -= segs.rows[s];
    }
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int k = c * BK + j * 8 + q * 2;
        float lo = (src && k < K) ? src[k] : 0.f;
        float hi = (src && k + 1 < K) ? src[k + 1] : 0.f;
        w[q] = pack_bf16x2(lo, hi);
    }
    char* tile = reinterpret_cast<char*>(out + packed_tile_offset(Ncols, n_chunks, p, c));
    *reinterpret_cast<uint4*>(tile + sw128_offset((uint32_t)r, (uint32_t)j)) = make_uint4(w[0], w[1], w[2], w[3]);
}

// ------------------------------------------------------------------------------------------
// the GEMM kernel
// ------------------------------------------------------------------------------------------
template <class Epi>
__global__ void __launch_bounds__(THREADS, 1) tc_gemm_kernel(GemmParams P, Epi epi) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* a_stage = smem;
    uint8_t* w_stage = smem + STAGES * A_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * (A_STAGE_BYTES + W_STAGE_BYTES));
    uint64_t* full = bars;                 // [STAGES]  producers + W bytes landed
    uint64_t* empty = bars + STAGES;       // [STAGES]  MMAs that read the stage retired
    uint64_t* tfull = bars + 2 * STAGES;   // [2]       accumulator complete
    uint64_t* tempty = tfull + 2;          // [2]       accumulator drained by the epilogue
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], P.a_img ? 1 : N_PROD_WARPS + 1); mbar_init(&empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], N_EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int64_t n_tiles = (P.M + BM - 1) / BM;
    const int n_pass = (P.Ncols + BN_MAX - 1) / BN_MAX;

    if (warp >= FIRST_PROD_WARP) {
        // ===== A producers: fp32 global -> bf16 swizzled smem (idle when A comes as tile images) =====
        const int pw = warp - FIRST_PROD_WARP;
        uint32_t it = 0;
        if (P.a_img == nullptr)
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            // lane l (< 16) keeps the pointer of tile row (pw + 8 l)
            const float* myptr = nullptr;
            if (lane < BM / N_PROD_WARPS) {
                int64_t row = tile * BM + pw + N_PROD_WARPS * lane;
                if (row < P.M) {
                    if (P.tm_R > 0) {
                        const int64_t t = row / P.tm_Rpad, pp = row - t * P.tm_Rpad;
                        if (pp < P.tm_R) {
                            const int64_t bb = pp / P.tm_N, nn = pp - bb * P.tm_N;
                            myptr = P.A + P.amap.offset((bb * P.tm_T + t) * P.tm_N + nn);
                        }
                    } else {
                        myptr = P.A + P.amap.offset(row);
                    }
                }
            }
            for (int p = 0; p < n_pass; ++p) {
                for (int c = 0; c < P.n_chunks; ++c, ++it) {
                    const int s = it % STAGES;
                    mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                    uint8_t* dst = a_stage + s * A_STAGE_BYTES;
                    const int k = c * BK + 2 * lane;
                    float v0[BM / N_PROD_WARPS], v1[BM / N_PROD_WARPS];
#pragma unroll
                    for (int l = 0; l < BM / N_PROD_WARPS; ++l) {
                        const float* rp = reinterpret_cast<const float*>(
                            __shfl_sync(0xffffffffu, reinterpret_cast<uintptr_t>(myptr), l));
                        float a = 0.f, b = 0.f;
                        if (rp != nullptr) {
                            if (k + 1 < P.K && ((reinterpret_cast<uintptr_t>(rp + k) & 7) == 0)) {
                                float2 t = __ldg(reinterpret_cast<const float2*>(rp + k));
                                a = t.x; b = t.y;
                            } else {
                                if (k < P.K) a = __ldg(rp + k);
                                if (k + 1 < P.K) b = __ldg(rp + k + 1);
                            }
                        }
                        v0[l] = a; v1[l] = b;
                    }
                    uint8_t* gimg = (P.a_img_out && p == 0)
                                        ? P.a_img_out + ((int64_t)tile * P.n_chunks + c) * A_STAGE_BYTES : nullptr;
#pragma unroll
                    for (int l = 0; l < BM / N_PROD_WARPS; ++l) {
                        const uint32_t r = pw + N_PROD_WARPS * l;
                        const uint32_t off = sw128_offset(r, lane >> 2) + (lane & 3) * 4;
                        const uint32_t w = pack_bf16x2(v0[l], v1[l]);
                        *reinterpret_cast<uint32_t*>(dst + off) = w;
                        if (gimg) *reinterpret_cast<uint32_t*>(gimg + off) = w;
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&full[s]);
                }
            }
        }
    } else if (warp == WLOAD_WARP) {
        // ===== W loader: one bulk copy per (pass, k-chunk) =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int p = 0; p < n_pass; ++p) {
                    const uint32_t bytes = (uint32_t)pass_cols(P.Ncols, p) * 128u;
                    for (int c = 0; c < P.n_chunks; ++c, ++it) {
                        const int s = it % STAGES;
                        mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                        mbar_arrive_expect_tx(&full[s], bytes + (P.a_img ? A_STAGE_BYTES : 0));
                        bulk_copy_g2s(w_stage + s * W_STAGE_BYTES, P.Wp + packed_tile_offset(P.Ncols, P.n_chunks, p, c),
                                      bytes, &full[s]);
                        if (P.a_img)
                            bulk_copy_g2s(a_stage + s * A_STAGE_BYTES, P.a_img + ((int64_t)tile * P.n_chunks + c) * A_STAGE_BYTES,
                                          A_STAGE_BYTES, &full[s]);
                    }
                }
        }
    } else if (warp == MMA_WARP) {
        // ===== MMA issuer =====
        if (lane == 0) {
            uint32_t it = 0, acc_it = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x)
                for (int p = 0; p < n_pass; ++p, ++acc_it) {
                    const int b = acc_it & 1;
                    const uint32_t idesc = umma_idesc_bf16(BM, pass_cols(P.Ncols, p), 0, 0);
                    mbar_wait(&tempty[b], ((acc_it >> 1) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t tmem_d = tmem_base + (uint32_t)b * BN_MAX;
                    for (int c = 0; c < P.n_chunks; ++c, ++it) {
                        const int s = it % STAGES;
                        mbar_wait(&full[s], (it / STAGES) & 1);
                        tc_fence_after();
                        const uint32_t a_addr = smem_u32(a_stage + s * A_STAGE_BYTES);
                        const uint32_t w_addr = smem_u32(w_stage + s * W_STAGE_BYTES);
#pragma unroll
                        for (int kk = 0; kk < BK / 16; ++kk) {
                            umma_bf16(tmem_d, umma_desc_sw128(a_addr + kk * 32, 16, 1024),
                                      umma_desc_sw128(w_addr + kk * 32, 16, 1024), idesc, (c | kk) != 0);
                        }
                        umma_commit(&empty[s]);
                    }
                    umma_commit(&tfull[b]);
                }
        }
    } else {
        // ===== epilogue: TMEM -> registers -> Epi =====
        uint32_t acc_it = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const int64_t m = tile * BM + warp * 32 + lane;
            const bool valid = m < P.M;
            typename Epi::Row row;
            epi.begin(row, m, valid);
            epi.attach(row, smem + STAGES * (A_STAGE_BYTES + W_STAGE_BYTES) + 256 + warp * (Epi::EXTRA_SMEM / N_EPI_WARPS));
            for (int p = 0; p < n_pass; ++p, ++acc_it) {
                const int b = acc_it & 1;
                const int ncols = pass_cols(P.Ncols, p);
                mbar_wait(&tfull[b], (acc_it >> 1) & 1);
                tc_fence_after();
                const uint32_t taddr = tmem_base + (uint32_t)b * BN_MAX + ((uint32_t)(warp * 32) << 16);
                for (int g = 0; g < ncols; g += 32) {
                    uint32_t v[32];
                    tmem_ld_32x32(taddr + g, v);
                    tmem_wait_ld();
                    epi.cols(row, m, valid, p * BN_MAX + g, v);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[b]);
            }
            epi.end(row, m, valid);
        }
        epi.finish();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------
// epilogues
// ------------------------------------------------------------------------------------------
struct PlainEpi {           // C[m*ldc + n] = acc + bias[n]
    static constexpr int EXTRA_SMEM = 0;
    template <class R> __device__ void attach(R&, uint8_t*) const {}
    __device__ void finish() const {}
    struct Row {};
    float* C; int64_t ldc; const float* bias; int Nreal;
    __device__ void begin(Row&, int64_t, bool) const {}
    __device__ void cols(Row&, int64_t m, bool valid, int col0, const uint32_t (&v)[32]) const {
        if (!valid) return;
#pragma unroll
        for (int j = 0; j < 32; ++j)
            if (col0 + j < Nreal) C[m * ldc + col0 + j] = __uint_as_float(v[j]) + (bias ? bias[col0 + j] : 0.f);
    }
    __device__ void end(Row&, int64_t, bool) const {}
};

// fc1 for the online and the target net in one GEMM: columns [0, 64) online, [64, 128) target.
//   x = relu(acc + tab_id[net][n][h] (bias folded in) + tab_act[net][a_prev][h])
struct Fc1Epi {
    static constexpr int EXTRA_SMEM = 0;
    template <class R> __device__ void attach(R&, uint8_t*) const {}
    __device__ void finish() const {}
    struct Row { int64_t out_off; int n; int a_prev; };
    const float* tab_act;       // [2][A][64]
    const float* tab_id;        // [2][N][64]   W_id[:, n] + b1 (or just b1 when obs_agent_id is off)
    const int64_t* actions; int64_t actions_sb;
    const int64_t* filled;  int64_t filled_sb;
    float* x_on; float* x_tg;   // [nt][R][64] time major
    int t0, nt, N, A, use_act;
    int64_t R;
    __device__ void begin(Row& r, int64_t m, bool valid) const {
        r.out_off = 0; r.n = 0; r.a_prev = -1;
        if (!valid) return;
        const int tn = nt * N;
        int64_t b = m / tn;
        int rem = (int)(m - b * tn);
        int tl = rem / N;
        r.n = rem - tl * N;
        int t = t0 + tl;
        if (use_act && t > 0 && filled[b * filled_sb + (t - 1)] != 0)
            r.a_prev = (int)actions[b * actions_sb + (int64_t)(t - 1) * N + r.n];
        r.out_off = ((int64_t)tl * R + b * N + r.n) * 64;
    }
    __device__ void cols(Row& r, int64_t, bool valid, int col0, const uint32_t (&v)[32]) const {
        if (!valid) return;
        const int net = col0 >> 6, h0 = col0 & 63;
        float* out = (net ? x_tg : x_on) + r.out_off + h0;
        const float4* tid = reinterpret_cast<const float4*>(tab_id + ((int64_t)net * N + r.n) * 64 + h0);
        const float4* tac = r.a_prev >= 0 ? reinterpret_cast<const float4*>(tab_act + ((int64_t)net * A + r.a_prev) * 64 + h0)
                                          : nullptr;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            float4 bi = __ldg(tid + q);
            float4 ac = tac ? __ldg(tac + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            float4 o;
            o.x = fmaxf(__uint_as_float(v[4 * q + 0]) + ac.x + bi.x, 0.f);
            o.y = fmaxf(__uint_as_float(v[4 * q + 1]) + ac.y + bi.y, 0.f);
            o.z = fmaxf(__uint_as_float(v[4 * q + 2]) + ac.z + bi.z, 0.f);
            o.w = fmaxf(__uint_as_float(v[4 * q + 3]) + ac.w + bi.w, 0.f);
            reinterpret_cast<float4*>(out)[q] = o;
        }
    }
    __device__ void end(Row&, int64_t, bool) const {}
};

// Same, but x is written as bf16 tile images [nt][n_tiles][16 KB] (the operand format of gru_tc.cu).
struct Fc1TiEpi {
    static constexpr int EXTRA_SMEM = 0;
    template <class R> __device__ void attach(R&, uint8_t*) const {}
    __device__ void finish() const {}
    struct Row { int64_t tile_off; uint32_t r; int n; int a_prev; };
    const float* tab_act; const float* tab_id;
    const int64_t* actions; int64_t actions_sb;
    const int64_t* filled;  int64_t filled_sb;
    uint8_t* x_on; uint8_t* x_tg;
    int t0, nt, N, A, use_act, n_tiles;
    int64_t R;
    uint32_t* relu_mask;        // optional [nt][n_tiles][2][128]: bit j of word (half, row) = online x[32*half + j] > 0
    // rows arrive in time-major tiled order: m = tl * (n_tiles*128) + p
    __device__ void begin(Row& r, int64_t m, bool valid) const {
        r.tile_off = 0; r.r = 0; r.n = 0; r.a_prev = -2;          // -2: padding row (nothing is written)
        if (!valid) return;
        const int64_t r_pad = (int64_t)n_tiles * 128;
        const int64_t tl = m / r_pad, p = m - tl * r_pad;
        if (p >= R) return;
        const int64_t b = p / N;
        r.n = (int)(p - b * N);
        r.a_prev = -1;
        const int t = t0 + (int)tl;
        if (use_act && t > 0 && filled[b * filled_sb + (t - 1)] != 0)
            r.a_prev = (int)actions[b * actions_sb + (int64_t)(t - 1) * N + r.n];
        r.tile_off = (tl * n_tiles + (p >> 7)) * 16384;
        r.r = (uint32_t)(p & 127);
    }
    __device__ void cols(Row& r, int64_t, bool valid, int col0, const uint32_t (&v)[32]) const {
        if (!valid || r.a_prev == -2) return;
        const int net = col0 >> 6, h0 = col0 & 63;
        uint8_t* tile = (net ? x_tg : x_on) + r.tile_off;
        const float4* tid = reinterpret_cast<const float4*>(tab_id + ((int64_t)net * N + r.n) * 64 + h0);
        const float4* tac = r.a_prev >= 0 ? reinterpret_cast<const float4*>(tab_act + ((int64_t)net * A + r.a_prev) * 64 + h0)
                                          : nullptr;
        uint32_t mbits = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {                 // 8 columns = one 16-byte chunk
            float o[8];
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                float4 bi = __ldg(tid + 2 * q + hh);
                float4 ac = tac ? __ldg(tac + 2 * q + hh) : make_float4(0.f, 0.f, 0.f, 0.f);
                o[4 * hh + 0] = fmaxf(__uint_as_float(v[8 * q + 4 * hh + 0]) + ac.x + bi.x, 0.f);
                o[4 * hh + 1] = fmaxf(__uint_as_float(v[8 * q + 4 * hh + 1]) + ac.y + bi.y, 0.f);
                o[4 * hh + 2] = fmaxf(__uint_as_float(v[8 * q + 4 * hh + 2]) + ac.z + bi.z, 0.f);
                o[4 * hh + 3] = fmaxf(__uint_as_float(v[8 * q + 4 * hh + 3]) + ac.w + bi.w, 0.f);
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) mbits |= (o[k] > 0.f ? 1u : 0u) << (8 * q + k);
            *reinterpret_cast<uint4*>(tile + sw128_offset(r.r, (uint32_t)(h0 / 8 + q))) =
                make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
        }
        if (relu_mask && net == 0) relu_mask[((r.tile_off >> 14) * 2 + (h0 >> 5)) * 128 + r.r] = mbits;
    }
    __device__ void end(Row&, int64_t, bool) const {}
};

// QMIX mixing on the hypernet outputs, E = 32.  Packed column order: [ w1 (N*32) | b1 | w_final | v0 ].
//   hidden = ELU(sum_n q[n] |w1[n, :]| + b1);  q_tot = hidden . |w_final| + V.2(ReLU(v0))
// Mixer epilogue for the image-fed path: GEMM rows are ALL (b, t) pairs, m' = b*T + t.  The online mixer
// (t_off = 0) uses rows t < T-1, the target mixer (t_off = 1) rows t >= 1; agent_qs / q_tot are indexed by
// mq = b*(T-1) + t - t_off.  raw_img (online only): hypernet outputs as bf16 tile images
// [row tile][(N+3)/2 column blocks of 64][16 KB], packed column order, kept for the backward.
struct MixImgEpi {
    // raw images leave through shared memory: every epilogue warp stages its 32 rows of a 64-column block (4 KB, image
    // layout) in its own double buffer and lane 0 bulk-stores it - no per-thread row-strided global stores
    static constexpr int EXTRA_SMEM = N_EPI_WARPS * 2 * 4096;
    struct Row { float hidden[32]; float y; int64_t mq; uint8_t* img; uint32_t r; uint8_t* stg; uint32_t nblk; };
    const float* bias; const float* agent_qs; const float* v2_w; const float* v2_b;
    float* q_tot; uint8_t* raw_img;
    int N, T, t_off, n_cblk;
    int64_t BT;
    __device__ void begin(Row& r, int64_t m, bool) const {
#pragma unroll
        for (int e = 0; e < 32; ++e) r.hidden[e] = 0.f;
        r.y = 0.f; r.mq = -1;
        // this warp's 32 rows of the tile: 4 KB inside every 16 KB block
        r.img = raw_img ? raw_img + (m >> 7) * (int64_t)n_cblk * 16384 + ((m & 127) & ~31) * 128 : nullptr;
        r.r = (uint32_t)(m & 127);
        r.nblk = 0;
        if (m < BT) {
            const int64_t b = m / T;
            const int t = (int)(m - b * T);
            if (t_off == 0 ? (t < T - 1) : (t >= 1)) r.mq = b * (T - 1) + t - t_off;
        }
    }
    __device__ void attach(Row& r, uint8_t* stg) const { r.stg = stg; }
    __device__ void flush(Row& r, int blk) const {              // whole warp
        fence_proxy_async_smem();
        __syncwarp();
        if ((threadIdx.x & 31) == 0) {
            bulk_copy_s2g(r.img + (int64_t)blk * 16384, r.stg + (r.nblk & 1) * 4096, 4096);
            bulk_commit_group();
            bulk_wait_group_read<1>();                          // the other buffer (previous block) has been read
        }
        __syncwarp();
        ++r.nblk;
    }
    __device__ void cols(Row& r, int64_t, bool, int col0, const uint32_t (&v)[32]) const {
        const int grp = col0 >> 5;
        float raw[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) raw[e] = __uint_as_float(v[e]) + __ldg(bias + col0 + e);
        if (r.img) {                                   // every row is written (finite values; the backward zeroes unused rows)
            uint8_t* blk = r.stg + (r.nblk & 1) * 4096;
            const uint32_t ch0 = (uint32_t)((col0 & 63) >> 3);
#pragma unroll
            for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(blk + sw128_offset(r.r & 31u, ch0 + q)) =
                    make_uint4(pack_bf16x2(raw[8 * q], raw[8 * q + 1]), pack_bf16x2(raw[8 * q + 2], raw[8 * q + 3]),
                               pack_bf16x2(raw[8 * q + 4], raw[8 * q + 5]), pack_bf16x2(raw[8 * q + 6], raw[8 * q + 7]));
            if (col0 & 32) flush(r, col0 >> 6);        // second half of a 64-column block
        }
        if (grp < N) {
            const float qn = r.mq >= 0 ? __ldg(agent_qs + r.mq * N + grp) : 0.f;
#pragma unroll
            for (int e = 0; e < 32; ++e) r.hidden[e] = fmaf(qn, fabsf(raw[e]), r.hidden[e]);
        } else if (grp == N) {
#pragma unroll
            for (int e = 0; e < 32; ++e) {
                float pre = r.hidden[e] + raw[e];
                r.hidden[e] = pre > 0.f ? pre : expm1f(pre);
            }
        } else if (grp == N + 1) {
#pragma unroll
            for (int e = 0; e < 32; ++e) r.y = fmaf(r.hidden[e], fabsf(raw[e]), r.y);
        } else if (grp == N + 2) {
#pragma unroll
            for (int e = 0; e < 32; ++e) r.y = fmaf(fmaxf(raw[e], 0.f), __ldg(v2_w + e), r.y);
        }
    }
    __device__ void end(Row& r, int64_t, bool) const {
        if (r.mq >= 0) q_tot[r.mq] = r.y + __ldg(v2_b);
        // (N + 3) odd: the last 64-column block was only half produced (its other half is padding the backward ignores)
        if (r.img) {
            if ((N + 3) & 1) flush(r, (N + 3) >> 1);
            // the next tile starts again with buffer 0: both buffers must have been read
            if ((threadIdx.x & 31) == 0) bulk_wait_group_read<0>();
            __syncwarp();
        }
    }
    __device__ void finish() const {
        if ((threadIdx.x & 31) == 0) bulk_wait_group<0>();
    }
};

template <class Epi>
int launch_tc_gemm(const GemmParams& P, const Epi& epi, cudaStream_t s) {
    if (P.M <= 0) return PMB_OK;
    auto kern = tc_gemm_kernel<Epi>;
    PMB_SMEM_ATTR(kern, SMEM_BYTES + Epi::EXTRA_SMEM);
    int64_t n_tiles = (P.M + BM - 1) / BM;
    int grid = (int)(n_tiles < sm_count() ? n_tiles : sm_count());
    kern<<<grid, THREADS, SMEM_BYTES + Epi::EXTRA_SMEM, s>>>(P, epi);
    PMB_LAUNCH_CHECK("tc_gemm_kernel");
    return PMB_OK;
}


// ------------------------------------------------------------------------------------------
// fc1 for both nets as a STREAMING kernel (obs is 70 % of the learner step's HBM bytes)
// ------------------------------------------------------------------------------------------
// The generic kernel above feeds A through eight producer warps that load 8 bytes per lane (obs rows are 4-byte
// aligned only: 285 floats) and convert synchronously, chunk by chunk: ~28 % of the HBM ceiling (ncu, profiles/).
// Here the copy engine does the streaming:
//   producer warp : walks the rows of a group (time-major tile order: a group is 1-2 contiguous runs of [B,T,N,O]
//                   memory, one per episode), issues ONE cp.async.bulk per run, widened to 16-byte boundaries, into a
//                   ring of staging slots in the obs element type.  3 slots x 18 KB in flight per SM.
//                   A group is 16 rows of fp32 obs or 32 rows of bf16 obs (pmb_batch.obs_dtype): a slot holds about the
//                   same bytes either way, and the stream is bound by the bytes in flight per SM.
//   8 converter warps : staging -> bf16 K-major/128B-swizzle A tile (all k-chunks of the tile, 80 KB); fp32 obs is
//                   rounded to nearest even here, bf16 obs is copied, and both give the same bytes for the same values.
//   MMA thread    : W (both nets, 128 columns, all chunks) stays resident; 4 tcgen05.mma per chunk, 2 TMEM buffers.
//   store thread  : the finished A tile IS the obs tile image the weight-gradient kernel wants: one 80 KB bulk store.
//   4 epilogue warps : Fc1TiEpi (one-hot gathers, bias, ReLU, bf16 x tile images of both nets, ReLU bit mask).
namespace fs {
constexpr int MAX_CHUNKS = 5;
// rows of a staging group (= one slot fill) for obs elements of ES bytes: 64 bytes of every row's 16-row share.
// (fp32: 8 rows x 6 slots measured no better than 16 x 3: 8.5 vs 8.2 ms)
// (bf16: 16 rows per group, half the bytes per slot, measured slower than 32: 8.61 against 8.08 ms, with the earlier
// converter; profiles/r03_obs_bf16.json)
constexpr int group_rows_of(int es) { return 64 / es; }
template <int ES> constexpr int group_rows() { return group_rows_of(ES); }
// staging bytes between two runs of a group: a run starts at the next 128-byte boundary (< 128) plus the 128-byte phase of
// its source (< 128), and its copy is widened by < 16 bytes - under 272 bytes, so the copies of the runs stay disjoint
constexpr int RUN_SLACK = 272;
constexpr int N_SLOTS = 3;                                   // learner step (both nets: W is 16 KB per k-chunk)
constexpr int N_SLOTS_1NET = 5;                              // rollout step: W of one net is half the size, two more slots fit
#ifndef PMB_FC1_NCONV
#define PMB_FC1_NCONV 8
#endif
constexpr int N_EPI = 4, MMA_W = 4, PROD_W = 5, N_CONV = PMB_FC1_NCONV;
// NS staging slots, one producer warp each (every producer warp owns one staging slot: parity waits are only safe one
// phase apart), then the converter warps
constexpr int threads_for(int ns) { return 32 * (PROD_W + ns + N_CONV); }
// a group's rows divide over the converter warps and into the 128-row tile, and the producer writes one row per lane
static_assert(group_rows<4>() % N_CONV == 0 && group_rows<2>() % N_CONV == 0, "group rows must divide over the converter warps");
static_assert(BM % group_rows<4>() == 0 && BM % group_rows<2>() == 0, "group rows must divide the tile");
static_assert(group_rows<4>() <= 32 && group_rows<2>() <= 32, "the producer writes one row table entry per lane");
}  // namespace fs

struct Fc1StreamParams {
    const int64_t* ep_index;       // optional batch row -> buffer episode
    const uint8_t* obs; int64_t obs_sb;   // fp32 or bf16 (the kernels' ES template argument), obs_sb in elements
    const __nv_bfloat16* Wp;       // packed [chunk][128 x 128 B]
    uint8_t* obs_img;              // optional [T*n_tiles][n_chunks][16 KB]
    int64_t R;
    int T, N, O, n_tiles, n_chunks, slot_bytes;
    // fold_id: the K padding of the last chunk carries one-hot(agent id) in columns O .. O+N-1 and 1.0 in column O+N;
    // the packed W holds the agent-id columns of fc1.weight and fc1.bias there, so the tensor core adds them.
    int fold_id;
    // epilogue
    const uint4* tab_act16;        // bf16 [A][net 2][64]: fc1.weight[:, O + a] of both nets
    const float* tab_id;           // fp32 [net 2][N][64] (used when !fold_id): W_id[:, n] + b1
    const int64_t* actions; int64_t actions_sb;
    const int64_t* filled;  int64_t filled_sb;
    uint8_t* x_on; uint8_t* x_tg;  // tile images [T][n_tiles][16 KB]
    uint32_t* relu_mask;           // [T][n_tiles][2][128]
    int use_act;
    int l2_prefetch;               // n > 0: prefetch the runs of the CTA's n-th next tile into L2 (off by default)
    int n_nets;                    // 2: online + target (learner step), 1: online only (rollout step)
    int t0;                        // batch timestep of item t = 0 (rollout: the step index; obs is addressed at t0 + t)
    int n_act;                     // A: rows of tab_act16
    // optional live-item schedule (learner step, pmb_dims.reserved bit 1): the grid walks items[k] instead of every item
    // k = t * n_tiles + tile, up to the first negative entry (the list is padded with -1 to T * n_tiles entries: a count
    // loaded in every role is hoisted above the role branch and spills in fc1_stream_ts_kernel).  Items not listed are
    // neither read nor written.
    const int32_t* items;
};

// the k-th item of the grid's walk, < 0 past the end of a live-item list (T * n_tiles < 2^31, validated on the host)
__device__ __forceinline__ int fc1_item(const Fc1StreamParams& P, int k) { return P.items ? __ldg(P.items + k) : k; }

__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_b32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_b32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// NC = number of 64-column k-chunks of the obs (compile time: the converters are instruction-latency bound - 8 warps,
// ~300 dependent instructions per 16-row group each - and with NC known the per-chunk predicates of all but the last
// chunk and the run-time "is this the last chunk" selects disappear)
// Per-role wait accounting (build with PMB_EXTRA_NVCC_FLAGS=-DPMB_FC1_PROFILE, read with tools/fc1_role_profile.py): cycles
// each role spends blocked on each barrier / in each converter phase, summed over CTAs.  This is what located the
// obs-image bulk store as the reason the converters idled between tiles.
// Slots: 0-7 and 10-15 role cycles (names in the tool), 8 kernel cycles, 9 CTAs, 15 producer warps (= staging slots).
#ifdef PMB_FC1_PROFILE
__device__ unsigned long long g_fc1_prof[16];
#define TWAIT(idx, bar, par) do { long long _t0 = clock64(); mbar_wait(bar, par); if (lane == 0) prof_acc[idx] += clock64() - _t0; } while (0)
#define TMARK(var) const long long var = clock64()
#define TADD(idx, expr) do { if (lane == 0) prof_acc[idx] += (expr); } while (0)
#define FC1_PROF_BEGIN long long prof_acc[16] = {}; const long long prof_t0 = clock64()
#define FC1_PROF_END(ns)                                                                                                  \
    do {                                                                                                                  \
        if (lane == 0)                                                                                                    \
            for (int i = 0; i < 15; ++i)                                                                                  \
                if (i != 8 && i != 9 && prof_acc[i]) atomicAdd(&g_fc1_prof[i], (unsigned long long)prof_acc[i]);          \
        if (threadIdx.x == 0) {                                                                                           \
            atomicAdd(&g_fc1_prof[8], (unsigned long long)(clock64() - prof_t0)); atomicAdd(&g_fc1_prof[9], 1ull);        \
            atomicAdd(&g_fc1_prof[15], (unsigned long long)(ns));                                                         \
        }                                                                                                                 \
    } while (0)
#else
#define TWAIT(idx, bar, par) mbar_wait(bar, par)
#define TMARK(var)
#define TADD(idx, expr)
#define FC1_PROF_BEGIN long long prof_acc[16]
#define FC1_PROF_END(ns) do { } while (0)
#endif
// The two roles the learner and the rollout kernels below share: the producer warps that stream the obs runs of a
// group into the staging ring, and the converter warps that turn a staged group into bf16 rows of the K-major /
// 128B-swizzle obs tile (and of the obs image).  ES = bytes of an obs element: 4 (fp32) or 2 (bf16).
struct Fc1Ring {
    uint8_t* stage;         // [NS][slot_bytes]
    int* rowinfo;           // [NS][group rows] byte offset of a row in its slot | agent index << 20 (fold_id only); -1: zeros
    uint64_t* st_full;      // [NS]
    uint64_t* st_empty;     // [NS]
};

template <int NC, int NS, int ES>
__device__ __forceinline__ void fc1_produce(const Fc1StreamParams& P, const Fc1Ring& ring, int pw, int lane,
                                            long long (&prof_acc)[16]) {
    using namespace fs;
    constexpr int N_SLOTS = NS, GROUP_ROWS = group_rows<ES>(), GROUPS = BM / GROUP_ROWS;
    uint8_t* stage = ring.stage;
    int* rowinfo = ring.rowinfo;
    uint64_t* st_full = ring.st_full;
    uint64_t* st_empty = ring.st_empty;
    const int n_items = P.T * P.n_tiles;
    const uint32_t row_bytes = (uint32_t)P.O * ES;

    // Lane i owns the i-th contiguous run of a group (one episode each) and computes its descriptor - global
    // address, staging offset, head / interior / tail split - in closed form, in parallel with the other lanes
    // and BEFORE the slot is free; once it is, every lane just issues its copies.  (The first version walked the
    // runs serially after the wait: ~1.5 us of dependent integer code per group during which the slot sat empty,
    // which bounded the stream at three slots per (walk + load + convert).)  A group has at most 32 runs (N = 1).
    uint32_t git = 0;
    for (int k = blockIdx.x; k < n_items; k += gridDim.x) {
        const int64_t item = fc1_item(P, k);
        if (item < 0) break;
        const int64_t t = item / P.n_tiles, tile = item - t * P.n_tiles;
        for (int g = 0; g < GROUPS; ++g, ++git) {
            const int slot = git % N_SLOTS;
            if (slot != pw) continue;
            TMARK(pp0);
            uint8_t* sl = stage + slot * P.slot_bytes;
            int* ri = rowinfo + slot * GROUP_ROWS;
            const int64_t p0 = tile * BM + g * GROUP_ROWS;
            int rows_here = P.R - p0 < GROUP_ROWS ? (int)(P.R - p0) : GROUP_ROWS;     // rows of this group below R
            if (rows_here < 0) rows_here = 0;
            const uint32_t b0 = (uint32_t)p0 / (uint32_t)P.N;               // B*N < 2^31 (validated on the host)
            const int n00 = (int)((uint32_t)p0 - b0 * (uint32_t)P.N);
            int first_cnt = P.N - n00;
            if (first_cnt > rows_here) first_cnt = rows_here;
            // run `lane`: rows [lr, lr + cnt) of the group, agent index n0 .. of episode b0 + lane
            const int lr = lane == 0 ? 0 : first_cnt + (lane - 1) * P.N;
            int cnt = lane == 0 ? first_cnt : (rows_here - lr < P.N ? rows_here - lr : P.N);
            if (cnt < 0) cnt = 0;
            const int n0 = lane == 0 ? n00 : 0;
            const uint8_t* ga = nullptr;
            uint32_t cur = 0, phase = 0, cp_bytes = 0;
            if (cnt > 0) {
                ga = P.obs + (ep_row(P.ep_index, (int64_t)b0 + lane) * P.obs_sb + ((t + P.t0) * P.N + n0) * (int64_t)P.O) * ES;
                phase = (uint32_t)(reinterpret_cast<uintptr_t>(ga) & 15);
                // staging offset: same 128-BYTE phase as the source (the copy engine then moves whole lines: with only the
                // 16-byte phase matched every line is split and shifted); RUN_SLACK bytes per run keep the runs - and
                // the up to 15 bytes copied before / after each of them - disjoint
                cur = (((uint32_t)lr * row_bytes + 127u) & ~127u) + (uint32_t)RUN_SLACK * lane +
                      (uint32_t)(reinterpret_cast<uintptr_t>(ga) & 127);
                // ONE bulk copy per run, widened to 16-byte boundaries on both sides (the extra bytes stay inside the
                // 16-byte granules the run touches anyway - never another page - and land in the slack).  The first
                // version copied the aligned interior and fetched head / tail with 4-byte cp.async: with the 32
                // no-increment barrier arrivals that needs, publishing a slot took ~1600 cycles.
                cp_bytes = (phase + (uint32_t)cnt * row_bytes + 15u) & ~15u;
            }
            const uint32_t tx = __reduce_add_sync(0xffffffffu, cp_bytes);
            // L2 prefetch of the same group of this CTA's NEXT tile: the staging ring is all the shared memory that is
            // left (3 x 18 KB in flight per SM), so the copies should see L2 latency, not loaded-HBM latency
            if (P.l2_prefetch && cnt > 0 && k + P.l2_prefetch * (int)gridDim.x < n_items) {
                const int64_t item2 = max(fc1_item(P, k + P.l2_prefetch * (int)gridDim.x), 0);
                const int64_t t2 = item2 / P.n_tiles, tile2 = item2 - t2 * P.n_tiles;
                const int64_t q0 = tile2 * BM + g * GROUP_ROWS;
                int rows2 = P.R - q0 < GROUP_ROWS ? (int)(P.R - q0) : GROUP_ROWS;
                if (rows2 < 0) rows2 = 0;
                const uint32_t c0 = (uint32_t)q0 / (uint32_t)P.N;
                const int m00 = (int)((uint32_t)q0 - c0 * (uint32_t)P.N);
                int fc = P.N - m00;
                if (fc > rows2) fc = rows2;
                const int lr2 = lane == 0 ? 0 : fc + (lane - 1) * P.N;
                int cnt2 = lane == 0 ? fc : (rows2 - lr2 < P.N ? rows2 - lr2 : P.N);
                if (cnt2 > 0) {
                    const uint8_t* gb = P.obs + (ep_row(P.ep_index, (int64_t)c0 + lane) * P.obs_sb +
                                                 ((t2 + P.t0) * P.N + (lane == 0 ? m00 : 0)) * (int64_t)P.O) * ES;
                    const uintptr_t a0 = (reinterpret_cast<uintptr_t>(gb) + 15) & ~(uintptr_t)15;
                    const uintptr_t a1 = (reinterpret_cast<uintptr_t>(gb) + (uint64_t)cnt2 * row_bytes) & ~(uintptr_t)15;
                    if (a1 > a0)
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a0), "r"((uint32_t)(a1 - a0)) : "memory");
                }
            }
            // row tables, one row per lane: row j belongs to run rj (run 0 holds first_cnt rows, the others N each)
            const int rj = lane < first_cnt ? 0 : 1 + (lane - first_cnt) / P.N;
            const int lrj = rj == 0 ? 0 : first_cnt + (rj - 1) * P.N;
            const uint32_t cur_j = __shfl_sync(0xffffffffu, cur, rj & 31);
            TADD(10, clock64() - pp0);                         // producer: descriptors of the group (before the slot wait)
            TWAIT(0, &st_empty[slot], ((git / N_SLOTS) & 1) ^ 1);
            TMARK(pp1);
            if (lane < GROUP_ROWS) {
                // the agent index is needed where one-hot(agent) goes into the K padding only (N < 64 there)
                const int nj = P.fold_id ? (rj == 0 ? n00 : 0) + (lane - lrj) : 0;
                ri[lane] = lane < rows_here ? (int)((cur_j + (uint32_t)(lane - lrj) * row_bytes) | ((uint32_t)nj << 20)) : -1;
            }
            if (cnt > 0) bulk_copy_g2s(sl + cur - phase, ga - phase, cp_bytes, &st_full[slot]);
            __syncwarp();
            if (lane == 0) {
                if (tx) mbar_arrive_expect_tx(&st_full[slot], tx); else mbar_arrive(&st_full[slot]);
            }
            TADD(11, clock64() - pp1);                         // producer: tables, copies, arrival
        }
    }
}

// converter warp cw owns rows RPW cw .. RPW cw + RPW - 1 of every group; arrives on a_full once per finished tile
template <int NC, int NS, int ES>
__device__ __forceinline__ void fc1_convert(const Fc1StreamParams& P, const Fc1Ring& ring, uint8_t* a_s, uint64_t* a_free,
                                            uint64_t* a_full, int cw, int lane, long long (&prof_acc)[16]) {
    using namespace fs;
    constexpr int N_SLOTS = NS, GROUP_ROWS = group_rows<ES>(), GROUPS = BM / GROUP_ROWS, RPW = GROUP_ROWS / N_CONV;
    constexpr int tile_bytes = NC * A_STAGE_BYTES;
    uint8_t* stage = ring.stage;
    int* rowinfo = ring.rowinfo;
    uint64_t* st_full = ring.st_full;
    uint64_t* st_empty = ring.st_empty;
    const int n_items = P.T * P.n_tiles;
    constexpr int c_last = NC - 1;
    // every column of the chunks before the last exists (O > 64 (NC-1)); the last chunk: per lane
    const bool okl0 = c_last * BK + 2 * lane < P.O, okl1 = c_last * BK + 2 * lane + 1 < P.O;
    const int j_pad = c_last * BK + 2 * lane - P.O;       // index of this lane's first column in the K padding
    const uint32_t a_s_u32 = smem_u32(a_s);
    const uint32_t a_base = a_s_u32 + ((uint32_t)(lane >> 2) << 4) + (lane & 3) * 4;   // + row*128, ^ swizzle
    uint32_t git = 0, ti = 0;
    for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++ti) {
        const int item = fc1_item(P, k);
        if (item < 0) break;
        for (int g = 0; g < GROUPS; ++g, ++git) {
            const int slot = git % N_SLOTS;
            TWAIT(1, &st_full[slot], (git / N_SLOTS) & 1);
            TMARK(pt1);
            // the lane's column pair 2 lane, 2 lane + 1 of chunk c sits at byte 2 ES lane + 64 ES c of the staged row
            const uint32_t sl = smem_u32(stage + slot * P.slot_bytes) + 2u * ES * lane;
            int offs[RPW], nns[RPW];
#pragma unroll
            for (int rr = 0; rr < RPW; ++rr) {
                const int info = rowinfo[slot * GROUP_ROWS + RPW * cw + rr];
                offs[rr] = info < 0 ? -1 : (info & 0xfffff);
                nns[rr] = info < 0 ? -1 : (info >> 20);
            }
            {
                // pack first (consumes every loaded value), release the staging slot, then write the A tile
                uint32_t pk[RPW][NC];
                if constexpr (ES == 4) {
                    float v0[RPW][NC], v1[RPW][NC];
#pragma unroll
                    for (int rr = 0; rr < RPW; ++rr) {           // all loads first
                        const int off = offs[rr];
                        const bool real = off >= 0;
                        const uint32_t src = sl + (uint32_t)(real ? off : 0);
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            v0[rr][c] = 0.f; v1[rr][c] = 0.f;
                            if (real && (c < c_last || okl0)) v0[rr][c] = lds_f32(src + c * 256);
                            if (real && (c < c_last || okl1)) v1[rr][c] = lds_f32(src + c * 256 + 4);
                        }
                    }
#pragma unroll
                    for (int rr = 0; rr < RPW; ++rr) {
                        const int off = offs[rr];
                        const int nn = nns[rr];
                        // one-hot(agent) and the bias column live in the K padding of the last chunk
                        const bool fold = P.fold_id && off >= 0;
                        const bool hit0 = fold && j_pad >= 0 && (j_pad == nn || j_pad == P.N);
                        const bool hit1 = fold && j_pad + 1 >= 0 && (j_pad + 1 == nn || j_pad + 1 == P.N);
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            float a = v0[rr][c], b = v1[rr][c];
                            if (c == c_last) { a = hit0 ? 1.0f : a; b = hit1 ? 1.0f : b; }
                            pk[rr][c] = pack_bf16x2(a, b);
                        }
                    }
                } else {
                    // bf16: the column pair is one packed word already.  A row of odd O starts at 2 mod 4 every other
                    // row, where the pair straddles two words: every lane loads the two aligned words around its pair and
                    // a per-row byte selector picks it out.  (Choosing between one load and two per row compiled to a
                    // branch around each chunk's loads, which serialised them: 8.1 against 6.5 ms for fp32 obs.)
                    uint32_t lo[RPW][NC], hi[RPW][NC];
#pragma unroll
                    for (int rr = 0; rr < RPW; ++rr) {           // all loads first
                        const int off = offs[rr];
                        const bool real = off >= 0;
                        const uint32_t src = sl + (uint32_t)(real ? (off & ~3) : 0);
#pragma unroll
                        for (int c = 0; c < NC; ++c) {
                            lo[rr][c] = 0u; hi[rr][c] = 0u;
                            if (real && (c < c_last || okl0)) {
                                lo[rr][c] = lds_b32(src + c * 128);
                                hi[rr][c] = lds_b32(src + c * 128 + 4);
                            }
                        }
                    }
#pragma unroll
                    for (int rr = 0; rr < RPW; ++rr) {
                        const int off = offs[rr];
                        const int nn = nns[rr];
                        const uint32_t sel = (off & 2) ? 0x5432u : 0x3210u;
#pragma unroll
                        for (int c = 0; c < NC; ++c) pk[rr][c] = __byte_perm(lo[rr][c], hi[rr][c], sel);
                        const bool fold = P.fold_id && off >= 0;
                        const bool hit0 = fold && j_pad >= 0 && (j_pad == nn || j_pad == P.N);
                        const bool hit1 = fold && j_pad + 1 >= 0 && (j_pad + 1 == nn || j_pad + 1 == P.N);
                        // last chunk: column O - 1 may share its word with the next row's first column; zero it, then
                        // bf16 1.0 (0x3f80) for the one-hot and bias columns
                        uint32_t w = pk[rr][c_last];
                        w = okl1 ? w : (w & 0xffffu);
                        w = hit0 ? ((w & 0xffff0000u) | 0x3f80u) : w;
                        w = hit1 ? ((w & 0xffffu) | 0x3f800000u) : w;
                        pk[rr][c_last] = w;
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&st_empty[slot]);
                TMARK(pt2);
                TADD(6, pt2 - pt1);                            // load + pack phase
                // the first group of a tile waits here (values already in registers, slot already released) until
                // the MMAs and the image store of the previous tile are done with the A tile
                if (g == 0) TWAIT(2, a_free, (ti & 1) ^ 1);
#pragma unroll
                for (int rr = 0; rr < RPW; ++rr) {
                    const uint32_t rt = (uint32_t)(g * GROUP_ROWS + RPW * cw + rr);
                    const uint32_t dst = (a_base + rt * 128u) ^ ((rt & 7u) << 4);
#pragma unroll
                    for (int c = 0; c < NC; ++c) sts_b32(dst + c * A_STAGE_BYTES, pk[rr][c]);
                    // the obs image leaves from here too: the warp's 32 words are one full 128-byte line of the image
                    // (a bulk store of the finished A tile kept the tile busy for ~2500 cycles after the MMAs were
                    // done with it: the converters of the next tile waited 22 % of the kernel time for it)
                    if (P.obs_img) {
                        uint8_t* img = P.obs_img + (int64_t)item * tile_bytes + (dst - a_s_u32);
#pragma unroll
                        for (int c = 0; c < NC; ++c) __stcs(reinterpret_cast<uint32_t*>(img + c * A_STAGE_BYTES), pk[rr][c]);
                    }
                }
                TADD(7, clock64() - pt2);                      // store phase (includes the a_free wait of group 0)
            }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(a_full);
    }
}

template <int NC, int NS, int ES>
__global__ void __launch_bounds__(fs::threads_for(NS), 1) fc1_stream_kernel(Fc1StreamParams P) {
    FC1_PROF_BEGIN;
    using namespace fs;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr int N_SLOTS = NS, N_PROD = NS, FIRST_CONV_W = PROD_W + NS;
    constexpr int tile_bytes = NC * A_STAGE_BYTES;
    // W of a k-chunk: 128 rows x 128 B (online | target); the rollout step keeps the online half only
    const int w_chunk = P.n_nets == 2 ? A_STAGE_BYTES : A_STAGE_BYTES / 2;
    uint8_t* w_s = smem;                                    // [n_chunks][w_chunk]
    uint8_t* a_s = smem + NC * w_chunk;                     // [n_chunks][16 KB]
    uint8_t* stage = a_s + tile_bytes;                      // [N_SLOTS][slot_bytes]
    int* rowinfo = reinterpret_cast<int*>(stage + N_SLOTS * P.slot_bytes);  // [N_SLOTS][group rows] (Fc1Ring)
    uint64_t* bars = reinterpret_cast<uint64_t*>(rowinfo + N_SLOTS * group_rows<ES>());
    uint64_t* w_full = bars;
    uint64_t* st_full = bars + 1;            // [N_SLOTS]
    uint64_t* st_empty = st_full + N_SLOTS;  // [N_SLOTS]
    uint64_t* a_full = st_empty + N_SLOTS;
    uint64_t* a_free = a_full + 1;
    uint64_t* tfull = a_free + 1;            // [2]
    uint64_t* tempty = tfull + 2;            // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int i = 0; i < N_SLOTS; ++i) { mbar_init(&st_full[i], 1); mbar_init(&st_empty[i], N_CONV); }
        mbar_init(a_full, N_CONV); mbar_init(a_free, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], N_EPI); }
        fence_barrier_init();
    }
    if (warp == MMA_W) tmem_alloc(tmem_slot, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_items = P.T * P.n_tiles;
    const Fc1Ring ring{stage, rowinfo, st_full, st_empty};
    // programmatic dependent launch (rollout step only; see gru_rollout_kernel): the next kernel may be scheduled as the
    // CTAs of this grid leave; this kernel reads nothing its predecessor writes and only its epilogue warps write something
    // the predecessor (the GRU step of the previous rollout step) may still be reading - the x images
    pdl_launch_dependents();

    if (warp >= PROD_W && warp < PROD_W + N_PROD) {
        // one producer warp per staging slot: the address walk of a warp is ~300 dependent integer instructions per
        // group (~1.5 us); ONE warp capped the stream at 2.9 TB/s, two at 4.6 TB/s.  A slot is always filled by the
        // same warp, so consecutive uses of a slot are program-ordered (a parity wait must never be two phases ahead).
        const int pw = warp - PROD_W;
        if (pw == 0 && lane == 0) {
            mbar_arrive_expect_tx(w_full, (uint32_t)(NC * w_chunk));
            for (int c = 0; c < NC; ++c)
                bulk_copy_g2s(w_s + c * w_chunk, reinterpret_cast<const uint8_t*>(P.Wp) + c * A_STAGE_BYTES, (uint32_t)w_chunk, w_full);
        }
        fc1_produce<NC, NS, ES>(P, ring, pw, lane, prof_acc);
    } else if (warp >= FIRST_CONV_W) {
        // ===== converters: warp cw owns rows RPW cw .. RPW cw + RPW - 1 of every group (RPW = 2 fp32, 4 bf16).  Everything that does not depend on the row
        // (which of a lane's two columns per chunk exist, where the one-hot padding columns are) is hoisted: the
        // first version spent ~2400 cycles per group in a serial chain of predicate / address arithmetic. =====
        fc1_convert<NC, NS, ES>(P, ring, a_s, a_free, a_full, warp - FIRST_CONV_W, lane, prof_acc);
    } else if (warp == MMA_W) {
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_bf16(BM, 64 * P.n_nets, 0, 0);
            mbar_wait(w_full, 0);
            uint32_t ti = 0;
            for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++ti) {
                if (fc1_item(P, k) < 0) break;
                const int b = ti & 1;
                TWAIT(3, a_full, ti & 1);
                TWAIT(4, &tempty[b], ((ti >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tm = tmem_base + 128u * b;
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const uint32_t a_addr = smem_u32(a_s + c * A_STAGE_BYTES), w_addr = smem_u32(w_s + c * w_chunk);
#pragma unroll
                    for (int kk = 0; kk < BK / 16; ++kk)
                        umma_bf16(tm, umma_desc_sw128(a_addr + kk * 32, 16, 1024), umma_desc_sw128(w_addr + kk * 32, 16, 1024),
                                  idesc, (c | kk) != 0);
                }
                umma_commit(a_free);
                umma_commit(&tfull[b]);
            }
        }
    } else {
        // (no store warp: the obs image is written by the converters.  One warp copying the finished A tile out with 16-byte
        // loads / stores took longer than the MMAs - 8.65 against 7.23 ms)
        // ===== epilogue: one row per thread; x = relu(acc [+ id/bias table] + act table) -> bf16 tile images + mask.
        // (Eight epilogue warps, one per row and net, measured slower: 7.21 -> 7.53 ms.) =====
        const uint32_t r = (uint32_t)(warp * 32 + lane);
        // the previous action of a row of the k-th item, fetched one item ahead (-1: none / step not filled, -2: padding row)
        auto fetch_prev = [&](int k, int& n_out) {
            n_out = 0;
            if (k >= n_items) return -2;
            const int64_t item = fc1_item(P, k);
            if (item < 0) return -2;
            const int64_t t = item / P.n_tiles, tile = item - t * P.n_tiles;
            const int64_t p = tile * BM + r;
            if (p >= P.R) return -2;
            const int64_t b = p / P.N;
            n_out = (int)(p - b * P.N);
            const int64_t tb = t + P.t0;                       // timestep in the batch
            if (!P.use_act || tb == 0) return -1;
            const int64_t be = ep_row(P.ep_index, b);
            const int64_t f = __ldg(P.filled + be * P.filled_sb + (tb - 1));
            const int a = (int)__ldg(P.actions + be * P.actions_sb + (tb - 1) * P.N + n_out);
            return f != 0 ? a : -1;
        };
        int n_cur, n_nxt;
        int a_prev = fetch_prev(blockIdx.x, n_cur);
        uint32_t ti = 0;
        pdl_wait();                                            // before the first store to the x images
        for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++ti) {
            const int64_t item = fc1_item(P, k);
            if (item < 0) break;
            const int b = ti & 1;
            const int a_next = fetch_prev(k + gridDim.x, n_nxt);
            TWAIT(5, &tfull[b], (ti >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + 128u * b + ((uint32_t)(warp * 32) << 16);
#pragma unroll
            for (int g = 0; g < 4; ++g) {                      // 32 accumulator columns: net = g / 2, h0 = 32 (g & 1)
                uint32_t v[32];
                tmem_ld_32x32(taddr + 32 * g, v);
                tmem_wait_ld();
                if (a_prev != -2 && g < 2 * P.n_nets) {
                    const int net = g >> 1, h0 = (g & 1) * 32;
                    uint8_t* tile_img = (net ? P.x_tg : P.x_on) + item * A_STAGE_BYTES;
                    const uint4* tac = a_prev >= 0 ? P.tab_act16 + ((int64_t)a_prev * 2 + net) * 8 + (h0 >> 3) : nullptr;
                    const float4* tid = P.fold_id ? nullptr
                                                  : reinterpret_cast<const float4*>(P.tab_id + ((int64_t)net * P.N + n_cur) * 64 + h0);
                    uint32_t mbits = 0;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {              // 8 columns = one 16-byte chunk
                        float o[8];
#pragma unroll
                        for (int k = 0; k < 8; ++k) o[k] = __uint_as_float(v[8 * q + k]);
                        if (tac) {
                            const uint4 w = __ldg(tac + q);
                            o[0] += __uint_as_float(w.x << 16); o[1] += __uint_as_float(w.x & 0xffff0000u);
                            o[2] += __uint_as_float(w.y << 16); o[3] += __uint_as_float(w.y & 0xffff0000u);
                            o[4] += __uint_as_float(w.z << 16); o[5] += __uint_as_float(w.z & 0xffff0000u);
                            o[6] += __uint_as_float(w.w << 16); o[7] += __uint_as_float(w.w & 0xffff0000u);
                        }
                        if (tid) {
                            const float4 b0 = __ldg(tid + 2 * q), b1 = __ldg(tid + 2 * q + 1);
                            o[0] += b0.x; o[1] += b0.y; o[2] += b0.z; o[3] += b0.w;
                            o[4] += b1.x; o[5] += b1.y; o[6] += b1.z; o[7] += b1.w;
                        }
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            o[k] = fmaxf(o[k], 0.f);
                            mbits |= (o[k] > 0.f ? 1u : 0u) << (8 * q + k);
                        }
                        *reinterpret_cast<uint4*>(tile_img + sw128_offset(r, (uint32_t)(h0 / 8 + q))) =
                            make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]),
                                       pack_bf16x2(o[6], o[7]));
                    }
                    if (P.relu_mask && net == 0) P.relu_mask[(item * 2 + (h0 >> 5)) * 128 + r] = mbits;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[b]);
            a_prev = a_next; n_cur = n_nxt;
        }
    }
    FC1_PROF_END(NS);
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_W) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256);
    }
}


// ------------------------------------------------------------------------------------------
// Learner fc1 of both nets with the weights in TENSOR memory.  The MMA runs transposed,
//   D[hidden, row] = W_tmem[hidden, k] . obs[row, k]^T     (M = 128 hidden units of both nets, N = 128 rows)
// so W (80 KB at K = 320) leaves shared memory; the obs tile is the B operand with the bytes and descriptor the
// A operand has in fc1_stream_kernel.  TMEM: [0, 256) two accumulators, [256, 256 + 32 NC) W.  The freed shared
// memory holds a five-slot staging ring (fc1_stream_kernel: three), the last-action table and a 2 x 16 KB stage
// from which each net's x tile leaves as ONE bulk store.  Producers and converters are those of fc1_stream_kernel.
// Epilogue: thread = (net, hidden unit) = accumulator lane, its 32 registers of a column block = 32 rows.
// fold_id only (the agent id / bias come in through the K padding), two nets only.
// ------------------------------------------------------------------------------------------
namespace fs {
constexpr int N_SLOTS_TS = 5;
constexpr int TS_TMEM_W = 256;            // first TMEM column of W
}  // namespace fs

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }   // the 4 epilogue warps

template <int NC, int ES>
__global__ void __launch_bounds__(fs::threads_for(fs::N_SLOTS_TS), 1) fc1_stream_ts_kernel(Fc1StreamParams P) {
    FC1_PROF_BEGIN;
    using namespace fs;
    constexpr int NS = N_SLOTS_TS, FIRST_CONV_W = PROD_W + NS;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* a_s = smem;                                    // [NC][16 KB] obs tile (B operand)
    uint8_t* xs = a_s + NC * A_STAGE_BYTES;                 // [net 2][16 KB] x tile images
    uint8_t* stage = xs + 2 * A_STAGE_BYTES;                // [NS][slot_bytes]
    float* tab_s = reinterpret_cast<float*>(stage + NS * P.slot_bytes);     // [A][128]: fc1.weight[h][O + a] of both nets
    int* prev_s = reinterpret_cast<int*>(tab_s + P.n_act * 128);            // [2][128] previous action of the tile's rows
    int* rowinfo = prev_s + 2 * BM;                         // [NS][group rows] (Fc1Ring)
    uint64_t* bars = reinterpret_cast<uint64_t*>(rowinfo + NS * group_rows<ES>());
    uint64_t* w_full = bars;                 // W is in TMEM (arrivals of the 4 epilogue warps)
    uint64_t* st_full = bars + 1;            // [NS]
    uint64_t* st_empty = st_full + NS;       // [NS]
    uint64_t* a_full = st_empty + NS;
    uint64_t* a_free = a_full + 1;
    uint64_t* tfull = a_free + 1;            // [2]
    uint64_t* tempty = tfull + 2;            // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(w_full, N_EPI);
        for (int i = 0; i < NS; ++i) { mbar_init(&st_full[i], 1); mbar_init(&st_empty[i], N_CONV); }
        mbar_init(a_full, N_CONV); mbar_init(a_free, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], N_EPI); }
        fence_barrier_init();
    }
    if (warp == MMA_W) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // (TMEM base and item count are read inside the roles: held across the role branch they spill at 112 registers)
    const Fc1Ring ring{stage, rowinfo, st_full, st_empty};

    if (warp >= PROD_W && warp < PROD_W + NS) {
        fc1_produce<NC, NS, ES>(P, ring, warp - PROD_W, lane, prof_acc);
    } else if (warp >= FIRST_CONV_W) {
        fc1_convert<NC, NS, ES>(P, ring, a_s, a_free, a_full, warp - FIRST_CONV_W, lane, prof_acc);
    } else if (warp == MMA_W) {
        if (lane == 0) {
            const uint32_t tmem_base = *tmem_slot;
            const int n_items = P.T * P.n_tiles;
            const uint32_t idesc = umma_idesc_bf16(BM, BM, 0, 0);
            mbar_wait(w_full, 0);
            tc_fence_after();
            uint32_t ti = 0;
            for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++ti) {
                if (fc1_item(P, k) < 0) break;
                const int b = ti & 1;
                TWAIT(3, a_full, ti & 1);
                TWAIT(4, &tempty[b], ((ti >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tm = tmem_base + 128u * b;
#pragma unroll
                for (int c = 0; c < NC; ++c) {
                    const uint32_t a_addr = smem_u32(a_s + c * A_STAGE_BYTES);
#pragma unroll
                    for (int kk = 0; kk < BK / 16; ++kk)
                        umma_bf16_ts(tm, tmem_base + TS_TMEM_W + (uint32_t)(c * (BK / 16) + kk) * 8u,
                                     umma_desc_sw128(a_addr + kk * 32, 16, 1024), idesc, (c | kk) != 0);
                }
                umma_commit(a_free);
                umma_commit(&tfull[b]);
            }
        }
    } else {
        // ===== epilogue: warp w reads accumulator lanes 32w .. 32w + 31 (its TMEM lane quarter) =====
        const int hl = warp * 32 + lane;                      // accumulator lane: online hidden 0-63 | target 64-127
        const int net = warp >> 1;
        const uint32_t tmem_base = *tmem_slot;
        const int n_items = P.T * P.n_tiles;
        TMARK(pe0);
        // W rows of this thread's hidden unit into TMEM: the packed image's 128-byte row, un-swizzled, is 32 columns
        {
            const uint8_t* wrow = reinterpret_cast<const uint8_t*>(P.Wp) + hl * 128;
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                uint32_t v[32];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint4 u = __ldg(reinterpret_cast<const uint4*>(wrow + c * A_STAGE_BYTES + ((j ^ (hl & 7)) << 4)));
                    v[4 * j] = u.x; v[4 * j + 1] = u.y; v[4 * j + 2] = u.z; v[4 * j + 3] = u.w;
                }
                tmem_st_32x32(tmem_base + TS_TMEM_W + 32u * c + ((uint32_t)(warp * 32) << 16), v);
            }
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(w_full);
        }
        {
            const uint16_t* ta = reinterpret_cast<const uint16_t*>(P.tab_act16);
            for (int i = hl; i < P.n_act * 128; i += 128) tab_s[i] = __uint_as_float((uint32_t)__ldg(ta + i) << 16);
        }
        TADD(14, clock64() - pe0);                             // epilogue: W into TMEM, table into shared memory
        // the previous action of row hl of the k-th item (-1: none / step not filled, -2: padding row)
        auto fetch_prev = [&](int k) {
            if (k >= n_items) return -2;
            const int64_t item = fc1_item(P, k);
            if (item < 0) return -2;
            const int64_t t = item / P.n_tiles, tile = item - t * P.n_tiles;
            const int64_t p = tile * BM + hl;
            if (p >= P.R) return -2;
            const int64_t b = p / P.N;
            const int n = (int)(p - b * P.N);
            const int64_t tb = t + P.t0;
            if (!P.use_act || tb == 0) return -1;
            const int64_t be = ep_row(P.ep_index, b);
            const int64_t f = __ldg(P.filled + be * P.filled_sb + (tb - 1));
            const int a = (int)__ldg(P.actions + be * P.actions_sb + (tb - 1) * P.N + n);
            return f != 0 ? a : -1;
        };
        int a_prev = fetch_prev(blockIdx.x);
        const uint32_t xs_u32 = smem_u32(xs + net * A_STAGE_BYTES);
        const uint32_t h2 = (uint32_t)(hl & 62);                // even hidden unit of the pair this lane stores
        const uint32_t xs_lane = xs_u32 + (h2 & 7) * 2;
        const uint32_t tab_u32 = smem_u32(tab_s + hl);
        uint32_t ti = 0;
        for (int k = blockIdx.x; k < n_items; k += gridDim.x, ++ti) {
            const int item = fc1_item(P, k);
            if (item < 0) break;
            const int b = ti & 1;
            const int a_next = fetch_prev(k + gridDim.x);
            const uint32_t pv_u32 = smem_u32(prev_s + b * BM);
            prev_s[b * BM + hl] = a_prev;
            TMARK(pe1);
            if (threadIdx.x == 0) bulk_wait_group_read<0>();    // the x stage of the previous item has been read
            epi_bar_sync();
            TADD(12, clock64() - pe1);                         // epilogue: stage free + prev table barrier
            TWAIT(5, &tfull[b], (ti >> 1) & 1);
            tc_fence_after();
            TMARK(pe2);
            const int tile = item % P.n_tiles;
            const int rows_valid = P.R - tile * BM < BM ? (int)(P.R - tile * BM) : BM;
            const uint32_t taddr = tmem_base + 128u * b + ((uint32_t)(warp * 32) << 16);
#pragma unroll 1
            for (int g = 0; g < 4; ++g) {                      // 32 accumulator columns = rows 32g .. 32g + 31
                uint32_t v[32];
                tmem_ld_32x32(taddr + 32 * g, v);
                tmem_wait_ld();
                if (g == 3) {                                  // the accumulator buffer is free for the tile after next
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty[b]);
                }
                // (explicit shared-space loads, no branches: generic loads and a branch per row made this loop a serial
                // chain of ~100 cycles per row)
                int pa[32];
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    int4 p4;
                    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(p4.x), "=r"(p4.y), "=r"(p4.z), "=r"(p4.w) : "r"(pv_u32 + (uint32_t)(32 * g + 4 * q) * 4u));
                    pa[4 * q] = p4.x; pa[4 * q + 1] = p4.y; pa[4 * q + 2] = p4.z; pa[4 * q + 3] = p4.w;
                }
                float o[32];
                uint32_t mword = 0;
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    const int a = pa[e];
                    const float t = lds_f32(tab_u32 + (uint32_t)(a > 0 ? a : 0) * 512u);
                    float x = __uint_as_float(v[e]);
                    x = a >= 0 ? x + t : x;
                    x = fmaxf(x, 0.f);
                    o[e] = x;
                    // the online net's ReLU word of (row, half) is the warp's vote: bit j = hidden unit 32 half + j
                    const uint32_t bal = __ballot_sync(0xffffffffu, x > 0.f);
                    mword = lane == e ? bal : mword;
                }
                if (net == 0 && P.relu_mask && 32 * g + lane < rows_valid)
                    P.relu_mask[((int64_t)item * 2 + warp) * 128 + 32 * g + lane] = mword;
                // bf16 pairs of adjacent hidden units: the even lane stores row e, the odd lane row e + 4 (the two rows
                // fall on disjoint 16-byte chunks of the swizzle, so the 32 stores of a step hit 32 banks)
#pragma unroll
                for (int e = 0; e < 32; ++e) {
                    if (e & 4) continue;
                    const bool odd = lane & 1;
                    const float send = odd ? o[e] : o[e + 4];
                    const float recv = __shfl_xor_sync(0xffffffffu, send, 1);
                    const uint32_t w = odd ? pack_bf16x2(recv, o[e + 4]) : pack_bf16x2(o[e], recv);
                    const uint32_t row = (uint32_t)(32 * g + e + (odd ? 4 : 0));
                    sts_b32(xs_lane + sw128_offset(row, h2 >> 3), w);
                }
            }
            fence_proxy_async_smem();
            epi_bar_sync();
            if (threadIdx.x == 0) {
                bulk_copy_s2g(P.x_on + (int64_t)item * A_STAGE_BYTES, xs, (uint32_t)rows_valid * 128u);
                bulk_copy_s2g(P.x_tg + (int64_t)item * A_STAGE_BYTES, xs + A_STAGE_BYTES, (uint32_t)rows_valid * 128u);
                bulk_commit_group();
            }
            TADD(13, clock64() - pe2);                         // epilogue: TMEM loads, tables, ReLU, mask, x stage
            a_prev = a_next;
        }
        if (threadIdx.x == 0) bulk_wait_group<0>();
    }
    FC1_PROF_END(NS);
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_W) {
        tc_fence_after();
        tmem_dealloc(*tmem_slot, 512);
    }
}

}  // namespace tc

// ------------------------------------------------------------------------------------------
// host entry points used by api.cu
// ------------------------------------------------------------------------------------------
int64_t tc_packed_elems(int Ncols, int K) {
    int n_chunks = (K + tc::BK - 1) / tc::BK;
    return (int64_t)Ncols * n_chunks * tc::BK;
}

int tc_pack_w(const float* const* ptrs, const int* rows, const int* lds, int nseg, int K, __nv_bfloat16* out,
              cudaStream_t s, int n_chunks_min) {
    tc::PackSegs segs;
    int Ncols = 0;
    segs.nseg = nseg;
    for (int i = 0; i < 4; ++i) {
        segs.ptr[i] = i < nseg ? ptrs[i] : nullptr;
        segs.rows[i] = i < nseg ? rows[i] : 0;
        segs.ld[i] = i < nseg ? lds[i] : 0;
        Ncols += segs.rows[i];
    }
    Ncols = (int)align_up(Ncols, 32);
    int n_chunks = (K + tc::BK - 1) / tc::BK;
    if (n_chunks < n_chunks_min) n_chunks = n_chunks_min;      // extra all-zero k-chunks (A images may be wider than K)
    int64_t total = (int64_t)Ncols * n_chunks * 8;
    tc::pack_w_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(segs, K, n_chunks, Ncols, out);
    PMB_LAUNCH_CHECK("pack_w_kernel");
    return PMB_OK;
}

// plain C = A . W^T + bias  (diagnostics / unit test of the tcgen05 pipeline)
int tc_gemm_plain(const float* A, RowMap amap, int64_t M, int K, const __nv_bfloat16* Wp, int Ncols_padded, int Nreal,
                  const float* bias, float* C, int64_t ldc, cudaStream_t s) {
    tc::GemmParams P{A, amap, M, K, (K + tc::BK - 1) / tc::BK, Wp, Ncols_padded, 0, 0, 0, 0, nullptr, nullptr};
    tc::PlainEpi epi{C, ldc, bias, Nreal};
    return tc::launch_tc_gemm(P, epi, s);
}

// tables for the fc1 epilogue: tab_act[net][a][h] = fc1_w[h][O + a];  tab_id[net][n][h] = fc1_w[h][O + A' + n] + b1[h]
__global__ void fc1_tables_kernel(const float* __restrict__ w_on, const float* __restrict__ b_on,
                                  const float* __restrict__ w_tg, const float* __restrict__ b_tg, int O, int A, int N,
                                  int D_in, int use_act, int use_id, float* __restrict__ tab_act,
                                  float* __restrict__ tab_id) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int n_act = 2 * A * 64, n_id = 2 * N * 64;
    if (i < n_act) {
        int net = i / (A * 64), r = i - net * A * 64, a = r / 64, h = r - a * 64;
        const float* w = net ? w_tg : w_on;
        tab_act[i] = use_act ? w[(int64_t)h * D_in + O + a] : 0.f;
    } else if (i < n_act + n_id) {
        int k = i - n_act;
        int net = k / (N * 64), r = k - net * N * 64, n = r / 64, h = r - n * 64;
        const float* w = net ? w_tg : w_on;
        const float* b = net ? b_tg : b_on;
        tab_id[k] = b[h] + (use_id ? w[(int64_t)h * D_in + O + (use_act ? A : 0) + n] : 0.f);
    }
}

int64_t tc_fc1_scratch_bytes(const pmb_dims* d);

// streaming fc1: packed W with the agent-id columns and the bias folded into the K padding (fold_id), and the
// last-action table of both nets as bf16 [A][net][64]
__global__ void fc1_stream_pack_kernel(const float* __restrict__ w_on, const float* __restrict__ b_on,
                                       const float* __restrict__ w_tg, const float* __restrict__ b_tg, int O, int A, int N,
                                       int D_in, int use_act, int use_id, int fold_id, int n_chunks,
                                       __nv_bfloat16* __restrict__ wp, __nv_bfloat16* __restrict__ tab_act16) {
    const int64_t n_w = (int64_t)128 * n_chunks * 8;          // one thread per 16-byte chunk of the packed image
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_w) {
        const int j = (int)(i & 7);
        const int col = (int)((i >> 3) & 127);
        const int c = (int)(i >> 10);
        const int net = col >> 6, h = col & 63;
        const float* w = (net ? w_tg : w_on) + (int64_t)h * D_in;
        const float bias = (net ? b_tg : b_on)[h];
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int k = c * 64 + j * 8 + e;
            float v = 0.f;
            if (k < O) v = w[k];
            else if (fold_id) {
                const int q = k - O;
                if (q < N) v = use_id ? w[O + (use_act ? A : 0) + q] : 0.f;
                else if (q == N) v = bias;
            }
            f[e] = v;
        }
        char* tile = reinterpret_cast<char*>(wp) + (int64_t)c * 16384;
        *reinterpret_cast<uint4*>(tile + tc::sw128_offset((uint32_t)col, (uint32_t)j)) =
            make_uint4(tc::pack_bf16x2(f[0], f[1]), tc::pack_bf16x2(f[2], f[3]), tc::pack_bf16x2(f[4], f[5]),
                       tc::pack_bf16x2(f[6], f[7]));
        return;
    }
    i -= n_w;
    if (i < (int64_t)A * 128) {
        const int a = (int)(i >> 7), net = (int)((i >> 6) & 1), h = (int)(i & 63);
        const float* w = net ? w_tg : w_on;
        tab_act16[i] = __float2bfloat16(use_act ? w[(int64_t)h * D_in + O + a] : 0.f);
    }
}

#ifdef PMB_FC1_PROFILE
extern "C" int pmb_debug_fc1_prof(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, tc::g_fc1_prof, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(tc::g_fc1_prof, z, sizeof(z)); }
    return 0;
}
#endif
// Shared-memory plan of the streaming fc1 kernels for obs elements of `es` bytes
struct Fc1StreamPlan {
    int n_chunks, slot_bytes, fold_id;
    int64_t smem_need;   // fc1_stream_kernel, both nets, N_SLOTS slots
    int64_t smem_1net;   // fc1_stream_kernel, one net (rollout), N_SLOTS_1NET slots
    int64_t smem_ts;     // fc1_stream_ts_kernel
    bool streams;        // tc_fc1_fwd_both with tile images runs a streaming kernel
};
static Fc1StreamPlan fc1_stream_plan(const pmb_dims* d, int es) {
    using namespace tc::fs;
    Fc1StreamPlan p;
    const int gr = group_rows_of(es);
    p.n_chunks = (d->O + tc::BK - 1) / tc::BK;
    // a group is at most (gr - 1) / N + 2 contiguous runs, each displaced by < RUN_SLACK bytes (see the producer)
    const int max_runs = std::min(gr, (gr - 1) / d->N + 2);
    p.slot_bytes = (int)align_up((int64_t)gr * d->O * es + (int64_t)RUN_SLACK * max_runs + 128, 128);
    p.fold_id = p.n_chunks * tc::BK - d->O >= d->N + 1;
    const int64_t tab = (int64_t)gr * 4;                     // row table bytes per slot
    p.smem_need = 1024 + 2 * (int64_t)p.n_chunks * tc::A_STAGE_BYTES + N_SLOTS * ((int64_t)p.slot_bytes + tab) + 256;
    p.smem_1net = 1024 + (int64_t)p.n_chunks * (tc::A_STAGE_BYTES / 2) + (int64_t)p.n_chunks * tc::A_STAGE_BYTES +
                  N_SLOTS_1NET * ((int64_t)p.slot_bytes + tab) + 256;
    p.smem_ts = 1024 + (int64_t)(p.n_chunks + 2) * tc::A_STAGE_BYTES + N_SLOTS_TS * ((int64_t)p.slot_bytes + tab) +
                (int64_t)d->A * 128 * 4 + 2 * tc::BM * 4 + 256;
    p.streams = p.n_chunks <= MAX_CHUNKS && p.smem_need <= 232448;
    return p;
}

bool tc_fc1_streams(const pmb_dims* d, int obs_dtype) {
    return fc1_stream_plan(d, obs_dtype == PMB_DTYPE_BF16 ? 2 : 4).streams;
}

// kind: 0 fc1_stream_ts_kernel, 1 fc1_stream_kernel with N_SLOTS_1NET slots (rollout, PDL), 2 with N_SLOTS slots
template <int NC, int ES>
static int launch_fc1_stream(const tc::Fc1StreamParams& Q, int kind, int64_t smem, int grid, cudaStream_t s) {
    using namespace tc::fs;
    if (kind == 0) {
        PMB_SMEM_ATTR((tc::fc1_stream_ts_kernel<NC, ES>), (int)smem);
        tc::fc1_stream_ts_kernel<NC, ES><<<grid, threads_for(N_SLOTS_TS), (size_t)smem, s>>>(Q);
    } else if (kind == 1) {
        PMB_SMEM_ATTR((tc::fc1_stream_kernel<NC, N_SLOTS_1NET, ES>), (int)smem);
        PMB_CUDA(launch_pdl(tc::fc1_stream_kernel<NC, N_SLOTS_1NET, ES>, dim3(grid), dim3(threads_for(N_SLOTS_1NET)),
                            (size_t)smem, s, rollout_pdl_enabled(), Q));
    } else {
        PMB_SMEM_ATTR((tc::fc1_stream_kernel<NC, N_SLOTS, ES>), (int)smem);
        tc::fc1_stream_kernel<NC, N_SLOTS, ES><<<grid, threads_for(N_SLOTS), (size_t)smem, s>>>(Q);
    }
    PMB_LAUNCH_CHECK("fc1_stream_kernel");
    return PMB_OK;
}

int tc_fc1_fwd_both(const pmb_dims* d, const pmb_batch* b, int t0, int nt, const AgentParams& on, const AgentParams& tg,
                    float* x_on, float* x_tg, int tile_images, uint8_t* obs_img_out, uint32_t* relu_mask, void* scratch,
                    int64_t scratch_bytes, cudaStream_t s, int weights_packed, const int32_t* live_items) {
    // scratch: packed W (128 x Kpad bf16) | tab_act | tab_id
    // live_items (may be NULL): the live (t, tile) items of a padded-step skipping learner step, -1 after the last one
    // (streaming kernels only)
    // weights_packed: the caller guarantees that `scratch` still holds the images / tables a previous call packed from
    // the SAME parameters (rollout steps between two learner updates): the pack launches are skipped
    const int D_in = d_in_of(d);
    int64_t wp_bytes = align_up(tc_packed_elems(128, d->O) * 2, 256);
    int64_t ta_bytes = align_up((int64_t)2 * d->A * 64 * 4, 256);
    int64_t ti_bytes = align_up((int64_t)2 * d->N * 64 * 4, 256);
    if (scratch_bytes < tc_fc1_scratch_bytes(d)) { set_error("tc_fc1: scratch too small"); return PMB_ERR_WORKSPACE; }
    __nv_bfloat16* wp = static_cast<__nv_bfloat16*>(scratch);
    float* tab_act = reinterpret_cast<float*>(static_cast<char*>(scratch) + wp_bytes);
    float* tab_id = reinterpret_cast<float*>(static_cast<char*>(scratch) + wp_bytes + ta_bytes);
    const bool bf16_obs = b->obs_dtype == PMB_DTYPE_BF16;
    // the streaming kernel packs its own W (fc1_stream_pack_kernel) and needs the agent-id table only when the one-hot
    // columns do not fit the K padding
    const Fc1StreamPlan sp = fc1_stream_plan(d, bf16_obs ? 2 : 4);
    const bool use_stream = tile_images && sp.streams;
    if (bf16_obs && !use_stream) { set_error("tc_fc1: bf16 obs needs the streaming fc1 kernel"); return PMB_ERR_INVALID; }
    int rc = PMB_OK;
    if (!use_stream) {
        const float* ptrs[2] = {on.fc1_w, tg.fc1_w};
        int rows[2] = {64, 64}, lds[2] = {D_in, D_in};
        rc = tc_pack_w(ptrs, rows, lds, 2, d->O, wp, s);
        if (rc) return rc;
    }
    if ((!use_stream || !sp.fold_id) && !(weights_packed && use_stream)) {
        int n_tab = 2 * (d->A + d->N) * 64;
        fc1_tables_kernel<<<(unsigned)ceil_div(n_tab, 256), 256, 0, s>>>(on.fc1_w, on.fc1_b, tg.fc1_w, tg.fc1_b, d->O, d->A,
                                                                         d->N, D_in, d->obs_last_action, d->obs_agent_id,
                                                                         tab_act, tab_id);
        PMB_LAUNCH_CHECK("fc1_tables_kernel");
    }
    const int64_t M = (int64_t)d->B * nt * d->N;
    RowMap map{b->obs_sb, (int64_t)d->N * d->O, (int64_t)d->O, nt, d->N};
    const float* obs_f32 = static_cast<const float*>(b->obs);
    tc::GemmParams P{obs_f32 + (int64_t)t0 * d->N * d->O, map, M, d->O, (d->O + tc::BK - 1) / tc::BK, wp, 128,
                     0, 0, 0, 0, nullptr, nullptr};
    if (tile_images) {
        // rows in time-major tiled order so that GEMM tiles coincide with the (t, tile) tile images
        const int64_t R = (int64_t)d->B * d->N;
        const int n_tiles = (int)ceil_div(R, 128);
        P.M = (int64_t)nt * n_tiles * 128;
        P.tm_R = R; P.tm_Rpad = (int64_t)n_tiles * 128; P.tm_N = d->N; P.tm_T = nt;
        P.a_img_out = obs_img_out;
        tc::Fc1TiEpi epi{tab_act, tab_id, b->actions, b->actions_sb, b->filled, b->filled_sb,
                         reinterpret_cast<uint8_t*>(x_on), reinterpret_cast<uint8_t*>(x_tg), t0, nt, d->N, d->A,
                         d->obs_last_action, n_tiles, R, relu_mask};
        if (use_stream) {
            const int n_chunks = sp.n_chunks, fold_id = sp.fold_id;
            __nv_bfloat16* tab_act16 = reinterpret_cast<__nv_bfloat16*>(static_cast<char*>(scratch) + wp_bytes + ta_bytes + ti_bytes);
            const int64_t n_pack = (int64_t)128 * n_chunks * 8 + (int64_t)d->A * 128;
            if (!weights_packed) {
                fc1_stream_pack_kernel<<<(unsigned)ceil_div(n_pack, 256), 256, 0, s>>>(
                    on.fc1_w, on.fc1_b, tg.fc1_w, tg.fc1_b, d->O, d->A, d->N, D_in, d->obs_last_action, d->obs_agent_id, fold_id,
                    n_chunks, wp, tab_act16);
                PMB_LAUNCH_CHECK("fc1_stream_pack_kernel");
            }
            tc::Fc1StreamParams Q;
            Q.ep_index = b->ep_index; Q.obs = static_cast<const uint8_t*>(b->obs); Q.obs_sb = b->obs_sb; Q.Wp = wp;
            Q.obs_img = obs_img_out; Q.R = R;
            Q.T = nt; Q.N = d->N; Q.O = d->O; Q.n_tiles = n_tiles; Q.n_chunks = n_chunks; Q.slot_bytes = sp.slot_bytes;
            Q.fold_id = fold_id; Q.tab_act16 = reinterpret_cast<const uint4*>(tab_act16); Q.tab_id = tab_id;
            Q.actions = b->actions; Q.actions_sb = b->actions_sb; Q.filled = b->filled; Q.filled_sb = b->filled_sb;
            Q.x_on = reinterpret_cast<uint8_t*>(x_on); Q.x_tg = reinterpret_cast<uint8_t*>(x_tg);
            Q.relu_mask = relu_mask; Q.use_act = d->obs_last_action;
            Q.n_nets = x_tg ? 2 : 1; Q.t0 = t0; Q.n_act = d->A;
            Q.items = live_items;
            // L2 prefetch of the CTA's next tile(s): measured (round 2, same box, alternating) as a LOSS - rollout step 0.196 ms
            // with one tile ahead, 0.217 ms with two, 0.190 ms without; learner fc1 8.1-8.4 / 8.8 / 8.0 ms - the copies of the
            // ring already keep the memory system busy and the prefetch instructions cost the producers issue time.
            // PMB_FC1_PREFETCH = tiles ahead keeps the experiment available.
            Q.l2_prefetch = 0;
            { const char* e = getenv("PMB_FC1_PREFETCH"); if (e) Q.l2_prefetch = atoi(e); }
            const int64_t n_items = (int64_t)nt * n_tiles;
            const int grid = (int)(n_items < sm_count() ? n_items : sm_count());
            // one net (rollout step): W takes half the shared memory, the staging ring gets two more slots when they fit -
            // the stream is bound by the bytes in flight per SM (slot turn-around ~3500 cycles: 3 x 18 KB give 4.6 TB/s)
            const bool wide_ring = Q.n_nets == 1 && sp.smem_1net <= 232448;
            // learner step: W of both nets in tensor memory (fc1_stream_ts_kernel) when the agent id is folded into the K
            // padding and its ring, x stage and last-action table fit; PMB_FC1_TS=0 selects fc1_stream_kernel (A/B switch,
            // read on every call so that one process can run both)
            const char* e_ts = getenv("PMB_FC1_TS");
            const bool use_ts = Q.n_nets == 2 && fold_id && sp.smem_ts <= 232448 && !(e_ts && e_ts[0] == '0');
            const int kind = use_ts ? 0 : (wide_ring ? 1 : 2);
            const int64_t smem = use_ts ? sp.smem_ts : (wide_ring ? sp.smem_1net : sp.smem_need);
#define PMB_FC1_STREAM_LAUNCH(NC)                                                                                          \
    case NC:                                                                                                               \
        return bf16_obs ? launch_fc1_stream<NC, 2>(Q, kind, smem, grid, s) : launch_fc1_stream<NC, 4>(Q, kind, smem, grid, s);
            switch (n_chunks) {
                PMB_FC1_STREAM_LAUNCH(1)
                PMB_FC1_STREAM_LAUNCH(2)
                PMB_FC1_STREAM_LAUNCH(3)
                PMB_FC1_STREAM_LAUNCH(4)
                PMB_FC1_STREAM_LAUNCH(5)
            }
#undef PMB_FC1_STREAM_LAUNCH
            set_error("tc_fc1: %d k-chunks", n_chunks);
            return PMB_ERR_INVALID;
        }
        if (b->ep_index || live_items) { set_error("tc_fc1: ep_index and live items need the streaming kernel (obs dim <= 320)"); return PMB_ERR_INVALID; }
        return tc::launch_tc_gemm(P, epi, s);
    }
    if (b->ep_index || live_items) { set_error("tc_fc1: ep_index and live items are not supported without tile images"); return PMB_ERR_INVALID; }
    tc::Fc1Epi epi{tab_act, tab_id, b->actions, b->actions_sb, b->filled, b->filled_sb, x_on, x_tg,
                   t0, nt, d->N, d->A, d->obs_last_action, (int64_t)d->B * d->N};
    return tc::launch_tc_gemm(P, epi, s);
}
int64_t tc_fc1_scratch_bytes(const pmb_dims* d) {
    return align_up(tc_packed_elems(128, d->O) * 2, 256) + align_up((int64_t)2 * d->A * 64 * 4, 256) +
           align_up((int64_t)2 * d->N * 64 * 4, 256) + align_up((int64_t)d->A * 128 * 2, 256);
}

// permuted bias for the mixer: packed order [w1 | b1 | w_final | v0] from flat order [w1 | w_final | b1 | v0]
__global__ void mix_bias_perm_kernel(const float* __restrict__ b_cat, int N, float* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int C = (N + 3) * 32;
    if (i >= C) return;
    int grp = i >> 5, e = i & 31;
    int src_grp = grp < N ? grp : (grp == N ? N + 1 : (grp == N + 1 ? N : N + 2));
    out[i] = b_cat[src_grp * 32 + e];
}

int64_t tc_mixer_scratch_bytes(const pmb_dims* d) {
    const int C = (d->N + 3) * 32;
    return align_up(tc_packed_elems((int)align_up(C, 32), d->S + 1) * 2, 256) + align_up((int64_t)C * 4, 256);
}

// ---- image-fed mixer path -------------------------------------------------------------------------
// state [B, T, S] fp32 or bf16 (ES = element size) -> bf16 tile images [ceil(B*T/128)][ceil((S+1)/64)][16 KB] over ALL
// (b, t) rows, m' = b*T + t.  Column S of every real row holds 1.0 (the bias-gradient column of the hypernet
// weight-gradient GEMM; the packed forward weights are zero there), everything else beyond S and all padding rows are
// zero.  fp32 state is rounded to bf16 here, so bf16 storage of the same rounded values gives the same images.
template <int ES>
__global__ void __launch_bounds__(256)
state_to_images_kernel(const uint8_t* __restrict__ state, int64_t state_sb, const int64_t* __restrict__ ep_index, int64_t BT,
                       int T, int S, int n_chunks, uint8_t* __restrict__ img) {
    static_assert(ES == 4 || ES == 2, "fp32 or bf16 state");
    // one thread per 16-byte chunk
    const int64_t total = ((BT + 127) / 128) * 128 * (int64_t)n_chunks * 8;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int j = (int)(i & 7);
    int64_t q = i >> 3;
    const int r = (int)(q & 127);
    q >>= 7;
    const int c = (int)(q % n_chunks);
    const int64_t tile = q / n_chunks;
    const int64_t m = tile * 128 + r;
    float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (m < BT) {
        const int64_t b = m / T;
        const int t = (int)(m - b * T);
        const uint8_t* src = state + (ep_row(ep_index, b) * state_sb + (int64_t)t * S + c * 64 + j * 8) * ES;
        const int nv = S - (c * 64 + j * 8);
        const uintptr_t al = reinterpret_cast<uintptr_t>(src);
        if (ES == 4 && nv >= 8 && (al & 7) == 0) {                          // the common fp32 case: four 8-byte loads
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(src) + e);
                f[2 * e] = v.x; f[2 * e + 1] = v.y;
            }
        } else if (ES == 2 && nv >= 8 && (al & 15) == 0) {                   // bf16: the whole chunk in one 16-byte load
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(src));
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) { f[2 * e] = __uint_as_float(w[e] << 16); f[2 * e + 1] = __uint_as_float(w[e] & 0xffff0000u); }
        } else if (ES == 2 && nv >= 8 && (al & 3) == 0) {                    // rows of 2 * S bytes, S even (27m: 2340)
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(src) + e);
                f[2 * e] = __uint_as_float(w << 16); f[2 * e + 1] = __uint_as_float(w & 0xffff0000u);
            }
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (e < nv) {
                    if (ES == 4) f[e] = __ldg(reinterpret_cast<const float*>(src) + e);
                    else f[e] = __uint_as_float((uint32_t)__ldg(reinterpret_cast<const unsigned short*>(src) + e) << 16);
                } else if (e == nv) {
                    f[e] = 1.0f;
                }
            }
        }
    }
    *reinterpret_cast<uint4*>(img + (tile * n_chunks + c) * 16384 + tc::sw128_offset((uint32_t)r, (uint32_t)j)) =
        make_uint4(tc::pack_bf16x2(f[0], f[1]), tc::pack_bf16x2(f[2], f[3]), tc::pack_bf16x2(f[4], f[5]),
                   tc::pack_bf16x2(f[6], f[7]));
}

int tc_state_to_images(const pmb_dims* d, const pmb_batch* b, uint8_t* img, cudaStream_t s) {
    const int64_t BT = (int64_t)d->B * d->T;
    const int n_chunks = tc_state_chunks(d);
    const int64_t total = ((BT + 127) / 128) * 128 * (int64_t)n_chunks * 8;
    const uint8_t* state = static_cast<const uint8_t*>(b->state);
    if (b->state_dtype == PMB_DTYPE_BF16)
        state_to_images_kernel<2><<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(state, b->state_sb, b->ep_index, BT, d->T,
                                                                                 d->S, n_chunks, img);
    else
        state_to_images_kernel<4><<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(state, b->state_sb, b->ep_index, BT, d->T,
                                                                                 d->S, n_chunks, img);
    PMB_LAUNCH_CHECK("state_to_images_kernel");
    return PMB_OK;
}

// QMIX forward from state images; raw_img != null keeps the hypernet outputs (online mixer)
int tc_mixer_fwd_img(const pmb_dims* d, const MixerParams& mp, const uint8_t* state_img, const float* agent_qs, int t_off,
                     uint8_t* raw_img, float* q_tot, void* scratch, int64_t scratch_bytes, cudaStream_t s) {
    const int N = d->N, S = d->S, C = (N + 3) * 32;
    const int n_chunks = tc_state_chunks(d);
    if (scratch_bytes < tc_mixer_scratch_bytes(d)) { set_error("tc_mixer: scratch too small"); return PMB_ERR_WORKSPACE; }
    __nv_bfloat16* wp = static_cast<__nv_bfloat16*>(scratch);
    float* bias = reinterpret_cast<float*>(static_cast<char*>(scratch) + align_up(tc_packed_elems(C, S + 1) * 2, 256));
    const float* ptrs[4] = {mp.w_cat, mp.w_cat + (int64_t)(N + 1) * 32 * S, mp.w_cat + (int64_t)N * 32 * S,
                            mp.w_cat + (int64_t)(N + 2) * 32 * S};
    int rows[4] = {N * 32, 32, 32, 32}, lds[4] = {S, S, S, S};
    int rc = tc_pack_w(ptrs, rows, lds, 4, S, wp, s, n_chunks);
    if (rc) return rc;
    mix_bias_perm_kernel<<<(unsigned)ceil_div(C, 256), 256, 0, s>>>(mp.b_cat, N, bias);
    PMB_LAUNCH_CHECK("mix_bias_perm_kernel");
    const int64_t BT = (int64_t)d->B * d->T;
    tc::GemmParams P{nullptr, dense_map(0), ((BT + 127) / 128) * 128, n_chunks * 64, n_chunks, wp, C,
                     0, 0, 0, 0, nullptr, state_img};
    tc::MixImgEpi epi{bias, agent_qs, mp.v2_w, mp.v2_b, q_tot, raw_img, N, d->T, t_off, tc_mix_cblks(d), BT};
    return tc::launch_tc_gemm(P, epi, s);
}

}  // namespace pmb
