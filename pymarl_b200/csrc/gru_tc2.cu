// bf16 tensor-core tier, second-generation recurrence kernels (learner step only).
//
//   gru_fwd2_kernel   : GRUCell unrolled over T for TWO 128-row tiles per CTA in ping-pong (one CTA per SM): while the
//                       eight epilogue warps do the gate math of one tile, the tensor core runs the 16 tcgen05.mma of
//                       the other.  No fc2 inside the recurrence (q is produced by q_select_kernel from the h images),
//                       so a step's dependency chain is MMA -> gate math -> MMA.  Everything that goes to HBM leaves
//                       through shared memory: the new h tile is the MMA operand tile itself, the four gate tiles are
//                       staged in the exact image layout, and ONE thread issues cp.async.bulk shared->global copies of
//                       16 KB each (the first version stored 16 bytes per thread at a 128-byte stride: 32 cache lines
//                       per warp instruction, which made the LSU the bottleneck - ncu, profiles/r01_*).
//   q_select_kernel   : q = fc2(h) for the online and the target net out of the h images (two tcgen05.mma groups per
//                       128-row tile) fused with learners/q_learner.py:55-78: chosen-action gather, avail masking
//                       (-9999999), double-Q arg-max (ties -> lowest index), target gather.  Q never goes to HBM
//                       unless a debug/test output pointer is given.
#include "common.cuh"
#include "tc_common.cuh"
#include "gru_tc.cuh"

namespace pmb {
namespace tc {

namespace {
constexpr int TILE_ROWS2 = 128;
constexpr int TILE_BYTES2 = 16384;

__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// sigmoid(x) = 0.5 tanh(0.5 x) + 0.5 : one MUFU op instead of ex2 + rcp
__device__ __forceinline__ float sigmoid_tanh(float x) { return fmaf(0.5f, tanh_approx(0.5f * x), 0.5f); }

__device__ __forceinline__ void ld_tmem_16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void ld_tmem_8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void lds_v4(uint32_t addr, float (&v)[4]) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}
// 16 fp32 values (columns 16*c16 .. +15 of row r) -> two 16-byte chunks of a tile image
__device__ __forceinline__ void st_row16(uint8_t* tile, uint32_t r, int c16, const float (&f)[16]) {
    uint4 a = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
    uint4 b = make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]), pack_bf16x2(f[12], f[13]),
                         pack_bf16x2(f[14], f[15]));
    *reinterpret_cast<uint4*>(tile + sw128_offset(r, 2 * c16)) = a;
    *reinterpret_cast<uint4*>(tile + sw128_offset(r, 2 * c16 + 1)) = b;
}
}  // namespace

// ------------------------------------------------------------------------------------------
// forward recurrence, two tiles per CTA
// ------------------------------------------------------------------------------------------
namespace g2 {
constexpr int WIH = 0, WHH = 24576;
constexpr int XB = 49152;                          // [tile 2][buf 2][16 KB]
constexpr int HT = XB + 4 * TILE_BYTES2;           // [tile 2][16 KB]   h operand tile = h image
constexpr int ST = HT + 2 * TILE_BYTES2;           // [4][16 KB]        gate staging (r, z, n, hn), shared by both tiles
constexpr int BIAS = ST + 4 * TILE_BYTES2;         // brz[128] | bin[64] | bhn[64]
constexpr int BARS = BIAS + 1024;
constexpr int SMEM_BYTES = 1024 + BARS + 256;
constexpr int N_EPI_WARPS = 16, MMA_WARP = 16, IO_WARP = 17;
constexpr int THREADS = 576;
}  // namespace g2

struct GruFwd2Params {
    const __nv_bfloat16* w_ih_img;   // 192 rows x 128 B
    const __nv_bfloat16* w_hh_img;
    const float *b_ih, *b_hh;
    const uint8_t* x_ti;             // [nt][n_tiles][16 KB]
    uint8_t* h_ti;                   // [(nt+1)][n_tiles][16 KB]   slot 0 = h_0 = 0 (written here), slot t+1 = h_t
    uint8_t* g_ti;                   // [nt][n_tiles][4][16 KB] (r, z, n, hn) or null
    int64_t R;
    int nt, n_tiles, tiles_per_cta;
    // optional (padded-step skipping): a CTA runs tile_steps[its first tile] steps.  Tiles are sorted by their step count,
    // descending, so a CTA's second tile never needs more; the steps it runs beyond its own count are never read.
    const int32_t* tile_steps;
};

// the steps a CTA runs sit in shared memory and are re-read at every step (held in a register, the count spills)
__device__ __forceinline__ int lds_s32(const int* p) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)));
    return v;
}

__global__ void __launch_bounds__(g2::THREADS, 1) gru_fwd2_kernel(GruFwd2Params P) {
    using namespace g2;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    float* bias = reinterpret_cast<float*>(smem + BIAS);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BARS);
    uint64_t* w_full = bars;                 // weights landed
    uint64_t* x_full = bars + 1;             // [tile][buf]
    uint64_t* x_empty = bars + 5;            // [tile][buf]
    uint64_t* gates_full = bars + 9;         // [tile]
    uint64_t* h_ready = bars + 11;           // [tile]  epilogue wrote the h tile and drained the accumulators
    uint64_t* ht_free = bars + 13;           // [tile]  the bulk store of the h tile has finished reading it
    uint64_t* st_ready = bars + 15;          // gate staging written
    uint64_t* st_free = bars + 16;           // the bulk store of the gate staging has finished reading it
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 17);
    int* nt_s = reinterpret_cast<int*>(bars + 18);   // steps this CTA runs (0: nothing but the h_0 image)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // tiles_per_cta = 2: ping-pong (the tensor core works on one tile while the epilogue warps do the other's gate math);
    // = 1 when there are fewer tiles than SMs: twice the CTAs, each with a shorter per-step chain
    const int tile0 = P.tiles_per_cta * blockIdx.x;
    const int n_my = P.n_tiles - tile0 >= P.tiles_per_cta ? P.tiles_per_cta : 1;
    const bool stash = P.g_ti != nullptr;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int i = 0; i < 4; ++i) { mbar_init(&x_full[i], 1); mbar_init(&x_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&gates_full[i], 1); mbar_init(&h_ready[i], N_EPI_WARPS); mbar_init(&ht_free[i], 1); }
        mbar_init(st_ready, N_EPI_WARPS); mbar_init(st_free, 1);
        *nt_s = P.tile_steps ? min(P.nt, __ldg(P.tile_steps + tile0)) : P.nt;
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc(tmem_slot, 512);
    for (int i = threadIdx.x; i < 128; i += THREADS) bias[i] = P.b_ih[i] + P.b_hh[i];
    for (int i = threadIdx.x; i < 64; i += THREADS) {
        bias[128 + i] = P.b_ih[128 + i];
        bias[192 + i] = P.b_hh[128 + i];
    }
    // h_0 = 0 in both operand tiles
    for (int i = threadIdx.x; i < 2 * TILE_BYTES2 / 16; i += THREADS)
        reinterpret_cast<uint4*>(smem + HT)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == IO_WARP) {
        // ===== loads (weights, x tiles) and bulk stores (h, gates) : one thread =====
        if (lane == 0) {
            mbar_arrive_expect_tx(w_full, 2 * 24576);
            bulk_copy_g2s(smem + WIH, P.w_ih_img, 24576, w_full);
            bulk_copy_g2s(smem + WHH, P.w_hh_img, 24576, w_full);
            auto load_x = [&](int i, int t) {
                const int b = t & 1;
                mbar_wait(&x_empty[2 * i + b], (uint32_t)(((t >> 1) & 1) ^ 1));
                mbar_arrive_expect_tx(&x_full[2 * i + b], TILE_BYTES2);
                bulk_copy_g2s(smem + XB + (2 * i + b) * TILE_BYTES2,
                              P.x_ti + ((int64_t)t * P.n_tiles + tile0 + i) * TILE_BYTES2, TILE_BYTES2, &x_full[2 * i + b]);
            };
            for (int t = 0; t < 2 && t < lds_s32(nt_s); ++t)
                for (int i = 0; i < n_my; ++i) load_x(i, t);
            // h_0 image (zeros) from the operand tiles
            for (int i = 0; i < n_my; ++i)
                bulk_copy_s2g(P.h_ti + (int64_t)(tile0 + i) * TILE_BYTES2, smem + HT + i * TILE_BYTES2, TILE_BYTES2);
            bulk_commit_group();
            bulk_wait_group_read<0>();
            for (int i = 0; i < n_my; ++i) mbar_arrive(&ht_free[i]);    // arrival #0: the h_0 stores no longer read HT
            uint32_t use = 0;
            for (int t = 0; t < lds_s32(nt_s); ++t)
                for (int i = 0; i < n_my; ++i, ++use) {
                    mbar_wait(&h_ready[i], (uint32_t)(t & 1));
                    const int64_t tt = (int64_t)t * P.n_tiles + tile0 + i;
                    bulk_copy_s2g(P.h_ti + (tt + P.n_tiles) * TILE_BYTES2, smem + HT + i * TILE_BYTES2, TILE_BYTES2);
                    bulk_commit_group();
                    if (t + 2 < lds_s32(nt_s)) load_x(i, t + 2);
                    if (stash) {
                        mbar_wait(st_ready, use & 1);
                        bulk_copy_s2g(P.g_ti + tt * 4 * TILE_BYTES2, smem + ST, 4 * TILE_BYTES2);
                        bulk_commit_group();
                        bulk_wait_group_read<1>();             // the h store (all but the newest group) is done reading
                        mbar_arrive(&ht_free[i]);
                        bulk_wait_group_read<0>();
                        mbar_arrive(st_free);
                    } else {
                        bulk_wait_group_read<0>();
                        mbar_arrive(&ht_free[i]);
                    }
                }
            bulk_wait_group<0>();
        }
    } else if (warp == MMA_WARP) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t wih = smem_u32(smem + WIH), whh = smem_u32(smem + WHH);
            const uint32_t id128 = umma_idesc_bf16(128, 128, 0, 0), id64 = umma_idesc_bf16(128, 64, 0, 0);
            mbar_wait(w_full, 0);
            for (int t = 0; t < lds_s32(nt_s); ++t)
                for (int i = 0; i < n_my; ++i) {
                    const int b = t & 1;
                    const uint32_t xt = smem_u32(smem + XB + (2 * i + b) * TILE_BYTES2);
                    const uint32_t ht = smem_u32(smem + HT + i * TILE_BYTES2);
                    const uint32_t tm = tmem_base + 256 * i;
                    mbar_wait(&x_full[2 * i + b], (uint32_t)((t >> 1) & 1));
                    if (t > 0) mbar_wait(&h_ready[i], (uint32_t)((t - 1) & 1));     // h_{t-1} written, gates(t-1) drained
                    tc_fence_after();
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)                 // r|z : x . W_i{r,z}^T
                        umma_bf16(tm, umma_desc_sw128(xt + kk * 32, 16, 1024), umma_desc_sw128(wih + kk * 32, 16, 1024),
                                  id128, kk != 0);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)                 // n, input part
                        umma_bf16(tm + 128, umma_desc_sw128(xt + kk * 32, 16, 1024),
                                  umma_desc_sw128(wih + 16384 + kk * 32, 16, 1024), id64, kk != 0);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)                 // r|z += h . W_h{r,z}^T
                        umma_bf16(tm, umma_desc_sw128(ht + kk * 32, 16, 1024), umma_desc_sw128(whh + kk * 32, 16, 1024),
                                  id128, 1);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)                 // n, hidden part
                        umma_bf16(tm + 192, umma_desc_sw128(ht + kk * 32, 16, 1024),
                                  umma_desc_sw128(whh + 16384 + kk * 32, 16, 1024), id64, kk != 0);
                    umma_commit(&x_empty[2 * i + b]);
                    umma_commit(&gates_full[i]);
                }
        }
    } else {
        // ===== epilogue: 16 warps (4 per scheduler, to hide the tcgen05.ld / MUFU / barrier latencies);
        // warp w owns TMEM lanes 32 (w & 3) .. +31 and hidden columns 16 (w >> 2) .. +15 =====
        const int q4 = warp & 3, c16 = warp >> 2;
        const uint32_t r = (uint32_t)(q4 * 32 + lane);
        const uint32_t tlane = tmem_base + ((uint32_t)(q4 * 32) << 16) + 16 * c16;
        float h[2][16];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
            for (int j = 0; j < 16; ++j) h[i][j] = 0.f;
        bool valid[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) valid[i] = (int64_t)(tile0 + i) * TILE_ROWS2 + r < P.R;
        const uint32_t bias_s = smem_u32(bias) + 64 * c16;     // this thread's 16 columns of brz | bin | bhn
        uint32_t use = 0;                                      // staging-buffer use counter (all tiles, all steps)
        for (int t = 0; t < lds_s32(nt_s); ++t) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                if (i < n_my) {
                    mbar_wait(&gates_full[i], (uint32_t)(t & 1));
                    mbar_wait(&ht_free[i], (uint32_t)(t & 1));   // the store of h_{t-1} (arrival #t) has read HT[i]
                    tc_fence_after();
                    uint8_t* hti = smem + HT + i * TILE_BYTES2;
                    const uint32_t ta = tlane + 256 * i;
                    uint32_t pr[8], pz[8], pn[8], phn[8];        // packed gates of the 16 columns, kept for the staging write
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {             // 8 columns at a time (register budget: 96 / thread)
                        uint32_t ar[8], az[8], ain[8], ahn[8];
                        ld_tmem_8(ta + 8 * hf, ar);
                        ld_tmem_8(ta + 64 + 8 * hf, az);
                        ld_tmem_8(ta + 128 + 8 * hf, ain);
                        ld_tmem_8(ta + 192 + 8 * hf, ahn);
                        float br[8], bz[8], bn[8], bh[8];
                        lds_v4(bias_s + 32 * hf, *reinterpret_cast<float(*)[4]>(&br[0]));
                        lds_v4(bias_s + 32 * hf + 16, *reinterpret_cast<float(*)[4]>(&br[4]));
                        lds_v4(bias_s + 256 + 32 * hf, *reinterpret_cast<float(*)[4]>(&bz[0]));
                        lds_v4(bias_s + 256 + 32 * hf + 16, *reinterpret_cast<float(*)[4]>(&bz[4]));
                        lds_v4(bias_s + 512 + 32 * hf, *reinterpret_cast<float(*)[4]>(&bn[0]));
                        lds_v4(bias_s + 512 + 32 * hf + 16, *reinterpret_cast<float(*)[4]>(&bn[4]));
                        lds_v4(bias_s + 768 + 32 * hf, *reinterpret_cast<float(*)[4]>(&bh[0]));
                        lds_v4(bias_s + 768 + 32 * hf + 16, *reinterpret_cast<float(*)[4]>(&bh[4]));
                        tmem_wait_ld();
                        uint32_t ph[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            float vr[2], vz[2], vn[2], vhn[2], vh[2];
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int j = 2 * k + e;
                                const float rg = sigmoid_tanh(__uint_as_float(ar[j]) + br[j]);
                                const float zg = sigmoid_tanh(__uint_as_float(az[j]) + bz[j]);
                                const float hn = __uint_as_float(ahn[j]) + bh[j];
                                const float ng = tanh_approx(fmaf(rg, hn, __uint_as_float(ain[j]) + bn[j]));
                                float hv = fmaf(zg, h[i][8 * hf + j] - ng, ng);
                                if (!valid[i]) hv = 0.f;
                                h[i][8 * hf + j] = hv;
                                vr[e] = rg; vz[e] = zg; vn[e] = ng; vhn[e] = hn; vh[e] = hv;
                            }
                            pr[4 * hf + k] = pack_bf16x2(vr[0], vr[1]); pz[4 * hf + k] = pack_bf16x2(vz[0], vz[1]);
                            pn[4 * hf + k] = pack_bf16x2(vn[0], vn[1]); phn[4 * hf + k] = pack_bf16x2(vhn[0], vhn[1]);
                            ph[k] = pack_bf16x2(vh[0], vh[1]);
                        }
                        *reinterpret_cast<uint4*>(hti + sw128_offset(r, (uint32_t)(2 * c16 + hf))) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                    }
                    // h is in place and the accumulators are drained: the next step's MMAs may start
                    tc_fence_before();
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&h_ready[i]);
                    if (stash) {
                        // the gate staging is shared by both tiles: wait until the previous use's store has read it
                        if (use > 0) mbar_wait(st_free, (use - 1) & 1);
#pragma unroll
                        for (int hf = 0; hf < 2; ++hf) {
                            const uint32_t off = sw128_offset(r, (uint32_t)(2 * c16 + hf));
                            const uint4 zero = make_uint4(0, 0, 0, 0);
                            const int k0 = 4 * hf;
                            *reinterpret_cast<uint4*>(smem + ST + off) =
                                valid[i] ? make_uint4(pr[k0], pr[k0 + 1], pr[k0 + 2], pr[k0 + 3]) : zero;
                            *reinterpret_cast<uint4*>(smem + ST + TILE_BYTES2 + off) =
                                valid[i] ? make_uint4(pz[k0], pz[k0 + 1], pz[k0 + 2], pz[k0 + 3]) : zero;
                            *reinterpret_cast<uint4*>(smem + ST + 2 * TILE_BYTES2 + off) =
                                valid[i] ? make_uint4(pn[k0], pn[k0 + 1], pn[k0 + 2], pn[k0 + 3]) : zero;
                            *reinterpret_cast<uint4*>(smem + ST + 3 * TILE_BYTES2 + off) =
                                valid[i] ? make_uint4(phn[k0], phn[k0 + 1], phn[k0 + 2], phn[k0 + 3]) : zero;
                        }
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(st_ready);
                    }
                    ++use;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------
// q = fc2(h) for both nets + chosen-action gather + double-Q target (q_learner.py:55-78)
// ------------------------------------------------------------------------------------------
namespace qs {
constexpr int STAGES = 2;                                  // x 2 CTAs per SM = 4 tiles in flight
constexpr int W2ON = 0, W2TG = 8192, STG = 16384;          // stage: h_on tile | h_tg tile
constexpr int STAGE_BYTES = 2 * TILE_BYTES2;
constexpr int BIAS = STG + STAGES * STAGE_BYTES;           // b2_on[64] | b2_tg[64]
constexpr int BARS = BIAS + 512;
constexpr int SMEM_BYTES = 1024 + BARS + 256;
constexpr int THREADS = 192;                               // warps 0-3 epilogue, 4 MMA, 5 loader
}  // namespace qs

struct QSelectParams {
    const __nv_bfloat16* w2_on_img;  // 64 rows x 128 B (rows >= A zero)
    const __nv_bfloat16* w2_tg_img;
    const float *b2_on, *b2_tg;
    const uint8_t* h_on_ti;          // [(T+1)][n_tiles][16 KB]
    const uint8_t* h_tg_ti;
    const void* avail; int64_t avail_sb;   // i32, or u8 (the kernel's AVB = 1)
    const int64_t* actions; int64_t actions_sb;
    const int64_t* ep_index;         // optional batch row -> buffer episode
    float* chosen;                   // [B][T-1][N]
    float* tmax;                     // [B][T-1][N]
    float* q_on_out;                 // optional fp32 [T][R][A] (tests / diagnostics)
    float* q_tg_out;
    int64_t R;
    int T, N, A, n_tiles, double_q;
    // optional (padded-step skipping): walk items[0 .. *n_live) instead of every t * n_tiles + tile, and write 0 to the
    // chosen / tmax entries of the (t, tile) items left out (t >= tile_steps[tile])
    const int32_t* items;
    const int32_t* n_live;
    const int32_t* tile_steps;
};

// One row's avail, columns c of [0, 64) as 16 words of 4 cells each.  i32 cells (AVB = 4): avv[c] is the cell; u8 cells
// (AVB = 1): byte c & 3 of word c >> 2.  The row's cells are loaded with the widest words its alignment allows, and no
// byte past column A - 1 is read; columns >= A read as 0.
template <int AVB> struct AvailRow;
template <> struct AvailRow<4> {
    int4 avv[16];
    __device__ __forceinline__ void load(const void* row, bool want, int A, bool vec_ok) {
        const int32_t* av = static_cast<const int32_t*>(row);
        const int n_q4 = (A + 3) >> 2;
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            avv[q] = make_int4(0, 0, 0, 0);
            if (want && q < n_q4) {
                if (vec_ok) avv[q] = __ldg(reinterpret_cast<const int4*>(av) + q);
                else {
                    avv[q].x = __ldg(av + 4 * q);
                    if (4 * q + 1 < A) avv[q].y = __ldg(av + 4 * q + 1);
                    if (4 * q + 2 < A) avv[q].z = __ldg(av + 4 * q + 2);
                    if (4 * q + 3 < A) avv[q].w = __ldg(av + 4 * q + 3);
                }
            }
        }
    }
    __device__ __forceinline__ bool ok(int a) const {
        const int4 w = avv[a >> 2];
        return ((a & 3) == 0 ? w.x : ((a & 3) == 1 ? w.y : ((a & 3) == 2 ? w.z : w.w))) != 0;
    }
};
template <> struct AvailRow<1> {
    uint32_t w[16];
    __device__ __forceinline__ void load(const void* row, bool want, int A, bool) {
        const uint8_t* av = static_cast<const uint8_t*>(row);
        const uintptr_t al = reinterpret_cast<uintptr_t>(av);
#pragma unroll
        for (int q = 0; q < 16; ++q) w[q] = 0u;
        if (!want) return;
#pragma unroll
        for (int g = 0; g < 4; ++g) {                      // 16-byte groups of columns
            const int c0 = 16 * g;
            if (c0 >= A) break;
            if (c0 + 16 <= A && (al & 15) == 0) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(av + c0));
                w[4 * g] = v.x; w[4 * g + 1] = v.y; w[4 * g + 2] = v.z; w[4 * g + 3] = v.w;
            } else if (c0 + 16 <= A && (al & 7) == 0) {
                const uint2 v0 = __ldg(reinterpret_cast<const uint2*>(av + c0)), v1 = __ldg(reinterpret_cast<const uint2*>(av + c0 + 8));
                w[4 * g] = v0.x; w[4 * g + 1] = v0.y; w[4 * g + 2] = v1.x; w[4 * g + 3] = v1.y;
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = c0 + 4 * k;
                    if (c + 4 <= A && (al & 3) == 0) w[4 * g + k] = __ldg(reinterpret_cast<const uint32_t*>(av + c));
                    else {
#pragma unroll
                        for (int e = 0; e < 4; ++e)
                            if (c + e < A) w[4 * g + k] |= (uint32_t)__ldg(av + c + e) << (8 * e);
                    }
                }
            }
        }
    }
    __device__ __forceinline__ bool ok(int a) const { return ((w[a >> 2] >> (8 * (a & 3))) & 0xffu) != 0u; }
};

template <int AVB>
__global__ void __launch_bounds__(qs::THREADS, 2) q_select_kernel(QSelectParams P) {
    using namespace qs;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    float* bias = reinterpret_cast<float*>(smem + BIAS);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BARS);
    uint64_t* w_full = bars;
    uint64_t* full = bars + 1;               // [STAGES]
    uint64_t* empty = bars + 1 + STAGES;     // [STAGES]
    uint64_t* tfull = bars + 1 + 2 * STAGES; // [2]
    uint64_t* tempty = tfull + 2;            // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int A_pad = (P.A + 15) & ~15;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
        fence_barrier_init();
    }
    if (warp == 4) tmem_alloc(tmem_slot, 256);
    for (int i = threadIdx.x; i < 128; i += THREADS) {
        const int a = i & 63;
        bias[i] = a < P.A ? (i < 64 ? P.b2_on[a] : P.b2_tg[a]) : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int64_t n_items = P.items ? (int64_t)__ldg(P.n_live) : (int64_t)P.T * P.n_tiles;

    if (warp == 5) {
        if (lane == 0) {
            mbar_arrive_expect_tx(w_full, 2 * 8192);
            bulk_copy_g2s(smem + W2ON, P.w2_on_img, 8192, w_full);
            bulk_copy_g2s(smem + W2TG, P.w2_tg_img, 8192, w_full);
            uint32_t it = 0;
            for (int64_t k = blockIdx.x; k < n_items; k += gridDim.x, ++it) {
                const int64_t item = P.items ? (int64_t)__ldg(P.items + k) : k;
                const int s = it % STAGES;
                mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
                mbar_arrive_expect_tx(&full[s], STAGE_BYTES);
                uint8_t* st = smem + STG + s * STAGE_BYTES;
                // item = t * n_tiles + tile ; h_t lives in slot t + 1
                bulk_copy_g2s(st, P.h_on_ti + (item + P.n_tiles) * TILE_BYTES2, TILE_BYTES2, &full[s]);
                bulk_copy_g2s(st + TILE_BYTES2, P.h_tg_ti + (item + P.n_tiles) * TILE_BYTES2, TILE_BYTES2, &full[s]);
            }
        }
    } else if (warp == 4) {
        if (lane == 0) {
            const uint32_t w_on = smem_u32(smem + W2ON), w_tg = smem_u32(smem + W2TG);
            const uint32_t idq = umma_idesc_bf16(128, A_pad, 0, 0);
            mbar_wait(w_full, 0);
            uint32_t it = 0;
            for (int64_t item = blockIdx.x; item < n_items; item += gridDim.x, ++it) {
                const int s = it % STAGES, b = it & 1;
                mbar_wait(&full[s], (it / STAGES) & 1);
                mbar_wait(&tempty[b], ((it >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t st = smem_u32(smem + STG + s * STAGE_BYTES);
                const uint32_t tm = tmem_base + 128 * b;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                    umma_bf16(tm, umma_desc_sw128(st + kk * 32, 16, 1024), umma_desc_sw128(w_on + kk * 32, 16, 1024), idq,
                              kk != 0);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                    umma_bf16(tm + 64, umma_desc_sw128(st + TILE_BYTES2 + kk * 32, 16, 1024),
                              umma_desc_sw128(w_tg + kk * 32, 16, 1024), idq, kk != 0);
                umma_commit(&empty[s]);
                umma_commit(&tfull[b]);
            }
        }
    } else {
        // ===== epilogue: one row per thread =====
        const uint32_t r = (uint32_t)(warp * 32 + lane);
        const uint32_t tl = tmem_base + ((uint32_t)(warp * 32) << 16);
        const bool vec_ok = (P.A & 3) == 0 && (P.avail_sb & 3) == 0 && (reinterpret_cast<uintptr_t>(P.avail) & 15) == 0;
        const uint32_t bias_s = smem_u32(bias);
        uint32_t it = 0;
        for (int64_t k = blockIdx.x; k < n_items; k += gridDim.x, ++it) {
            const int64_t item = P.items ? (int64_t)__ldg(P.items + k) : k;
            const int b2 = it & 1;
            const int t = (int)((uint32_t)item / (uint32_t)P.n_tiles);           // T * n_tiles < 2^31
            const int tile = (int)item - t * P.n_tiles;
            const int64_t p = (int64_t)tile * TILE_ROWS2 + r;
            const bool valid = p < P.R;
            const int64_t b = valid ? (int64_t)((uint32_t)p / (uint32_t)P.N) : 0;
            const int n = valid ? (int)(p - b * P.N) : 0;
            // issue the index / avail loads before waiting for the accumulator
            int a_taken = -1;
            const int64_t be = ep_row(P.ep_index, b);
            if (valid && t < P.T - 1) a_taken = (int)__ldg(P.actions + be * P.actions_sb + (int64_t)t * P.N + n);
            const void* av = static_cast<const uint8_t*>(P.avail) + (be * P.avail_sb + ((int64_t)t * P.N + n) * P.A) * AVB;
            const bool want_t = valid && t >= 1;
            // the whole avail row goes to registers (16-byte loads when the layout allows); columns >= A read as 0
            AvailRow<AVB> avr;
            avr.load(av, want_t, P.A, vec_ok);
            mbar_wait(&tfull[b2], (it >> 1) & 1);
            tc_fence_after();
            // padding columns (a >= A) have zero weights, zero bias and avail = 0: they are masked like unavailable
            // actions and can never win the arg-max against column 0 (strict >), so the loop needs no a < A tests
            float best = -INFINITY, chosen = 0.f, tsel = 0.f, mt0 = 0.f;
            int bidx = 0x7fffffff;
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const int c0 = 16 * cc;
                if (c0 < A_pad) {
                    uint32_t von[16], vtg[16];
                    ld_tmem_16(tl + 128 * b2 + c0, von);
                    ld_tmem_16(tl + 128 * b2 + 64 + c0, vtg);
                    float bo[16], bt[16];
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        lds_v4(bias_s + 4 * (c0 + 4 * j4), *reinterpret_cast<float(*)[4]>(&bo[4 * j4]));
                        lds_v4(bias_s + 256 + 4 * (c0 + 4 * j4), *reinterpret_cast<float(*)[4]>(&bt[4 * j4]));
                    }
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int a = c0 + j;
                        const float q_on = __uint_as_float(von[j]) + bo[j];
                        const float q_tg = __uint_as_float(vtg[j]) + bt[j];
                        chosen = a == a_taken ? q_on : chosen;
                        const bool ok = avr.ok(a);
                        const float mt = ok ? q_tg : kMaskValue;
                        const float v = P.double_q ? (ok ? q_on : kMaskValue) : mt;
                        if (a == 0) mt0 = mt;
                        if (v > best) { best = v; bidx = a; tsel = mt; }          // ascending a, strict >: lowest index wins
                    }
                    if (P.q_on_out != nullptr && valid) {                        // tests / diagnostics only
                        float* qo = P.q_on_out + ((int64_t)t * P.R + p) * P.A;
                        float* qt = P.q_tg_out + ((int64_t)t * P.R + p) * P.A;
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (c0 + j < P.A) { qo[c0 + j] = __uint_as_float(von[j]) + bo[j]; qt[c0 + j] = __uint_as_float(vtg[j]) + bt[j]; }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[b2]);
            if (valid && t < P.T - 1) P.chosen[(b * (P.T - 1) + t) * P.N + n] = chosen;
            if (want_t) {
                if (bidx >= P.A) { tsel = mt0; best = -INFINITY; }   // all-NaN row: index 0, as target_select_kernel
                P.tmax[(b * (P.T - 1) + (t - 1)) * P.N + n] = P.double_q ? tsel : best;
            }
        }
        if (P.tile_steps) {
            // the items the schedule left out: chosen of step t and tmax of step t - 1 are 0 there.  The mixers and the loss
            // read every (b, t) and the loss multiplies by a zero mask, so these entries must be finite; 0 is the cheapest.
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
                const int64_t p = (int64_t)tile * TILE_ROWS2 + r;
                if (p >= P.R) continue;
                const int64_t b = (int64_t)((uint32_t)p / (uint32_t)P.N);
                const int n = (int)(p - b * P.N);
                float* ch = P.chosen + b * (P.T - 1) * P.N + n;
                float* tm = P.tmax + b * (P.T - 1) * P.N + n;
                for (int t = __ldg(P.tile_steps + tile); t < P.T; ++t) {
                    if (t < P.T - 1) ch[(int64_t)t * P.N] = 0.f;
                    if (t >= 1) tm[(int64_t)(t - 1) * P.N] = 0.f;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 256);
    }
}


// ------------------------------------------------------------------------------------------
// backward recurrence (BPTT), one tile per CTA, double-buffered bulk-copied inputs
// ------------------------------------------------------------------------------------------
//   stage buffer (80 KB): [r | z | n | hn | h_prev] tile images of step t, brought in by two bulk copies; x_t in a
//   sixth, single-buffered slot (refilled as soon as the step's MMAs have completed, prefetched into L2 a step ahead).
//   The gate gradients are written IN PLACE (dr -> r, dz -> z, dn -> n, dn*r -> hn: every thread overwrites exactly
//   the elements it has just read) and are (a) the K-major A operands of 24 tcgen05.mma (dx = dg . W_ih, dh_rec =
//   dg' . W_hh; B = the weight images read MN-major), (b) the MN-major A operands of the weight-gradient MMAs
//   [da_r|da_z]^T [x|h_prev] and [da_n|da_n r]^T [x|h_prev] (N = 128: the x slot and the h_prev slot as two 64-column
//   blocks of one B operand) and of the bias column sums (B = a block of ones), accumulated over the whole kernel in
//   288 TMEM columns.  They never go to HBM; the only store per step is dpre1 = relu'(x) dx, staged in the h_prev
//   slot.  dh stays in fp32 registers; the fc2.weight row of the step's action comes out of the bf16 image in global
//   memory (L1), fetched one step ahead.
__device__ __forceinline__ uint32_t (&ax_lo(uint32_t (&v)[32]))[16] { return *reinterpret_cast<uint32_t (*)[16]>(&v[0]); }
__device__ __forceinline__ uint32_t (&ax_hi(uint32_t (&v)[32]))[16] { return *reinterpret_cast<uint32_t (*)[16]>(&v[16]); }

namespace b2 {
// 227 KB of shared memory, to the byte: both weight images (48 KB), ONE x slot (16 KB), two 5-tile stages (160 KB), a
// 2 KB block of ones (bias column sums on the tensor core) and the barriers.  There is no room for the usual 1 KB of
// alignment slack: the kernel has no static shared memory, so the dynamic window starts 1024-aligned (checked, traps).
constexpr int WIH = 0, WHH = 24576;
constexpr int XS = 49152;                          // x_t tile (single slot: only the weight-gradient MMAs read it)
constexpr int BUF = XS + TILE_BYTES2;              // [2][5][16 KB]   r | z | n | hn | h_prev
constexpr int BUF_BYTES = 5 * TILE_BYTES2;
constexpr int ONES = BUF + 2 * BUF_BYTES;          // bf16 1.0, 16 rows x 128 B
constexpr int BARS = ONES + 2048;
constexpr int SMEM_BYTES = BARS + 128;
constexpr int N_EPI_WARPS = 8, MMA_WARP = 8, IO_WARP = 9;
constexpr int THREADS = 320;
// per-tile partial: weight_ih [192][64] | weight_hh [192][64] | bias r,z (ih = hh) [128] | bias_ih n [64] | bias_hh n [64]
constexpr int PARTIAL_FLOATS = 2 * 192 * 64 + 256;
static_assert(SMEM_BYTES <= 232448, "gru_bwd2 shared memory");
}  // namespace b2

struct GruBwd2Params {
    const __nv_bfloat16* w_ih_img;
    const __nv_bfloat16* w_hh_img;
    const uint8_t* w2_img;           // fc2.weight image: row a at a * 128 B, 16-byte chunk j at (j ^ (a & 7))
    const uint8_t* x_ti;             // [T][n_tiles][16 KB]       x_t = relu(fc1), the GRU input (weight_ih gradient operand)
    const uint8_t* h_ti;             // [(T+1)][n_tiles][16 KB]   slot t = h_{t-1}
    const uint8_t* g_ti;             // [T][n_tiles][4][16 KB]    r, z, n, hn of the forward pass
    uint8_t* dpre1_ti;               // [T][n_tiles][16 KB]
    const uint32_t* relu_mask;       // [T][n_tiles][2][128]: bit j of word (half, row) = fc1 output column 32*half + j > 0
    const float* d_chosen;           // [B][T-1][N]
    const int64_t* actions; int64_t actions_sb;
    const int64_t* ep_index;         // optional batch row -> buffer episode
    float* partial;                  // [n_tiles][b2::PARTIAL_FLOATS]
    int64_t R;
    int T, N, A, n_tiles;
    // optional (padded-step skipping): tile `tile` runs steps t = tile_steps[tile] - 1 .. 0 only.  dh = 0 at the start is
    // exact: d_chosen is 0 for every row of the tile at every later step.  A tile with no steps writes zero partials.
    const int32_t* tile_steps;
};

// BPTT through the GRU over one 128-row tile, fused with ALL recurrent weight gradients: per step the gate gradients
// are written in place over the stashed gates and feed (a) 24 MMAs for dx and the recurrent part of dh_prev, (b) 16
// MMAs [da_r|da_z]^T [x|h_prev] and [da_n|da_n r]^T [x|h_prev] (M = 128 gate columns, N = 128, K = the tile's 128 rows)
// whose TMEM accumulators live for the whole kernel, (c) 16 N=16 MMAs against a block of ones for the bias column sums.
// The gate gradients never reach HBM.
__global__ void __launch_bounds__(b2::THREADS, 1) gru_bwd2_kernel(GruBwd2Params P) {
    using namespace b2;
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BARS);
    uint64_t* w_full = bars;
    uint64_t* in_full = bars + 1;            // [2]  stage buffer landed
    uint64_t* x_full = bars + 3;             // x slot landed
    uint64_t* dg_ready = bars + 4;           // gate gradients written (8 warps)
    uint64_t* mma_done = bars + 5;
    uint64_t* dp_ready = bars + 6;           // dpre1 staged (8 warps)
    uint64_t* ld_done = bars + 7;            // dx / dh_rec read out of TMEM (8 warps)
    uint64_t* dw_done = bars + 8;            // weight-gradient MMAs of the step complete: its six tiles are dead
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x;
    const int steps = P.tile_steps ? __ldg(P.tile_steps + tile) : P.T;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        mbar_init(&in_full[0], 1); mbar_init(&in_full[1], 1); mbar_init(x_full, 1);
        mbar_init(dg_ready, N_EPI_WARPS); mbar_init(mma_done, 1); mbar_init(dp_ready, N_EPI_WARPS);
        mbar_init(ld_done, N_EPI_WARPS); mbar_init(dw_done, 1);
        fence_barrier_init();
    }
    if (warp == MMA_WARP) tmem_alloc(tmem_slot, 512);
    if (threadIdx.x < 128)
        reinterpret_cast<uint4*>(smem + ONES)[threadIdx.x] = make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // epilogue-warp coordinates (used again in the common tail): warp w owns rows 32 (w & 3) .. +31 and hidden
    // columns 32 ((w >> 2) & 1) .. +31
    const int q4 = warp & 3, ch = (warp >> 2) & 1;
    const uint32_t r = (uint32_t)(q4 * 32 + lane);
    const uint32_t tlane = tmem_base + ((uint32_t)(q4 * 32) << 16) + 32 * ch;

    if (steps == 0) {
        // no live step: zero partials for gru_bwd2_reduce_kernel
        for (int i = threadIdx.x; i < PARTIAL_FLOATS; i += THREADS) P.partial[(int64_t)tile * PARTIAL_FLOATS + i] = 0.f;
    } else if (warp == IO_WARP) {
        if (lane == 0) {
            mbar_arrive_expect_tx(w_full, 2 * 24576);
            bulk_copy_g2s(smem + WIH, P.w_ih_img, 24576, w_full);
            bulk_copy_g2s(smem + WHH, P.w_hh_img, 24576, w_full);
            auto load = [&](int i) {                            // step index i <-> t = T-1-i, buffer i & 1
                const int t = steps - 1 - i;
                const int64_t tt = (int64_t)t * P.n_tiles + tile;
                uint8_t* buf = smem + BUF + (i & 1) * BUF_BYTES;
                mbar_arrive_expect_tx(&in_full[i & 1], BUF_BYTES);
                bulk_copy_g2s(buf, P.g_ti + tt * 4 * TILE_BYTES2, 4 * TILE_BYTES2, &in_full[i & 1]);
                bulk_copy_g2s(buf + 4 * TILE_BYTES2, P.h_ti + tt * TILE_BYTES2, TILE_BYTES2, &in_full[i & 1]);
            };
            auto load_x = [&](int i) {
                const int64_t tt = (int64_t)(steps - 1 - i) * P.n_tiles + tile;
                mbar_arrive_expect_tx(x_full, TILE_BYTES2);
                bulk_copy_g2s(smem + XS, P.x_ti + tt * TILE_BYTES2, TILE_BYTES2, x_full);
                if (i + 1 < steps)                                // the next one comes out of L2
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(P.x_ti + (tt - P.n_tiles) * TILE_BYTES2),
                                 "r"((uint32_t)TILE_BYTES2) : "memory");
            };
            auto prefetch = [&](int i) {                        // stage i into L2: its buffer frees late, the copy must be short
                const int64_t tt = (int64_t)(steps - 1 - i) * P.n_tiles + tile;
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(P.g_ti + tt * 4 * TILE_BYTES2),
                             "r"((uint32_t)(4 * TILE_BYTES2)) : "memory");
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(P.h_ti + tt * TILE_BYTES2),
                             "r"((uint32_t)TILE_BYTES2) : "memory");
            };
            load(0);
            load_x(0);
            if (steps > 1) load(1);
            if (steps > 2) prefetch(2);
            for (int i = 0; i < steps; ++i) {
                if (i + 3 < steps) prefetch(i + 3);
                const int64_t tt = (int64_t)(steps - 1 - i) * P.n_tiles + tile;
                uint8_t* buf = smem + BUF + (i & 1) * BUF_BYTES;
                mbar_wait(dw_done, (uint32_t)(i & 1));          // the x slot is free: refill it first
                if (i + 1 < steps) load_x(i + 1);
                mbar_wait(dp_ready, (uint32_t)(i & 1));
                bulk_copy_s2g(P.dpre1_ti + tt * TILE_BYTES2, buf + 4 * TILE_BYTES2, TILE_BYTES2);
                bulk_commit_group();
                bulk_wait_group_read<0>();                     // buffer i & 1 is free again
                if (i + 2 < steps) load(i + 2);
            }
            bulk_wait_group<0>();
        }
    } else if (warp == MMA_WARP) {
        if (lane == 0) {
            const uint32_t wih = smem_u32(smem + WIH), whh = smem_u32(smem + WHH);
            const uint32_t xs = smem_u32(smem + XS), ones = smem_u32(smem + ONES);
            const uint32_t idesc = umma_idesc_bf16(128, 64, 0, 1);          // A K-major, B MN-major
            const uint32_t idesc2 = umma_idesc_bf16(128, 128, 0, 1);
            const uint32_t idesc_dw = umma_idesc_bf16(128, 128, 1, 1);      // both MN-major: reduction over the 128 rows
            const uint32_t idesc_b = umma_idesc_bf16(128, 16, 1, 1);
            const uint64_t b_one = umma_desc_sw128(ones, TILE_BYTES2, 1024);
            mbar_wait(w_full, 0);
            for (int i = 0; i < steps; ++i) {
                const uint32_t dg = smem_u32(smem + BUF + (i & 1) * BUF_BYTES);
                const uint32_t xh_lbo = dg + 4 * TILE_BYTES2 - xs;          // [x | h_prev]: two 64-column blocks this far apart
                mbar_wait(dg_ready, (uint32_t)(i & 1));
                tc_fence_after();
                // [dx | dh_rec] = da_r [W_ir | W_hr] + da_z [W_iz | W_hz]: the r and z gate gradients feed both products, so the
                // two weight images are read as ONE N = 128 operand (W_ih block, W_hh block 24 KB further)
#pragma unroll
                for (int g = 0; g < 2; ++g)
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16(tmem_base, umma_desc_sw128(dg + g * TILE_BYTES2 + kk * 32, 16, 1024),
                                  umma_desc_sw128(wih + g * 8192 + kk * 2048, WHH - WIH, 1024), idesc2, (g | kk) != 0);
                // dx += da_n W_in ;  dh_rec += (da_n r) W_hn
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    umma_bf16(tmem_base, umma_desc_sw128(dg + 2 * TILE_BYTES2 + kk * 32, 16, 1024),
                              umma_desc_sw128(wih + 2 * 8192 + kk * 2048, 8192, 1024), idesc, 1);
                    umma_bf16(tmem_base + 64, umma_desc_sw128(dg + 3 * TILE_BYTES2 + kk * 32, 16, 1024),
                              umma_desc_sw128(whh + 2 * 8192 + kk * 2048, 8192, 1024), idesc, 1);
                }
                umma_commit(mma_done);
                // weight gradients, accumulated over all steps: [da_r|da_z]^T [x|h_prev], [da_n|da_n r]^T [x|h_prev], and
                // the column sums of the four gate-gradient tiles (biases).  Off the dh chain: issued once the epilogue has
                // read dx / dh_rec out of TMEM, they run while it does the gate-gradient math of the next step.
                mbar_wait(x_full, (uint32_t)(i & 1));
                mbar_wait(ld_done, (uint32_t)(i & 1));
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    const uint32_t acc = (i | kk) != 0;
                    const uint64_t b_xh = umma_desc_sw128(xs + kk * 2048, xh_lbo, 1024);
                    const uint64_t a_rz = umma_desc_sw128(dg + kk * 2048, TILE_BYTES2, 1024);
                    const uint64_t a_n = umma_desc_sw128(dg + 2 * TILE_BYTES2 + kk * 2048, TILE_BYTES2, 1024);
                    umma_bf16(tmem_base + 128, a_rz, b_xh, idesc_dw, acc);
                    umma_bf16(tmem_base + 256, a_n, b_xh, idesc_dw, acc);
                    umma_bf16(tmem_base + 384, a_rz, b_one, idesc_b, acc);
                    umma_bf16(tmem_base + 400, a_n, b_one, idesc_b, acc);
                }
                umma_commit(dw_done);
            }
        }
    } else {
        // ===== 8 warps: gate-gradient math, dh update =====
        const int64_t row = (int64_t)tile * TILE_ROWS2 + r;
        const bool valid = row < P.R;
        const int64_t b = valid ? row / P.N : 0;
        const int n = valid ? (int)(row - b * P.N) : 0;
        float dh[32], zk[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) dh[j] = 0.f;
        // per-step scalars and the fc2.weight row of the step's action (32 bf16 of this warp's column half), fetched one
        // step ahead
        auto fetch_dq = [&](int t) { return (valid && t >= 0 && t < P.T - 1) ? __ldg(P.d_chosen + (b * (P.T - 1) + t) * P.N + n) : 0.f; };
        const int64_t be = ep_row(P.ep_index, b);
        auto fetch_a = [&](int t) { return (valid && t >= 0 && t < P.T - 1) ? (int)__ldg(P.actions + be * P.actions_sb + (int64_t)t * P.N + n) : 0; };
        auto fetch_m = [&](int t) { return t >= 0 ? __ldg(P.relu_mask + (((int64_t)t * P.n_tiles + tile) * 2 + ch) * 128 + r) : 0u; };
        auto fetch_w2 = [&](int a, uint4 (&w)[4]) {
            const uint8_t* wr = P.w2_img + a * 128;
#pragma unroll
            for (int c = 0; c < 4; ++c)
                w[c] = __ldg(reinterpret_cast<const uint4*>(wr + (((uint32_t)(4 * ch + c) ^ ((uint32_t)a & 7u)) << 4)));
        };
        float dq = fetch_dq(steps - 1);
        uint32_t xm = fetch_m(steps - 1);
        uint4 w2[4];
        uint32_t dpk[16];                                       // dpre1 of the previous step (bf16 pairs), staged late
        fetch_w2(fetch_a(steps - 1), w2);
        int act_n = fetch_a(steps - 2);
        for (int i = 0; i < steps; ++i) {
            const int t = steps - 1 - i;
            uint8_t* buf = smem + BUF + (i & 1) * BUF_BYTES;
            const float dq_n = fetch_dq(t - 1);
            const uint32_t xm_n = fetch_m(t - 1);
            // chosen-action gradient enters through fc2: dh += dq * fc2_w[a, :]
            if (dq != 0.f) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const uint32_t ww[4] = {w2[c].x, w2[c].y, w2[c].z, w2[c].w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        dh[8 * c + 2 * k] = fmaf(dq, __uint_as_float(ww[k] << 16), dh[8 * c + 2 * k]);
                        dh[8 * c + 2 * k + 1] = fmaf(dq, __uint_as_float(ww[k] & 0xffff0000u), dh[8 * c + 2 * k + 1]);
                    }
                }
            }
            fetch_w2(act_n, w2);                                // row for step i + 1 (L1-resident table)
            act_n = fetch_a(t - 2);
            mbar_wait(&in_full[i & 1], (uint32_t)((i >> 1) & 1));
#pragma unroll
            for (int c = 0; c < 4; ++c) {                       // 4 chunks of 8 columns
                const uint32_t off = sw128_offset(r, (uint32_t)(4 * ch + c));
                const uint4 vr = *reinterpret_cast<const uint4*>(buf + off);
                const uint4 vz = *reinterpret_cast<const uint4*>(buf + TILE_BYTES2 + off);
                const uint4 vn = *reinterpret_cast<const uint4*>(buf + 2 * TILE_BYTES2 + off);
                const uint4 vh = *reinterpret_cast<const uint4*>(buf + 3 * TILE_BYTES2 + off);
                const uint4 vp = *reinterpret_cast<const uint4*>(buf + 4 * TILE_BYTES2 + off);
                const uint32_t wr_[4] = {vr.x, vr.y, vr.z, vr.w}, wz_[4] = {vz.x, vz.y, vz.z, vz.w};
                const uint32_t wn_[4] = {vn.x, vn.y, vn.z, vn.w}, wh_[4] = {vh.x, vh.y, vh.z, vh.w};
                const uint32_t wp_[4] = {vp.x, vp.y, vp.z, vp.w};
                uint32_t o_r[4], o_z[4], o_n[4], o_nr[4];
                const f32x2 ONE = f2_make(1.f, 1.f), M1 = f2_make(-1.f, -1.f);
#pragma unroll
                for (int k = 0; k < 4; ++k) {                   // two columns per iteration, packed fp32 pairs (FFMA2)
                    const int jj = 8 * c + 2 * k;
                    const f32x2 fr = f2_from_bf16x2(wr_[k]), fz = f2_from_bf16x2(wz_[k]), fn = f2_from_bf16x2(wn_[k]);
                    const f32x2 fhn = f2_from_bf16x2(wh_[k]), fhp = f2_from_bf16x2(wp_[k]);
                    const f32x2 d = f2_make(dh[jj], dh[jj + 1]);
                    const f32x2 omz = f2_fma(fz, M1, ONE);                              // 1 - z
                    const f32x2 omn2 = f2_fma(f2_mul(fn, fn), M1, ONE);                 // 1 - n^2
                    const f32x2 da_n = f2_mul(f2_mul(d, omz), omn2);
                    const f32x2 dr = f2_mul(f2_mul(f2_mul(da_n, fhn), fr), f2_fma(fr, M1, ONE));
                    const f32x2 dz = f2_mul(f2_mul(f2_mul(d, f2_fma(fn, M1, fhp)), fz), omz);
                    const f32x2 dnr = f2_mul(da_n, fr);
                    float a0, a1;
                    f2_split(dr, a0, a1); o_r[k] = pack_bf16x2(a0, a1);
                    f2_split(dz, a0, a1); o_z[k] = pack_bf16x2(a0, a1);
                    f2_split(da_n, a0, a1); o_n[k] = pack_bf16x2(a0, a1);
                    f2_split(dnr, a0, a1); o_nr[k] = pack_bf16x2(a0, a1);
                    f2_split(fz, zk[jj], zk[jj + 1]);
                }
                *reinterpret_cast<uint4*>(buf + off) = make_uint4(o_r[0], o_r[1], o_r[2], o_r[3]);
                *reinterpret_cast<uint4*>(buf + TILE_BYTES2 + off) = make_uint4(o_z[0], o_z[1], o_z[2], o_z[3]);
                *reinterpret_cast<uint4*>(buf + 2 * TILE_BYTES2 + off) = make_uint4(o_n[0], o_n[1], o_n[2], o_n[3]);
                *reinterpret_cast<uint4*>(buf + 3 * TILE_BYTES2 + off) = make_uint4(o_nr[0], o_nr[1], o_nr[2], o_nr[3]);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(dg_ready);

            // dpre1 of the previous step goes to its h_prev slot now: the weight-gradient MMAs that read the slot ran
            // during the math above
            auto stage_dp = [&](int ip) {
                uint8_t* hp = smem + BUF + (ip & 1) * BUF_BYTES + 4 * TILE_BYTES2;
                mbar_wait(dw_done, (uint32_t)(ip & 1));
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    *reinterpret_cast<uint4*>(hp + sw128_offset(r, (uint32_t)(4 * ch + c))) =
                        make_uint4(dpk[4 * c], dpk[4 * c + 1], dpk[4 * c + 2], dpk[4 * c + 3]);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(dp_ready);
            };
            if (i > 0) stage_dp(i - 1);

            mbar_wait(mma_done, (uint32_t)(i & 1));
            tc_fence_after();
            {
                uint32_t ax[32], ah[32];
                ld_tmem_16(tlane, ax_lo(ax));
                ld_tmem_16(tlane + 16, ax_hi(ax));
                ld_tmem_16(tlane + 64, ax_lo(ah));
                ld_tmem_16(tlane + 80, ax_hi(ah));
                tmem_wait_ld();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(ld_done);
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    const float d0 = (xm >> j) & 1u ? __uint_as_float(ax[j]) : 0.f;
                    const float d1 = (xm >> (j + 1)) & 1u ? __uint_as_float(ax[j + 1]) : 0.f;
                    dpk[j >> 1] = pack_bf16x2(d0, d1);
                    dh[j] = fmaf(dh[j], zk[j], __uint_as_float(ah[j]));
                    dh[j + 1] = fmaf(dh[j + 1], zk[j + 1], __uint_as_float(ah[j + 1]));
                }
            }
            if (i == steps - 1) stage_dp(i);
            dq = dq_n; xm = xm_n;
        }
    }
    // ---- end of the tile: every role is done (all MMAs complete, the IO thread has drained its bulk stores) ----
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp < N_EPI_WARPS && steps > 0) {
        // accumulator row = gate column (r < 64: first gate of the pair, else the second), accumulator columns 0..63 =
        // x columns (weight_ih), 64..127 = h_{t-1} columns (weight_hh): warp half ch takes the x resp. the h block
        float* part = P.partial + (int64_t)tile * PARTIAL_FLOATS;
        float* w = part + (ch ? 192 * 64 : 0);
        const uint32_t tl = tmem_base + ((uint32_t)(q4 * 32) << 16);
        const bool n_row = ch == 0 ? r < 64 : r >= 64;           // [da_n]^T x  resp.  [da_n r]^T h_prev
        float* o1 = w + (int64_t)r * 64;                          // rows r (0..63), z (64..127)
        float* o2 = w + (int64_t)(128 + (r & 63)) * 64;           // rows n
#pragma unroll
        for (int sc = 0; sc < 4; ++sc) {
            uint32_t a1[16], a2[16];
            ld_tmem_16(tl + 128 + 64 * ch + 16 * sc, a1);
            ld_tmem_16(tl + 256 + 64 * ch + 16 * sc, a2);
            tmem_wait_ld();
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
                *reinterpret_cast<float4*>(o1 + 16 * sc + 4 * j4) =
                    make_float4(__uint_as_float(a1[4 * j4]), __uint_as_float(a1[4 * j4 + 1]), __uint_as_float(a1[4 * j4 + 2]),
                                __uint_as_float(a1[4 * j4 + 3]));
                if (n_row)
                    *reinterpret_cast<float4*>(o2 + 16 * sc + 4 * j4) =
                        make_float4(__uint_as_float(a2[4 * j4]), __uint_as_float(a2[4 * j4 + 1]),
                                    __uint_as_float(a2[4 * j4 + 2]), __uint_as_float(a2[4 * j4 + 3]));
            }
        }
        if (ch == 0) {
            uint32_t b1[8], b2_[8];
            ld_tmem_8(tl + 384, b1);
            ld_tmem_8(tl + 400, b2_);
            tmem_wait_ld();
            float* bias = part + 2 * 192 * 64;
            bias[r] = __uint_as_float(b1[0]);                     // r, z: bias_ih = bias_hh
            bias[128 + r] = __uint_as_float(b2_[0]);              // 128..191 bias_ih[n], 192..255 bias_hh[n]
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_WARP) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// rnn gradients from the per-tile partials of gru_bwd2.  Block = 32 outputs x 8 slices of the tile range; fixed summation
// order (slice-local ascending, then slices ascending): deterministic
__global__ void __launch_bounds__(256) gru_bwd2_reduce_kernel(const float* __restrict__ partial, int n_part, float* __restrict__ w_ih,
                                                              float* __restrict__ w_hh, float* __restrict__ b_ih,
                                                              float* __restrict__ b_hh) {
    constexpr int PF = b2::PARTIAL_FLOATS;
    __shared__ float red[8][33];
    const int o = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + o;
    const int per = (n_part + 7) / 8;
    const int c0 = sl * per, c1 = c0 + per < n_part ? c0 + per : n_part;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (i < PF) {
        int c = c0;
        for (; c + 4 <= c1; c += 4) {
            s0 += partial[(int64_t)c * PF + i];
            s1 += partial[(int64_t)(c + 1) * PF + i];
            s2 += partial[(int64_t)(c + 2) * PF + i];
            s3 += partial[(int64_t)(c + 3) * PF + i];
        }
        for (; c < c1; ++c) s0 += partial[(int64_t)c * PF + i];
    }
    red[sl][o] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (sl != 0 || i >= PF) return;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][o];
    if (i < 192 * 64) w_ih[i] = s;
    else if (i < 2 * 192 * 64) w_hh[i - 192 * 64] = s;
    else {
        const int k = i - 2 * 192 * 64;
        if (k < 128) { b_ih[k] = s; b_hh[k] = s; }
        else if (k < 192) b_ih[k] = s;
        else b_hh[k - 64] = s;
    }
}

}  // namespace tc

int tc_gru_fwd2(const __nv_bfloat16* w_ih_img, const __nv_bfloat16* w_hh_img, const float* b_ih, const float* b_hh,
                const uint8_t* x_ti, uint8_t* h_ti, uint8_t* g_ti, int64_t R, int nt, int n_tiles, cudaStream_t s,
                int tiles_per_cta, const int32_t* tile_steps) {
    tc::GruFwd2Params P;
    P.w_ih_img = w_ih_img; P.w_hh_img = w_hh_img; P.b_ih = b_ih; P.b_hh = b_hh;
    P.x_ti = x_ti; P.h_ti = h_ti; P.g_ti = g_ti; P.R = R; P.nt = nt; P.n_tiles = n_tiles;
    P.tiles_per_cta = tiles_per_cta == 1 ? 1 : 2;
    P.tile_steps = tile_steps;
    PMB_SMEM_ATTR(tc::gru_fwd2_kernel, tc::g2::SMEM_BYTES);
    tc::gru_fwd2_kernel<<<(n_tiles + P.tiles_per_cta - 1) / P.tiles_per_cta, tc::g2::THREADS, tc::g2::SMEM_BYTES, s>>>(P);
    PMB_LAUNCH_CHECK("gru_fwd2_kernel");
    return PMB_OK;
}

int tc_q_select(const pmb_dims* d, const pmb_batch* b, const __nv_bfloat16* w2_on_img, const __nv_bfloat16* w2_tg_img,
                const float* b2_on, const float* b2_tg, const uint8_t* h_on_ti, const uint8_t* h_tg_ti, int n_tiles,
                float* chosen, float* tmax, float* q_on_out, float* q_tg_out, cudaStream_t s, const int32_t* live_items,
                const int32_t* n_live, const int32_t* tile_steps) {
    tc::QSelectParams P;
    P.w2_on_img = w2_on_img; P.w2_tg_img = w2_tg_img; P.b2_on = b2_on; P.b2_tg = b2_tg;
    P.h_on_ti = h_on_ti; P.h_tg_ti = h_tg_ti;
    P.avail = b->avail; P.avail_sb = b->avail_sb; P.actions = b->actions; P.actions_sb = b->actions_sb;
    P.ep_index = b->ep_index;
    P.chosen = chosen; P.tmax = tmax; P.q_on_out = q_on_out; P.q_tg_out = q_tg_out;
    P.R = (int64_t)d->B * d->N; P.T = d->T; P.N = d->N; P.A = d->A; P.n_tiles = n_tiles; P.double_q = d->double_q;
    P.items = live_items; P.n_live = n_live; P.tile_steps = tile_steps;
    const int64_t n_items = (int64_t)d->T * n_tiles;
    int grid = 2 * sm_count();
    if (grid > n_items) grid = (int)n_items;
    if (b->avail_dtype == PMB_DTYPE_U8) {
        PMB_SMEM_ATTR(tc::q_select_kernel<1>, tc::qs::SMEM_BYTES);
        tc::q_select_kernel<1><<<grid, tc::qs::THREADS, tc::qs::SMEM_BYTES, s>>>(P);
    } else {
        PMB_SMEM_ATTR(tc::q_select_kernel<4>, tc::qs::SMEM_BYTES);
        tc::q_select_kernel<4><<<grid, tc::qs::THREADS, tc::qs::SMEM_BYTES, s>>>(P);
    }
    PMB_LAUNCH_CHECK("q_select_kernel");
    return PMB_OK;
}

int64_t tc_gru_bwd2_partial_bytes(int n_tiles) {
    return align_up((int64_t)n_tiles * tc::b2::PARTIAL_FLOATS * 4, 256);
}

int tc_gru_bwd2(const __nv_bfloat16* w_ih_img, const __nv_bfloat16* w_hh_img, const __nv_bfloat16* w2_img,
                const uint8_t* x_ti, const uint8_t* h_ti, const uint8_t* g_ti, uint8_t* dpre1_ti, const uint32_t* relu_mask,
                const float* d_chosen, const int64_t* actions, int64_t actions_sb, const int64_t* ep_index, int64_t R, int T,
                int N, int A, int n_tiles, float* partial, cudaStream_t s, const int32_t* tile_steps) {
    tc::GruBwd2Params P;
    P.w_ih_img = w_ih_img; P.w_hh_img = w_hh_img; P.w2_img = reinterpret_cast<const uint8_t*>(w2_img);
    P.x_ti = x_ti; P.h_ti = h_ti; P.g_ti = g_ti; P.dpre1_ti = dpre1_ti;
    P.relu_mask = relu_mask; P.d_chosen = d_chosen; P.actions = actions; P.actions_sb = actions_sb;
    P.partial = partial; P.ep_index = ep_index;
    P.R = R; P.T = T; P.N = N; P.A = A; P.n_tiles = n_tiles; P.tile_steps = tile_steps;
    PMB_SMEM_ATTR(tc::gru_bwd2_kernel, tc::b2::SMEM_BYTES);
    tc::gru_bwd2_kernel<<<n_tiles, tc::b2::THREADS, tc::b2::SMEM_BYTES, s>>>(P);
    PMB_LAUNCH_CHECK("gru_bwd2_kernel");
    return PMB_OK;
}

// rnn.weight_ih / weight_hh / bias_ih / bias_hh gradients out of the partials
int tc_gru_bwd2_reduce(const float* partial, int n_tiles, float* w_ih, float* w_hh, float* b_ih, float* b_hh, cudaStream_t s) {
    tc::gru_bwd2_reduce_kernel<<<(unsigned)ceil_div(tc::b2::PARTIAL_FLOATS, 32), 256, 0, s>>>(partial, n_tiles, w_ih, w_hh,
                                                                                              b_ih, b_hh);
    PMB_LAUNCH_CHECK("gru_bwd2_reduce_kernel");
    return PMB_OK;
}

}  // namespace pmb
