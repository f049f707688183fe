// bf16 tensor-core tier: the RNNAgent recurrence on tcgen05.
//
// Activations of this tier are stored as bf16 "tile images": a [rows x 64] matrix is cut into tiles of
// 128 rows; a tile is the exact shared-memory image of a K-major / 128-byte-swizzle UMMA operand
// (row r at byte r*128, 16-byte chunk j at ((j ^ (r & 7)) << 4)), 16 KB.  One bulk async copy brings
// a tile in, and the same bytes serve as K-major A operand (forward) and as MN-major operand (weight
// gradients) - only the descriptor changes.
//
//   gru_rollout: the ROLLOUT step kernel (fp32 hidden state in and out, fc2 and the epsilon-greedy selection inside):
//                one persistent CTA per SM with two 128-row tiles in flight, W_ih / W_hh / fc2 images resident in shared
//                memory, hidden state in fp32 registers and in a bf16 operand tile.  Per tile: 16 tcgen05.mma for the
//                gates (r|z fused over [x|h], n input part, n hidden part), gate math out of TMEM, 4 mma for fc2, q out
//                of TMEM.  (The learner step uses gru_fwd2 / gru_bwd2 / q_select in gru_tc2.cu.)
//   agent_dw_tc: fc1 / fc2 weight gradients as one image-fed GEMM kernel.  (The rnn.* gradients are accumulated
//                inside gru_bwd2, gru_tc2.cu.)
#include <cuda.h>
#include "common.cuh"
#include "tc_common.cuh"
#include "gru_tc.cuh"

namespace pmb {
namespace tc {

constexpr int TILE_ROWS = 128;
constexpr int TILE_BYTES = TILE_ROWS * 128;      // 16 KB

// sigmoid(x) = 0.5 tanh(0.5 x) + 0.5 : one MUFU op instead of ex2 + rcp (same form as gru_fwd2 in gru_tc2.cu, so the
// rollout step and the learner's unroll round identically)
__device__ __forceinline__ float fast_sigmoid(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(0.5f * x));
    return fmaf(0.5f, y, 0.5f);
}
__device__ __forceinline__ float fast_tanh(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }

// Philox4x32-10 and the (0, 1] mapping: identical to select.cu (the fused selection must draw the same numbers)
__device__ __forceinline__ uint4 gf_philox4x32_10(uint4 ctr, uint2 key) {
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
__device__ __forceinline__ float gf_u01(uint32_t x) { return ((float)(x >> 8) + 1.0f) * (1.0f / 16777216.0f); }

// position of the n-th (0-based) set bit of m; needs popc(m) > n.  Five popc steps instead of the fns.b32 emulation.
__device__ __forceinline__ int nth_set_bit(uint32_t m, int n) {
    int pos = 0;
    int c = __popc(m & 0xffffu);
    if (n >= c) { n -= c; pos += 16; m >>= 16; }
    c = __popc(m & 0xffu);
    if (n >= c) { n -= c; pos += 8; m >>= 8; }
    c = __popc(m & 0xfu);
    if (n >= c) { n -= c; pos += 4; m >>= 4; }
    c = __popc(m & 0x3u);
    if (n >= c) { n -= c; pos += 2; m >>= 2; }
    c = (int)(m & 1u);
    if (n >= c) pos += 1;
    return pos;
}

// 16 fp32 values (columns 16c .. 16c+15 of row r) -> two 16-byte chunks of a tile image
__device__ __forceinline__ void store_row16(uint8_t* tile, uint32_t r, int c16, const float (&f)[16]) {
    uint4 a = make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
    uint4 b = make_uint4(pack_bf16x2(f[8], f[9]), pack_bf16x2(f[10], f[11]), pack_bf16x2(f[12], f[13]),
                         pack_bf16x2(f[14], f[15]));
    *reinterpret_cast<uint4*>(tile + sw128_offset(r, 2 * c16)) = a;
    *reinterpret_cast<uint4*>(tile + sw128_offset(r, 2 * c16 + 1)) = b;
}
__device__ __forceinline__ void load_row16(const uint8_t* tile, uint32_t r, int c16, float (&f)[16]) {
    uint4 a = *reinterpret_cast<const uint4*>(tile + sw128_offset(r, 2 * c16));
    uint4 b = *reinterpret_cast<const uint4*>(tile + sw128_offset(r, 2 * c16 + 1));
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) { f[2 * i] = bf16_lo(w[i]); f[2 * i + 1] = bf16_hi(w[i]); }
}

// ------------------------------------------------------------------------------------------
// rollout step: one GRU step + fc2 + epsilon-greedy selection for all rows
// ------------------------------------------------------------------------------------------
// One persistent CTA per SM with TWO tiles in flight (slots).  Everything a tile needs from HBM arrives by bulk copy
// while the other tile computes: the x tile image (one 16 KB bulk copy), the fp32 hidden state (two tensor-map copies,
// 128 rows x 32 columns each, landing 128-byte-swizzled so that the row-per-thread 16-byte accesses of the epilogue are
// conflict-free; rows beyond R arrive as zeros) and the avail rows (one bulk copy per env the tile touches).  The new
// hidden state goes back through the same staging tiles: each warp stages its 32 rows and writes them out with
// coalesced 16-byte stores.  Measured on the way: per-thread row-strided global accesses with 2 CTAs per SM and nothing
// prefetched (first version) 176 us for 16384 x 27 rows; one 256-byte bulk copy per row 320 us (the copy engine's
// per-operation cost); 16-byte cp.async by one loader warp 244 us (too few bytes in flight per warp).
// Warps 0-7 / 8-15: epilogue of slot 0 / 1 (TWO threads per row, 32 hidden columns each in fp32 registers: with one
// thread per row the 2 epilogue warps per scheduler could not hide the gate-math latencies), warp 16: MMA issuer, warp 17:
// loader, warp 18: avail loader.  What the per-role wait profile (tools/ro_role_profile.py) changed: a slot's chain per
// tile was loads -> h_0 operand -> 16 gate MMAs -> gate math -> new hidden state out -> fc2 -> q + selection, 14.5 k cycles,
// with the selection (one thread per row, 5.3 k cycles) and the wait for the gate MMAs (4.9 k) the longest links.  Now (1)
// the x halves of the gate MMAs are issued as soon as the tile's inputs have landed, before the epilogue has written the
// h_0 operand; (2) the two threads of a row split the q chunks / availability bits / Philox draws of the selection and
// the column-half-1 thread hands its partial result over through 16 bytes of shared memory and a 64-thread named barrier;
// the availability bits and the draws are computed BEFORE the fc2 MMAs are waited for; (3) the new hidden state leaves
// through the staging tiles with two tensor-map bulk STORES issued by the loader thread (rows beyond R are clipped by the
// tensor map) instead of 8 x (LDS + coalesced STG) per epilogue thread.
namespace ro {
constexpr int WIH = 0, WHH = 24576, W2 = 49152;
constexpr int SLOT0 = 57344;
constexpr int S_X = 0, S_HT = 16384, S_HS = 32768, S_AV = S_HS + 32768;      // S_HS: two fp32 tiles (columns 0-31, 32-63)
constexpr int AV_BYTES = 18432;                               // staged avail rows: 128 * A * 4 <= this (i32, A <= 36)
constexpr int AV8_SLACK = 48;                                 // u8: bytes per env run beyond its cells (av8_run)
constexpr int S_XC = S_AV + AV_BYTES;                         // 16 bytes per row: selection hand-over between the two threads of a row
constexpr int SLOT_BYTES = S_XC + 2048;                       // 86016 = 84 KB (multiple of 1024)
constexpr int BIAS = SLOT0 + 2 * SLOT_BYTES;
constexpr int BIAS_FLOATS = 128 + 64 + 64 + 64;               // brz | bin | bhn | b2
constexpr int BARS = BIAS + BIAS_FLOATS * 4;
constexpr int SMEM_BYTES = BARS + 256;                      // 17 barriers + the TMEM slot
constexpr int THREADS = 608;
constexpr int MMA_W = 16, LOAD_W = 17, AV_W = 18;
static_assert(SLOT_BYTES % 1024 == 0 && SMEM_BYTES <= 232448, "rollout kernel shared memory");
}  // namespace ro

// Per-role wait / phase accounting (build with PMB_EXTRA_NVCC_FLAGS=-DPMB_RO_PROFILE, read with tools/ro_role_profile.py)
#ifdef PMB_RO_PROFILE
__device__ unsigned long long g_ro_prof[16];
#define RWAIT(idx, bar, par) do { long long _t0 = clock64(); mbar_wait(bar, par); if (lane == 0) prof_acc[idx] += clock64() - _t0; } while (0)
#define RMARK(var) long long var = clock64()
#define RADD(idx, expr) do { if (lane == 0) prof_acc[idx] += (expr); } while (0)
#else
#define RWAIT(idx, bar, par) mbar_wait(bar, par)
#define RMARK(var)
#define RADD(idx, expr)
#endif
// u8 avail staging.  A bulk copy moves 16-byte-aligned, 16-byte-granular runs, and an env's N x A bytes (972 at 27m) are
// neither, so the loader copies the aligned superset of each env's run [lo, hi): every 16-byte word of it holds a byte
// of the run, so no word lies outside the allocation.  Env e of the tile (k = e - e0) lands at the 16-aligned
// dst = 16 floor(x / 16) + 48 k, x = (first row of e in the tile - row0) * A; with L <= len + 30 bytes per superset the
// next env starts at least len + 33 bytes later, so the runs never overlap, and the whole area is under
// 128 A + 48 (envs per tile).  A row's cells sit at dst + (start & 15) + (row - ra) A: same alignment as in memory.
struct Av8Run { const uint8_t* lo; uint32_t dst, bytes, phase; };
__device__ __forceinline__ Av8Run av8_run(const GruFwdParams& P, int64_t e, int64_t row0, int64_t row_end) {
    const int64_t ra = e * P.N > row0 ? e * P.N : row0;                        // rows of env e inside the tile
    const int64_t rb = (e + 1) * P.N < row_end ? (e + 1) * P.N : row_end;
    const uintptr_t start = reinterpret_cast<uintptr_t>(P.avail) + e * P.avail_sb + (ra - e * P.N) * P.A;
    const uintptr_t lo = start & ~(uintptr_t)15, hi = (start + (rb - ra) * P.A + 15) & ~(uintptr_t)15;
    const int64_t e0 = (int64_t)((uint32_t)row0 / (uint32_t)P.N);
    Av8Run run;
    run.lo = reinterpret_cast<const uint8_t*>(lo);
    run.dst = (uint32_t)((((ra - row0) * P.A) & ~(int64_t)15) + ro::AV8_SLACK * (e - e0));
    run.bytes = (uint32_t)(hi - lo);
    run.phase = (uint32_t)(start & 15);
    return run;
}

// availability bits of cells c0 .. c0 + 15 of a row (generic pointer: staged in shared memory or in global memory);
// cells >= A read as 0 and are not read.  vec (i32): the row is 16-byte aligned and A % 4 == 0.
template <int AVB>
__device__ __forceinline__ uint32_t avail_bits16(const uint8_t* row, int c0, int A, bool vec) {
    uint32_t oks = 0u;
    if (AVB == 4) {
        const int32_t* av = reinterpret_cast<const int32_t*>(row);
        int avj[16];
        if (vec && c0 + 16 <= A) {
#pragma unroll
            for (int j4 = 0; j4 < 4; ++j4) {
                const int4 w4 = *(reinterpret_cast<const int4*>(av + c0) + j4);
                avj[4 * j4] = w4.x; avj[4 * j4 + 1] = w4.y; avj[4 * j4 + 2] = w4.z; avj[4 * j4 + 3] = w4.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) avj[j] = c0 + j < A ? av[c0 + j] : 0;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) oks |= (avj[j] != 0 ? 1u : 0u) << j;
    } else {
        const uint8_t* av = row + c0;
        const uintptr_t al = reinterpret_cast<uintptr_t>(av);
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (c0 + 16 <= A && (al & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(av);
            w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = c0 + 4 * k;
                if (c + 4 <= A && (al & 3) == 0) w[k] = *reinterpret_cast<const uint32_t*>(av + 4 * k);
                else {
#pragma unroll
                    for (int e = 0; e < 4; ++e)
                        if (c + e < A) w[k] |= (uint32_t)av[4 * k + e] << (8 * e);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) oks |= (((w[j >> 2] >> (8 * (j & 3))) & 0xffu) != 0u ? 1u : 0u) << j;
    }
    return oks;
}

template <int AVB>
__global__ void __launch_bounds__(ro::THREADS, 1) gru_rollout_kernel(GruFwdParams P, int av_smem,
                                                                     const __grid_constant__ CUtensorMap tmap_h0,
                                                                     const __grid_constant__ CUtensorMap tmap_h1) {
#ifdef PMB_RO_PROFILE
    long long prof_acc[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    const long long prof_t0 = clock64();
#endif
    using namespace ro;
    extern __shared__ __align__(1024) uint8_t smem[];
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    float* bias = reinterpret_cast<float*>(smem + BIAS);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BARS);
    uint64_t* w_full = bars;
    uint64_t* in_full = bars + 1;        // [2] x tile and h_0 tiles landed
    uint64_t* xh_free = bars + 3;        // [2] x tile dead, new hidden state staged (8 epilogue warps): store it, refill the slot
    uint64_t* hb_ready = bars + 5;       // [2] bf16 h operand written: arrival pair per tile (h_0, then h_1)
    uint64_t* gates_full = bars + 7;     // [2]
    uint64_t* q_full = bars + 9;         // [2]
    uint64_t* tmem_free = bars + 11;     // [2] q drained (8 warps)
    uint64_t* av_full = bars + 13;       // [2] avail rows landed
    uint64_t* av_free = bars + 15;       // [2] selection done with the avail rows (8 warps)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 17);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int A_pad = (P.A + 15) & ~15;
    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&in_full[i], 1); mbar_init(&xh_free[i], 8); mbar_init(&hb_ready[i], 8);
            mbar_init(&av_full[i], 1); mbar_init(&av_free[i], 8);
            mbar_init(&gates_full[i], 1); mbar_init(&q_full[i], 1); mbar_init(&tmem_free[i], 8);
        }
        fence_barrier_init();
    }
    if (warp == MMA_W) tmem_alloc(tmem_slot, 512);
    for (int i = threadIdx.x; i < 128; i += THREADS) bias[i] = P.b_ih[i] + P.b_hh[i];
    for (int i = threadIdx.x; i < 64; i += THREADS) {
        bias[128 + i] = P.b_ih[128 + i];
        bias[192 + i] = P.b_hh[128 + i];
        bias[256 + i] = i < P.A ? P.b2[i] : 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_my = (P.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // tiles of this CTA
    // Programmatic dependent launch, both ways.  The next kernel of the stream (the streaming fc1 of the next rollout
    // step) may be scheduled onto SMs as the CTAs of this grid leave them; it waits before it overwrites the x images.
    // This kernel was itself scheduled while the fc1 of this step was finishing: everything above (barriers, TMEM,
    // biases - parameters, not written by fc1) ran under its tail; the two loader threads wait before the first byte of
    // x / hidden state / avail is fetched, and every other role only ever acts on what they fetched.
    pdl_launch_dependents();
#ifdef PMB_RO_PROFILE
    if (threadIdx.x == 0) prof_acc[13] = clock64() - prof_t0;      // prologue
#endif

    if (warp == LOAD_W) {
        // ===== loader =====
        if (lane == 0) {
            mbar_arrive_expect_tx(w_full, 24576 + 24576 + 8192);
            bulk_copy_g2s(smem + WIH, P.w_ih_img, 24576, w_full);
            bulk_copy_g2s(smem + WHH, P.w_hh_img, 24576, w_full);
            bulk_copy_g2s(smem + W2, P.w2_img, 8192, w_full);
        }
        // the staging of a slot is released in two steps (x / hidden state after the gate math, avail after the selection),
        // so the next tile's big copies are in flight while the current one still selects; avail has its own warp.
        // Use k of a slot starts by storing the new hidden state the slot's previous tile (k - 2) left in the staging tiles.
        if (lane == 0) {
            pdl_wait();
            for (int k = 0; k < n_my + 2; ++k) {
                const int s = k & 1, u = k >> 1;
                if (k >= 2 && k - 2 >= n_my) continue;
                const int64_t tile = (int64_t)blockIdx.x + (int64_t)k * gridDim.x;
                uint8_t* sl = smem + SLOT0 + s * SLOT_BYTES;
                RWAIT(0, &xh_free[s], (uint32_t)((u & 1) ^ 1));
                if (k >= 2 && P.h_last) {
                    const int64_t ptile = tile - 2 * (int64_t)gridDim.x;
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                                         reinterpret_cast<uint64_t>(&tmap_h1)),
                                     "r"(32 * hf), "r"((int)(ptile * TILE_ROWS)), "r"(smem_u32(sl + S_HS + hf * TILE_BYTES))
                                     : "memory");
                    bulk_commit_group();
                    bulk_wait_group_read<0>();                     // the staging tiles may be refilled
                }
                if (k >= n_my) continue;
                // the slot's NEXT tile into L2 now: its copies can only start when this tile's gate math is over, and the
                // chain math -> store -> load -> h_0 operand -> gate MMAs -> math of a slot is what bounds the kernel
                if (k + 2 < n_my) {
                    const int64_t ntile = tile + 2 * (int64_t)gridDim.x;
                    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(P.x_ti + ntile * TILE_BYTES), "r"(TILE_BYTES) : "memory");
                    if (P.h0) {
                        const int64_t nrow0 = ntile * TILE_ROWS;
                        const int64_t nrows = P.R - nrow0 < TILE_ROWS ? P.R - nrow0 : TILE_ROWS;
                        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(P.h0 + nrow0 * 64), "r"((uint32_t)(nrows * 256)) : "memory");
                    }
                }
                mbar_arrive_expect_tx(&in_full[s], TILE_BYTES + (P.h0 ? 2 * TILE_BYTES : 0));
                bulk_copy_g2s(sl + S_X, P.x_ti + tile * TILE_BYTES, TILE_BYTES, &in_full[s]);
                if (P.h0) {
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        asm volatile(
                            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                                smem_u32(sl + S_HS + hf * TILE_BYTES)),
                            "l"(reinterpret_cast<uint64_t>(&tmap_h0)), "r"(32 * hf), "r"((int)(tile * TILE_ROWS)),
                            "r"(smem_u32(&in_full[s]))
                            : "memory");
                }
            }
            bulk_wait_group<0>();                                  // the hidden-state stores have completed
        }
    } else if (warp == AV_W) {
        // ===== avail loader: one copy per env the tile touches (an env's N x A block is contiguous; the batch stride is free) =====
        if (av_smem) {
            pdl_wait();
            for (int k = 0; k < n_my; ++k) {
                const int s = k & 1, u = k >> 1;
                const int64_t tile = (int64_t)blockIdx.x + (int64_t)k * gridDim.x;
                uint8_t* sl = smem + SLOT0 + s * SLOT_BYTES;
                const int64_t row0 = tile * TILE_ROWS;
                const int rows_here = (int)(P.R - row0 < TILE_ROWS ? P.R - row0 : TILE_ROWS);
                RWAIT(1, &av_free[s], (uint32_t)((u & 1) ^ 1));
                const int64_t e0 = (int64_t)((uint32_t)row0 / (uint32_t)P.N);
                if (AVB == 4) {
                    if (lane == 0) mbar_arrive_expect_tx(&av_full[s], (uint32_t)(rows_here * P.A * 4));
                    __syncwarp();
                    const int32_t* avail = static_cast<const int32_t*>(P.avail);
                    for (int64_t e = e0 + lane; e * P.N < row0 + rows_here; e += 32) {
                        const int64_t ra = e * P.N > row0 ? e * P.N : row0;                  // rows of env e inside the tile
                        const int64_t rb = (e + 1) * P.N < row0 + rows_here ? (e + 1) * P.N : row0 + rows_here;
                        bulk_copy_g2s(sl + S_AV + (ra - row0) * P.A * 4, avail + e * P.avail_sb + (ra - e * P.N) * P.A,
                                      (uint32_t)((rb - ra) * P.A * 4), &av_full[s]);
                    }
                } else {
                    uint32_t bytes = 0;
                    for (int64_t e = e0 + lane; e * P.N < row0 + rows_here; e += 32) bytes += av8_run(P, e, row0, row0 + rows_here).bytes;
                    bytes = __reduce_add_sync(0xffffffffu, bytes);
                    if (lane == 0) mbar_arrive_expect_tx(&av_full[s], bytes);
                    __syncwarp();
                    for (int64_t e = e0 + lane; e * P.N < row0 + rows_here; e += 32) {
                        const Av8Run run = av8_run(P, e, row0, row0 + rows_here);
                        bulk_copy_g2s(sl + S_AV + run.dst, run.lo, run.bytes, &av_full[s]);
                    }
                }
            }
        }
    } else if (warp == MMA_W) {
        // ===== MMA issuer: gates of tile k, then fc2 of tile k-1 (its new hidden state is ready by then) =====
        if (lane == 0) {
            const uint32_t wih = smem_u32(smem + WIH), whh = smem_u32(smem + WHH), w2 = smem_u32(smem + W2);
            const uint32_t id128 = umma_idesc_bf16(128, 128, 0, 0), id64 = umma_idesc_bf16(128, 64, 0, 0);
            const uint32_t idq = umma_idesc_bf16(128, A_pad, 0, 0);
            auto fc2 = [&](int j) {
                const int s = j & 1;
                const uint32_t ht = smem_u32(smem + SLOT0 + s * SLOT_BYTES + S_HT);
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
                    umma_bf16(tmem_base + 256 * s, umma_desc_sw128(ht + kk * 32, 16, 1024), umma_desc_sw128(w2 + kk * 32, 16, 1024),
                              idq, kk != 0);
                umma_commit(&q_full[s]);
            };
            auto gates_x = [&](int k) {                            // the halves that only need the x tile
                const int s = k & 1;
                const uint32_t xt = smem_u32(smem + SLOT0 + s * SLOT_BYTES + S_X);
                const uint32_t tm = tmem_base + 256 * s;
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)                     // r|z : x . W_i{r,z}^T
                    umma_bf16(tm, umma_desc_sw128(xt + kk * 32, 16, 1024), umma_desc_sw128(wih + kk * 32, 16, 1024), id128,
                              kk != 0);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)                     // n, input part
                    umma_bf16(tm + 128, umma_desc_sw128(xt + kk * 32, 16, 1024),
                              umma_desc_sw128(wih + 16384 + kk * 32, 16, 1024), id64, kk != 0);
            };
            auto gates_h = [&](int k) {                            // the halves that need the h_0 operand; commits both
                const int s = k & 1;
                const uint32_t ht = smem_u32(smem + SLOT0 + s * SLOT_BYTES + S_HT);
                const uint32_t tm = tmem_base + 256 * s;
                tc_fence_after();
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)                     // r|z += h . W_h{r,z}^T
                    umma_bf16(tm, umma_desc_sw128(ht + kk * 32, 16, 1024), umma_desc_sw128(whh + kk * 32, 16, 1024), id128, 1);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)                     // n, hidden part
                    umma_bf16(tm + 192, umma_desc_sw128(ht + kk * 32, 16, 1024),
                              umma_desc_sw128(whh + 16384 + kk * 32, 16, 1024), id64, kk != 0);
                umma_commit(&gates_full[s]);
            };
            mbar_wait(w_full, 0);
            // Whatever is ready is issued: the x halves of the gates of the next tile (inputs landed, accumulators drained),
            // the h halves of the oldest tile whose h_0 operand is written, or fc2 of the oldest tile whose new hidden state
            // is written.  A fixed order (gates k, fc2 k-1) made fc2 of one tile wait for the LOADS of the next one.  The
            // tests are ordered so that no parity test can see a stale phase: in_full(u) implies the slot's previous use
            // is over; the h halves are only tried after the tile's x halves, fc2 only after its h halves; hb_ready
            // alternates h_0 (parity 0) / h_1 (parity 1) per tile and the epilogue writes the next h_0 only after q_full.
            int kx = 0, kg = 0, kf = 0;
            while (kf < n_my) {
                if (kx < n_my) {
                    const int s = kx & 1, u = kx >> 1;
                    if (mbar_try_wait(&in_full[s], (uint32_t)(u & 1)) && mbar_try_wait(&tmem_free[s], (uint32_t)((u & 1) ^ 1))) {
                        RMARK(tg0);
                        gates_x(kx);
                        RADD(2, clock64() - tg0);
                        ++kx;
                    }
                }
                if (kg < kx && mbar_try_wait(&hb_ready[kg & 1], 0)) {
                    RMARK(tg0);
                    gates_h(kg);
                    RADD(2, clock64() - tg0);
                    ++kg;
                }
                if (kf < kg && mbar_try_wait(&hb_ready[kf & 1], 1)) {
                    RMARK(tf0);
                    fc2(kf);
                    RADD(2, clock64() - tf0);
                    ++kf;
                }
            }
        }
    } else if (warp < 8) {
        // ===== gate group: EVERY tile of the CTA, slots alternating.  Gate math out of TMEM, new hidden state (bf16 operand
        // of fc2 and fp32 staging tile).  The h_0 operand of a tile is written by the selection group, a tile ahead. =====
        const int q4 = warp & 3, ch = warp >> 2;
        const uint32_t r = q4 * 32 + lane;                        // tile row of this thread; it owns columns 32 ch .. +31
        const float* bias_c = bias + 32 * ch;
        for (int k = 0; k < n_my; ++k) {
            const int s = k & 1, u = k >> 1;
            uint8_t* sl = smem + SLOT0 + s * SLOT_BYTES;
            uint8_t* hs = sl + S_HS + ch * TILE_BYTES;            // the fp32 staging tile of this column half
            const uint32_t tlane = tmem_base + 256 * s + ((uint32_t)(q4 * 32) << 16);
            RWAIT(3, &in_full[s], (uint32_t)(u & 1));          // (complete long before the gate MMAs are: makes the staged h_0 visible here)
#ifdef PMB_RO_PROFILE
            if (threadIdx.x == 0 && k == 0) prof_acc[14] = clock64() - prof_t0;      // kernel entry -> first tile landed
#endif
            RWAIT(4, &gates_full[s], (uint32_t)(u & 1));
            RMARK(tm0);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t ar[16], az[16], ain[16], ahn[16];
                tmem_ld_32x16(tlane + 32 * ch + 16 * c, ar);
                tmem_ld_32x16(tlane + 64 + 32 * ch + 16 * c, az);
                tmem_ld_32x16(tlane + 128 + 32 * ch + 16 * c, ain);
                tmem_ld_32x16(tlane + 192 + 32 * ch + 16 * c, ahn);
                tmem_wait_ld();
                // four columns at a time: biases (16-byte loads, same address in all lanes) and h_0 (again from the staging
                // tile: not kept in registers across the MMA wait) are loaded right where they are used
                uint32_t pk[8];
#pragma unroll
                for (int j4 = 0; j4 < 4; ++j4) {
                    const float4 br = *reinterpret_cast<const float4*>(bias_c + 16 * c + 4 * j4);
                    const float4 bz = *reinterpret_cast<const float4*>(bias_c + 64 + 16 * c + 4 * j4);
                    const float4 bn = *reinterpret_cast<const float4*>(bias_c + 128 + 16 * c + 4 * j4);
                    const float4 bh = *reinterpret_cast<const float4*>(bias_c + 192 + 16 * c + 4 * j4);
                    float4 h4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    float* hp = reinterpret_cast<float*>(hs + sw128_offset(r, (uint32_t)(4 * c + j4)));
                    if (P.h0) h4 = *reinterpret_cast<const float4*>(hp);
                    const float brv[4] = {br.x, br.y, br.z, br.w}, bzv[4] = {bz.x, bz.y, bz.z, bz.w};
                    const float bnv[4] = {bn.x, bn.y, bn.z, bn.w}, bhv[4] = {bh.x, bh.y, bh.z, bh.w};
                    const float hv4[4] = {h4.x, h4.y, h4.z, h4.w};
                    float o[4];
#pragma unroll
                    for (int jj = 0; jj < 4; ++jj) {
                        const int j = 4 * j4 + jj;
                        const float rg = fast_sigmoid(__uint_as_float(ar[j]) + brv[jj]);
                        const float zg = fast_sigmoid(__uint_as_float(az[j]) + bzv[jj]);
                        const float hn = __uint_as_float(ahn[j]) + bhv[jj];
                        const float ng = fast_tanh(__uint_as_float(ain[j]) + bnv[jj] + rg * hn);
                        o[jj] = ng + zg * (hv4[jj] - ng);
                    }
                    pk[2 * j4] = pack_bf16x2(o[0], o[1]);
                    pk[2 * j4 + 1] = pack_bf16x2(o[2], o[3]);
                    // new hidden state: in place in the staging tile of this column half, in the layout the tensor map
                    // describes; the loader thread stores both staging tiles with two bulk tensor copies once all 8 warps arrived
                    if (P.h_last) *reinterpret_cast<float4*>(hp) = make_float4(o[0], o[1], o[2], o[3]);
                }
                *reinterpret_cast<uint4*>(sl + S_HT + sw128_offset(r, (uint32_t)(2 * (2 * ch + c)))) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                *reinterpret_cast<uint4*>(sl + S_HT + sw128_offset(r, (uint32_t)(2 * (2 * ch + c) + 1))) = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&hb_ready[s]);                         // h_1 operand written: fc2 may be issued
                mbar_arrive(&xh_free[s]);                          // gate MMAs complete, new hidden state staged
            }
            RADD(8, clock64() - tm0);
        }
    } else {
        // ===== selection group: q = fc2(h) out of TMEM and the epsilon-greedy selection of EVERY tile, one tile behind the
        // gate group.  The two threads of a row split the 16-action chunks: column half 0 takes chunks 0 and 2, column half 1
        // chunks 1 and 3 and the Philox draws.  Everything that does not need q (the availability bits, the draws) is done
        // before the fc2 MMAs are waited for.
        const int q4 = warp & 3, ch = (warp >> 2) & 1;
        const uint32_t r = q4 * 32 + lane;
        const bool q_vec = (P.A & 3) == 0 && (reinterpret_cast<uintptr_t>(P.q) & 15) == 0;
        // h_0 of tile k2 (fp32 staging tile, or zeros) -> bf16 operand tile of its slot.  Done while the gate group is still
        // busy with tile k2 - 1, so the gate MMAs of k2 are complete when the gate group gets there.  The operand tile is free:
        // its last readers, the fc2 MMAs of tile k2 - 2, completed before this group selected for that tile.
        auto h0_operand = [&](int k2) {
            const int s2 = k2 & 1, u2 = k2 >> 1;
            uint8_t* sl2 = smem + SLOT0 + s2 * SLOT_BYTES;
            const uint8_t* hs2 = sl2 + S_HS + ch * TILE_BYTES;
            RWAIT(15, &in_full[s2], (uint32_t)(u2 & 1));
            RMARK(tp0);
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                float f[16];
                if (P.h0) {
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4)
                        *reinterpret_cast<float4*>(&f[4 * j4]) = *reinterpret_cast<const float4*>(hs2 + sw128_offset(r, (uint32_t)(4 * c + j4)));
                } else {
#pragma unroll
                    for (int j = 0; j < 16; ++j) f[j] = 0.f;
                }
                store_row16(sl2 + S_HT, r, 2 * ch + c, f);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&hb_ready[s2]);
            RADD(7, clock64() - tp0);
        };
        if (n_my > 0) h0_operand(0);
        for (int k = 0; k < n_my; ++k) {
            const int s = k & 1, u = k >> 1;
            uint8_t* sl = smem + SLOT0 + s * SLOT_BYTES;
            const uint32_t tlane = tmem_base + 256 * s + ((uint32_t)(q4 * 32) << 16);
            const int64_t tile = (int64_t)blockIdx.x + (int64_t)k * gridDim.x;
            const int64_t row = tile * TILE_ROWS + r;
            const bool valid = row < P.R;
            const bool select = P.actions_out != nullptr && valid;
            float* qo = P.q ? P.q + row * P.A : nullptr;
            const uint8_t* av = nullptr;
            bool av_vec = true;
            // first what the gate group will wait for next: the h_0 operand of the next tile (its inputs landed while this
            // group selected for the previous tile)
            if (k + 1 < n_my) h0_operand(k + 1);
            if (av_smem) RWAIT(6, &av_full[s], (uint32_t)(u & 1));
            RMARK(tq0);
            uint32_t oks2[2] = {0u, 0u};                           // availability bits of the own chunks ch, ch + 2
            uint32_t rnd_x = 0u, rnd_y = 0u;
            if (select) {
                const int64_t bb = (int64_t)((uint32_t)row / (uint32_t)P.N);
                if (av_smem && AVB == 4) av = sl + S_AV + r * P.A * 4;
                else if (av_smem) {
                    const int64_t row0 = tile * TILE_ROWS;
                    const Av8Run run = av8_run(P, bb, row0, row0 + TILE_ROWS);
                    const int64_t ra = bb * P.N > row0 ? bb * P.N : row0;
                    av = sl + S_AV + run.dst + run.phase + (row - ra) * P.A;
                } else {
                    av = static_cast<const uint8_t*>(P.avail) + (bb * P.avail_sb + (row - bb * P.N) * P.A) * AVB;
                    av_vec = (P.A & 3) == 0 && (P.avail_sb & 3) == 0 && (reinterpret_cast<uintptr_t>(P.avail) & 15) == 0;
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int c0 = 16 * (ch + 2 * i);
                    if (c0 < A_pad) {
                        uint32_t oks = avail_bits16<AVB>(av, c0, P.A, av_vec);
                        const int left = P.A - c0;                                   // actions of this chunk that exist
                        oks &= left >= 16 ? 0xffffu : ((1u << (left > 0 ? left : 0)) - 1u);
                        oks2[i] = oks;
                    }
                }
                if (ch == 1 && !P.expo) {
                    // Philox mode (same arithmetic as epsilon_greedy_kernel): word x -> epsilon test, word y -> rank
                    const uint4 r0 = gf_philox4x32_10(make_uint4((uint32_t)P.offset, (uint32_t)(P.offset >> 32), (uint32_t)row,
                                                                 ((uint32_t)(row >> 32) << 16)),
                                                      make_uint2((uint32_t)P.seed, (uint32_t)(P.seed >> 32)));
                    rnd_x = r0.x; rnd_y = r0.y;
                }
            }
            RADD(10, clock64() - tq0);
            RWAIT(5, &q_full[s], (uint32_t)(u & 1));
            RMARK(tq1);
            tc_fence_after();
            float best = -INFINITY;
            int bidx = 0x7fffffff;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int c0 = 16 * (ch + 2 * i);
                if (c0 < A_pad) {
                    uint32_t aq[16];
                    tmem_ld_32x16(tlane + c0, aq);
                    float bq[16];
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4)
                        *reinterpret_cast<float4*>(&bq[4 * j4]) = *reinterpret_cast<const float4*>(bias + 256 + c0 + 4 * j4);
                    tmem_wait_ld();
                    if (valid) {
                        float qv[16];
#pragma unroll
                        for (int j = 0; j < 16; ++j) qv[j] = __uint_as_float(aq[j]) + bq[j];
                        if (qo) {
                            if (q_vec) {
#pragma unroll
                                for (int j4 = 0; j4 < 4; ++j4)
                                    if (c0 + 4 * j4 < P.A)
                                        *reinterpret_cast<float4*>(qo + c0 + 4 * j4) =
                                            make_float4(qv[4 * j4], qv[4 * j4 + 1], qv[4 * j4 + 2], qv[4 * j4 + 3]);
                            } else {
#pragma unroll
                                for (int j = 0; j < 16; ++j)
                                    if (c0 + j < P.A) qo[c0 + j] = qv[j];
                            }
                        }
                        if (select) {
                            // arg-max of the chunk as a tournament (depth 4 instead of a 16-long dependent chain); the lower
                            // index is kept unless the higher one is strictly greater: lowest index wins, as in a scan
                            const uint32_t oks = oks2[i];
                            float tv[16];
                            int ti[16];
#pragma unroll
                            for (int j = 0; j < 16; ++j) { tv[j] = (oks >> j) & 1u ? qv[j] : -INFINITY; ti[j] = j; }
#pragma unroll
                            for (int st = 1; st < 16; st <<= 1)
#pragma unroll
                                for (int j = 0; j < 16; j += 2 * st)
                                    if (tv[j + st] > tv[j]) { tv[j] = tv[j + st]; ti[j] = ti[j + st]; }
                            if (tv[0] > best) { best = tv[0]; bidx = c0 + ti[0]; }    // chunks ascending, strict >
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_free[s]);
            if (P.actions_out) {
                // hand-over: 16 bytes per row (best q bits | index | availability bits of chunks 1, 3 | draws) and a
                // 64-thread named barrier per row quarter.  Both warps wait on it, so the half-1 warp never runs a tile ahead
                // of its partner: neither the barrier nor the slot's hand-over block can be reused early.
                uint4* xc = reinterpret_cast<uint4*>(sl + S_XC) + r;
                const int bar_id = 1 + q4;
                if (ch == 1) {
                    const uint32_t explore = (1.0f - gf_u01(rnd_x)) < P.epsilon ? 1u : 0u;      // u in [0, 1)
                    *xc = make_uint4(__float_as_uint(best), (uint32_t)bidx, oks2[0] | (oks2[1] << 16), (rnd_y & ~1u) | explore);
                }
                asm volatile("bar.sync %0, 64;" ::"r"(bar_id) : "memory");
                if (ch == 0 && select) {
                    const uint4 o = *xc;
                    const float best1 = __uint_as_float(o.x);
                    const int bidx1 = (int)o.y;
                    if (bidx1 != 0x7fffffff && (best1 > best || (best1 == best && bidx1 < bidx))) { best = best1; bidx = bidx1; }
                    const uint32_t ok_lo = oks2[0] | (o.z << 16);                // available actions 0..31
                    const uint32_t ok_hi = oks2[1] | (o.z & 0xffff0000u);        //                   32..63
                    const int cnt = __popc(ok_lo) + __popc(ok_hi);
                    if (bidx == 0x7fffffff) bidx = 0;                              // all -inf / NaN: first index
                    int ridx;
                    bool explore;
                    if (P.expo) {
                        // reference arithmetic with injected draws: argmax_a (avail[a] / cnt) / Exp(1)[a]
                        const float prob = __fdiv_rn(1.0f, (float)cnt);
                        float rbest = -INFINITY;
                        ridx = 0x7fffffff;
                        for (int a = 0; a < P.A; ++a) {
                            const bool oka = ((a < 32 ? ok_lo >> a : ok_hi >> (a - 32)) & 1u) != 0u;
                            const float ratio = __fdiv_rn(oka ? prob : 0.0f, __ldg(P.expo + row * P.A + a));
                            if (ratio > rbest) { rbest = ratio; ridx = a; }
                        }
                        if (ridx == 0x7fffffff) ridx = 0;
                        explore = __ldg(P.u + row) < P.epsilon;
                    } else {
                        explore = (o.w & 1u) != 0u;
                        int kq = (int)((1.0f - gf_u01(o.w)) * (float)cnt);
                        if (kq >= cnt) kq = cnt - 1;
                        // the kq-th set bit of the availability mask
                        const int c_lo = __popc(ok_lo);
                        ridx = cnt <= 0 ? 0 : (kq < c_lo ? nth_set_bit(ok_lo, kq) : 32 + nth_set_bit(ok_hi, kq - c_lo));
                    }
                    int pick = (cnt > 0 && explore) ? ridx : bidx;
                    if (pick >= P.A) pick = 0;
                    P.actions_out[row] = pick;
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&av_free[s]);
            RADD(9, clock64() - tq1);
        }
    }
#ifdef PMB_RO_PROFILE
    if (lane == 0) {
        for (int i = 0; i < 11; ++i) if (prof_acc[i]) atomicAdd(&g_ro_prof[i], (unsigned long long)prof_acc[i]);
        for (int i = 13; i < 16; ++i) if (prof_acc[i]) atomicAdd(&g_ro_prof[i], (unsigned long long)prof_acc[i]);
        if (threadIdx.x == 0) { atomicAdd(&g_ro_prof[11], (unsigned long long)(clock64() - prof_t0)); atomicAdd(&g_ro_prof[12], 1ull); }
    }
#endif
    tc_fence_before();
    __syncthreads();
    if (warp == MMA_W) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

// ------------------------------------------------------------------------------------------
// fc1 / fc2 weight gradients from tile images, one-hot operands generated on the fly.
//   item = (t, tile, half): 64 rows.  A1 = [dpre1 | Q1], A2 = [P1 | (ignored)] (MN-major, M = 128), where
//     Q1[row, a]  = dq[row]        if a == action[row]          (-> fc2.weight / fc2.bias)
//     P1[row, a]  = 1              if a == action[row at t-1] and that step was filled (-> fc1 last-action columns)
//   D_obs = A1 x obs image (rows 0..63: fc1.weight[:, :O]; the image carries one-hot(agent) and a ones column in its K
//   padding - written by the streaming fc1 kernel - so columns O.. give the agent-id columns and fc1.bias),
//   D_h = A1 x h_t (fc2.weight in rows 64..), D_one = A1 x 1 (fc2.bias in rows 64..), D_a2 = A2 x dpre1 (rows 0..63:
//   last-action columns).  Three 72 KB stages.
// ------------------------------------------------------------------------------------------
namespace ad {
constexpr int HALF = 8192;                                   // 64 rows x 128 B
constexpr int MAX_CHUNKS = 5;                                // obs width <= 320
constexpr int STAGES = 3;
constexpr int STAGE_BYTES = (4 + MAX_CHUNKS) * HALF;         // dpre1 | Q1 | P1 | h_t | obs chunks
constexpr int ONES = STAGES * STAGE_BYTES;
constexpr int BARS = ONES + HALF;
constexpr int SMEM_BYTES = 1024 + BARS + 128;
constexpr int N_PAIR = STAGES;                                // generator warp pairs (warps 0-3 and 6-7): pair p owns stage p
static_assert(N_PAIR == STAGES, "a pair per stage: its parity waits on the stage barrier are then never two phases apart");
constexpr int THREADS = 32 * (6 + 2 * (N_PAIR - 2));
constexpr int OBS_LD = MAX_CHUNKS * 64;                      // 320
constexpr int PARTIAL_FLOATS = 64 * OBS_LD + 64 * 64 + 128 + 128 * 64;   // dW1obs | dW2 | (db1|db2) | (dW1act|dW1id)
}  // namespace ad

struct AgentDwParams {
    const uint8_t* dpre1_ti; const uint8_t* h_ti; const uint8_t* obs_ti;
    const float* d_chosen; const int64_t* actions; int64_t actions_sb; const int64_t* filled; int64_t filled_sb;
    const int64_t* ep_index;
    float* partial;
    int64_t R, n_items, items_per_cta;
    int T, N, A, n_tiles, n_chunks, use_act, use_id;
    // optional (padded-step skipping): the (t, tile) items are live[0 .. *n_live) (t * n_tiles + tile), each two half
    // items; the split over the grid is then computed here from the device count.  The list must hold every live item
    // and nothing else: the dpre1 images of the other items are stale x values of the target net.
    const int32_t* live;
    const int32_t* n_live;
};

__global__ void __launch_bounds__(ad::THREADS, 1) agent_dw_tc_kernel(AgentDwParams P) {
    using namespace ad;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BARS);
    uint64_t* full = bars;               // [STAGES]: loader bytes + 2 generator warps
    uint64_t* empty = bars + STAGES;     // [STAGES]
    uint64_t* done = bars + 2 * STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 3); mbar_init(&empty[i], 1); }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == 4) tmem_alloc(tmem_slot, 512);
    for (int i = threadIdx.x; i < HALF / 16; i += THREADS)
        reinterpret_cast<uint4*>(smem + ONES)[i] = make_uint4(0x3f803f80u, 0x3f803f80u, 0x3f803f80u, 0x3f803f80u);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int64_t n_items = P.live ? 2 * (int64_t)__ldg(P.n_live) : P.n_items;
    const int64_t items_per_cta = P.live ? (n_items + gridDim.x - 1) / gridDim.x : P.items_per_cta;
    const int64_t beg = (int64_t)blockIdx.x * items_per_cta;
    const int64_t end = beg + items_per_cta < n_items ? beg + items_per_cta : n_items;
    const int64_t n_my = end > beg ? end - beg : 0;
    const int n_obs_cols = P.n_chunks * 64;

    if (warp == 5) {
        if (lane == 0) {
            for (int64_t i = 0; i < n_my; ++i) {
                const int s = (int)(i % STAGES);
                const int64_t item = beg + i;
                const int64_t tt = P.live ? (int64_t)__ldg(P.live + (item >> 1)) : item >> 1;   // t * n_tiles + tile
                const int half = (int)(item & 1);
                const int64_t t = tt / P.n_tiles, tile = tt - t * P.n_tiles;
                mbar_wait(&empty[s], (uint32_t)(((i / STAGES) & 1) ^ 1));
                mbar_arrive_expect_tx(&full[s], (2 + P.n_chunks) * HALF);
                uint8_t* st = smem + s * STAGE_BYTES;
                bulk_copy_g2s(st, P.dpre1_ti + tt * TILE_BYTES + half * HALF, HALF, &full[s]);
                bulk_copy_g2s(st + 3 * HALF, P.h_ti + ((t + 1) * P.n_tiles + tile) * TILE_BYTES + half * HALF, HALF, &full[s]);
                for (int c = 0; c < P.n_chunks; ++c)
                    bulk_copy_g2s(st + (4 + c) * HALF, P.obs_ti + (tt * P.n_chunks + c) * TILE_BYTES + half * HALF, HALF,
                                  &full[s]);
            }
        }
    } else if (warp == 4) {
        if (lane == 0 && n_my > 0) {
            const int n1 = n_obs_cols > 256 ? 256 : n_obs_cols, n2 = n_obs_cols - n1;
            const uint32_t id_o1 = umma_idesc_bf16(128, n1, 1, 1), id_o2 = umma_idesc_bf16(128, n2 > 0 ? n2 : 16, 1, 1);
            const uint32_t id64 = umma_idesc_bf16(128, 64, 1, 1), id16 = umma_idesc_bf16(128, 16, 1, 1);
            const uint32_t ones = smem_u32(smem + ONES);
            for (int64_t i = 0; i < n_my; ++i) {
                const int s = (int)(i % STAGES);
                mbar_wait(&full[s], (uint32_t)((i / STAGES) & 1));
                tc_fence_after();
                const uint32_t st = smem_u32(smem + s * STAGE_BYTES);
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {               // 64 rows = 4 x (K = 16)
                    const uint32_t acc = (i | kk) != 0;
                    const uint64_t a1 = umma_desc_sw128(st + kk * 2048, HALF, 1024);              // [dpre1 | Q1]
                    const uint64_t a2 = umma_desc_sw128(st + 2 * HALF + kk * 2048, HALF, 1024);   // [P1 | h (rows 64.. unused)]
                    umma_bf16(tmem_base, a1, umma_desc_sw128(st + 4 * HALF + kk * 2048, HALF, 1024), id_o1, acc);
                    if (n2 > 0)
                        umma_bf16(tmem_base + 256, a1, umma_desc_sw128(st + 8 * HALF + kk * 2048, HALF, 1024), id_o2, acc);
                    umma_bf16(tmem_base + 320, a1, umma_desc_sw128(st + 3 * HALF + kk * 2048, HALF, 1024), id64, acc);
                    umma_bf16(tmem_base + 384, a1, umma_desc_sw128(ones + kk * 2048, HALF, 1024), id16, acc);
                    umma_bf16(tmem_base + 400, a2, umma_desc_sw128(st + kk * 2048, HALF, 1024), id64, acc);
                }
                umma_commit(&empty[s]);
            }
            umma_commit(done);
        }
    } else {
        // ===== one-hot generators (one row per thread): warps 0-1 take the even items of this CTA, warps 2-3 the odd
        // ones; the index loads of a warp's next item are issued before the current item is written (software
        // pipeline: the generators, not the copies or the MMAs, were the critical path).  All four warps: final epilogue.
        {
            const int rr = (warp & 1) * 32 + lane;             // row within the half tile
            // RAW loaded values: nothing in fetch() depends on a load (in-order issue: the warp would stall right there)
            struct Idx { long long a, ap, f; float dq; };
            auto fetch = [&](int64_t i) {
                Idx x{-1, -1, 0, 0.f};
                if (i >= n_my) return x;
                const int64_t item = beg + i;
                const int64_t tt = P.live ? (int64_t)__ldg(P.live + (item >> 1)) : item >> 1;
                const int half = (int)(item & 1);
                const int64_t t = tt / P.n_tiles, tile = tt - t * P.n_tiles;
                const int64_t p = tile * TILE_ROWS + half * 64 + rr;
                if (p < P.R) {
                    const int64_t b = (int64_t)((uint32_t)p / (uint32_t)P.N);
                    const int n = (int)(p - b * P.N);
                    const int64_t be = ep_row(P.ep_index, b);
                    if (t < P.T - 1) {
                        x.dq = __ldg(P.d_chosen + (b * (P.T - 1) + t) * P.N + n);
                        x.a = __ldg(P.actions + be * P.actions_sb + t * P.N + n);
                    }
                    if (P.use_act && t > 0) {
                        x.f = __ldg(P.filled + be * P.filled_sb + (t - 1));
                        x.ap = __ldg(P.actions + be * P.actions_sb + (t - 1) * P.N + n);
                    }
                }
                return x;
            };
            // write the one-hot tiles of item i from the resolved indices, publish the stage
            auto emit = [&](int64_t i, const Idx& x) {
                const int s = (int)(i % STAGES);
                const int a = (int)x.a, ap = x.f != 0 ? (int)x.ap : -1;
                const uint32_t dqb = pack_bf16x2(x.dq, 0.f) & 0xffffu;        // bf16 bits of dq
                mbar_wait(&empty[s], (uint32_t)(((i / STAGES) & 1) ^ 1));
                uint8_t* st = smem + s * STAGE_BYTES;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const uint32_t off = sw128_offset((uint32_t)rr, (uint32_t)j);
                    uint32_t q[4] = {0, 0, 0, 0}, pp[4] = {0, 0, 0, 0};
                    if ((a >> 3) == j) q[(a & 7) >> 1] = dqb << (16 * (a & 1));
                    if ((ap >> 3) == j) pp[(ap & 7) >> 1] = 0x3f80u << (16 * (ap & 1));
                    *reinterpret_cast<uint4*>(st + 1 * HALF + off) = make_uint4(q[0], q[1], q[2], q[3]);
                    *reinterpret_cast<uint4*>(st + 2 * HALF + off) = make_uint4(pp[0], pp[1], pp[2], pp[3]);
                }
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(&full[s]);
            };
            // Two items in flight per warp, their loads issued AFTER the proxy fence of emit() (it compiles to MEMBAR.ALL.CTA
            // + FENCE.VIEW.ASYNC and waits for every load the thread has in flight) and by two distinct sets of load
            // instructions (a scoreboard is a counter: a wait on one item's values also waits for newer loads on it).
            // Role profile (clock64 around every wait): the generators, not the copies or the MMAs, bound this kernel -
            // the MMA warp waits for their tiles ~38 % of the time; most of a generator's time is load latency that the
            // fence or the next use exposes.  Separate index-loader warps feeding the writers through a two-slot ring were
            // measured at 6.0-6.5 ms against 3.27 (the ring is too shallow; there is no shared memory for a deeper one).
            // (one pair per stage: with two pairs, a pair's budget per item - two item times - was spent almost entirely on
            // exposed load latency and the MMA warp waited for the tiles 38 % of the time; four pairs over three stages
            // let a pair run two barrier phases ahead - a parity wait cannot tell - and corrupted a stage)
            const int64_t i0 = warp < 4 ? (warp >> 1) : 2 + ((warp - 6) >> 1);
            Idx x0 = fetch(i0), x1 = fetch(i0 + N_PAIR);
            for (int64_t i = i0; i < n_my; i += 2 * N_PAIR) {
                emit(i, x0);
                x0 = fetch(i + 2 * N_PAIR);
                if (i + N_PAIR < n_my) emit(i + N_PAIR, x1);
                x1 = fetch(i + 3 * N_PAIR);
            }
        }
        if (warp >= 4) goto tail;                               // the final epilogue: warps 0-3 (one TMEM lane quarter each)
        float* out = P.partial + (int64_t)blockIdx.x * PARTIAL_FLOATS;
        float* p_obs = out, *p_w2 = out + 64 * OBS_LD, *p_b = p_w2 + 64 * 64, *p_a2 = p_b + 128;
        const int c = warp * 32 + lane;                        // accumulator row 0..127
        if (n_my > 0) {
            mbar_wait(done, 0);
            tc_fence_after();
            const uint32_t tl = tmem_base + ((uint32_t)(warp * 32) << 16);
            for (int g = 0; g < n_obs_cols; g += 32) {          // D_obs: rows 0..63 = fc1.weight[:, :O]
                uint32_t v[32];
                tmem_ld_32x32(tl + g, v);
                tmem_wait_ld();
                if (c < 64) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) p_obs[c * OBS_LD + g + j] = __uint_as_float(v[j]);
                }
            }
            for (int g = 0; g < 64; g += 32) {
                uint32_t v[32], w[32];
                tmem_ld_32x32(tl + 320 + g, v);                 // D_h: rows 64.. = fc2.weight[a, :]
                tmem_ld_32x32(tl + 400 + g, w);                 // D_a2: rows 0..63 last-action, 64.. agent-id
                tmem_wait_ld();
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (c >= 64) p_w2[(c - 64) * 64 + g + j] = __uint_as_float(v[j]);
                    p_a2[c * 64 + g + j] = __uint_as_float(w[j]);
                }
            }
            uint32_t b1[16];
            tmem_ld_32x16(tl + 384, b1);
            tmem_wait_ld();
            p_b[c] = __uint_as_float(b1[0]);
        } else {
            for (int i = threadIdx.x; i < PARTIAL_FLOATS; i += 128) out[i] = 0.f;
        }
    }
tail:
    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
}

__global__ void agent_dw_reduce_kernel(const float* __restrict__ partial, int n_cta, int O, int A, int N, int D_in,
                                       int use_act, int use_id, float* __restrict__ fc1_w, float* __restrict__ fc1_b,
                                       float* __restrict__ fc2_w, float* __restrict__ fc2_b) {
    using namespace ad;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= PARTIAL_FLOATS) return;
    float s = 0.f;
    for (int c = 0; c < n_cta; ++c) s += partial[(int64_t)c * PARTIAL_FLOATS + i];
    if (i < 64 * OBS_LD) {
        int j = i / OBS_LD, k = i - j * OBS_LD;
        if (k < O) fc1_w[(int64_t)j * D_in + k] = s;
        else if (k - O < N) { if (use_id) fc1_w[(int64_t)j * D_in + O + (use_act ? A : 0) + (k - O)] = s; }   // one-hot(agent) columns
        else if (k - O == N) fc1_b[j] = s;                                                                   // ones column
    } else if (i < 64 * OBS_LD + 64 * 64) {
        int q = i - 64 * OBS_LD, a = q / 64, j = q - a * 64;
        if (a < A) fc2_w[a * 64 + j] = s;
    } else if (i < 64 * OBS_LD + 64 * 64 + 128) {
        int q = i - (64 * OBS_LD + 64 * 64);
        if (q >= 64 && q - 64 < A) fc2_b[q - 64] = s;
    } else {
        int q = i - (64 * OBS_LD + 64 * 64 + 128), r = q / 64, j = q - r * 64;
        if (r < 64 && use_act && r < A) fc1_w[(int64_t)j * D_in + O + r] = s;
    }
}

// zero the padding rows (row >= R) of the last tile of every timestep of a tile-image buffer
__global__ void ti_zero_pad_kernel(uint8_t* buf, int n_t, int n_tiles, int64_t R) {
    const int pad0 = (int)(R - (int64_t)(n_tiles - 1) * TILE_ROWS);      // first padding row of the last tile
    const int n_pad = TILE_ROWS - pad0;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;          // one 16-byte chunk each
    int64_t total = (int64_t)n_t * n_pad * 8;
    if (i >= total) return;
    int j = (int)(i & 7);
    int64_t q = i >> 3;
    int rr = pad0 + (int)(q % n_pad);
    int64_t t = q / n_pad;
    uint8_t* tile = buf + (t * n_tiles + (n_tiles - 1)) * TILE_BYTES;
    *reinterpret_cast<uint4*>(tile + sw128_offset((uint32_t)rr, (uint32_t)j)) = make_uint4(0, 0, 0, 0);
}

}  // namespace tc

int tc_gru_fwd(const tc::GruFwdParams& P, cudaStream_t s) {
    if (P.nt != 1 || P.h_ti || P.g_ti) { set_error("tc_gru_fwd: the rollout kernel does one step and keeps no stash"); return PMB_ERR_INVALID; }
    if ((reinterpret_cast<uintptr_t>(P.h0) & 15) || (reinterpret_cast<uintptr_t>(P.h_last) & 15)) {
        set_error("tc_gru_fwd: hidden state must be 16-byte aligned");
        return PMB_ERR_INVALID;
    }
    // avail rows are staged through shared memory by bulk copies when they fit and (i32) are 16-byte granular; u8 rows
    // are staged as the aligned superset of each env's run, which fits for every A <= 64
    const int envs_per_tile = 127 / P.N + 2 < 128 ? 127 / P.N + 2 : 128;
    const int av_smem = P.actions_out && P.avail &&
                        (P.avail_u8 ? 128 * P.A + tc::ro::AV8_SLACK * envs_per_tile <= tc::ro::AV_BYTES
                                    : (P.A & 3) == 0 && 128 * P.A * 4 <= tc::ro::AV_BYTES && (P.avail_sb & 3) == 0 &&
                                          ((int64_t)P.N * P.A & 3) == 0 && (reinterpret_cast<uintptr_t>(P.avail) & 15) == 0);
    // tensor maps of the fp32 hidden state [R][64], in and out: boxes of 128 rows x 32 columns, 128-byte swizzle; loads
    // fill rows beyond R with zeros, stores clip them
    CUtensorMap tmap, tmap_out;
    memset(&tmap, 0, sizeof(tmap));
    memset(&tmap_out, 0, sizeof(tmap_out));
    if (P.h0 || P.h_last) {
        typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                     const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        static std::atomic<EncodeFn> encode_cache{nullptr};   // process-wide driver entry point; racing initialisers store the same value
        EncodeFn encode = encode_cache.load(std::memory_order_acquire);
        if (!encode) {
            void* fn = nullptr;
            cudaDriverEntryPointQueryResult qres;
            PMB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
            if (!fn || qres != cudaDriverEntryPointSuccess) { set_error("tc_gru_fwd: cuTensorMapEncodeTiled not available"); return PMB_ERR_CUDA; }
            encode = reinterpret_cast<EncodeFn>(fn);
            encode_cache.store(encode, std::memory_order_release);
        }
        const cuuint64_t gdim[2] = {64, (cuuint64_t)P.R};
        const cuuint64_t gstride[1] = {256};
        const cuuint32_t box[2] = {32, 128};
        const cuuint32_t estr[2] = {1, 1};
        for (int io = 0; io < 2; ++io) {
            const float* base = io ? P.h_last : P.h0;
            if (!base) continue;
            const CUresult cr = encode(io ? &tmap_out : &tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim,
                                       gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (cr != CUDA_SUCCESS) { set_error("tc_gru_fwd: cuTensorMapEncodeTiled failed"); return PMB_ERR_CUDA; }
        }
    }
    const auto kern = P.avail_u8 ? tc::gru_rollout_kernel<1> : tc::gru_rollout_kernel<4>;
    PMB_SMEM_ATTR(kern, tc::ro::SMEM_BYTES);
    const int grid = P.n_tiles < sm_count() ? P.n_tiles : sm_count();
    PMB_CUDA(launch_pdl(kern, dim3(grid), dim3(tc::ro::THREADS), tc::ro::SMEM_BYTES, s, rollout_pdl_enabled(), P, av_smem, tmap, tmap_out));
    PMB_LAUNCH_CHECK("gru_rollout_kernel");
    return PMB_OK;
}

#ifdef PMB_RO_PROFILE
extern "C" int pmb_debug_ro_prof(unsigned long long* out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, tc::g_ro_prof, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(tc::g_ro_prof, z, sizeof(z)); }
    return 0;
}
#endif


// one partial block per CTA of the persistent grid (grid <= SM count of the current device), with 2x head room
int64_t tc_agent_dw_scratch_bytes() { return align_up((int64_t)sm_count() * 2 * tc::ad::PARTIAL_FLOATS * 4, 256); }

int tc_agent_dw(const pmb_dims* d, const pmb_batch* b, const uint8_t* dpre1_ti, const uint8_t* h_ti, const uint8_t* obs_ti,
                const float* d_chosen, int n_tiles, float* fc1_w, float* fc1_b, float* fc2_w, float* fc2_b, void* scratch,
                int64_t scratch_bytes, cudaStream_t s, const int32_t* live_items, const int32_t* n_live) {
    tc::AgentDwParams P;
    P.dpre1_ti = dpre1_ti; P.h_ti = h_ti; P.obs_ti = obs_ti; P.d_chosen = d_chosen;
    P.actions = b->actions; P.actions_sb = b->actions_sb; P.filled = b->filled; P.filled_sb = b->filled_sb;
    P.ep_index = b->ep_index;
    P.R = (int64_t)d->B * d->N; P.T = d->T; P.N = d->N; P.A = d->A; P.n_tiles = n_tiles;
    P.n_chunks = (d->O + 63) / 64; P.use_act = d->obs_last_action; P.use_id = d->obs_agent_id;
    P.n_items = (int64_t)d->T * n_tiles * 2;
    P.live = live_items; P.n_live = n_live;
    int grid = (int)(P.n_items < sm_count() ? P.n_items : sm_count());
    if ((int64_t)grid * tc::ad::PARTIAL_FLOATS * 4 > scratch_bytes) { set_error("tc_agent_dw: scratch too small"); return PMB_ERR_WORKSPACE; }
    P.items_per_cta = ceil_div(P.n_items, grid);
    P.partial = static_cast<float*>(scratch);
    PMB_SMEM_ATTR(tc::agent_dw_tc_kernel, tc::ad::SMEM_BYTES);
    tc::agent_dw_tc_kernel<<<grid, tc::ad::THREADS, tc::ad::SMEM_BYTES, s>>>(P);
    PMB_LAUNCH_CHECK("agent_dw_tc_kernel");
    tc::agent_dw_reduce_kernel<<<(unsigned)ceil_div(tc::ad::PARTIAL_FLOATS, 256), 256, 0, s>>>(
        P.partial, grid, d->O, d->A, d->N, d_in_of(d), d->obs_last_action, d->obs_agent_id, fc1_w, fc1_b, fc2_w, fc2_b);
    PMB_LAUNCH_CHECK("agent_dw_reduce_kernel");
    return PMB_OK;
}

int tc_ti_zero_pad(uint8_t* buf, int n_t, int n_tiles, int64_t R, cudaStream_t s) {
    if (R % tc::TILE_ROWS == 0) return PMB_OK;
    int n_pad = (int)((int64_t)n_tiles * tc::TILE_ROWS - R);
    int64_t total = (int64_t)n_t * n_pad * 8;
    tc::ti_zero_pad_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(buf, n_t, n_tiles, R);
    PMB_LAUNCH_CHECK("ti_zero_pad_kernel");
    return PMB_OK;
}


}  // namespace pmb
