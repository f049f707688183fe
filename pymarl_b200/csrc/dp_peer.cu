// Data-parallel exchange fused with the optimiser step over NVLink peer memory (SURVEY.md section 8e).
//
// Every rank (one process per GPU) holds its un-normalised gradient and the five loss sums in an exchange buffer that
// the other ranks map through CUDA IPC.  ONE kernel per rank and step then does what used to be pack -> NCCL all-reduce
// -> unpack -> grad-norm -> clip + RMSprop (five launches and a host-side collective call):
//   P0  block 0 packs the local loss sums behind the gradient and raises `ready[rank] = step` in every peer's flag block;
//       all blocks wait until every peer's `ready` flag in the LOCAL flag block reached `step`
//   P1  one-shot all-reduce: element i = sum over ranks r = 0 .. world-1 (fixed order -> bit-identical on every rank) of
//       peer r's buffer, read over NVLink with 16-byte volatile loads; the block's sum of squares goes to a partial array
//   --  grid barrier (all blocks are resident: the grid is at most the SM count)
//   P2  block 0 raises `done[rank] = step` at the peers (their buffers are no longer read); every block derives
//       1 / sum(mask), the global norm and the clip coefficient from the ordered partials and applies RMSprop (+ hard
//       target sync) to its slice of the REPLICATED parameters
//   P3  after every peer's `done` flag arrived the local buffer receives the global (normalised, clipped) gradient, so
//       `.grad` holds what torch's optimiser would have seen
// A spin that exceeds ~2 s (a dead peer) sets an error word instead of hanging the GPU.
#include <string.h>
#include "common.cuh"

namespace pmb {
namespace {

constexpr int PX_MAX_WORLD = 8;
constexpr int PX_THREADS = 256;
constexpr long long PX_SPIN_LIMIT = 4000000000ll;          // cycles (~2 s)

struct PeerArgs {
    float* buf[PX_MAX_WORLD];            // exchange buffers (own + IPC-mapped peers): [n grads | 16 tail floats]
    long long* flags[PX_MAX_WORLD];      // per buffer: ready[8] | done[8]
    int world, rank;
    int64_t n;                           // gradient elements (tail excluded)
};

__device__ __forceinline__ bool spin_until(const volatile long long* flag, long long value, int* err) {
    const long long t0 = clock64();
    while (*flag < value) {
        if (clock64() - t0 > PX_SPIN_LIMIT) { *err = 1; return false; }
        __nanosleep(64);
    }
    return true;
}

__global__ void __launch_bounds__(PX_THREADS)
dp_fused_kernel(PeerArgs A, long long step, unsigned long long epoch, float* __restrict__ p, float* __restrict__ sq,
                float* __restrict__ target, int do_sync, float* __restrict__ g_red, double* __restrict__ stats,
                double* __restrict__ partial, unsigned long long* __restrict__ grid_bar, int* __restrict__ err, float lr,
                float alpha, float eps, float clip) {
    __shared__ double sh[PX_THREADS / 32];
    __shared__ float s_scale, s_coef;
    const int world = A.world, rank = A.rank;
    float* mine = A.buf[rank];
    long long* my_flags = A.flags[rank];

    // ---- P0: publish, then wait for everybody's gradients ----
    if (blockIdx.x == 0) {
        if (threadIdx.x < 5)                                    // loss sums as (hi, lo) float pairs behind the gradient
            dp_pack_sum(threadIdx.x, stats[threadIdx.x], mine + A.n + 2 * threadIdx.x);
        __syncthreads();
        __threadfence_system();
        if (threadIdx.x < world) {
            volatile long long* f = A.flags[threadIdx.x] + rank;              // ready[rank] in peer threadIdx.x's block
            *f = step;
        }
    }
    if (threadIdx.x < world) spin_until(my_flags + threadIdx.x, step, err);
    __syncthreads();
    __threadfence_system();

    // ---- P1: ordered one-shot all-reduce + sum of squares ----
    const int64_t n4 = A.n / 4;
    double ss = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 acc = __ldcv(reinterpret_cast<const float4*>(A.buf[0]) + i);
        for (int r = 1; r < world; ++r) {
            const float4 v = __ldcv(reinterpret_cast<const float4*>(A.buf[r]) + i);
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
        reinterpret_cast<float4*>(g_red)[i] = acc;
        ss += (double)acc.x * acc.x + (double)acc.y * acc.y + (double)acc.z * acc.z + (double)acc.w * acc.w;
    }
    if (blockIdx.x == 0) {                                      // tail elements and the loss sums
        for (int64_t i = n4 * 4 + threadIdx.x; i < A.n; i += blockDim.x) {
            float acc = __ldcv(A.buf[0] + i);
            for (int r = 1; r < world; ++r) acc += __ldcv(A.buf[r] + i);
            g_red[i] = acc;
            ss += (double)acc * acc;
        }
        if (threadIdx.x < 5) {
            double hi = 0.0, lo = 0.0;
            float fh = 0.f, fl = 0.f;                           // summed in fp32 in rank order, like the NCCL path;
                                                                // mask_sum's pairs add exactly (dp_pack_sum)
            for (int r = 0; r < world; ++r) { fh += __ldcv(A.buf[r] + A.n + 2 * threadIdx.x); fl += __ldcv(A.buf[r] + A.n + 2 * threadIdx.x + 1); }
            hi = (double)fh; lo = (double)fl;
            stats[threadIdx.x] = hi + lo;
        }
    }
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < PX_THREADS / 32; ++w) tot += sh[w];
        partial[blockIdx.x] = tot;
        __threadfence();
        atomicAdd(grid_bar, 1ULL);
        const unsigned long long want = (epoch + 1) * gridDim.x;
        const long long t0 = clock64();
        while (*reinterpret_cast<volatile unsigned long long*>(grid_bar) < want)
            if (clock64() - t0 > PX_SPIN_LIMIT) { *err = 2; break; }
        __threadfence();
    }
    __syncthreads();

    // ---- P2: peers may reuse their buffers; identical update of the replicated parameters ----
    if (blockIdx.x == 0 && threadIdx.x < world) {
        __threadfence_system();
        volatile long long* f = A.flags[threadIdx.x] + PX_MAX_WORLD + rank;   // done[rank] at peer threadIdx.x
        *f = step;
    }
    if (threadIdx.x == 0) {
        const volatile double* pv = partial;
        double tot = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) tot += pv[b];
        const double mask_sum = *reinterpret_cast<const volatile double*>(stats + PMB_S_MASK_SUM);
        const float scale = (float)(1.0 / mask_sum);
        const float norm = (float)(sqrt(tot) / mask_sum);
        float coef = clip / (norm + 1e-6f);
        coef = coef < 1.f ? coef : 1.f;
        s_scale = scale; s_coef = coef;
        if (blockIdx.x == 0) {
            stats[PMB_S_GRAD_NORM] = (double)norm;
            stats[PMB_S_CLIP_COEF] = (double)coef;
            stats[PMB_S_LOSS] = stats[PMB_S_TD2_SUM] / mask_sum;
        }
    }
    __syncthreads();
    const float scale = s_scale, coef = s_coef;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (int64_t)gridDim.x * blockDim.x) {
        const float gv = (g_red[i] * scale) * coef;
        const float v = sq[i] * alpha + ((1.f - alpha) * gv) * gv;
        const float avg = sqrtf(v) + eps;
        const float pv2 = p[i] + (-lr * gv) / avg;
        g_red[i] = gv;
        sq[i] = v;
        p[i] = pv2;
        if (do_sync && target) target[i] = pv2;
    }

    // ---- P3: the local exchange buffer gets the global gradient once nobody reads it any more ----
    if (threadIdx.x < world) spin_until(my_flags + PX_MAX_WORLD + threadIdx.x, step, err);
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (int64_t)gridDim.x * blockDim.x)
        mine[i] = g_red[i];
}

}  // namespace
}  // namespace pmb

using namespace pmb;

extern "C" {

int pmb_ipc_export(const void* dev_ptr, void* handle_out, int64_t* offset_out) {
    PMB_REQUIRE(dev_ptr && handle_out && offset_out, "ipc_export: NULL pointer");
    cudaPointerAttributes attr;
    PMB_CUDA(cudaPointerGetAttributes(&attr, dev_ptr));
    PMB_REQUIRE(attr.type == cudaMemoryTypeDevice, "ipc_export: not a device pointer");
    // the handle names the whole cudaMalloc allocation: find its base to report the offset of dev_ptr inside it
    void* base = nullptr;
    size_t size = 0;
    {
        typedef int (*RangeFn)(unsigned long long*, size_t*, unsigned long long);
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        PMB_CUDA(cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q));
        PMB_REQUIRE(fn && q == cudaDriverEntryPointSuccess, "ipc_export: cuMemGetAddressRange not available");
        unsigned long long b = 0;
        const int rc = reinterpret_cast<RangeFn>(fn)(&b, &size, (unsigned long long)(uintptr_t)dev_ptr);
        PMB_REQUIRE(rc == 0, "ipc_export: cuMemGetAddressRange failed (%d)", rc);
        base = reinterpret_cast<void*>((uintptr_t)b);
    }
    cudaIpcMemHandle_t h;
    PMB_CUDA(cudaIpcGetMemHandle(&h, base));
    memcpy(handle_out, &h, sizeof(h));
    *offset_out = (int64_t)((const char*)dev_ptr - (const char*)base);
    return PMB_OK;
}

int pmb_ipc_open(const void* handle, int64_t offset, void** ptr_out) {
    PMB_REQUIRE(handle && ptr_out && offset >= 0, "ipc_open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void* base = nullptr;
    PMB_CUDA(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
    *ptr_out = static_cast<char*>(base) + offset;
    return PMB_OK;
}

int pmb_ipc_close(void* mapped_ptr, int64_t offset) {
    if (!mapped_ptr) return PMB_OK;
    PMB_CUDA(cudaIpcCloseMemHandle(static_cast<char*>(mapped_ptr) - offset));
    return PMB_OK;
}

int64_t pmb_dp_exchange_floats(int64_t n) {
    // [n gradients | PMB_DP_TAIL_FLOATS loss sums | pad to 16 B | flags: ready[8] + done[8] int64]
    return align_up(n + PMB_DP_TAIL_FLOATS, 4) + 2 * PX_MAX_WORLD * 2;
}

int pmb_dp_fused_allreduce_update(int32_t world, int32_t rank, void* const* bufs, int64_t n, int64_t step, float* flat_p,
                                  float* flat_sq, float* flat_target, int32_t do_target_sync, double* stats, float lr,
                                  float alpha, float eps, float grad_norm_clip, void* scratch, int64_t scratch_bytes,
                                  pmb_stream stream) {
    PMB_REQUIRE(world >= 2 && world <= PX_MAX_WORLD && rank >= 0 && rank < world && bufs && n > 0 && step > 0,
                "dp_fused: world must be 2..%d, step ids start at 1", PX_MAX_WORLD);
    PMB_REQUIRE(flat_p && flat_sq && stats && scratch, "dp_fused: NULL pointer");
    int grid = sm_count() / 2;
    if (grid > 64) grid = 64;
    if (grid < 1) grid = 1;
    // scratch: [g_red n floats][partial grid doubles][grid barrier counter u64][error word]; the counter only ever grows, so
    // the scratch must be zeroed once (by the owner) and then kept for the life of the exchange
    const int64_t need = align_up(n * 4, 256) + 1024 + 64;
    if (scratch_bytes < need) { set_error("dp_fused: scratch too small (%lld < %lld)", (long long)scratch_bytes, (long long)need); return PMB_ERR_WORKSPACE; }
    char* base = static_cast<char*>(scratch);
    float* g_red = reinterpret_cast<float*>(base);
    double* partial = reinterpret_cast<double*>(base + align_up(n * 4, 256));
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(base + align_up(n * 4, 256) + 1024);
    int* err = reinterpret_cast<int*>(bar + 2);
    PeerArgs A;
    A.world = world; A.rank = rank; A.n = n;
    const int64_t flag_off = align_up(n + PMB_DP_TAIL_FLOATS, 4);
    for (int r = 0; r < PX_MAX_WORLD; ++r) {
        A.buf[r] = r < world ? static_cast<float*>(bufs[r]) : nullptr;
        A.flags[r] = r < world ? reinterpret_cast<long long*>(static_cast<float*>(bufs[r]) + flag_off) : nullptr;
        PMB_REQUIRE(r >= world || bufs[r], "dp_fused: peer buffer %d is NULL", r);
    }
    dp_fused_kernel<<<grid, PX_THREADS, 0, (cudaStream_t)stream>>>(A, (long long)step, (unsigned long long)(step - 1), flat_p,
                                                                   flat_sq, flat_target, do_target_sync, g_red, stats, partial,
                                                                   bar, err, lr, alpha, eps, grad_norm_clip);
    PMB_LAUNCH_CHECK("dp_fused_kernel");
    return PMB_OK;
}

}  // extern "C"
