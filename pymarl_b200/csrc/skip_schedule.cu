// Padded-step skipping for the tensor-core learner step (pmb_dims.reserved bit 1): the schedule, built on the device.
//
// A ragged batch is truncated to its longest episode only, so most episodes end before the last step of the batch.
// Batch row b needs F_b = min(T, l_b + 2) forward steps, l_b = the last t with filled[b, t] = 1 (F_b = 0 when there is
// none): the mask of the loss is 0 beyond l_b, and the double-Q target at t = l_b reads both nets' Q at l_b + 1.
//   skip_steps_kernel : F_b, one warp per row, scanning `filled` from the end (the last filled step, not the sum of
//                       `filled`: a hole must not shorten an episode).
//   skip_sort_kernel  : ONE CTA.  A stable counting sort of the rows by F_b, descending (ties keep batch order: the
//                       schedule is deterministic and a full-length batch keeps the identity order), then the per-tile
//                       step counts and the list of live (t, tile) items.  With rows sorted, the rows live at step t
//                       are a prefix of the time-major row range p = b * N + n, so the live tiles of step t are
//                       [0, live_tiles(t)) and a tile's step count is that of its first episode.  The list is padded
//                       with -1 to T * n_tiles entries.
// Both launches are sized by the full rectangle and read nothing from the host: a captured CUDA graph stays correct
// when the next batch has other lengths.
#include "common.cuh"
#include "gru_tc.cuh"

namespace pmb {
namespace {

constexpr int kSortThreads = 1024;

__global__ void __launch_bounds__(256) skip_steps_kernel(const int64_t* __restrict__ filled, int64_t filled_sb,
                                                         const int64_t* __restrict__ ep_index, int B, int T,
                                                         int32_t* __restrict__ steps) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= B) return;
    const int64_t* f = filled + ep_row(ep_index, w) * filled_sb;
    int last = -1;
    for (int t0 = T - 1; t0 >= 0 && last < 0; t0 -= 32) {       // warp-uniform: `last` comes from a ballot
        const int t = t0 - lane;
        const unsigned m = __ballot_sync(0xffffffffu, t >= 0 && __ldg(f + t) != 0);
        if (m) last = t0 - (__ffs((int)m) - 1);                   // lowest lane = latest step
    }
    if (lane == 0) steps[w] = last < 0 ? 0 : min(T, last + 2);
}

// exclusive prefix sums over v[0 .. n) by one warp, in place; returns the total.  desc: sum from the top (v[n-1] first).
__device__ int warp_exclusive_scan(int* v, int n, bool desc, int lane) {
    int running = 0;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = desc ? n - 1 - (i0 + lane) : i0 + lane;
        const bool ok = i0 + lane < n;
        const int x = ok ? v[i] : 0;
        int inc = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (ok) v[i] = running + inc - x;
        running += __shfl_sync(0xffffffffu, inc, 31);
    }
    __syncwarp();
    return running;
}

// shared memory: base[T + 1] (per-key start of the sorted range, then the first list position of each step) | live[T]
__global__ void __launch_bounds__(kSortThreads, 1) skip_sort_kernel(const int32_t* __restrict__ steps,
                                                                     const int64_t* __restrict__ ep_index, int B, int T, int N,
                                                                     int n_tiles, SkipSchedule S) {
    extern __shared__ int sm[];
    int* base = sm;                 // [T + 1]
    int* live = sm + T + 1;         // [T]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int k = tid; k <= T; k += kSortThreads) base[k] = 0;
    __syncthreads();
    for (int b = tid; b < B; b += kSortThreads) atomicAdd(&base[__ldg(steps + b)], 1);
    __syncthreads();
    if (warp == 0) {
        // key k starts after every row with a larger key
        warp_exclusive_scan(base, T + 1, true, lane);
        // stable placement, 32 rows at a time in batch order: a row's rank among equal keys of its group + the rows of
        // that key already placed
        int key_next = lane < B ? __ldg(steps + lane) : -1;
        for (int b0 = 0; b0 < B; b0 += 32) {
            const int b = b0 + lane;
            const int key = key_next;
            key_next = b + 32 < B ? __ldg(steps + b + 32) : -1;
            const unsigned peers = __match_any_sync(0xffffffffu, key);
            if (key >= 0) {
                const int pos = base[key] + __popc(peers & ((1u << lane) - 1u));
                S.steps_sorted[pos] = key;
                S.ep_order[pos] = ep_index ? __ldg(ep_index + b) : (int64_t)b;
            }
            __syncwarp();
            if (key >= 0 && lane == __ffs((int)peers) - 1) base[key] += __popc(peers);
            __syncwarp();
        }
    }
    __syncthreads();
    // the first row of a tile belongs to the tile's longest episode
    for (int tile = tid; tile < n_tiles; tile += kSortThreads)
        S.tile_steps[tile] = S.steps_sorted[(int)(((int64_t)tile * 128) / N)];
    __syncthreads();
    // live_tiles(t) = number of tiles with more than t steps (tile_steps is non-increasing)
    for (int t = tid; t < T; t += kSortThreads) {
        int lo = 0, hi = n_tiles;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (S.tile_steps[mid] > t) lo = mid + 1; else hi = mid;
        }
        live[t] = lo;
        base[t] = lo;
    }
    __syncthreads();
    if (warp == 0) {
        const int total = warp_exclusive_scan(base, T, false, lane);
        if (lane == 0) { base[T] = total; *S.n_items = total; }
    }
    __syncthreads();
    // -1 behind the last live item: the fc1 kernels walk the list up to its first negative entry
    for (int i = base[T] + tid; i < T * n_tiles; i += kSortThreads) S.items[i] = -1;
    for (int t = warp; t < T; t += kSortThreads / 32) {
        int32_t* dst = S.items + base[t];
        const int32_t row0 = t * n_tiles;
        for (int tile = lane; tile < live[t]; tile += 32) dst[tile] = row0 + tile;
    }
}

}  // namespace

int64_t skip_schedule_bytes(int B, int T, int n_tiles) {
    return align_up((int64_t)B * 8, 256) + align_up((int64_t)n_tiles * 4, 256) + align_up((int64_t)T * n_tiles * 4, 256) + 256 +
           2 * align_up((int64_t)B * 4, 256);
}

SkipSchedule skip_schedule_views(void* base, int B, int T, int n_tiles) {
    char* p = static_cast<char*>(base);
    SkipSchedule S;
    S.ep_order = reinterpret_cast<int64_t*>(p);        p += align_up((int64_t)B * 8, 256);
    S.tile_steps = reinterpret_cast<int32_t*>(p);      p += align_up((int64_t)n_tiles * 4, 256);
    S.items = reinterpret_cast<int32_t*>(p);           p += align_up((int64_t)T * n_tiles * 4, 256);
    S.n_items = reinterpret_cast<int32_t*>(p);         p += 256;
    S.steps = reinterpret_cast<int32_t*>(p);           p += align_up((int64_t)B * 4, 256);
    S.steps_sorted = reinterpret_cast<int32_t*>(p);
    return S;
}

int tc_skip_schedule(const pmb_dims* d, const pmb_batch* b, const SkipSchedule& S, int n_tiles, cudaStream_t s) {
    const int B = d->B, T = d->T;
    skip_steps_kernel<<<(unsigned)ceil_div((int64_t)B * 32, 256), 256, 0, s>>>(b->filled, b->filled_sb, b->ep_index, B, T, S.steps);
    PMB_LAUNCH_CHECK("skip_steps_kernel");
    const int smem = (2 * T + 1) * 4;
    PMB_REQUIRE(smem <= 232448, "skip schedule: T = %d is too long for the one-CTA sort", T);
    if (smem > 48 * 1024) PMB_SMEM_ATTR(skip_sort_kernel, smem);
    skip_sort_kernel<<<1, kSortThreads, smem, s>>>(S.steps, b->ep_index, B, T, d->N, n_tiles, S);
    PMB_LAUNCH_CHECK("skip_sort_kernel");
    return PMB_OK;
}

}  // namespace pmb
