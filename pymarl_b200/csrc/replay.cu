// Replay-buffer side of the path (SURVEY.md section 8f, rank 1): ReplayBuffer.sample / EpisodeBatch.__getitem__ with an
// array of episode ids (components/episode_buffer.py:205-217,291-298) and max_t_filled (:255-256) for a buffer that
// lives in HBM.  The reference gathers every field with one advanced-indexing kernel per field; here ONE launch copies
// whole episodes (contiguous [T, ...] blocks) of all fields with 16-byte accesses: a pure HBM-bandwidth kernel
// (read + write of the sampled bytes).
#include "common.cuh"

namespace pmb {
namespace {

constexpr int GATHER_MAX_FIELDS = 16;
struct GatherArgs {
    const char* src[GATHER_MAX_FIELDS];
    char* dst[GATHER_MAX_FIELDS];
    int64_t bytes[GATHER_MAX_FIELDS];        // per episode
    int32_t vec[GATHER_MAX_FIELDS];          // 16, 8, 4 or 1: widest access the pointers and the size allow
    int32_t n_fields;
    const int64_t* ids;
    int64_t n_src;                           // episodes in the source (ids are checked against it)
};

// Block x of gridDim.x copies the contiguous span [x, x+1) * ceil(n_vec / gridDim.x) of the field: consecutive threads
// take consecutive vectors, eight independent loads in flight per thread.
template <typename V>
__device__ __forceinline__ void copy_span(const char* __restrict__ s, char* __restrict__ d, int64_t n_vec) {
    const V* sv = reinterpret_cast<const V*>(s);
    V* dv = reinterpret_cast<V*>(d);
    const int64_t span = (n_vec + gridDim.x - 1) / gridDim.x;
    const int64_t beg = (int64_t)blockIdx.x * span;
    const int64_t end = beg + span < n_vec ? beg + span : n_vec;
    int64_t i = beg + threadIdx.x;
    constexpr int U = 8;
    for (; i + (U - 1) * 256 < end; i += U * 256) {
        V v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = __ldcs(sv + i + u * 256);
#pragma unroll
        for (int u = 0; u < U; ++u) __stcs(dv + i + u * 256, v[u]);
    }
    for (; i < end; i += 256) __stcs(dv + i, __ldcs(sv + i));
}

// grid: (blocks per episode, n_ids).  Block (x, j) copies its share of episode ids[j] of every field.
__global__ void __launch_bounds__(256) gather_episodes_kernel(GatherArgs A) {
    const int64_t j = blockIdx.y;
    const int64_t id = A.ids[j];
    if (id < 0 || id >= A.n_src) return;                 // invalid id: leave the destination untouched (checked on the host too)
    for (int f = 0; f < A.n_fields; ++f) {
        const char* s = A.src[f] + id * A.bytes[f];
        char* d = A.dst[f] + j * A.bytes[f];
        switch (A.vec[f]) {
            case 16: copy_span<uint4>(s, d, A.bytes[f] / 16); break;
            case 8: copy_span<uint2>(s, d, A.bytes[f] / 8); break;
            case 4: copy_span<uint32_t>(s, d, A.bytes[f] / 4); break;
            case 2: copy_span<uint16_t>(s, d, A.bytes[f] / 2); break;
            default: copy_span<uint8_t>(s, d, A.bytes[f]); break;
        }
    }
}

// ---- the first `steps` timesteps of sampled episodes, from HBM or over PCIe (pmb_gather_episode_steps) ----------------
// A replay buffer in pinned host memory is read by this kernel through its device alias, so the copy is PCIe-bound and
// the read side decides the rate.  One episode's timesteps of one field are ONE contiguous run in source and destination.
// The source run is read in aligned 16-byte words only: a bf16 obs cell at odd O starts 2-byte aligned, and a narrower
// read of mapped host memory is a PCIe request of its own.  The words of a tile are staged in shared memory and shifted
// into place with funnel shifts; destination rows start 16-byte aligned, so every store is a full 16-byte word.  (The
// copy loop of gather_episodes above needs both sides equally aligned, which these runs are not.)
// A CTA's unit of work is a group of up to STEPS_TILES_PER_GROUP tiles of one episode, so trim mode reads the episode's
// `filled` row once per group, not once per tile.  Tiles past the trimmed length F_j are zero-filled without a read.
constexpr int STEPS_MAX_FIELDS = 8;
constexpr int STEPS_THREADS = 256;
constexpr int STEPS_UNROLL = 4;                                  // independent 16-byte loads in flight per thread
constexpr int STEPS_TILE = STEPS_THREADS * STEPS_UNROLL;         // destination words of one tile (16 KB)
constexpr int STEPS_TILES_PER_GROUP = 16;

struct StepsArgs {
    const char* src[STEPS_MAX_FIELDS];       // device addresses
    char* dst[STEPS_MAX_FIELDS];
    int64_t cell[STEPS_MAX_FIELDS];          // bytes of one timestep
    int64_t src_ep[STEPS_MAX_FIELDS];        // T_src * cell
    int64_t dst_sb[STEPS_MAX_FIELDS];        // destination row stride (bytes, multiple of 16)
    int32_t tile0[STEPS_MAX_FIELDS + 1];     // first tile of field f in an episode's tile list; [n_fields] = tiles per episode
    int32_t n_fields, groups_per_ep, steps;
    const int64_t* ids;
    int64_t n_ids, n_src;
    const int64_t* filled;                   // trim mode: [n_src][filled_sb] int64; NULL: copy all `steps`
    int64_t filled_sb;
};

__global__ void __launch_bounds__(STEPS_THREADS) gather_steps_kernel(StepsArgs A) {
    __shared__ uint4 stage[STEPS_TILE + 1];
    __shared__ int copy_steps;
    const int tid = threadIdx.x;
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    const int64_t n_groups = A.n_ids * A.groups_per_ep;
    for (int64_t g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const int64_t j = g / A.groups_per_ep;
        const int q = (int)(g - j * A.groups_per_ep);
        const int64_t id = __ldg(A.ids + j);
        if (id < 0 || id >= A.n_src) continue;                    // invalid id: leave the row untouched (block-uniform)
        if (tid < 32) {
            int F = A.steps;
            if (A.filled) {                                       // F_j = min(steps, l_j + 2), as skip_steps_kernel
                const int64_t* fr = A.filled + id * A.filled_sb;
                int last = -1;
                for (int t0 = A.steps - 1; t0 >= 0 && last < 0; t0 -= 32) {
                    const int t = t0 - tid;
                    const unsigned m = __ballot_sync(0xffffffffu, t >= 0 && fr[t] != 0);
                    if (m) last = t0 - (__ffs((int)m) - 1);
                }
                F = last < 0 ? 0 : min(A.steps, last + 2);
            }
            if (tid == 0) copy_steps = F;
        }
        __syncthreads();
        const int F = copy_steps;
        const int r_end = min((q + 1) * STEPS_TILES_PER_GROUP, A.tile0[A.n_fields]);
        int f = 0;
        for (int r = q * STEPS_TILES_PER_GROUP; r < r_end; ++r) {
            while (r >= A.tile0[f + 1]) ++f;
            const int64_t k0 = (int64_t)(r - A.tile0[f]) * STEPS_TILE;     // first destination word of the tile
            const int64_t n_copy = (int64_t)F * A.cell[f];
            const int64_t n_words = ceil_div((int64_t)A.steps * A.cell[f], 16);
            uint4* d = reinterpret_cast<uint4*>(A.dst[f] + j * A.dst_sb[f]);
            if (16 * k0 >= n_copy) {                              // trimmed tail: zeros, no read
                for (int i = tid; i < STEPS_TILE && k0 + i < n_words; i += STEPS_THREADS) d[k0 + i] = zero;
                continue;
            }
            const char* s = A.src[f] + id * A.src_ep[f];
            const int a = (int)(reinterpret_cast<uintptr_t>(s) & 15);
            const uint4* sv = reinterpret_cast<const uint4*>(s - a);
            const int64_t n_src_words = ceil_div(a + n_copy, 16);          // aligned words holding a byte of the copy
            uint4 v[STEPS_UNROLL];
#pragma unroll
            for (int u = 0; u < STEPS_UNROLL; ++u) {
                const int64_t m = k0 + tid + u * STEPS_THREADS;
                v[u] = m < n_src_words ? __ldcs(sv + m) : zero;
            }
            if (tid == 0) stage[STEPS_TILE] = k0 + STEPS_TILE < n_src_words ? __ldcs(sv + k0 + STEPS_TILE) : zero;
#pragma unroll
            for (int u = 0; u < STEPS_UNROLL; ++u) stage[tid + u * STEPS_THREADS] = v[u];
            __syncthreads();
            // destination word k = source bytes [a + 16 k, a + 16 k + 16) of the aligned stream
            const uint32_t* w32 = reinterpret_cast<const uint32_t*>(stage);
            const unsigned sh = 8u * (unsigned)(a & 3);
#pragma unroll
            for (int u = 0; u < STEPS_UNROLL; ++u) {
                const int i = tid + u * STEPS_THREADS;
                const int64_t k = k0 + i;
                if (k >= n_words) break;
                const int w = 4 * i + (a >> 2);
                uint32_t o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) o[e] = __funnelshift_r(w32[w + e], w32[w + e + 1], sh);
                const int64_t valid = n_copy - 16 * k;            // bytes of this word inside the copied prefix
                if (valid < 16) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int64_t keep = valid - 4 * e;
                        o[e] = keep <= 0 ? 0u : (keep >= 4 ? o[e] : o[e] & ((1u << (8 * keep)) - 1u));
                    }
                }
                d[k] = make_uint4(o[0], o[1], o[2], o[3]);
            }
            __syncthreads();
        }
        __syncthreads();                                          // copy_steps is rewritten by the next group
    }
}

// max_b sum_t filled[b, t]  (episode_buffer.py:255-256), one block per 256 episodes + atomicMax
__global__ void __launch_bounds__(256) max_t_filled_kernel(const int64_t* __restrict__ filled, int64_t B, int T, int64_t sb,
                                                           unsigned long long* __restrict__ out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    long long s = 0;
    if (b < B)
        for (int t = 0; t < T; ++t) s += filled[b * sb + t];
    for (int o = 16; o > 0; o >>= 1) {
        long long v = __shfl_xor_sync(0xffffffffu, s, o);
        s = v > s ? v : s;
    }
    if ((threadIdx.x & 31) == 0 && s > 0) atomicMax(out, (unsigned long long)s);
}

// ---- EpisodeBatch.update on the device (SURVEY.md section 8f, rank 2) -------------------------------------------
// One launch writes every field of an `update(data, bs, ts)` call (components/episode_buffer.py:98-154): cell (i, j) of
// the dense source [nb][nt][cell] goes to episode row(i) / timestep t0 + j of the destination field; `filled` is marked;
// the OneHot preprocess (transforms.py:12-21) is fused: an int64 index cell [G][1] becomes a float32 cell [G][dim].
constexpr int UPDATE_MAX_FIELDS = 12;
struct UpdateArgs {
    const char* src[UPDATE_MAX_FIELDS];
    char* dst[UPDATE_MAX_FIELDS];
    int64_t cell[UPDATE_MAX_FIELDS];         // bytes of one source cell
    int64_t sb[UPDATE_MAX_FIELDS];           // destination batch stride (bytes)
    int64_t st[UPDATE_MAX_FIELDS];           // destination time stride (bytes; 0: episode-constant field)
    int32_t vec[UPDATE_MAX_FIELDS];
    int32_t onehot[UPDATE_MAX_FIELDS];       // > 0: fused OneHot of this width
    int32_t n_fields;
    const int64_t* b_index;                  // device ids of the nb episodes, or NULL: b0 + i * b_step
    int64_t b0, b_step, nb, n_rows, t0, nt;
    int64_t* filled; int64_t filled_sb;      // elements
};

template <typename V>
__device__ __forceinline__ void copy_cell(const char* __restrict__ s, char* __restrict__ d, int64_t n_vec) {
    const V* sv = reinterpret_cast<const V*>(s);
    V* dv = reinterpret_cast<V*>(d);
    for (int64_t i = threadIdx.x; i < n_vec; i += blockDim.x) dv[i] = sv[i];
}

// one block per (episode i, timestep j) cell
__global__ void __launch_bounds__(128) batch_update_kernel(UpdateArgs A) {
    const int64_t c = blockIdx.x;
    const int64_t i = c / A.nt, j = c - i * A.nt;
    const int64_t b = A.b_index ? A.b_index[i] : A.b0 + i * A.b_step;
    if (b < 0 || b >= A.n_rows) return;                   // checked on the host as well
    const int64_t t = A.t0 + j;
    if (A.filled && threadIdx.x == 0) A.filled[b * A.filled_sb + t] = 1;
    for (int f = 0; f < A.n_fields; ++f) {
        const char* s = A.src[f] + c * A.cell[f];
        char* d = A.dst[f] + b * A.sb[f] + t * A.st[f];
        if (A.onehot[f] > 0) {
            const int dim = A.onehot[f];
            const int64_t G = A.cell[f] / 8;              // int64 indices in the cell
            const int64_t* idx = reinterpret_cast<const int64_t*>(s);
            float* o = reinterpret_cast<float*>(d);
            for (int64_t e = threadIdx.x; e < G * dim; e += blockDim.x) {
                const int64_t g = e / dim;
                o[e] = (idx[g] == e - g * dim) ? 1.f : 0.f;
            }
        } else {
            switch (A.vec[f]) {
                case 16: copy_cell<uint4>(s, d, A.cell[f] / 16); break;
                case 8: copy_cell<uint2>(s, d, A.cell[f] / 8); break;
                case 4: copy_cell<uint32_t>(s, d, A.cell[f] / 4); break;
                case 2: copy_cell<uint16_t>(s, d, A.cell[f] / 2); break;
                default: copy_cell<uint8_t>(s, d, A.cell[f]); break;
            }
        }
        // fields are applied in call order like the reference's loop over data.items(): a later field that targets the same
        // cells (insert_episode_batch copies actions_onehot AFTER the preprocess of actions produced it) wins
        __syncthreads();
    }
}

}  // namespace
}  // namespace pmb

using namespace pmb;

// widest copy unit (16, 8, 4, 2 or 1 bytes) that divides every address and size of a field: a bf16 obs cell of an odd obs
// dim (570 bytes at O = 285) moves in 2-byte words instead of bytes
static int vec_width(uintptr_t bits) {
    return (bits & 15) == 0 ? 16 : ((bits & 7) == 0 ? 8 : ((bits & 3) == 0 ? 4 : ((bits & 1) == 0 ? 2 : 1)));
}

extern "C" {

int pmb_gather_episodes(const pmb_gather_field* fields, int32_t n_fields, const int64_t* ep_ids, int64_t n_ids,
                        int64_t n_src_episodes, pmb_stream stream) {
    PMB_REQUIRE(fields && ep_ids && n_fields > 0 && n_fields <= GATHER_MAX_FIELDS, "gather_episodes: 1..%d fields", GATHER_MAX_FIELDS);
    PMB_REQUIRE(n_ids >= 0 && n_ids < 65536 && n_src_episodes > 0, "gather_episodes: 0 <= n_ids < 65536");
    if (n_ids == 0) return PMB_OK;
    GatherArgs A;
    A.n_fields = n_fields; A.ids = ep_ids; A.n_src = n_src_episodes;
    int64_t biggest = 0;
    for (int f = 0; f < n_fields; ++f) {
        PMB_REQUIRE(fields[f].src && fields[f].dst && fields[f].bytes_per_episode > 0, "gather_episodes: field %d is empty", f);
        A.src[f] = static_cast<const char*>(fields[f].src);
        A.dst[f] = static_cast<char*>(fields[f].dst);
        A.bytes[f] = fields[f].bytes_per_episode;
        const uintptr_t bits = reinterpret_cast<uintptr_t>(fields[f].src) | reinterpret_cast<uintptr_t>(fields[f].dst) |
                               (uintptr_t)fields[f].bytes_per_episode;
        A.vec[f] = vec_width(bits);
        if (A.bytes[f] > biggest) biggest = A.bytes[f];
    }
    // enough blocks per episode to give every thread ~32 vectors of the biggest field, at least 4 waves in total
    int64_t bx = ceil_div(biggest / 16, (int64_t)256 * 32);
    const int64_t want = ceil_div((int64_t)4 * sm_count(), n_ids);
    if (bx < want) bx = want;
    if (bx > 1024) bx = 1024;
    if (bx < 1) bx = 1;
    dim3 grid((unsigned)bx, (unsigned)n_ids);
    gather_episodes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(A);
    PMB_LAUNCH_CHECK("gather_episodes_kernel");
    return PMB_OK;
}

// The address the device reads `p` at: device memory as it is, pinned host memory through its mapped alias.  Pageable
// host memory has no device address; a kernel that read it would fault, so it is refused here.
static int device_alias(const void* p, bool host_ok, const void** out, const char* what, int f) {
    cudaPointerAttributes at;
    PMB_CUDA(cudaPointerGetAttributes(&at, p));
    if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) {
        *out = p;
        return PMB_OK;
    }
    PMB_REQUIRE(at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeUnregistered,
                "gather_episode_steps: %s of field %d: unknown memory type", what, f);
    PMB_REQUIRE(host_ok, "gather_episode_steps: %s of field %d must be device memory", what, f);
    PMB_REQUIRE(at.type == cudaMemoryTypeHost,
                "gather_episode_steps: %s of field %d is pageable host memory; the GPU reads a host buffer only when it "
                "is pinned and mapped (ReplayBuffer(..., pin_memory=True) or pin_memory_())", what, f);
    void* d = at.devicePointer;
    if (!d && cudaHostGetDevicePointer(&d, const_cast<void*>(p), 0) != cudaSuccess) {
        (void)cudaGetLastError();
        d = nullptr;
    }
    PMB_REQUIRE(d, "gather_episode_steps: %s of field %d is pinned host memory that is not mapped into the device", what, f);
    *out = d;
    return PMB_OK;
}

int pmb_gather_episode_steps(const pmb_step_field* fields, int32_t n_fields, const int64_t* ep_ids, int64_t n_ids,
                             int64_t n_src_episodes, int32_t T_src, int32_t steps, const int64_t* filled, int32_t trim,
                             pmb_stream stream) {
    PMB_REQUIRE(fields && n_fields > 0 && n_fields <= STEPS_MAX_FIELDS, "gather_episode_steps: 1..%d fields", STEPS_MAX_FIELDS);
    PMB_REQUIRE(n_ids >= 0 && n_src_episodes > 0 && steps > 0 && steps <= T_src, "gather_episode_steps: need n_ids >= 0, "
                "n_src_episodes > 0 and 0 < steps <= T_src");
    PMB_REQUIRE(!trim || filled, "gather_episode_steps: trim mode needs the buffer's filled field");
    if (n_ids == 0) return PMB_OK;
    PMB_REQUIRE(ep_ids, "gather_episode_steps: ep_ids is NULL");
    StepsArgs A;
    A.n_fields = n_fields; A.steps = steps; A.ids = ep_ids; A.n_ids = n_ids; A.n_src = n_src_episodes;
    A.filled = nullptr; A.filled_sb = T_src;
    if (trim) {
        const void* fd = nullptr;
        if (int rc = device_alias(filled, true, &fd, "filled", -1)) return rc;
        A.filled = static_cast<const int64_t*>(fd);
    }
    int64_t tiles = 0;
    for (int f = 0; f < n_fields; ++f) {
        const pmb_step_field& u = fields[f];
        PMB_REQUIRE(u.src && u.dst && u.cell_bytes > 0, "gather_episode_steps: field %d is NULL or empty", f);
        PMB_REQUIRE(u.dst_stride_bytes % 16 == 0 && reinterpret_cast<uintptr_t>(u.dst) % 16 == 0 &&
                    u.dst_stride_bytes >= steps * u.cell_bytes,
                    "gather_episode_steps: field %d: dst must be 16-byte aligned with a stride that is a multiple of 16 "
                    "and holds steps * cell_bytes", f);
        const void* s = nullptr;
        const void* d = nullptr;
        if (int rc = device_alias(u.src, true, &s, "src", f)) return rc;
        if (int rc = device_alias(u.dst, false, &d, "dst", f)) return rc;
        A.src[f] = static_cast<const char*>(s);
        A.dst[f] = static_cast<char*>(const_cast<void*>(d));
        A.cell[f] = u.cell_bytes; A.src_ep[f] = (int64_t)T_src * u.cell_bytes; A.dst_sb[f] = u.dst_stride_bytes;
        A.tile0[f] = (int32_t)tiles;
        tiles += ceil_div(ceil_div((int64_t)steps * u.cell_bytes, 16), STEPS_TILE);
    }
    PMB_REQUIRE(tiles < ((int64_t)1 << 30), "gather_episode_steps: episodes too large");
    A.tile0[n_fields] = (int32_t)tiles;
    A.groups_per_ep = (int32_t)ceil_div(tiles, STEPS_TILES_PER_GROUP);
    // one CTA per SM: 16 KB of loads in flight per SM covers the PCIe round trip many times over, and the CTAs leave
    // room on every SM for the compute kernels of the other chunk of a streamed learner step
    const int64_t n_groups = n_ids * A.groups_per_ep;
    const unsigned grid = (unsigned)(n_groups < sm_count() ? n_groups : sm_count());
    gather_steps_kernel<<<grid, STEPS_THREADS, 0, (cudaStream_t)stream>>>(A);
    PMB_LAUNCH_CHECK("gather_steps_kernel");
    return PMB_OK;
}

int pmb_host_alloc(int64_t bytes, void** out) {
    PMB_REQUIRE(out && bytes > 0, "host_alloc: bytes must be > 0");
    *out = nullptr;
    PMB_CUDA(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocPortable | cudaHostAllocMapped));
    return PMB_OK;
}

int pmb_host_free(void* p) {
    if (p) PMB_CUDA(cudaFreeHost(p));
    return PMB_OK;
}

int pmb_batch_update(const pmb_update_field* fields,int32_t n_fields, const int64_t* b_index, int64_t b0, int64_t b_step,
                     int64_t nb, int64_t n_rows, int64_t t0, int64_t nt, int64_t* filled, int64_t filled_sb, pmb_stream stream) {
    PMB_REQUIRE(fields && n_fields > 0 && n_fields <= UPDATE_MAX_FIELDS, "batch_update: 1..%d fields", UPDATE_MAX_FIELDS);
    PMB_REQUIRE(nb >= 0 && nt > 0 && t0 >= 0 && n_rows > 0 && nb * nt < ((int64_t)1 << 31), "batch_update: bad index range");
    PMB_REQUIRE(b_index || (b0 >= 0 && b_step > 0 && b0 + (nb - 1) * b_step < n_rows), "batch_update: episode range outside the batch");
    if (nb == 0) return PMB_OK;
    UpdateArgs A;
    A.n_fields = n_fields; A.b_index = b_index; A.b0 = b0; A.b_step = b_step; A.nb = nb; A.n_rows = n_rows; A.t0 = t0; A.nt = nt;
    A.filled = filled; A.filled_sb = filled_sb;
    for (int f = 0; f < n_fields; ++f) {
        const pmb_update_field& u = fields[f];
        PMB_REQUIRE(u.src && u.dst && u.cell_bytes > 0, "batch_update: field %d is empty", f);
        PMB_REQUIRE(u.onehot_dim <= 0 || u.cell_bytes % 8 == 0, "batch_update: a one-hot source cell holds int64 indices");
        A.src[f] = static_cast<const char*>(u.src); A.dst[f] = static_cast<char*>(u.dst);
        A.cell[f] = u.cell_bytes; A.sb[f] = u.dst_batch_stride_bytes; A.st[f] = u.dst_time_stride_bytes;
        A.onehot[f] = u.onehot_dim;
        const uintptr_t bits = reinterpret_cast<uintptr_t>(u.src) | reinterpret_cast<uintptr_t>(u.dst) | (uintptr_t)u.cell_bytes |
                               (uintptr_t)u.dst_batch_stride_bytes | (uintptr_t)u.dst_time_stride_bytes;
        A.vec[f] = vec_width(bits);
    }
    batch_update_kernel<<<(unsigned)(nb * nt), 128, 0, (cudaStream_t)stream>>>(A);
    PMB_LAUNCH_CHECK("batch_update_kernel");
    return PMB_OK;
}

int pmb_max_t_filled(const int64_t* filled, int64_t B, int32_t T, int64_t filled_sb, int64_t* out, pmb_stream stream) {
    PMB_REQUIRE(filled && out && B > 0 && T > 0, "max_t_filled: bad arguments");
    cudaStream_t s = (cudaStream_t)stream;
    PMB_CUDA(cudaMemsetAsync(out, 0, sizeof(int64_t), s));
    max_t_filled_kernel<<<(unsigned)ceil_div(B, 256), 256, 0, s>>>(filled, B, T, filled_sb,
                                                                  reinterpret_cast<unsigned long long*>(out));
    PMB_LAUNCH_CHECK("max_t_filled_kernel");
    return PMB_OK;
}

}  // extern "C"
