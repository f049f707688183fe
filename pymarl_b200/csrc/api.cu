#include <cstdlib>
// extern "C" surface of libpymarl_b200.so (see include/pymarl_b200.h) and the orchestration of
// the whole learner step (learners/q_learner.py:37-107).
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <atomic>
#include <mutex>
#include <vector>
#include <cuda_bf16.h>
#include "common.cuh"
#include "gru_tc.cuh"
#include "mixer_tc.cuh"

namespace pmb {

// launchers defined in the other translation units
int gru_fwd_dispatch(const pmb_dims* d, const AgentParams& p, int64_t R, int nt, const float* x, const float* h0,
                     float* h_stash, float* gates, float* q, float* h_last, cudaStream_t s);
int gru_bwd_dispatch(const pmb_dims* d, const pmb_batch* b, const AgentParams& p, const float* x,
                     const float* h_stash, float* gates, const float* d_chosen, float* dpre1, cudaStream_t s,
                     const float* dq_full = nullptr);
int64_t scatter_scratch_bytes(const pmb_dims* d);
int scatter_grads_dispatch(const pmb_dims* d, const pmb_batch* b, const float* h_stash, const float* dpre1,
                           const float* d_chosen, AgentGrads gr, void* scratch, int64_t scratch_bytes, cudaStream_t s,
                           int ti_tiles = 0);
int launch_target_select(const pmb_dims* d, const pmb_batch* b, const float* q_on, const float* q_tg, float* chosen,
                         float* tmax, int32_t* cur_max, cudaStream_t s);
int launch_epsilon_greedy(int64_t rows, int N, int A, const float* q, const int32_t* avail, int64_t avail_sb,
                          float epsilon, const float* u, const float* expo, uint64_t seed, uint64_t offset,
                          int64_t* actions_out, cudaStream_t s);
int launch_mixer_fwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs,
                     int t_off, float* raw, float* q_tot, cudaStream_t s);
int64_t mixer_bwd_scratch_bytes(const pmb_dims* d);
int launch_mixer_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs, float* raw,
                     const float* g, float* d_agent_qs, float* flat_grad_mixer, void* scratch, int64_t scratch_bytes,
                     cudaStream_t s);
int launch_td_loss(const pmb_dims* d, const pmb_batch* b, const float* q_tot, const float* t_tot, float gamma,
                   float* g_out, double* stats, cudaStream_t s, double* partials = nullptr, int64_t partial_bytes = 0);
int launch_stats_reset(double* stats, cudaStream_t s);
int launch_dp_pack(const double* stats, float* tail, cudaStream_t s);
int launch_dp_unpack(const float* tail, double* stats, cudaStream_t s);
// coma.cu
int coma_launch_inputs(const pmb_dims* d, const pmb_batch* b, int t0, int nt, float* out, cudaStream_t s);
int coma_launch_gather_taken(const pmb_dims* d, const pmb_batch* b, int t0, int nt, const float* q, float* taken, cudaStream_t s);
int coma_launch_td_lambda(const pmb_dims* d, const pmb_batch* b, float gamma, float lam, const float* taken, float* targets,
                          cudaStream_t s);
int coma_launch_critic_td(const pmb_dims* d, const pmb_batch* b, int t, const float* q_t, const float* targets, float* q_vals,
                          float* dqv, int32_t* dqa, double* stats_row, double* partials, cudaStream_t s);
int coma_launch_critic_bwd_pointwise(int64_t R, int A, int Hc, const float* dqv, const int32_t* dqa, const float* w3,
                                     const float* x2, float* dq_dense, float* dx2, cudaStream_t s);
int launch_relu_mask(int64_t n, const float* x, float* dx, cudaStream_t s);
int launch_transpose(int rows, int cols, const float* in, float* out, cudaStream_t s);
int coma_launch_policy(const pmb_dims* d, const pmb_batch* b, float eps, const float* logits, const float* q_vals,
                       float* dlogits, float* pi_out, double* stats_row, double* partials, cudaStream_t s);
int launch_policy_head(int64_t rows, int A, float eps, int test_mode, const float* logits, const int32_t* avail, float* probs,
                       cudaStream_t s);
int launch_multinomial(int64_t rows, int A, const float* probs, const int32_t* avail, const float* expo, int greedy,
                       uint64_t seed, uint64_t offset, int64_t* out, cudaStream_t s);
int launch_clip_rmsprop(int64_t n, float* p, float* g, float* sq, float* target, int do_sync, double* stats, float lr,
                        float alpha, float eps, float clip, float* scratch, cudaStream_t s, int skip_if_empty = 0);

// tc_gemm.cu (bf16 tcgen05 tier)
int tc_gemm_plain(const float* A, RowMap amap, int64_t M, int K, const __nv_bfloat16* Wp, int Ncols_padded, int Nreal,
                  const float* bias, float* C, int64_t ldc, cudaStream_t s);
int tc_fc1_fwd_both(const pmb_dims* d, const pmb_batch* b, int t0, int nt, const AgentParams& on, const AgentParams& tg,
                    float* x_on, float* x_tg, int tile_images, uint8_t* obs_img_out, uint32_t* relu_mask, void* scratch,
                    int64_t scratch_bytes, cudaStream_t s, int weights_packed = 0, const int32_t* live_items = nullptr);
// tc_atb.cu (tile-image D operand)
int tc_gemm_atb_ti(const uint8_t* d_ti, int T, int N, int64_t R, int n_tiles, const float* A, RowMap amap, int K,
                   float* out, int64_t ldo, float* bias_out, void* scratch, int64_t scratch_bytes, cudaStream_t s);
int64_t tc_atb_ti_scratch_bytes(int T, int n_tiles, int K);
int64_t tc_fc1_scratch_bytes(const pmb_dims* d);
bool tc_fc1_streams(const pmb_dims* d, int obs_dtype);

static thread_local char g_err[512] = "";
std::atomic<long long> g_launch_count{0};

// ---- optional per-phase timing (pmb_profile_begin / pmb_profile_end) --------------------------
// When armed, the step records a CUDA event on the launch stream between its kernels; the
// host reads the elapsed times after the step.  Disarmed (the default) it costs one branch.
// Per host thread (the thread that arms the timer is the thread that launches); up to kMaxPhases phases per
// begin/end pair, i.e. several steps of the learner can be profiled back to back inside one timed region.
constexpr int kMaxPhases = 1024;
struct PhaseTimer {
    bool armed = false;
    int n = 0;
    int created = 0;                       // events created so far (lazily, only as many as are used)
    cudaEvent_t ev[kMaxPhases + 1];
    const char* name[kMaxPhases];
};
static thread_local PhaseTimer g_timer;

static void phase_mark(cudaStream_t s, const char* name) {
    PhaseTimer& t = g_timer;
    if (!t.armed) return;
    if (t.n > kMaxPhases) return;
    while (t.created <= t.n) cudaEventCreate(&t.ev[t.created++]);
    cudaEventRecord(t.ev[t.n], s);           // event i closes phase i-1 and opens phase i
    if (t.n < kMaxPhases) t.name[t.n] = name;
    t.n++;
}
#define PHASE(s, name) phase_mark(s, name)

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    set_error("CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorName(e), file, line, what);
    return PMB_ERR_CUDA;
}

bool rollout_pdl_enabled() {
    static const bool on = [] { const char* e = getenv("PMB_ROLLOUT_PDL"); return !(e && e[0] == '0'); }();
    return on;
}

// SM count of the CURRENT device (cached per device ordinal)
int sm_count() {
    constexpr int kMaxDev = 64;
    static std::atomic<int> cached[kMaxDev];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDev) return 148;
    int n = cached[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;   // B200
        cached[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device, size) instead of on every launch
cudaError_t set_smem_attr(const void* func, int bytes) {
    struct Key { const void* f; int dev, bytes; };
    static std::mutex mu;
    static std::vector<Key> done;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    for (const Key& k : done)
        if (k.f == func && k.dev == dev && k.bytes >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done.push_back(Key{func, dev, bytes});
    return e;
}

// Side stream + fork / join events of the CURRENT device, created on first use (never while a graph is being captured:
// the learner runs every new configuration once eagerly before it captures).  The forward pass forks the target net's
// recurrence onto the side stream when both recurrences fit on the device side by side.
struct SideStream { cudaStream_t stream = nullptr; cudaEvent_t fork = nullptr, join = nullptr, fork2 = nullptr, join2 = nullptr; };
static int side_stream(SideStream** out) {
    constexpr int kMaxDev = 64;
    static SideStream table[kMaxDev];
    static std::mutex mu;
    int dev = 0;
    PMB_CUDA(cudaGetDevice(&dev));
    PMB_REQUIRE(dev >= 0 && dev < kMaxDev, "device ordinal %d out of range", dev);
    std::lock_guard<std::mutex> lock(mu);
    SideStream& e = table[dev];
    if (!e.stream) {
        PMB_CUDA(cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking));
        PMB_CUDA(cudaEventCreateWithFlags(&e.fork, cudaEventDisableTiming));
        PMB_CUDA(cudaEventCreateWithFlags(&e.join, cudaEventDisableTiming));
        PMB_CUDA(cudaEventCreateWithFlags(&e.fork2, cudaEventDisableTiming));
        PMB_CUDA(cudaEventCreateWithFlags(&e.join2, cudaEventDisableTiming));
    }
    *out = &e;
    return PMB_OK;
}

int validate_dims(const pmb_dims* d) {
    PMB_REQUIRE(d != nullptr, "dims is NULL");
    PMB_REQUIRE(d->B > 0 && d->T > 0 && d->N > 0 && d->O > 0 && d->A > 0, "B, T, N, O, A must be positive");
    PMB_REQUIRE(d->H == 16 || d->H == 32 || d->H == 64, "rnn_hidden_dim %d unsupported (16, 32, 64)", d->H);
    PMB_REQUIRE(d->mixer >= PMB_MIXER_NONE && d->mixer <= PMB_MIXER_QMIX, "unknown mixer id %d", d->mixer);
    if (d->mixer == PMB_MIXER_QMIX) {
        PMB_REQUIRE(d->S > 0, "QMIX needs a positive state dim");
        PMB_REQUIRE(d->E > 0 && d->E <= 64, "mixing_embed_dim %d unsupported (1..64)", d->E);
    }
    return PMB_OK;
}

void compute_layout(const pmb_dims* d, pmb_layout* L) {
    const int64_t H = d->H, A = d->A, Din = d_in_of(d), S = d->S, N = d->N, E = d->E;
    int64_t numel[PMB_P_COUNT] = {H * Din, H, 3 * H * H, 3 * H * H, 3 * H, 3 * H, A * H, A,
                                  N * E * S, E * S, E * S, E * S, N * E, E, E, E, E, 1};
    int64_t off = 0;
    for (int i = 0; i < PMB_P_COUNT; ++i) {
        bool is_mixer = i >= PMB_P_HW1_W;
        L->numel[i] = (is_mixer && d->mixer != PMB_MIXER_QMIX) ? 0 : numel[i];
        L->offset[i] = off;
        off += L->numel[i];
        if (i == PMB_P_FC2_B) L->n_agent = off;
    }
    L->n_total = off;
}

namespace {

struct WsPlan {
    int64_t off[18];
    int64_t scratch_bytes;
    int64_t mixdw_bytes;
    int64_t sched_bytes;           // the padded-step skipping schedule (0 when pmb_dims.reserved bit 1 is not honoured)
    int64_t total;
};

// The fused tensor-core path: tcgen05 agent kernels, the image-fed QMIX mixer (VDN and IQL need none), the streaming fc1
// kernel (obs dim <= 320) with one-hot(agent) + ones folded into the K padding.  Zero-copy replay sampling (ep_index)
// and padded-step skipping need it.
bool fused_tc_path(const pmb_dims* d) {
    const bool tc_agent = d->precision == PMB_PREC_BF16 && d->H == 64 && d->A <= 64;
    const bool tc_mixer = d->precision == PMB_PREC_BF16 && d->mixer == PMB_MIXER_QMIX && d->E == 32;
    return tc_agent && (d->mixer != PMB_MIXER_QMIX || tc_mixer) && d->O <= 320 && ((d->O + 63) / 64) * 64 - d->O >= d->N + 1;
}

// pmb_dims.reserved bit 1 (pmb_qlearner_train_step): skip the padded steps of a ragged batch.  Ignored off the fused path.
bool skip_padding(const pmb_dims* d) { return (d->reserved & 2) && fused_tc_path(d); }

bool rollout_tc_ok(const pmb_dims* d) {
    return d->precision == PMB_PREC_BF16 && d->H == 64 && d->A <= 64 && d->O <= 320;
}

// Where the kernels read bf16 obs (pmb_batch.obs_dtype) natively: the streaming fc1 kernels are the only obs readers of
// the fused learner step (the fc1 / fc2 weight gradients read the obs tile images they write) and of the tensor-core
// rollout step.
bool obs_bf16_native(const pmb_dims* d, int entry) {
    if (entry == PMB_ENTRY_TRAIN_STEP) return fused_tc_path(d) && tc_fc1_streams(d, PMB_DTYPE_BF16);
    if (entry == PMB_ENTRY_SELECT_ACTIONS) return rollout_tc_ok(d) && tc_fc1_streams(d, PMB_DTYPE_BF16);
    return false;
}

static_assert(sizeof(pmb_batch) == 128, "pmb_batch: state_dtype / avail_dtype live in the former tail padding");

// Where the kernels read compact state / avail natively: the q-select epilogue is the only avail reader of the
// tensor-core agent's learner step, state_to_images_kernel the only state reader of the tensor-core mixer, and the
// rollout kernel the only avail reader of the tensor-core rollout step.
bool field_dtype_native(const pmb_dims* d, int entry, int field, int dtype) {
    if (field < PMB_FIELD_OBS || field > PMB_FIELD_AVAIL) return false;
    if (dtype == PMB_DTYPE_F32) return entry == PMB_ENTRY_TRAIN_STEP || entry == PMB_ENTRY_SELECT_ACTIONS;
    const bool tc_agent = d->precision == PMB_PREC_BF16 && d->H == 64 && d->A <= 64;
    const bool tc_mixer = d->precision == PMB_PREC_BF16 && d->mixer == PMB_MIXER_QMIX && d->E == 32;
    if (field == PMB_FIELD_OBS) return dtype == PMB_DTYPE_BF16 && obs_bf16_native(d, entry);
    if (field == PMB_FIELD_STATE) return dtype == PMB_DTYPE_BF16 && entry == PMB_ENTRY_TRAIN_STEP && tc_mixer;
    if (field == PMB_FIELD_AVAIL && dtype == PMB_DTYPE_U8)
        return (entry == PMB_ENTRY_TRAIN_STEP && tc_agent) || (entry == PMB_ENTRY_SELECT_ACTIONS && rollout_tc_ok(d));
    return false;
}

// batch.{obs,state,avail}_dtype of a call to `who`: the reference types always, compact ones where `entry` reads them
// natively (entry < 0: nowhere)
int check_dtypes(const pmb_dims* d, const pmb_batch* b, int entry, const char* who) {
    PMB_REQUIRE(b->obs_dtype == PMB_DTYPE_F32 || b->obs_dtype == PMB_DTYPE_BF16, "%s: unknown batch.obs_dtype %d", who,
                (int)b->obs_dtype);
    PMB_REQUIRE(b->obs_dtype == PMB_DTYPE_F32 || (entry >= 0 && obs_bf16_native(d, entry)),
                "%s: bf16 obs is not read natively for these dims (see pmb_obs_bf16_supported); convert obs to fp32", who);
    PMB_REQUIRE(b->state_dtype == PMB_DTYPE_F32 || b->state_dtype == PMB_DTYPE_BF16, "%s: unknown batch.state_dtype %d",
                who, (int)b->state_dtype);
    PMB_REQUIRE(b->state_dtype == PMB_DTYPE_F32 || field_dtype_native(d, entry, PMB_FIELD_STATE, b->state_dtype),
                "%s: bf16 state is not read natively for these dims (see pmb_field_dtype_supported); convert state to fp32",
                who);
    PMB_REQUIRE(b->avail_dtype == PMB_DTYPE_F32 || b->avail_dtype == PMB_DTYPE_U8, "%s: unknown batch.avail_dtype %d",
                who, (int)b->avail_dtype);
    PMB_REQUIRE(b->avail_dtype == PMB_DTYPE_F32 || field_dtype_native(d, entry, PMB_FIELD_AVAIL, b->avail_dtype),
                "%s: uint8 avail is not read natively for these dims (see pmb_field_dtype_supported); convert avail to int32",
                who);
    return PMB_OK;
}

// the fields of an entry point that accepted the reference types only
const float* obs_f32(const pmb_batch* b) { return static_cast<const float*>(b->obs); }
const int32_t* avail_i32(const pmb_batch* b) { return static_cast<const int32_t*>(b->avail); }

int64_t agent_bwd_scratch(const pmb_dims* d) {
    const int64_t rows = (int64_t)d->T * d->B * d->N;
    int64_t a = atb_scratch_bytes(d->precision, 3 * d->H, d->H, rows);
    int64_t b = atb_scratch_bytes(d->precision, d->H, d->O, rows);
    int64_t c = scatter_scratch_bytes(d);
    int64_t m = a > b ? a : b;
    return m > c ? m : c;
}

WsPlan plan_workspace(const pmb_dims* d) {
    const int64_t R = (int64_t)d->B * d->N, T = d->T, H = d->H, A = d->A, N = d->N;
    const int64_t M = (int64_t)d->B * (T - 1);
    const int64_t C = (int64_t)(N + 3) * d->E;
    const bool qmix = d->mixer == PMB_MIXER_QMIX, iql = d->mixer == PMB_MIXER_NONE;
    const int64_t W = iql ? N : 1;
    // the bf16 tier stores x / h / gates as bf16 tile images (128-row tiles, 16 KB each); take the larger size
    const int64_t n_tiles = ceil_div(R, 128), ti = d->precision == PMB_PREC_BF16 ? 4096 : 0;   // floats per tile
    auto mx = [](int64_t a, int64_t b) { return a > b ? a : b; };
    const bool tc_mix = qmix && d->precision == PMB_PREC_BF16 && d->E == 32;
    int64_t sizes[18] = {
        mx(T * R * H, T * n_tiles * ti),               // 0 x_on
        mx(T * R * H, T * n_tiles * ti),               // 1 x_tg (reused as dpre1 in the backward)
        mx((T + 1) * R * H, (T + 1) * n_tiles * ti),   // 2 h_stash
        mx(T * R * 4 * H, T * n_tiles * 4 * ti),       // 3 gates
        T * R * A,                 // 4 q_on
        T * R * A,                 // 5 q_tg
        M * N,                     // 6 chosen
        M * N,                     // 7 tmax
        // 8 raw: hypernet outputs of the online mixer (bf16 tier: tile images, see mixer_tc.cuh)
        qmix ? (tc_mix ? tc_raw_img_bytes(d) / 4 : M * C) : 0,
        // 9 obs tile images [T][n_tiles][ceil(O/64)][16 KB] written by the fc1 GEMM, read by agent_dw_tc
        (d->precision == PMB_PREC_BF16 && d->H == 64) ? T * n_tiles * ((d->O + 63) / 64) * ti : 0,
        iql ? 0 : M,               // 10 q_tot
        iql ? 0 : M,               // 11 t_tot
        M * W,                     // 12 g
        iql ? 0 : M * N,           // 13 d_chosen
        tc_mix ? tc_state_img_bytes(d) / 4 : 0,   // 14 state tile images (bf16 tier)
        // 15 h images of the TARGET net (bf16 tier: q = fc2(h) is computed from the images by q_select)
        (d->precision == PMB_PREC_BF16 && d->H == 64) ? (T + 1) * n_tiles * ti : 0,
        // 16 ReLU mask of the online fc1 output, one bit per element: [T][n_tiles][2][128] words
        (d->precision == PMB_PREC_BF16 && d->H == 64) ? T * n_tiles * 256 : 0,
        0                          // 17 scratch (bytes, below)
    };
    WsPlan p;
    int64_t off = 0;
    for (int i = 0; i < 17; ++i) {
        p.off[i] = off;
        off += align_up(sizes[i] * 4, 256);
    }
    int64_t sc = agent_bwd_scratch(d);
    int64_t mb = mixer_bwd_scratch_bytes(d);
    if (mb > sc) sc = mb;
    if (d->precision == PMB_PREC_BF16) {
        int64_t f = tc_fc1_scratch_bytes(d);
        if (f > sc) sc = f;
        int64_t g = 131072 + tc_gru_bwd2_partial_bytes((int)ceil_div((int64_t)d->B * d->N, 128));
        if (g > sc) sc = g;
        int64_t a2 = tc_atb_ti_scratch_bytes(d->T, (int)ceil_div((int64_t)d->B * d->N, 128), d->O);
        if (a2 > sc) sc = a2;
        if (tc_agent_dw_scratch_bytes() > sc) sc = tc_agent_dw_scratch_bytes();
        if (tc_mix) {
            int64_t m2 = tc_mixer_scratch_bytes(d); if (m2 > sc) sc = m2;
            int64_t m3 = tc_mixer_bwd_img_scratch_bytes(d); if (m3 > sc) sc = m3;
        }
    }
    if (sc < 65536) sc = 65536;                  // >= the per-block partial sums of td_loss (8 x SMs x 5 doubles)
    p.off[17] = off;
    p.scratch_bytes = align_up(sc, 256);
    // behind the scratch area: the slice partials of the hypernet weight-gradient GEMM when it runs on the side stream next
    // to the agent's BPTT (which owns the scratch area then)
    p.mixdw_bytes = (tc_mix && d->H == 64) ? tc_mixer_dw_scratch_bytes(d) : 0;
    p.sched_bytes = skip_padding(d) ? skip_schedule_bytes(d->B, d->T, (int)n_tiles) : 0;
    p.total = off + p.scratch_bytes + p.mixdw_bytes + p.sched_bytes;
    return p;
}

void fill_views(const pmb_dims* d, void* ws, const WsPlan& p, pmb_ws_views* v) {
    char* base = static_cast<char*>(ws);
    auto f = [&](int i) { return reinterpret_cast<float*>(base + p.off[i]); };
    const bool iql = d->mixer == PMB_MIXER_NONE;
    v->x_on = f(0); v->x_tg = f(1); v->h_stash = f(2); v->gates = f(3); v->q_on = f(4); v->q_tg = f(5);
    v->chosen = f(6); v->tmax = f(7); v->raw_on = f(8); v->raw_tg = f(8);
    v->q_tot = iql ? v->chosen : f(10);
    v->t_tot = iql ? v->tmax : f(11);
    v->g = f(12);
    v->d_chosen = iql ? v->g : f(13);
    v->scratch = f(17);
    v->relu_mask = f(16);
    v->state_img = f(14);
    v->h_tg = f(15);
    v->scratch_bytes = p.scratch_bytes;
    v->obs_img = f(9);
    v->ep_order = nullptr;
    v->tile_steps = nullptr;
    if (p.sched_bytes) {
        SkipSchedule S = skip_schedule_views(base + p.total - p.sched_bytes, d->B, d->T, (int)ceil_div((int64_t)d->B * d->N, 128));
        v->ep_order = S.ep_order;
        v->tile_steps = S.tile_steps;
    }
}

int fc1_fwd(const pmb_dims* d, const pmb_batch* b, int t0, int nt, const AgentParams& ap, float* x_out,
            cudaStream_t s) {
    const int64_t M = (int64_t)d->B * nt * d->N;
    RowMap map{b->obs_sb, (int64_t)d->N * d->O, (int64_t)d->O, nt, d->N};
    Fc1Epilogue ep;
    ep.fc1_w = ap.fc1_w; ep.fc1_b = ap.fc1_b;
    ep.actions = b->actions; ep.actions_sb = b->actions_sb;
    ep.filled = b->filled; ep.filled_sb = b->filled_sb;
    ep.x_out = x_out;
    ep.T_batch = d->T; ep.t0 = t0; ep.nt = nt; ep.N = d->N; ep.O = d->O; ep.A = d->A; ep.H = d->H;
    ep.D_in = d_in_of(d); ep.use_act = d->obs_last_action; ep.use_id = d->obs_agent_id;
    ep.R = (int64_t)d->B * d->N;
    return launch_fc1_gemm(obs_f32(b) + (int64_t)t0 * d->N * d->O, map, M, d->O, ap.fc1_w, ep.D_in, d->H, ep, s);
}

int agent_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_agent, const float* x_on, const float* h_stash,
              float* gates, const float* d_chosen, float* dpre1, float* flat_grad_agent, void* scratch,
              int64_t scratch_bytes, cudaStream_t s, const float* dq_full = nullptr) {
    AgentParams ap = agent_params(d, flat_agent);
    AgentGrads gr = agent_grads(d, flat_grad_agent);
    const int64_t R = (int64_t)d->B * d->N, rows = (int64_t)d->T * R;
    const int H = d->H;
    PHASE(s, "gru_unroll_bwd");
    int rc = gru_bwd_dispatch(d, b, ap, x_on, h_stash, gates, d_chosen, dpre1, s, dq_full);
    if (rc) return rc;
    PHASE(s, "dW_rnn_gemm_atb");
    // rnn.weight_ih / bias_ih:  [da_r | da_z | da_n]^T . x
    const int prec = d->precision;
    rc = gemm_atb_any(prec, gates, dense_map(4 * H), 3 * H, x_on, dense_map(H), H, rows, gr.w_ih, H, gr.b_ih, scratch,
                      scratch_bytes, s);
    if (rc) return rc;
    // rnn.weight_hh / bias_hh:  [da_r | da_z | da_n * r]^T . h_{t-1}   (h_stash slot t holds h_{t-1})
    rc = gemm_atb_any(prec, gates, dense_map(4 * H), 2 * H, h_stash, dense_map(H), H, rows, gr.w_hh, H, gr.b_hh, scratch,
                      scratch_bytes, s);
    if (rc) return rc;
    rc = gemm_atb_any(prec, gates + 3 * H, dense_map(4 * H), H, h_stash, dense_map(H), H, rows,
                      gr.w_hh + (int64_t)2 * H * H, H, gr.b_hh + 2 * H, scratch, scratch_bytes, s);
    if (rc) return rc;
    PHASE(s, "dW_fc1_gemm_atb");
    // fc1.weight[:, :O] / fc1.bias:  dpre1^T . obs   (dpre1 time major, obs batch major)
    RowMap dmap{(int64_t)d->N * H, R * H, (int64_t)H, d->T, d->N};
    RowMap omap{b->obs_sb, (int64_t)d->N * d->O, (int64_t)d->O, d->T, d->N};
    rc = gemm_atb_any(prec, dpre1, dmap, H, obs_f32(b), omap, d->O, rows, gr.fc1_w, d_in_of(d), gr.fc1_b, scratch,
                      scratch_bytes, s);
    if (rc) return rc;
    PHASE(s, "agent_scatter_grads");
    rc = scatter_grads_dispatch(d, b, h_stash, dpre1, dq_full ? nullptr : d_chosen, gr, scratch, scratch_bytes, s);
    if (rc || !dq_full) return rc;
    // dense dq (COMA): fc2.weight / fc2.bias = dq^T . h_t over all (t, row); h_stash slot t + 1 holds h_t
    return gemm_atb_any(PMB_PREC_FP32, dq_full, dense_map(d->A), d->A, h_stash + R * H, dense_map(H), H, rows, gr.fc2_w, H,
                        gr.fc2_b, scratch, scratch_bytes, s);
}

// GRU / fc2 weight images of one agent: [w_ih 24 KB | w_hh 24 KB | fc2 8 KB] (bf16, K-major, 128B swizzle)
int pack_gru_images(const pmb_dims* d, const AgentParams& ap, char* base, cudaStream_t s) {
    // ONE launch: rnn.weight_ih (192 rows) | rnn.weight_hh (192) | fc2.weight (A rows, zero rows up to 64) stacked into one
    // [448 x 64] image = the three images at byte offsets 0 / 24576 / 49152
    const float* p[4] = {ap.w_ih, ap.w_hh, ap.fc2_w, nullptr};
    int r[4] = {192, 192, d->A, 64 - d->A}, l[4] = {64, 64, 64, 64};
    return tc_pack_w(p, r, l, 4, 64, reinterpret_cast<__nv_bfloat16*>(base), s);
}

}  // namespace
}  // namespace pmb

using namespace pmb;

extern "C" {

const char* pmb_last_error(void) { return g_err; }

int64_t pmb_launch_count(void) { return (int64_t)g_launch_count; }

int pmb_profile_begin(void) {
    g_timer.armed = true;
    g_timer.n = 0;
    return PMB_OK;
}

int pmb_profile_end(float* ms_host, char* names_host, int32_t names_stride, int32_t max_phases, int32_t* n_out) {
    PhaseTimer& t = g_timer;
    t.armed = false;
    int n = t.n > 0 ? t.n - 1 : 0;                 // n+1 events delimit n phases
    if (n > kMaxPhases) n = kMaxPhases;
    if (n > 0) PMB_CUDA(cudaEventSynchronize(t.ev[n]));
    int m = n < max_phases ? n : max_phases;
    for (int i = 0; i < m; ++i) {
        float ms = 0.f;
        PMB_CUDA(cudaEventElapsedTime(&ms, t.ev[i], t.ev[i + 1]));
        if (ms_host) ms_host[i] = ms;
        if (names_host && names_stride > 0) {
            strncpy(names_host + (size_t)i * names_stride, t.name[i], names_stride - 1);
            names_host[(size_t)i * names_stride + names_stride - 1] = 0;
        }
    }
    if (n_out) *n_out = m;
    t.n = 0;
    return PMB_OK;
}
int pmb_version(void) { return 200; }

int pmb_h2d_rows(void* dst_dev, const void* src_host, int64_t rows, int64_t row_bytes, int64_t src_pitch_bytes,
                 pmb_stream stream) {
    PMB_REQUIRE(dst_dev && src_host && rows > 0 && row_bytes > 0 && src_pitch_bytes >= row_bytes, "h2d_rows: bad arguments");
    PMB_CUDA(cudaMemcpy2DAsync(dst_dev, (size_t)row_bytes, src_host, (size_t)src_pitch_bytes, (size_t)row_bytes, (size_t)rows,
                               cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return PMB_OK;
}

int pmb_device_info(int32_t* sm, int32_t* cc_major, int32_t* cc_minor, int64_t* smem_optin) {
    int dev = 0;
    PMB_CUDA(cudaGetDevice(&dev));
    int v = 0;
    PMB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev)); if (sm) *sm = v;
    PMB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev)); if (cc_major) *cc_major = v;
    PMB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev)); if (cc_minor) *cc_minor = v;
    PMB_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev)); if (smem_optin) *smem_optin = v;
    return PMB_OK;
}

int pmb_flat_layout(const pmb_dims* d, pmb_layout* out) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(out != nullptr, "layout out is NULL");
    compute_layout(d, out);
    return PMB_OK;
}

int pmb_obs_bf16_supported(const pmb_dims* d, int32_t entry) {
    if (validate_dims(d)) return 0;
    return obs_bf16_native(d, entry) ? 1 : 0;
}

int pmb_field_dtype_supported(const pmb_dims* d, int32_t entry, int32_t field, int32_t dtype) {
    if (validate_dims(d)) return 0;
    return field_dtype_native(d, entry, field, dtype) ? 1 : 0;
}

int64_t pmb_learner_workspace_bytes(const pmb_dims* d) {
    if (validate_dims(d) || d->T < 2) return -1;
    return plan_workspace(d).total;
}

int pmb_learner_workspace_views(const pmb_dims* d, void* workspace, int64_t workspace_bytes, pmb_ws_views* out) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2, "T must be >= 2");
    WsPlan p = plan_workspace(d);
    if (workspace_bytes < p.total) { set_error("workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)p.total); return PMB_ERR_WORKSPACE; }
    fill_views(d, workspace, p, out);
    return PMB_OK;
}

int pmb_agent_fc1_fwd(const pmb_dims* d, const pmb_batch* b, int32_t t0, int32_t nt, const float* flat_agent,
                      float* x_out, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(b && b->obs && flat_agent && x_out, "fc1_fwd: NULL pointer");
    PMB_REQUIRE(b == nullptr || b->ep_index == nullptr, "pmb_agent_fc1_fwd: batch.ep_index is only supported by pmb_qlearner_train_step");
    PMB_REQUIRE(t0 >= 0 && nt > 0 && t0 + nt <= d->T, "fc1_fwd: bad time range [%d, %d) for T = %d", t0, t0 + nt, d->T);
    PMB_REQUIRE(!d->obs_last_action || (b->actions && b->filled), "fc1_fwd: obs_last_action needs actions and filled");
    if ((rc = check_dtypes(d, b, -1, "pmb_agent_fc1_fwd"))) return rc;
    return fc1_fwd(d, b, t0, nt, agent_params(d, flat_agent), x_out, (cudaStream_t)stream);
}

int pmb_agent_fc1_dense_fwd(const pmb_dims* d, int64_t rows, int32_t d_in, const float* inputs, const float* flat_agent,
                            float* x_out, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(inputs && flat_agent && x_out, "fc1_dense_fwd: NULL pointer");
    PMB_REQUIRE(d_in == d_in_of(d), "fc1_dense_fwd: input width %d != %d", d_in, d_in_of(d));
    AgentParams ap = agent_params(d, flat_agent);
    return launch_gemm_tn(inputs, dense_map(d_in), rows, d_in, ap.fc1_w, d_in, d->H, ap.fc1_b, x_out, d->H, 1,
                          (cudaStream_t)stream);
}

int pmb_agent_gru_unroll_fwd(const pmb_dims* d, int64_t rows, int32_t nt, const float* flat_agent, const float* x,
                             const float* h0, float* h_stash, float* gates, float* q, float* h_last,
                             pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(flat_agent && x && q, "gru_unroll_fwd: NULL pointer");
    PMB_REQUIRE(rows > 0 && nt > 0, "gru_unroll_fwd: rows and nt must be positive");
    return gru_fwd_dispatch(d, agent_params(d, flat_agent), rows, nt, x, h0, h_stash, gates, q, h_last,
                            (cudaStream_t)stream);
}

int pmb_target_select(const pmb_dims* d, const pmb_batch* b, const float* q_on, const float* q_tg, float* chosen,
                      float* tmax, int32_t* cur_max, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2, "target_select: T must be >= 2");
    PMB_REQUIRE(b && b->avail && b->actions && q_on && q_tg && chosen && tmax, "target_select: NULL pointer");
    PMB_REQUIRE(b == nullptr || b->ep_index == nullptr, "pmb_target_select: batch.ep_index is only supported by pmb_qlearner_train_step");
    if ((rc = check_dtypes(d, b, -1, "pmb_target_select"))) return rc;
    return launch_target_select(d, b, q_on, q_tg, chosen, tmax, cur_max, (cudaStream_t)stream);
}

int pmb_mixer_fwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs,
                  int32_t t_off, float* raw, float* q_tot, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2 && (t_off == 0 || t_off == 1), "mixer_fwd: bad T / t_off");
    PMB_REQUIRE(agent_qs && q_tot, "mixer_fwd: NULL pointer");
    PMB_REQUIRE(b == nullptr || b->ep_index == nullptr, "mixer_fwd: batch.ep_index is only supported by pmb_qlearner_train_step");
    if (b && (rc = check_dtypes(d, b, -1, "pmb_mixer_fwd"))) return rc;
    return launch_mixer_fwd(d, b, flat_mixer, agent_qs, t_off, raw, q_tot, (cudaStream_t)stream);
}

int pmb_stats_reset(double* stats, pmb_stream stream) {
    PMB_REQUIRE(stats, "stats is NULL");
    return launch_stats_reset(stats, (cudaStream_t)stream);
}

int pmb_td_loss(const pmb_dims* d, const pmb_batch* b, const float* q_tot, const float* t_tot, float gamma,
                float* g_out, double* stats, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2, "td_loss: T must be >= 2");
    PMB_REQUIRE(b && b->reward && b->terminated && b->filled && q_tot && t_tot && g_out && stats, "td_loss: NULL pointer");
    if ((rc = check_dtypes(d, b, -1, "pmb_td_loss"))) return rc;
    return launch_td_loss(d, b, q_tot, t_tot, gamma, g_out, stats, (cudaStream_t)stream);
}

int64_t pmb_mixer_bwd_workspace_bytes(const pmb_dims* d) {
    if (validate_dims(d) || d->T < 2) return -1;
    return mixer_bwd_scratch_bytes(d);
}

int pmb_mixer_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs, float* raw,
                  const float* g, float* d_agent_qs, float* flat_grad_mixer, void* scratch, int64_t scratch_bytes,
                  pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2 && g && d_agent_qs, "mixer_bwd: bad arguments");
    PMB_REQUIRE(b == nullptr || b->ep_index == nullptr, "mixer_bwd: batch.ep_index is only supported by pmb_qlearner_train_step");
    if (b && (rc = check_dtypes(d, b, -1, "pmb_mixer_bwd"))) return rc;
    return launch_mixer_bwd(d, b, flat_mixer, agent_qs, raw, g, d_agent_qs, flat_grad_mixer, scratch, scratch_bytes,
                            (cudaStream_t)stream);
}

int64_t pmb_agent_bwd_workspace_bytes(const pmb_dims* d) {
    if (validate_dims(d)) return -1;
    return agent_bwd_scratch(d);
}

int pmb_agent_unroll_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_agent, const float* x_on,
                         const float* h_stash, float* gates, const float* d_chosen, float* dpre1,
                         float* flat_grad_agent, void* scratch, int64_t scratch_bytes, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2, "agent_unroll_bwd: T must be >= 2");
    PMB_REQUIRE(b == nullptr || b->ep_index == nullptr, "pmb_agent_unroll_bwd: batch.ep_index is only supported by pmb_qlearner_train_step");
    PMB_REQUIRE(b && b->obs && b->actions && b->filled && flat_agent && x_on && h_stash && gates && d_chosen && dpre1 &&
                    flat_grad_agent && scratch, "agent_unroll_bwd: NULL pointer");
    if ((rc = check_dtypes(d, b, -1, "pmb_agent_unroll_bwd"))) return rc;
    return agent_bwd(d, b, flat_agent, x_on, h_stash, gates, d_chosen, dpre1, flat_grad_agent, scratch, scratch_bytes,
                     (cudaStream_t)stream);
}

int pmb_clip_rmsprop_update(int64_t n, float* flat_p, float* flat_g, float* flat_sq, float* flat_target,
                            int32_t do_target_sync, double* stats, float lr, float alpha, float eps,
                            float grad_norm_clip, float* scratch, pmb_stream stream) {
    PMB_REQUIRE(n > 0 && flat_p && flat_g && flat_sq && stats && scratch, "clip_rmsprop_update: bad arguments");
    return launch_clip_rmsprop(n, flat_p, flat_g, flat_sq, flat_target, do_target_sync, stats, lr, alpha, eps,
                               grad_norm_clip, scratch, (cudaStream_t)stream);
}

int pmb_dp_pack(int64_t n, float* flat_g, const double* stats, pmb_stream stream) {
    PMB_REQUIRE(n > 0 && flat_g && stats, "dp_pack: bad arguments");
    return launch_dp_pack(stats, flat_g + n, (cudaStream_t)stream);
}

int pmb_dp_unpack(int64_t n, const float* flat_g, double* stats, pmb_stream stream) {
    PMB_REQUIRE(n > 0 && flat_g && stats, "dp_unpack: bad arguments");
    return launch_dp_unpack(flat_g + n, stats, (cudaStream_t)stream);
}

int pmb_epsilon_greedy(int64_t rows, int32_t A, const float* q, const int32_t* avail, float epsilon, const float* u,
                       const float* expo, uint64_t seed, uint64_t offset, int64_t* actions_out, pmb_stream stream) {
    PMB_REQUIRE(rows >= 0 && A > 0 && q && avail && actions_out, "epsilon_greedy: bad arguments");
    PMB_REQUIRE((u == nullptr) == (expo == nullptr), "epsilon_greedy: inject both u and expo or neither");
    return launch_epsilon_greedy(rows, 1, A, q, avail, A, epsilon, u, expo, seed, offset, actions_out,
                                 (cudaStream_t)stream);
}

int64_t pmb_select_actions_workspace_bytes(const pmb_dims* d) {
    if (validate_dims(d)) return -1;
    const int64_t R = (int64_t)d->B * d->N;
    int64_t n = align_up(R * d->H * 4, 256) + align_up(R * d->A * 4, 256);
    if (rollout_tc_ok(d))          // x tile images | GRU weight images | fc1 scratch
        n += align_up(ceil_div(R, 128) * 16384, 256) + 65536 + align_up(tc_fc1_scratch_bytes(d), 256);
    return n;
}

int pmb_select_actions_step(const pmb_dims* d, const pmb_batch* b, int32_t t, const float* flat_agent, float* hidden,
                            float epsilon, const float* u, const float* expo, uint64_t seed, uint64_t offset,
                            int64_t* actions_out, float* q_out, void* scratch, int64_t scratch_bytes,
                            pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(b && b->obs && b->avail && flat_agent && hidden && scratch, "select_actions_step: NULL pointer");
    PMB_REQUIRE(b == nullptr || b->ep_index == nullptr, "pmb_select_actions_step: batch.ep_index is only supported by pmb_qlearner_train_step");
    PMB_REQUIRE(t >= 0 && t < d->T, "select_actions_step: t = %d outside [0, %d)", t, d->T);
    PMB_REQUIRE((u == nullptr) == (expo == nullptr), "select_actions_step: inject both u and expo or neither");
    if ((rc = check_dtypes(d, b, PMB_ENTRY_SELECT_ACTIONS, "pmb_select_actions_step"))) return rc;
    if (scratch_bytes < pmb_select_actions_workspace_bytes(d)) { set_error("select_actions_step: scratch too small"); return PMB_ERR_WORKSPACE; }
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t R = (int64_t)d->B * d->N;
    float* x = static_cast<float*>(scratch);
    float* q = q_out ? q_out : reinterpret_cast<float*>(static_cast<char*>(scratch) + align_up(R * d->H * 4, 256));
    AgentParams ap = agent_params(d, flat_agent);
    if (rollout_tc_ok(d)) {
        // bf16 tier: streaming fc1 (online net only) -> x tile images -> one tcgen05 GRU step with fc2
        char* base = static_cast<char*>(scratch) + align_up(R * d->H * 4, 256) + align_up(R * d->A * 4, 256);
        const int n_tiles = (int)ceil_div(R, 128);
        uint8_t* x_ti = reinterpret_cast<uint8_t*>(base);
        char* gru_img = base + align_up((int64_t)n_tiles * 16384, 256);
        void* fc1_scr = gru_img + 65536;
        // (no zeroing of the padding rows of the last x tile: tile rows are independent in every MMA of this path and the
        // rollout kernel neither stores nor selects for rows >= R)
        // pmb_dims.reserved bit 0: the weight images in `scratch` are current (same parameters, same scratch as the
        // previous step of this rollout) - the two pack launches are skipped
        const int packed = d->reserved & 1;
        if ((rc = tc_fc1_fwd_both(d, b, t, 1, ap, ap, reinterpret_cast<float*>(x_ti), nullptr, 1, nullptr, nullptr, fc1_scr,
                                  align_up(tc_fc1_scratch_bytes(d), 256), s, packed))) return rc;
        if (!packed && (rc = pack_gru_images(d, ap, gru_img, s))) return rc;
        tc::GruFwdParams fp;
        fp.w_ih_img = reinterpret_cast<const __nv_bfloat16*>(gru_img);
        fp.w_hh_img = reinterpret_cast<const __nv_bfloat16*>(gru_img + 24576);
        fp.w2_img = reinterpret_cast<const __nv_bfloat16*>(gru_img + 49152);
        fp.b_ih = ap.b_ih; fp.b_hh = ap.b_hh; fp.b2 = ap.fc2_b;
        fp.x_ti = x_ti; fp.h0 = hidden; fp.h_ti = nullptr; fp.g_ti = nullptr; fp.q = q; fp.h_last = hidden;
        fp.R = R; fp.nt = 1; fp.A = d->A; fp.n_tiles = n_tiles;
        // epsilon-greedy fused into the q epilogue (no q round trip through HBM); q itself only when the caller wants it
        fp.avail = static_cast<const uint8_t*>(b->avail) + ((int64_t)t * d->N * d->A << (b->avail_dtype == PMB_DTYPE_U8 ? 0 : 2));
        fp.avail_u8 = b->avail_dtype == PMB_DTYPE_U8; fp.avail_sb = b->avail_sb; fp.N = d->N; fp.epsilon = epsilon;
        fp.u = u; fp.expo = expo; fp.seed = seed; fp.offset = offset; fp.actions_out = actions_out;
        if (actions_out && !q_out) fp.q = nullptr;
        if ((rc = tc_gru_fwd(fp, s))) return rc;
        return PMB_OK;
    } else {
        rc = fc1_fwd(d, b, t, 1, ap, x, s);
        if (rc) return rc;
        rc = gru_fwd_dispatch(d, ap, R, 1, x, hidden, nullptr, nullptr, q, hidden, s);
        if (rc) return rc;
    }
    if (!actions_out) return PMB_OK;
    return launch_epsilon_greedy(R, d->N, d->A, q, avail_i32(b) + (int64_t)t * d->N * d->A, b->avail_sb, epsilon, u, expo,
                                 seed, offset, actions_out, s);
}

int64_t pmb_gemm_bf16_workspace_bytes(int32_t n, int32_t k) {
    return align_up(tc_packed_elems((int)align_up(n, 32), k) * 2, 256);
}

int pmb_gemm_bf16_tn(int64_t m, int32_t n, int32_t k, const float* a, const float* w, const float* bias, float* c,
                     void* scratch, int64_t scratch_bytes, pmb_stream stream) {
    PMB_REQUIRE(m > 0 && n > 0 && k > 0 && a && w && c && scratch, "gemm_bf16_tn: bad arguments");
    if (scratch_bytes < pmb_gemm_bf16_workspace_bytes(n, k)) { set_error("gemm_bf16_tn: scratch too small"); return PMB_ERR_WORKSPACE; }
    cudaStream_t s = (cudaStream_t)stream;
    __nv_bfloat16* wp = static_cast<__nv_bfloat16*>(scratch);
    const float* ptrs[1] = {w};
    int rows[1] = {n}, lds[1] = {k};
    int rc = tc_pack_w(ptrs, rows, lds, 1, k, wp, s);
    if (rc) return rc;
    return tc_gemm_plain(a, dense_map(k), m, k, wp, (int)align_up(n, 32), n, bias, c, n, s);
}

int64_t pmb_gemm_bf16_atb_workspace_bytes(int64_t m, int32_t c, int32_t k) { return tc_atb_scratch_bytes(c, k, m); }

int pmb_gemm_bf16_atb(int64_t m, int32_t c, int32_t k, const float* d, int64_t ldd, const float* a, int64_t lda,
                      float* out, float* bias_out, void* scratch, int64_t scratch_bytes, pmb_stream stream) {
    PMB_REQUIRE(m > 0 && c > 0 && k > 0 && d && a && out && scratch, "gemm_bf16_atb: bad arguments");
    return tc_gemm_atb(d, dense_map(ldd), c, a, dense_map(lda), k, m, out, k, bias_out, scratch, scratch_bytes,
                       (cudaStream_t)stream);
}

int pmb_qlearner_train_step(const pmb_dims* d, const pmb_batch* b, const pmb_hparams* hp, float* flat_p, float* flat_g,
                            float* flat_sq, float* flat_target, void* workspace, int64_t workspace_bytes,
                            double* stats, pmb_stream stream) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2, "train_step: T must be >= 2");
    PMB_REQUIRE(b && hp && flat_p && flat_g && flat_sq && flat_target && workspace && stats, "train_step: NULL pointer");
    PMB_REQUIRE(b->obs && b->actions && b->avail && b->reward && b->terminated && b->filled, "train_step: batch field is NULL");
    PMB_REQUIRE(d->mixer != PMB_MIXER_QMIX || b->state, "train_step: QMIX needs batch.state");
    if ((rc = check_dtypes(d, b, PMB_ENTRY_TRAIN_STEP, "pmb_qlearner_train_step"))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    WsPlan plan = plan_workspace(d);
    if (workspace_bytes < plan.total) { set_error("workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)plan.total); return PMB_ERR_WORKSPACE; }
    pmb_ws_views v;
    fill_views(d, workspace, plan, &v);
    pmb_layout L;
    compute_layout(d, &L);
    const int64_t R = (int64_t)d->B * d->N;
    AgentParams on = agent_params(d, flat_p), tg = agent_params(d, flat_target);

    if ((rc = launch_stats_reset(stats, s))) return rc;
    // q_learner.py:47-52 / 58-62: both nets over all T steps
    const bool tc_agent = d->precision == PMB_PREC_BF16 && d->H == 64 && d->A <= 64;
    const bool tc_mixer = d->precision == PMB_PREC_BF16 && d->mixer == PMB_MIXER_QMIX && d->E == 32;
    PMB_REQUIRE(b->ep_index == nullptr || fused_tc_path(d),
                "train_step: batch.ep_index (zero-copy replay sampling) needs the tensor-core tier with the fused kernels");
    const int n_tiles = (int)ceil_div(R, 128);
    // Padded-step skipping: sort the episodes by the steps they need (longest first) on the device; from here on the step
    // reads the batch in that order (ep_order composes the incoming ep_index), and the agent kernels walk the live
    // (t, tile) items only.  Launch sizes stay those of the full rectangle.
    pmb_batch sorted_batch;
    SkipSchedule sched{};
    const bool skip = skip_padding(d);
    if (skip) sched = skip_schedule_views(static_cast<char*>(workspace) + plan.total - plan.sched_bytes, d->B, d->T, n_tiles);
    const int32_t* live_items = skip ? sched.items : nullptr;
    const int32_t* n_live = skip ? sched.n_items : nullptr;
    const int32_t* tile_steps = skip ? sched.tile_steps : nullptr;
    uint8_t *x_on_ti = reinterpret_cast<uint8_t*>(v.x_on), *x_tg_ti = reinterpret_cast<uint8_t*>(v.x_tg);
    uint8_t *h_ti = reinterpret_cast<uint8_t*>(v.h_stash), *g_ti = reinterpret_cast<uint8_t*>(v.gates);
    uint8_t* hg_ti = reinterpret_cast<uint8_t*>(v.h_tg);
    // GRU weight images live at the start of the scratch area: [online: w_ih | w_hh | w2][target: same]
    auto pack_gru = [&](const AgentParams& ap, char* base) -> int { return pack_gru_images(d, ap, base, s); };
    char* gru_img = reinterpret_cast<char*>(v.scratch);
    // fc1/fc2 weight gradients as one image-fed GEMM kernel (needs the obs tile images written by fc1)
    // needs the obs images of the streaming fc1 kernel with one-hot(agent) + ones folded into the K padding
    const bool fused_dw = tc_agent && d->O <= 320 && d->N <= 64 && ((d->O + 63) / 64) * 64 - d->O >= d->N + 1;
    uint8_t* obs_ti = reinterpret_cast<uint8_t*>(v.obs_img);
    if (tc_agent) {
        if ((rc = tc_ti_zero_pad(x_on_ti, d->T, n_tiles, R, s))) return rc;
        if ((rc = tc_ti_zero_pad(x_tg_ti, d->T, n_tiles, R, s))) return rc;
        if (skip) {                                      // (skip implies the tensor-core agent)
            PHASE(s, "skip_schedule");
            if ((rc = tc_skip_schedule(d, b, sched, n_tiles, s))) return rc;
            sorted_batch = *b;
            sorted_batch.ep_index = sched.ep_order;
            b = &sorted_batch;
        }
        PHASE(s, "fc1_fwd_both_tc");
        if ((rc = tc_fc1_fwd_both(d, b, 0, d->T, on, tg, v.x_on, v.x_tg, 1, fused_dw ? obs_ti : nullptr,
                                  reinterpret_cast<uint32_t*>(v.relu_mask), v.scratch, v.scratch_bytes, s, 0, live_items)))
            return rc;
        // The two recurrences are independent.  Each runs ceil(n_tiles / 2) CTAs (one per SM): when both fit on the device
        // at once (small configs, or a batch sharded over many GPUs) the target net's pass is forked onto a side stream and
        // the two chains of T dependent steps run side by side instead of back to back.
        // With very few tiles (2 passes x n_tiles CTAs fit) every CTA takes ONE tile: no ping-pong, shorter per-step chain.
        const int tpc = 2 * n_tiles <= sm_count() ? 1 : 2;
        const int gru_ctas = (n_tiles + tpc - 1) / tpc;
        static const int fork_mode = []() { const char* e = getenv("PMB_FORK"); return e ? atoi(e) : -1; }();   // A/B switch: 0 never, 1 always
        const bool fork_tg = fork_mode >= 0 ? fork_mode != 0 : 4 * 2 * gru_ctas <= 5 * sm_count();   // up to 1.25 x the SMs: the few CTAs that wait start when the first (shorter) target CTAs retire - measured 4.22 -> 3.79 ms on MMM2 / 2048 (160 CTAs)
        PHASE(s, fork_tg ? "gru_unroll_fwd_both_tc" : "gru_unroll_fwd_online_tc");
        if ((rc = pack_gru(on, gru_img))) return rc;
        if ((rc = pack_gru(tg, gru_img + 57344))) return rc;
        auto img = [&](int64_t off) { return reinterpret_cast<const __nv_bfloat16*>(gru_img + off); };
        SideStream* side = nullptr;
        if (fork_tg) {
            if ((rc = side_stream(&side))) return rc;
            PMB_CUDA(cudaEventRecord(side->fork, s));
            PMB_CUDA(cudaStreamWaitEvent(side->stream, side->fork, 0));
            if ((rc = tc_gru_fwd2(img(57344), img(57344 + 24576), tg.b_ih, tg.b_hh, x_tg_ti, hg_ti, nullptr, R, d->T, n_tiles,
                                  side->stream, tpc, tile_steps))) return rc;
            PMB_CUDA(cudaEventRecord(side->join, side->stream));
        }
        if ((rc = tc_gru_fwd2(img(0), img(24576), on.b_ih, on.b_hh, x_on_ti, h_ti, g_ti, R, d->T, n_tiles, s, tpc, tile_steps)))
            return rc;
        if (fork_tg) {
            PMB_CUDA(cudaStreamWaitEvent(s, side->join, 0));
        } else {
            PHASE(s, "gru_unroll_fwd_target_tc");
            if ((rc = tc_gru_fwd2(img(57344), img(57344 + 24576), tg.b_ih, tg.b_hh, x_tg_ti, hg_ti, nullptr, R, d->T, n_tiles,
                                  s, 2, tile_steps))) return rc;
        }
        // :55-78 fused with fc2 of both nets
        PHASE(s, "q_select_tc");
        if ((rc = tc_q_select(d, b, img(49152), img(57344 + 49152), on.fc2_b, tg.fc2_b, h_ti, hg_ti, n_tiles, v.chosen,
                              v.tmax, (hp->keep_q & 1) ? v.q_on : nullptr, (hp->keep_q & 1) ? v.q_tg : nullptr, s, live_items,
                              n_live, tile_steps))) return rc;
    } else {
        PHASE(s, "fc1_fwd_online");
        if ((rc = fc1_fwd(d, b, 0, d->T, on, v.x_on, s))) return rc;
        PHASE(s, "fc1_fwd_target");
        if ((rc = fc1_fwd(d, b, 0, d->T, tg, v.x_tg, s))) return rc;
    }
    if (!tc_agent) {
        PHASE(s, "gru_unroll_fwd_online");
        if ((rc = gru_fwd_dispatch(d, on, R, d->T, v.x_on, nullptr, v.h_stash, v.gates, v.q_on, nullptr, s))) return rc;
        PHASE(s, "gru_unroll_fwd_target");
        if ((rc = gru_fwd_dispatch(d, tg, R, d->T, v.x_tg, nullptr, nullptr, nullptr, v.q_tg, nullptr, s))) return rc;
    }
    // :55-78
    if (!tc_agent) {
        PHASE(s, "target_select");
        if ((rc = launch_target_select(d, b, v.q_on, v.q_tg, v.chosen, v.tmax, nullptr, s))) return rc;
    }
    // :81-83 (target mixer first: both passes share the raw buffer, the online one must survive)
    uint8_t* state_img = reinterpret_cast<uint8_t*>(v.state_img);
    uint8_t* raw_img = reinterpret_cast<uint8_t*>(v.raw_on);
    if (tc_mixer) {
        PHASE(s, "state_to_images");
        if ((rc = tc_state_to_images(d, b, state_img, s))) return rc;
        PHASE(s, "mixer_fwd_target_tc");
        if ((rc = tc_mixer_fwd_img(d, mixer_params(d, flat_target + L.n_agent), state_img, v.tmax, 1, nullptr, v.t_tot,
                                   v.scratch, v.scratch_bytes, s))) return rc;
        PHASE(s, "mixer_fwd_online_tc");
        if ((rc = tc_mixer_fwd_img(d, mixer_params(d, flat_p + L.n_agent), state_img, v.chosen, 0, raw_img, v.q_tot,
                                   v.scratch, v.scratch_bytes, s))) return rc;
    } else if (d->mixer != PMB_MIXER_NONE) {
        PHASE(s, "mixer_fwd_target");
        if ((rc = launch_mixer_fwd(d, b, flat_target + L.n_agent, v.tmax, 1, v.raw_tg, v.t_tot, s))) return rc;
        PHASE(s, "mixer_fwd_online");
        if ((rc = launch_mixer_fwd(d, b, flat_p + L.n_agent, v.chosen, 0, v.raw_on, v.q_tot, s))) return rc;
    }
    // :86-97
    PHASE(s, "td_loss");
    // the scratch area is free between the mixer forward and the mixer backward: per-block loss sums -> fixed-order total
    if ((rc = launch_td_loss(d, b, v.q_tot, v.t_tot, hp->gamma, v.g, stats, s, reinterpret_cast<double*>(v.scratch),
                             v.scratch_bytes))) return rc;
    if (hp->keep_q & 2) {              // debug: forward pass + loss sums only, intermediates stay in the workspace
        PHASE(s, "end");
        return PMB_OK;
    }
    // :100-101 backward
    PHASE(s, "mixer_bwd");
    // The hypernet weight-gradient GEMM (d_raw^T . [state | 1]) feeds nothing but the optimiser.  When the agent's BPTT kernel
    // (one CTA per row tile) leaves SMs idle - small configs, or a batch sharded over many GPUs - it runs on the side stream
    // on those SMs, with its own partial-sum area behind the scratch, and joins before the clip / RMSprop kernels.
    SideStream* side_dw = nullptr;
    if (tc_mixer) {
        static const int dw_fork_mode = []() { const char* e = getenv("PMB_DW_FORK"); return e ? atoi(e) : -1; }();   // A/B: 0 never, 1 whenever it fits
        const int free_sms = sm_count() - n_tiles;
        const bool fork_dw = tc_agent && plan.mixdw_bytes > 0 && dw_fork_mode != 0 && free_sms >= tc_mixer_dw_ctas(d);
        if (!fork_dw) {
            if ((rc = tc_mixer_bwd_img(d, mixer_params(d, flat_p + L.n_agent), state_img, raw_img, v.chosen, v.g, v.d_chosen,
                                       flat_g + L.offset[PMB_P_HW1_W], flat_g + L.offset[PMB_P_HW1_B],
                                       flat_g + L.offset[PMB_P_V2_W], flat_g + L.offset[PMB_P_V2_B], v.scratch,
                                       v.scratch_bytes, s))) return rc;
        } else {
            if ((rc = tc_mixer_bwd_img_dq(d, mixer_params(d, flat_p + L.n_agent), raw_img, v.chosen, v.g, v.d_chosen,
                                          flat_g + L.offset[PMB_P_V2_W], flat_g + L.offset[PMB_P_V2_B], v.scratch,
                                          v.scratch_bytes, s))) return rc;
            if ((rc = side_stream(&side_dw))) return rc;
            PMB_CUDA(cudaEventRecord(side_dw->fork2, s));
            PMB_CUDA(cudaStreamWaitEvent(side_dw->stream, side_dw->fork2, 0));
            if ((rc = tc_mixer_dw(d, state_img, raw_img, flat_g + L.offset[PMB_P_HW1_W], flat_g + L.offset[PMB_P_HW1_B],
                                  reinterpret_cast<char*>(v.scratch) + plan.scratch_bytes, plan.mixdw_bytes, free_sms,
                                  side_dw->stream))) return rc;
            PMB_CUDA(cudaEventRecord(side_dw->join2, side_dw->stream));
        }
    } else if (d->mixer != PMB_MIXER_NONE) {
        if ((rc = launch_mixer_bwd(d, b, flat_p + L.n_agent, v.chosen, v.raw_on, v.g, v.d_chosen, flat_g + L.n_agent,
                                   v.scratch, v.scratch_bytes, s))) return rc;
    }
    if (tc_agent) {
        AgentGrads gr = agent_grads(d, flat_g);
        PHASE(s, "gru_unroll_bwd_tc");
        if ((rc = pack_gru(on, gru_img))) return rc;
        float* rnn_part = reinterpret_cast<float*>(reinterpret_cast<char*>(v.scratch) + 131072);
        auto img = [&](int64_t off) { return reinterpret_cast<const __nv_bfloat16*>(gru_img + off); };
        if ((rc = tc_gru_bwd2(img(0), img(24576), img(49152), x_on_ti, h_ti, g_ti, x_tg_ti,
                              reinterpret_cast<const uint32_t*>(v.relu_mask), v.d_chosen, b->actions, b->actions_sb, b->ep_index,
                              R, d->T, d->N, d->A, n_tiles, rnn_part, s, tile_steps))) return rc;
        PHASE(s, "dW_rnn_tc");
        if ((rc = tc_gru_bwd2_reduce(rnn_part, n_tiles, gr.w_ih, gr.w_hh, gr.b_ih, gr.b_hh, s))) return rc;
        if (fused_dw) {
            PHASE(s, "dW_fc1_fc2_tc");
            if ((rc = tc_agent_dw(d, b, x_tg_ti, h_ti, obs_ti, v.d_chosen, n_tiles, gr.fc1_w, gr.fc1_b, gr.fc2_w, gr.fc2_b,
                                  v.scratch, v.scratch_bytes, s, live_items, n_live))) return rc;
        } else {
            PHASE(s, "dW_fc1_tc");
            RowMap omap{b->obs_sb, (int64_t)d->N * d->O, (int64_t)d->O, d->T, d->N};
            if ((rc = tc_gemm_atb_ti(x_tg_ti, d->T, d->N, R, n_tiles, obs_f32(b), omap, d->O, gr.fc1_w, d_in_of(d), gr.fc1_b,
                                     v.scratch, v.scratch_bytes, s))) return rc;
            PHASE(s, "agent_scatter_grads");
            if ((rc = scatter_grads_dispatch(d, b, v.h_stash, v.x_tg, v.d_chosen, gr, v.scratch, v.scratch_bytes, s,
                                             n_tiles))) return rc;
        }
    } else if ((rc = agent_bwd(d, b, flat_p, v.x_on, v.h_stash, v.gates, v.d_chosen, v.x_tg, flat_g, v.scratch,
                               v.scratch_bytes, s))) return rc;
    if (side_dw) PMB_CUDA(cudaStreamWaitEvent(s, side_dw->join2, 0));
    // :102-107
    PHASE(s, "clip_rmsprop_update");
    if (!hp->skip_update) {
        if ((rc = launch_clip_rmsprop(L.n_total, flat_p, flat_g, flat_sq, flat_target, hp->do_target_sync, stats, hp->lr,
                                      hp->alpha, hp->eps, hp->grad_norm_clip, v.scratch, s))) return rc;
    }
    PHASE(s, "end");
    return PMB_OK;
}

}  // extern "C"

/* ---- COMA (SURVEY.md section 8f rank 4) ------------------------------------------------------------------------ */
namespace pmb {
namespace {
struct ComaPlan {
    int64_t D, Hc, R, Tp, chunk_nt, chunk_rows;
    int64_t off[24];
    int64_t scratch_bytes, total;
};
ComaPlan coma_plan(const pmb_dims* d) {
    ComaPlan p;
    p.D = (int64_t)d->S + d->O + 2 * (int64_t)d->N * d->A + d->N;
    p.Hc = d->E;
    p.R = (int64_t)d->B * d->N;
    p.Tp = d->T - 1;
    // the target critic runs over all T timesteps in chunks whose input matrix stays below ~256 MB
    int64_t nt = ((int64_t)64 << 20) / (p.R * p.D);
    if (nt < 1) nt = 1;
    if (nt > d->T) nt = d->T;
    p.chunk_nt = nt;
    p.chunk_rows = p.R * nt;
    const int64_t H = d->H, A = d->A;
    int64_t sizes[24] = {
        p.chunk_rows * p.D,            // 0 inp
        p.chunk_rows * p.Hc,           // 1 x1
        p.chunk_rows * p.Hc,           // 2 x2
        p.chunk_rows * A,              // 3 qtmp
        p.R * d->T,                    // 4 taken [B][T][N]
        p.R * p.Tp,                    // 5 targets [B][T-1][N]
        p.R * p.Tp * A,                // 6 q_vals [B][T-1][N][A]
        p.R,                           // 7 dqv
        p.R,                           // 8 dqa (int32)
        p.R * A,                       // 9 dq dense
        p.R * p.Hc,                    // 10 dx2
        p.R * p.Hc,                    // 11 dx1
        p.Hc * p.Hc,                   // 12 w2t
        p.Tp * p.R * H,                // 13 x (agent fc1 out)
        (p.Tp + 1) * p.R * H,          // 14 h_stash
        p.Tp * p.R * 4 * H,            // 15 gates
        p.Tp * p.R * A,                // 16 logits
        p.Tp * p.R * A,                // 17 dlogits
        p.Tp * p.R * H,                // 18 dpre1
        p.Tp * p.R * A,                // 19 pi (diagnostics / tests)
        0, 0, 0, 0};
    int64_t off = 0;
    for (int i = 0; i < 24; ++i) { p.off[i] = off; off += align_up(sizes[i] * 4, 256); }
    pmb_dims da = *d;
    da.T = (int32_t)p.Tp; da.precision = PMB_PREC_FP32; da.mixer = PMB_MIXER_NONE;
    int64_t sc = p.Tp > 0 ? agent_bwd_scratch(&da) : 0;
    int64_t c1 = gemm_atb_scratch_bytes((int)A, (int)p.Hc, p.R), c2 = gemm_atb_scratch_bytes((int)p.Hc, (int)p.Hc, p.R),
            c3 = gemm_atb_scratch_bytes((int)p.Hc, (int)p.D, p.R);
    if (c1 > sc) sc = c1;
    if (c2 > sc) sc = c2;
    if (c3 > sc) sc = c3;
    if (sc < 65536) sc = 65536;                  // >= the per-block partial sums of the td / policy kernels
    p.scratch_bytes = align_up(sc, 256);
    p.total = off + p.scratch_bytes;
    return p;
}
struct CriticParams { const float *w1, *b1, *w2, *b2, *w3, *b3; };
struct CriticGrads { float *w1, *b1, *w2, *b2, *w3, *b3; };
template <class P, class F>
P critic_views(F* flat, int64_t D, int64_t Hc, int64_t A) {
    F* w1 = flat; F* b1 = w1 + Hc * D; F* w2 = b1 + Hc; F* b2 = w2 + Hc * Hc; F* w3 = b2 + Hc; F* b3 = w3 + A * Hc;
    return P{w1, b1, w2, b2, w3, b3};
}
int critic_fwd(const CriticParams& c, const float* inp, int64_t rows, int64_t D, int Hc, int A, float* x1, float* x2, float* q,
               cudaStream_t s) {
    int rc;
    if ((rc = launch_gemm_tn(inp, dense_map(D), rows, (int)D, c.w1, (int)D, Hc, c.b1, x1, Hc, 1, s))) return rc;
    if ((rc = launch_gemm_tn(x1, dense_map(Hc), rows, Hc, c.w2, Hc, Hc, c.b2, x2, Hc, 1, s))) return rc;
    return launch_gemm_tn(x2, dense_map(Hc), rows, Hc, c.w3, Hc, A, c.b3, q, A, 0, s);
}
int validate_coma(const pmb_dims* d) {
    int rc = validate_dims(d);
    if (rc) return rc;
    PMB_REQUIRE(d->T >= 2 && d->S > 0 && d->E > 0 && d->E <= 1024 && d->A <= 64, "coma: need T >= 2, a state, critic width 1..1024, n_actions <= 64");
    return PMB_OK;
}
}  // namespace
}  // namespace pmb

extern "C" {

int64_t pmb_coma_critic_numel(const pmb_dims* d) {
    if (validate_coma(d)) return -1;
    const int64_t D = (int64_t)d->S + d->O + 2 * (int64_t)d->N * d->A + d->N, Hc = d->E;
    return Hc * D + Hc + Hc * Hc + Hc + (int64_t)d->A * Hc + d->A;
}

int64_t pmb_coma_workspace_bytes(const pmb_dims* d) {
    if (validate_coma(d)) return -1;
    return coma_plan(d).total;
}

int pmb_coma_workspace_views(const pmb_dims* d, void* workspace, float** q_vals, float** targets, float** pi, float** logits) {
    if (validate_coma(d)) return PMB_ERR_INVALID;
    ComaPlan p = coma_plan(d);
    char* base = static_cast<char*>(workspace);
    if (q_vals) *q_vals = reinterpret_cast<float*>(base + p.off[6]);
    if (targets) *targets = reinterpret_cast<float*>(base + p.off[5]);
    if (pi) *pi = reinterpret_cast<float*>(base + p.off[19]);
    if (logits) *logits = reinterpret_cast<float*>(base + p.off[16]);
    return PMB_OK;
}

int pmb_coma_train_step(const pmb_dims* d, const pmb_batch* b, const pmb_coma_hparams* hp, float* agent_p, float* agent_g,
                        float* agent_sq, float* critic_p, float* critic_g, float* critic_sq, const float* target_critic_p,
                        void* workspace, int64_t workspace_bytes, double* stats, pmb_stream stream) {
    int rc = validate_coma(d);
    if (rc) return rc;
    PMB_REQUIRE(b && hp && agent_p && agent_g && agent_sq && critic_p && critic_g && critic_sq && target_critic_p && workspace && stats,
                "coma_train_step: NULL pointer");
    PMB_REQUIRE(b->obs && b->state && b->actions && b->avail && b->reward && b->terminated && b->filled && !b->ep_index,
                "coma_train_step: batch field is NULL (or ep_index given)");
    if ((rc = check_dtypes(d, b, -1, "pmb_coma_train_step"))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    ComaPlan P = coma_plan(d);
    if (workspace_bytes < P.total) { set_error("coma workspace too small: %lld < %lld", (long long)workspace_bytes, (long long)P.total); return PMB_ERR_WORKSPACE; }
    char* base = static_cast<char*>(workspace);
    auto f = [&](int i) { return reinterpret_cast<float*>(base + P.off[i]); };
    float *inp = f(0), *x1 = f(1), *x2 = f(2), *qtmp = f(3), *taken = f(4), *targets = f(5), *q_vals = f(6), *dqv = f(7);
    int32_t* dqa = reinterpret_cast<int32_t*>(f(8));
    float *dq = f(9), *dx2 = f(10), *dx1 = f(11), *w2t = f(12), *x = f(13), *h_stash = f(14), *gates = f(15), *logits = f(16),
          *dlogits = f(17), *dpre1 = f(18), *pi = f(19);
    void* scratch = base + P.total - P.scratch_bytes;
    const int64_t D = P.D, R = P.R;
    const int Hc = (int)P.Hc, A = d->A, Tp = (int)P.Tp;
    const int64_t n_critic = pmb_coma_critic_numel(d);
    CriticParams cp = critic_views<CriticParams, const float>(critic_p, D, Hc, A);
    CriticParams tp = critic_views<CriticParams, const float>(target_critic_p, D, Hc, A);
    CriticGrads cg = critic_views<CriticGrads, float>(critic_g, D, Hc, A);
    PMB_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * PMB_S_COUNT * (Tp + 1), s));

    // coma_learner.py:105-109: target critic over all timesteps -> Q of the taken actions -> td-lambda targets
    for (int t0 = 0; t0 < d->T; t0 += (int)P.chunk_nt) {
        const int nt = d->T - t0 < P.chunk_nt ? d->T - t0 : (int)P.chunk_nt;
        if ((rc = coma_launch_inputs(d, b, t0, nt, inp, s))) return rc;
        if ((rc = critic_fwd(tp, inp, R * nt, D, Hc, A, x1, x2, qtmp, s))) return rc;
        if ((rc = coma_launch_gather_taken(d, b, t0, nt, qtmp, taken, s))) return rc;
    }
    if ((rc = coma_launch_td_lambda(d, b, hp->gamma, hp->td_lambda, taken, targets, s))) return rc;

    // :118-146: one critic optimiser step per timestep, backwards in time
    for (int t = Tp - 1; t >= 0; --t) {
        double* st = stats + (int64_t)t * PMB_S_COUNT;
        if ((rc = coma_launch_inputs(d, b, t, 1, inp, s))) return rc;
        if ((rc = critic_fwd(cp, inp, R, D, Hc, A, x1, x2, qtmp, s))) return rc;
        if ((rc = coma_launch_critic_td(d, b, t, qtmp, targets, q_vals, dqv, dqa, st, static_cast<double*>(scratch), s))) return rc;
        if ((rc = coma_launch_critic_bwd_pointwise(R, A, Hc, dqv, dqa, cp.w3, x2, dq, dx2, s))) return rc;
        if ((rc = launch_gemm_atb(dq, dense_map(A), A, x2, dense_map(Hc), Hc, R, cg.w3, Hc, cg.b3, scratch, P.scratch_bytes, s))) return rc;
        if ((rc = launch_gemm_atb(dx2, dense_map(Hc), Hc, x1, dense_map(Hc), Hc, R, cg.w2, Hc, cg.b2, scratch, P.scratch_bytes, s))) return rc;
        if ((rc = launch_transpose(Hc, Hc, cp.w2, w2t, s))) return rc;
        if ((rc = launch_gemm_tn(dx2, dense_map(Hc), R, Hc, w2t, Hc, Hc, nullptr, dx1, Hc, 0, s))) return rc;
        if ((rc = launch_relu_mask(R * Hc, x1, dx1, s))) return rc;
        if ((rc = launch_gemm_atb(dx1, dense_map(Hc), Hc, inp, dense_map(D), (int)D, R, cg.w1, D, cg.b1, scratch, P.scratch_bytes, s))) return rc;
        if ((rc = launch_clip_rmsprop(n_critic, critic_p, critic_g, critic_sq, nullptr, 0, st, hp->critic_lr, hp->alpha, hp->eps,
                                      hp->grad_norm_clip, static_cast<float*>(scratch), s, 1))) return rc;
    }

    // :55-90: agent unroll over t = 0 .. T-2, policy head, COMA loss, policy gradient, clip + RMSprop
    pmb_dims da = *d;
    da.T = Tp; da.precision = PMB_PREC_FP32; da.mixer = PMB_MIXER_NONE;
    AgentParams ap = agent_params(&da, agent_p);
    if ((rc = fc1_fwd(&da, b, 0, Tp, ap, x, s))) return rc;
    if ((rc = gru_fwd_dispatch(&da, ap, R, Tp, x, nullptr, h_stash, gates, logits, nullptr, s))) return rc;
    double* sa = stats + (int64_t)Tp * PMB_S_COUNT;
    if ((rc = coma_launch_policy(d, b, hp->epsilon, logits, q_vals, dlogits, pi, sa, static_cast<double*>(scratch), s))) return rc;
    if ((rc = agent_bwd(&da, b, agent_p, x, h_stash, gates, nullptr, dpre1, agent_g, scratch, P.scratch_bytes, s, dlogits))) return rc;
    pmb_layout L;
    compute_layout(&da, &L);
    return launch_clip_rmsprop(L.n_agent, agent_p, agent_g, agent_sq, nullptr, 0, sa, hp->lr, hp->alpha, hp->eps,
                               hp->grad_norm_clip, static_cast<float*>(scratch), s, 0);
}

int pmb_coma_critic_fwd(const pmb_dims* d, const pmb_batch* b, const float* critic_p, int32_t t0, int32_t nt, float* q_out,
                        void* workspace, int64_t workspace_bytes, pmb_stream stream) {
    int rc = validate_coma(d);
    if (rc) return rc;
    PMB_REQUIRE(b && critic_p && q_out && workspace && b->obs && b->state && b->actions && b->filled && !b->ep_index,
                "coma_critic_fwd: NULL pointer");
    if ((rc = check_dtypes(d, b, -1, "pmb_coma_critic_fwd"))) return rc;
    PMB_REQUIRE(t0 >= 0 && nt > 0 && t0 + nt <= d->T, "coma_critic_fwd: bad time range");
    cudaStream_t s = (cudaStream_t)stream;
    ComaPlan P = coma_plan(d);
    if (workspace_bytes < P.total) { set_error("coma workspace too small"); return PMB_ERR_WORKSPACE; }
    char* base = static_cast<char*>(workspace);
    auto f = [&](int i) { return reinterpret_cast<float*>(base + P.off[i]); };
    CriticParams cp = critic_views<CriticParams, const float>(critic_p, P.D, P.Hc, d->A);
    // q_out [B][nt][N][A]; chunks of timesteps keep the materialised input matrix bounded (rows are (b, tt, n) per chunk,
    // so a chunk's rows are scattered into q_out per episode)
    for (int c0 = 0; c0 < nt; c0 += (int)P.chunk_nt) {
        const int cn = nt - c0 < P.chunk_nt ? nt - c0 : (int)P.chunk_nt;
        if ((rc = coma_launch_inputs(d, b, t0 + c0, cn, f(0), s))) return rc;
        if ((rc = critic_fwd(cp, f(0), P.R * cn, P.D, (int)P.Hc, d->A, f(1), f(2), f(3), s))) return rc;
        PMB_CUDA(cudaMemcpy2DAsync(q_out + (int64_t)c0 * d->N * d->A, sizeof(float) * nt * d->N * d->A, f(3),
                                   sizeof(float) * cn * d->N * d->A, sizeof(float) * cn * d->N * d->A, (size_t)d->B,
                                   cudaMemcpyDeviceToDevice, s));
    }
    return PMB_OK;
}

int pmb_policy_head(int64_t rows, int32_t A, float epsilon, int32_t test_mode, const float* logits, const int32_t* avail,
                    float* probs, pmb_stream stream) {
    PMB_REQUIRE(rows >= 0 && A > 0 && A <= 64 && logits && avail && probs, "policy_head: bad arguments");
    return launch_policy_head(rows, A, epsilon, test_mode, logits, avail, probs, (cudaStream_t)stream);
}

int pmb_multinomial(int64_t rows, int32_t A, const float* probs, const int32_t* avail, const float* expo, int32_t greedy,
                    uint64_t seed, uint64_t offset, int64_t* actions_out, pmb_stream stream) {
    PMB_REQUIRE(rows >= 0 && A > 0 && probs && avail && actions_out, "multinomial: bad arguments");
    return launch_multinomial(rows, A, probs, avail, expo, greedy, seed, offset, actions_out, (cudaStream_t)stream);
}

}  // extern "C"
