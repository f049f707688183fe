// Backward of COMACritic.forward (fc1 -> ReLU -> fc2 -> ReLU -> fc3 over the generated critic input, coma.py:22-59),
// fp32 on every tier: what autograd through COMACritic needs when a user's actor-critic learner calls loss.backward() on
// a loss of the critic's q (coma_learner.py:118-146 is the reference's pattern).  The forward is pmb_coma_critic_fwd's
// own launches (coma_inputs_kernel + three gemm_tn) with the two hidden activations kept.
//
//   critic_row_bwd_kernel : per row, dx2 = (dq W3) * [x2 > 0], then dx1 = (dx2 W2) * [x1 > 0].  The weights are read
//                           through L1 / L2; a tile's dq and dx2 rows sit in shared memory.  It also copies dq into the
//                           saved row order for the fc3 weight gradient.
//   critic_dw_kernel      : every weight gradient in one launch, a grouped sum over rows:
//                             fc3 (dq, x2) and fc2 (dx2, x1): dense 64 x 64 output tiles;
//                             fc1 state columns: dx1 summed over the N agents of an (episode, step) first, since
//                               they share the state, then a 64 x 64 tile over the (episode, step) groups;
//                             fc1 obs columns: dense tiles, obs read from the batch;
//                             fc1 one-hot action columns (actions at t, own block zero; actions at t-1): a scatter by
//                               index - a thread owns (agent m, hidden unit c) and adds the group's dx1 sum into the
//                               column of the action agent m took, in shared memory;
//                             fc1 agent-id columns: a per-agent sum of dx1.
//                           The [rows x D] input matrix is never built.  Rows go in fixed slices of (episode, step)
//                           groups; with more than one slice critic_dw_reduce_kernel adds the partials in slice order.
// No float atomics: two identical calls give identical bits.
#include "common.cuh"

namespace pmb {

namespace {

// saved row r <-> (b, t, n): the forward's order, chunk by chunk of `cnt` timesteps (coma_plan's chunk_nt), (b, tt, n)
// inside a chunk.  A group g = r / N is one (episode, step).
struct CriticRows {
    int B, N, t0, nt, cnt;
    __device__ __forceinline__ void group(int64_t g, int64_t& b, int& t) const {
        const int64_t per = (int64_t)B * cnt;
        const int64_t c = g / per;
        const int64_t loc = g - c * per;
        const int c0 = (int)c * cnt;
        const int cn = nt - c0 < cnt ? nt - c0 : cnt;
        b = loc / cn;
        t = t0 + c0 + (int)(loc - b * cn);
    }
};

// ------------------------------------------------------------------------------------------
// per-row backward through fc3 and fc2
// ------------------------------------------------------------------------------------------
constexpr int RNT = 128;

template <int RT>
__global__ void __launch_bounds__(RNT)
critic_row_bwd_kernel(CriticRows rw, int64_t R, int E, int A, const float* __restrict__ w2, const float* __restrict__ w3,
                      const float* __restrict__ x1, const float* __restrict__ x2, const float* __restrict__ dq,
                      float* __restrict__ dqr, float* __restrict__ dx2, float* __restrict__ dx1) {
    extern __shared__ float rsm[];                         // dq tile [RT][A] | dx2 tile [RT][E]
    float* dqs = rsm;
    float* d2s = rsm + RT * A;
    const int64_t row0 = (int64_t)blockIdx.x * RT;
    for (int i = threadIdx.x; i < RT * A; i += RNT) {
        const int rl = i / A, a = i - rl * A;
        const int64_t r = row0 + rl;
        float v = 0.f;
        if (r < R) {
            const int64_t g = r / rw.N;
            const int n = (int)(r - g * rw.N);
            int64_t b;
            int t;
            rw.group(g, b, t);
            v = __ldg(dq + ((b * rw.nt + (t - rw.t0)) * rw.N + n) * A + a);      // dq [B][nt][N][A]
            dqr[r * A + a] = v;
        }
        dqs[i] = v;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < E; j += RNT) {
        float acc[RT];
#pragma unroll
        for (int i = 0; i < RT; ++i) acc[i] = 0.f;
        for (int a = 0; a < A; ++a) {
            const float w = __ldg(w3 + (int64_t)a * E + j);
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = fmaf(dqs[i * A + a], w, acc[i]);
        }
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            const int64_t r = row0 + i;
            const float v = (r < R && __ldg(x2 + r * E + j) > 0.f) ? acc[i] : 0.f;
            d2s[i * E + j] = v;
            if (r < R) dx2[r * E + j] = v;
        }
    }
    __syncthreads();
    for (int j = threadIdx.x; j < E; j += RNT) {
        float acc[RT];
#pragma unroll
        for (int i = 0; i < RT; ++i) acc[i] = 0.f;
#pragma unroll 4
        for (int k = 0; k < E; ++k) {
            const float w = __ldg(w2 + (int64_t)k * E + j);
#pragma unroll
            for (int i = 0; i < RT; ++i) acc[i] = fmaf(d2s[i * E + k], w, acc[i]);
        }
#pragma unroll
        for (int i = 0; i < RT; ++i) {
            const int64_t r = row0 + i;
            if (r < R) dx1[r * E + j] = __ldg(x1 + r * E + j) > 0.f ? acc[i] : 0.f;
        }
    }
}

// ------------------------------------------------------------------------------------------
// grouped weight gradients
// ------------------------------------------------------------------------------------------
constexpr int NT = 256, TC = 64, TK = 64, TM = 16, MQ = 4, MAXP = 7;
enum Kind { K_ROWS = 0, K_STATE, K_OBS, K_CUR, K_LAST, K_ID };

struct DwProblem {
    int kind;
    const float* D;          // K_ROWS: D [R][C]
    const float* A;          // K_ROWS: A [R][K]
    int C, K;
    float* out; int64_t ldo; // out[c * ldo + k]
    float* bias;             // [C] or NULL
    int tile0, k_tiles;      // first tile in the grid; tiles along k (K_CUR / K_LAST / K_ID: agent quads)
    int64_t part0;           // offset in one slice's partials (C K, + C with a bias)
};
struct DwProblems {
    DwProblem p[MAXP];
    int n;
};
struct CriticIn {
    CriticRows rw;
    const float* dx1;
    const float* state; int64_t state_sb;
    const float* obs; int64_t obs_sb;
    const int64_t* actions; int64_t actions_sb;
    const int64_t* filled; int64_t filled_sb;
    int E, S, O, A;
};

__device__ __forceinline__ void put(const DwProblem& pr, bool direct, float* Pp, int c, int k, float v) {
    if (direct) pr.out[(int64_t)c * pr.ldo + k] = v;
    else Pp[(int64_t)c * pr.K + k] = v;
}

// 64 x 64 output tile of a dense-form problem over rows (K_ROWS, K_OBS) or groups (K_STATE) [mbeg, mend)
__device__ __forceinline__ void dense_tile(const DwProblem& pr, const CriticIn& in, int tile, int64_t mbeg, int64_t mend,
                                           bool direct, float* Pp) {
    __shared__ __align__(16) float Ds[TM][TC + 4];
    __shared__ __align__(16) float As[TM][TK + 4];
    const int k0 = (tile % pr.k_tiles) * TK, c0 = (tile / pr.k_tiles) * TC;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int l_row = tid >> 4, l_q = (tid & 15) * 4;
    const int N = in.rw.N;
    float acc[4][4], bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int64_t mb = mbeg; mb < mend; mb += TM) {
        const int64_t m = mb + l_row;
        const bool ok = m < mend;
        const float* arow = nullptr;
        if (ok && pr.kind != K_ROWS) {
            const int64_t g = pr.kind == K_STATE ? m : m / N;
            int64_t b;
            int t;
            in.rw.group(g, b, t);
            arow = pr.kind == K_STATE ? in.state + b * in.state_sb + (int64_t)t * in.S
                                      : in.obs + b * in.obs_sb + ((int64_t)t * N + (m - g * N)) * in.O;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = c0 + l_q + i, k = k0 + l_q + i;
            float dv = 0.f, av = 0.f;
            if (ok && c < pr.C) {
                if (pr.kind == K_STATE) {                  // the N agents of the group share the state
                    const float* d = in.dx1 + m * N * (int64_t)in.E + c;
                    for (int n = 0; n < N; ++n) dv += __ldg(d + (int64_t)n * in.E);
                } else {
                    dv = __ldg((pr.kind == K_ROWS ? pr.D : in.dx1) + m * pr.C + c);
                }
            }
            if (ok && k < pr.K) av = __ldg(pr.kind == K_ROWS ? pr.A + m * pr.K + k : arow + k);
            Ds[l_row][l_q + i] = dv;
            As[l_row][l_q + i] = av;
        }
        __syncthreads();
#pragma unroll
        for (int mm = 0; mm < TM; ++mm) {
            const float4 dv = *reinterpret_cast<const float4*>(&Ds[mm][ty * 4]);
            const float4 av = *reinterpret_cast<const float4*>(&As[mm][tx * 4]);
            const float d4[4] = {dv.x, dv.y, dv.z, dv.w};
            const float a4[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                bsum[i] += d4[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(d4[i], a4[j], acc[i][j]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = c0 + ty * 4 + i;
        if (c >= pr.C) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k < pr.K) put(pr, direct, Pp, c, k, acc[i][j]);
        }
        if (pr.bias && k0 == 0 && tx == 0) {
            if (direct) pr.bias[c] = bsum[i];
            else Pp[(int64_t)pr.C * pr.K + c] = bsum[i];
        }
    }
}

// one-hot columns of fc1 for agents m0 .. m0+3 and hidden units c0 .. c0+63 over groups [gbeg, gend).  Thread (q, cl)
// owns agent m = m0 + q and unit c = c0 + cl; in K_CUR / K_LAST it owns acc[q][*][cl] in shared memory, so the scatter
// by action index needs no atomics and adds in group order.
__device__ __forceinline__ void onehot_tile(const DwProblem& pr, const CriticIn& in, int tile, int64_t gbeg, int64_t gend,
                                            bool direct, float* Pp, float* acc) {
    const int N = in.rw.N, A = in.A, E = in.E;
    const int m0 = (tile % pr.k_tiles) * MQ, c0 = (tile / pr.k_tiles) * TC;
    const int q = threadIdx.x / TC, cl = threadIdx.x - q * TC;
    const int m = m0 + q, c = c0 + cl;
    if (m >= N || c >= E) return;                          // no barrier below
    float* my = acc + (int64_t)q * A * TC + cl;            // acc[q][a][cl]
    if (pr.kind != K_ID)
        for (int a = 0; a < A; ++a) my[a * TC] = 0.f;
    float id_sum = 0.f;
    for (int64_t g = gbeg; g < gend; ++g) {
        const float* d = in.dx1 + g * N * (int64_t)E + c;
        if (pr.kind == K_ID) {
            id_sum += __ldg(d + (int64_t)m * E);
            continue;
        }
        int64_t b;
        int t;
        in.rw.group(g, b, t);
        const int ts = pr.kind == K_CUR ? t : t - 1;       // K_CUR: actions at t; K_LAST: actions at t - 1
        if (ts < 0 || __ldg(in.filled + b * in.filled_sb + ts) == 0) continue;
        const int a = (int)__ldg(in.actions + b * in.actions_sb + (int64_t)ts * N + m);
        if (a < 0 || a >= A) continue;
        float v = 0.f;
        for (int n = 0; n < N; ++n)
            if (pr.kind == K_LAST || n != m) v += __ldg(d + (int64_t)n * E);
        my[a * TC] += v;
    }
    if (pr.kind == K_ID) put(pr, direct, Pp, c, m, id_sum);
    else
        for (int a = 0; a < A; ++a) put(pr, direct, Pp, c, m * A + a, my[a * TC]);
}

__global__ void __launch_bounds__(NT)
critic_dw_kernel(DwProblems P, CriticIn in, int64_t G, int64_t groups_per_slice, float* __restrict__ partial,
                 int64_t part_stride) {
    extern __shared__ float oh_acc[];                      // [MQ][A][TC] for the one-hot tiles
    int pi = 0;
    while (pi + 1 < P.n && (int)blockIdx.x >= P.p[pi + 1].tile0) ++pi;
    const DwProblem& pr = P.p[pi];
    const int tile = blockIdx.x - pr.tile0;
    const int64_t gbeg = (int64_t)blockIdx.y * groups_per_slice;
    const int64_t gend = gbeg + groups_per_slice < G ? gbeg + groups_per_slice : G;
    const bool direct = gridDim.y == 1;
    float* Pp = partial + (int64_t)blockIdx.y * part_stride + pr.part0;
    if (pr.kind == K_CUR || pr.kind == K_LAST || pr.kind == K_ID) {
        onehot_tile(pr, in, tile, gbeg, gend, direct, Pp, oh_acc);
    } else {
        const int64_t rows = pr.kind == K_STATE ? 1 : in.rw.N;
        dense_tile(pr, in, tile, gbeg * rows, gend * rows, direct, Pp);
    }
}

__global__ void critic_dw_reduce_kernel(DwProblems P, const float* __restrict__ partial, int slices, int64_t part_stride) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= part_stride) return;
    int pi = 0;
    while (pi + 1 < P.n && i >= P.p[pi + 1].part0) ++pi;
    const DwProblem& pr = P.p[pi];
    float s = 0.f;
    for (int sl = 0; sl < slices; ++sl) s += partial[(int64_t)sl * part_stride + i];
    const int64_t e = i - pr.part0, ck = (int64_t)pr.C * pr.K;
    if (e < ck) {
        const int c = (int)(e / pr.K), k = (int)(e - (int64_t)c * pr.K);
        pr.out[(int64_t)c * pr.ldo + k] = s;
    } else {
        pr.bias[e - ck] = s;
    }
}

// the seven problems; returns the floats of one slice's partials
int64_t dw_problems(const pmb_dims* d, const float* dqr, const float* x1, const float* x2, const float* dx2,
                    const CriticGrads& g, DwProblems* P) {
    const int E = d->E, A = d->A, N = d->N, S = d->S, O = d->O;
    const int64_t D = (int64_t)S + O + 2 * (int64_t)N * A + N;
    float* oh = g.w1 + S + O;
    DwProblem p[MAXP] = {
        {K_ROWS, dqr, x2, A, E, g.w3, E, g.b3, 0, 0, 0},                   // fc3.weight / bias
        {K_ROWS, dx2, x1, E, E, g.w2, E, g.b2, 0, 0, 0},                   // fc2.weight / bias
        {K_STATE, nullptr, nullptr, E, S, g.w1, D, g.b1, 0, 0, 0},         // fc1 state columns; fc1.bias = sum of dx1
        {K_OBS, nullptr, nullptr, E, O, g.w1 + S, D, nullptr, 0, 0, 0},    // fc1 obs columns
        {K_CUR, nullptr, nullptr, E, N * A, oh, D, nullptr, 0, 0, 0},      // other agents' actions at t
        {K_LAST, nullptr, nullptr, E, N * A, oh + N * A, D, nullptr, 0, 0, 0},   // every agent's action at t - 1
        {K_ID, nullptr, nullptr, E, N, oh + 2 * N * A, D, nullptr, 0, 0, 0},     // agent id
    };
    int tiles = 0;
    int64_t part = 0;
    for (int i = 0; i < MAXP; ++i) {
        const bool oh_kind = p[i].kind >= K_CUR;
        p[i].tile0 = tiles;
        p[i].k_tiles = (int)(oh_kind ? ceil_div(N, MQ) : ceil_div(p[i].K, TK));
        p[i].part0 = part;
        tiles += p[i].k_tiles * (int)ceil_div(p[i].C, TC);
        part += (int64_t)p[i].C * p[i].K + (p[i].bias ? p[i].C : 0);
        P->p[i] = p[i];
    }
    P->n = MAXP;
    return part;
}

int dw_tiles(const DwProblems& P) {
    const DwProblem& l = P.p[P.n - 1];
    return l.tile0 + l.k_tiles * (int)ceil_div(l.C, TC);
}

// row slices: enough CTAs for two waves, at least 128 rows each
int dw_slices(int tiles, int64_t R, int64_t G) {
    int64_t s = ceil_div((int64_t)2 * sm_count(), tiles), mx = ceil_div(R, 128);
    if (s > mx) s = mx;
    if (s > G) s = G;
    if (s > 64) s = 64;
    return (int)(s < 1 ? 1 : s);
}

struct BwdPlan {
    int64_t R, G, part, off_dx2, off_dx1, off_part, total;
    int slices;
};
BwdPlan bwd_plan(const pmb_dims* d, int nt, DwProblems* P, const float* dqr = nullptr, const float* x1 = nullptr,
                 const float* x2 = nullptr, const float* dx2 = nullptr, const CriticGrads& g = CriticGrads{}) {
    BwdPlan b;
    b.G = (int64_t)d->B * nt;
    b.R = b.G * d->N;
    b.part = dw_problems(d, dqr, x1, x2, dx2, g, P);
    b.slices = dw_slices(dw_tiles(*P), b.R, b.G);
    b.off_dx2 = align_up(b.R * d->A * 4, 256);
    b.off_dx1 = b.off_dx2 + align_up(b.R * d->E * 4, 256);
    b.off_part = b.off_dx1 + align_up(b.R * d->E * 4, 256);
    b.total = b.off_part + (b.slices > 1 ? align_up(b.slices * b.part * 4, 256) : 0);
    return b;
}

template <int RT>
int launch_row_bwd(const CriticRows& rw, int64_t R, int E, int A, const float* w2, const float* w3, const float* x1,
                   const float* x2, const float* dq, float* dqr, float* dx2, float* dx1, cudaStream_t s) {
    const size_t smem = (size_t)RT * (A + E) * sizeof(float);
    auto kern = critic_row_bwd_kernel<RT>;
    PMB_SMEM_ATTR(kern, smem);
    kern<<<(unsigned)ceil_div(R, RT), RNT, smem, s>>>(rw, R, E, A, w2, w3, x1, x2, dq, dqr, dx2, dx1);
    PMB_LAUNCH_CHECK("critic_row_bwd_kernel");
    return PMB_OK;
}

}  // namespace

int64_t critic_step_bwd_scratch(const pmb_dims* d, int nt) {
    DwProblems P;
    return bwd_plan(d, nt, &P).total;
}

int critic_step_bwd(const pmb_dims* d, const pmb_batch* b, int t0, int nt, int chunk_nt, const CriticParams& cp,
                    const float* x1, const float* x2, const float* dq, const CriticGrads& g, void* scratch,
                    int64_t scratch_bytes, cudaStream_t s) {
    const int E = d->E, A = d->A;
    char* base = static_cast<char*>(scratch);
    DwProblems P;
    BwdPlan pl = bwd_plan(d, nt, &P);
    if (scratch_bytes < pl.total) {
        set_error("coma_critic_step_bwd: scratch too small (%lld < %lld)", (long long)scratch_bytes, (long long)pl.total);
        return PMB_ERR_WORKSPACE;
    }
    float* dqr = reinterpret_cast<float*>(base);
    float* dx2 = reinterpret_cast<float*>(base + pl.off_dx2);
    float* dx1 = reinterpret_cast<float*>(base + pl.off_dx1);
    float* partial = reinterpret_cast<float*>(base + pl.off_part);
    pl = bwd_plan(d, nt, &P, dqr, x1, x2, dx2, g);
    const CriticRows rw{d->B, d->N, t0, nt, chunk_nt};
    // 16-row tiles once they give every SM a block, else 4-row tiles (a single step: B N rows)
    const int rc = ceil_div(pl.R, 16) >= sm_count()
                       ? launch_row_bwd<16>(rw, pl.R, E, A, cp.w2, cp.w3, x1, x2, dq, dqr, dx2, dx1, s)
                       : launch_row_bwd<4>(rw, pl.R, E, A, cp.w2, cp.w3, x1, x2, dq, dqr, dx2, dx1, s);
    if (rc) return rc;

    CriticIn in{};
    in.rw = rw;
    in.dx1 = dx1;
    in.state = static_cast<const float*>(b->state); in.state_sb = b->state_sb;
    in.obs = static_cast<const float*>(b->obs); in.obs_sb = b->obs_sb;
    in.actions = b->actions; in.actions_sb = b->actions_sb;
    in.filled = b->filled; in.filled_sb = b->filled_sb;
    in.E = E; in.S = d->S; in.O = d->O; in.A = A;
    const int tiles = dw_tiles(P);
    const int64_t per_slice = ceil_div(pl.G, pl.slices);
    const size_t smem = (size_t)MQ * A * TC * sizeof(float);
    PMB_SMEM_ATTR(critic_dw_kernel, smem);
    critic_dw_kernel<<<dim3((unsigned)tiles, (unsigned)pl.slices), NT, smem, s>>>(P, in, pl.G, per_slice, partial, pl.part);
    PMB_LAUNCH_CHECK("critic_dw_kernel");
    if (pl.slices == 1) return PMB_OK;
    critic_dw_reduce_kernel<<<(unsigned)ceil_div(pl.part, 256), 256, 0, s>>>(P, partial, pl.slices, pl.part);
    PMB_LAUNCH_CHECK("critic_dw_reduce_kernel");
    return PMB_OK;
}

}  // namespace pmb
