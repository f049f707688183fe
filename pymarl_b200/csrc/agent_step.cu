// Backward of ONE agent step (fc1 -> ReLU -> GRUCell -> fc2), fp32 on every tier: what autograd through RNNAgent.forward
// and BasicMAC.forward needs when a user's learner differentiates through them (one graph node per timestep).
//
//   agent_step_bwd_kernel : fused per-row backward.  dh = dh_in + dq W_2; the GRU-cell gate gradients
//                           (da_r | da_z | da_n | da_n * r) -> dg [R][4H]; dh_prev = dh z + [da_r | da_z | da_n r] W_hh;
//                           dpre1 = relu'(x) * ([da_r | da_z | da_n] W_ih).  A single step has no recurrence, so the weights
//                           are read through L1 / L2 instead of being staged: one kernel for every rnn_hidden_dim.
//   step_dw_kernel        : every weight gradient of the step in one launch - a grouped out[c][k] = sum_m D[m][c] A[m][k]
//                           (+ bias[c] = sum_m D[m][c]) over five problems (W_ih, the two W_hh row blocks, fc2, fc1).
//                           fc1's A operand is the step's virtual input [obs | last-action one-hot | agent-id one-hot]
//                           generated from the batch, or a dense input matrix.  64 x 64 output tiles, rows split into fixed
//                           slices; with more than one slice step_dw_reduce_kernel adds the partials in slice order.
// No float atomics: two identical calls give identical bits.
//
// reference: modules/agents/rnn_agent.py:27-36, controllers/basic_controller.py:100-135 and torch autograd through them.
#include "common.cuh"

namespace pmb {

namespace {

constexpr int NT = 256;

template <int H, int RW>
__global__ void __launch_bounds__(NT)
agent_step_bwd_kernel(AgentParams p, int A, int64_t R, const float* __restrict__ x, const float* __restrict__ h_prev,
                      const float* __restrict__ gates, const float* __restrict__ dq, const float* __restrict__ dh_in,
                      float* __restrict__ dg, float* __restrict__ dpre1, float* __restrict__ dh_prev) {
    constexpr int JW = H / 16, LDD = 4 * H + 1;
    extern __shared__ float dgs[];                                    // [16 RW][4H+1] the tile's gate gradients
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int j0 = tx * JW;
    const int64_t row0 = (int64_t)blockIdx.x * 16 * RW;

    float dhz[RW][JW];
#pragma unroll
    for (int i = 0; i < RW; ++i) {
        const int rl = ty * RW + i;
        const int64_t row = row0 + rl;
        float dr_[JW], dz_[JW], dn_[JW], dnr_[JW];
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) { dr_[jj] = dz_[jj] = dn_[jj] = dnr_[jj] = 0.f; dhz[i][jj] = 0.f; }
        if (row < R) {
            float d[JW];
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) d[jj] = dh_in ? __ldg(dh_in + row * H + j0 + jj) : 0.f;
            if (dq) {
                for (int a = 0; a < A; ++a) {
                    const float g = __ldg(dq + row * A + a);
#pragma unroll
                    for (int jj = 0; jj < JW; ++jj) d[jj] = fmaf(g, __ldg(p.fc2_w + a * H + j0 + jj), d[jj]);
                }
            }
            const float* gr = gates + row * 4 * H + j0;
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                const float r = __ldg(gr + jj), z = __ldg(gr + H + jj), n = __ldg(gr + 2 * H + jj);
                const float ghn = __ldg(gr + 3 * H + jj), hp = __ldg(h_prev + row * H + j0 + jj);
                // torch GRUCell: h' = n + z (h - n)
                const float da_n = d[jj] * (1.f - z) * (1.f - n * n);
                dr_[jj] = (da_n * ghn) * r * (1.f - r);
                dz_[jj] = d[jj] * (hp - n) * z * (1.f - z);
                dn_[jj] = da_n;
                dnr_[jj] = da_n * r;
                dhz[i][jj] = d[jj] * z;
            }
            float* o = dg + row * 4 * H + j0;
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) { o[jj] = dr_[jj]; o[H + jj] = dz_[jj]; o[2 * H + jj] = dn_[jj]; o[3 * H + jj] = dnr_[jj]; }
        }
        float* s = dgs + rl * LDD + j0;
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) { s[jj] = dr_[jj]; s[H + jj] = dz_[jj]; s[2 * H + jj] = dn_[jj]; s[3 * H + jj] = dnr_[jj]; }
    }
    __syncthreads();

    float dx[RW][JW], dhp[RW][JW];
#pragma unroll
    for (int i = 0; i < RW; ++i)
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) { dx[i][jj] = 0.f; dhp[i][jj] = dhz[i][jj]; }
    // dx += da_c W_ih[c];  dh_prev += (c < 2H ? da_c : da_n r) W_hh[c]
#pragma unroll 2
    for (int c = 0; c < 3 * H; ++c) {
        float wi[JW], wh[JW], di[RW], dh[RW];
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) { wi[jj] = __ldg(p.w_ih + c * H + j0 + jj); wh[jj] = __ldg(p.w_hh + c * H + j0 + jj); }
#pragma unroll
        for (int i = 0; i < RW; ++i) {
            di[i] = dgs[(ty * RW + i) * LDD + c];
            dh[i] = dgs[(ty * RW + i) * LDD + (c < 2 * H ? c : c + H)];
        }
#pragma unroll
        for (int i = 0; i < RW; ++i)
#pragma unroll
            for (int jj = 0; jj < JW; ++jj) {
                dx[i][jj] = fmaf(di[i], wi[jj], dx[i][jj]);
                dhp[i][jj] = fmaf(dh[i], wh[jj], dhp[i][jj]);
            }
    }
#pragma unroll
    for (int i = 0; i < RW; ++i) {
        const int64_t row = row0 + ty * RW + i;
        if (row >= R) continue;
#pragma unroll
        for (int jj = 0; jj < JW; ++jj) {
            dpre1[row * H + j0 + jj] = __ldg(x + row * H + j0 + jj) > 0.f ? dx[i][jj] : 0.f;
            if (dh_prev) dh_prev[row * H + j0 + jj] = dhp[i][jj];
        }
    }
}

// ------------------------------------------------------------------------------------------
// grouped weight gradients
// ------------------------------------------------------------------------------------------
constexpr int TC = 64, TK = 64, TM = 16, MAXP = 5;

struct DwProblem {
    const float* D; int64_t ldd;       // D[m][c] (NULL: zero, e.g. no gradient reached q)
    const float* A; int64_t lda;       // A[m][k] (NULL: the step's virtual input, see StepInput)
    int C, K;
    float* out; int64_t ldo;           // out[c * ldo + k]
    float* bias;                       // [C]
    int tile0, k_tiles;                // first tile of the problem in the grid, tiles along k
    int64_t part0;                     // offset of the problem in one slice's partials (C K + C floats)
};
struct DwProblems {
    DwProblem p[MAXP];
    int n;
};

// the fc1 input of row m = b N + n at batch time t, as pmb_agent_fc1_fwd reads it (controllers/basic_controller.py:100-135)
struct StepInput {
    const float* obs; int64_t obs_sb;
    const int64_t* actions; int64_t actions_sb;
    const int64_t* filled; int64_t filled_sb;
    int t, N, O, A, use_act, use_id;
    __device__ __forceinline__ int last_action(int64_t m) const {
        const int64_t b = m / N;
        const int n = (int)(m - b * N);
        if (!use_act || t == 0 || __ldg(filled + b * filled_sb + (t - 1)) == 0) return -1;
        return (int)__ldg(actions + b * actions_sb + (int64_t)(t - 1) * N + n);
    }
    __device__ __forceinline__ float at(int64_t m, int k, int a_prev) const {
        const int64_t b = m / N;
        const int n = (int)(m - b * N);
        if (k < O) return __ldg(obs + b * obs_sb + ((int64_t)t * N + n) * O + k);
        k -= O;
        if (use_act) {
            if (k < A) return k == a_prev ? 1.f : 0.f;
            k -= A;
        }
        return k == n ? 1.f : 0.f;
    }
};

__global__ void __launch_bounds__(NT)
step_dw_kernel(DwProblems P, StepInput in, int64_t M, int64_t rows_per_slice, float* __restrict__ partial,
               int64_t part_stride) {
    __shared__ __align__(16) float Ds[TM][TC + 4];
    __shared__ __align__(16) float As[TM][TK + 4];
    int pi = 0;
    while (pi + 1 < P.n && (int)blockIdx.x >= P.p[pi + 1].tile0) ++pi;
    const DwProblem& pr = P.p[pi];
    const int tile = blockIdx.x - pr.tile0;
    const int k0 = (tile % pr.k_tiles) * TK, c0 = (tile / pr.k_tiles) * TC;
    const int64_t mbeg = (int64_t)blockIdx.y * rows_per_slice;
    const int64_t mend = mbeg + rows_per_slice < M ? mbeg + rows_per_slice : M;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int l_row = tid >> 4, l_q = (tid & 15) * 4;

    float acc[4][4], bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int64_t mb = mbeg; mb < mend; mb += TM) {
        const int64_t m = mb + l_row;
        const bool ok = m < mend;
        const int a_prev = (ok && !pr.A) ? in.last_action(m) : -1;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int c = c0 + l_q + i, k = k0 + l_q + i;
            Ds[l_row][l_q + i] = (ok && pr.D && c < pr.C) ? __ldg(pr.D + m * pr.ldd + c) : 0.f;
            As[l_row][l_q + i] = (ok && k < pr.K) ? (pr.A ? __ldg(pr.A + m * pr.lda + k) : in.at(m, k, a_prev)) : 0.f;
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
    // one slice: straight into the gradient block; else this slice's partials
    const bool direct = gridDim.y == 1;
    float* Pp = partial + (int64_t)blockIdx.y * part_stride + pr.part0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = c0 + ty * 4 + i;
        if (c >= pr.C) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k >= pr.K) continue;
            if (direct) pr.out[(int64_t)c * pr.ldo + k] = acc[i][j];
            else Pp[(int64_t)c * pr.K + k] = acc[i][j];
        }
        if (k0 == 0 && tx == 0) {
            if (direct) pr.bias[c] = bsum[i];
            else Pp[(int64_t)pr.C * pr.K + c] = bsum[i];
        }
    }
}

__global__ void step_dw_reduce_kernel(DwProblems P, const float* __restrict__ partial, int slices, int64_t part_stride) {
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

// the five problems of one step; returns the floats of one slice's partials
int64_t dw_problems(const pmb_dims* d, int64_t R, const float* inputs, const float* x, const float* h_stash, const float* dq,
                    const float* dg, const float* dpre1, AgentGrads gr, DwProblems* P) {
    const int H = d->H, A = d->A, D_in = d_in_of(d);
    const float* h_prev = h_stash;
    const float* h = h_stash + R * H;
    DwProblem p[MAXP] = {
        {dg, 4 * H, x, H, 3 * H, H, gr.w_ih, H, gr.b_ih, 0, 0, 0},                            // rnn.weight_ih / bias_ih
        {dg, 4 * H, h_prev, H, 2 * H, H, gr.w_hh, H, gr.b_hh, 0, 0, 0},                       // rnn.weight_hh rows r, z
        {dg + 3 * H, 4 * H, h_prev, H, H, H, gr.w_hh + 2 * H * H, H, gr.b_hh + 2 * H, 0, 0, 0},   // rows n: (da_n r) h_prev
        {dq, A, h, H, A, H, gr.fc2_w, H, gr.fc2_b, 0, 0, 0},                                  // fc2
        {dpre1, H, inputs, D_in, H, D_in, gr.fc1_w, D_in, gr.fc1_b, 0, 0, 0},                 // fc1 (whole D_in)
    };
    int tiles = 0;
    int64_t part = 0;
    for (int i = 0; i < MAXP; ++i) {
        p[i].tile0 = tiles;
        p[i].k_tiles = (int)ceil_div(p[i].K, TK);
        p[i].part0 = part;
        tiles += p[i].k_tiles * (int)ceil_div(p[i].C, TC);
        part += (int64_t)p[i].C * p[i].K + p[i].C;
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
int dw_slices(int tiles, int64_t R) {
    int64_t s = ceil_div((int64_t)2 * sm_count(), tiles), mx = ceil_div(R, 128);
    if (s > mx) s = mx;
    if (s > 64) s = 64;
    return (int)(s < 1 ? 1 : s);
}

template <int H, int RW>
int launch_step_bwd(const AgentParams& p, int A, int64_t R, const float* x, const float* h_prev, const float* gates,
                    const float* dq, const float* dh, float* dg, float* dpre1, float* dh_prev, cudaStream_t s) {
    const size_t smem = (size_t)16 * RW * (4 * H + 1) * sizeof(float);
    auto kern = agent_step_bwd_kernel<H, RW>;
    PMB_SMEM_ATTR(kern, smem);
    kern<<<(unsigned)ceil_div(R, 16 * RW), NT, smem, s>>>(p, A, R, x, h_prev, gates, dq, dh, dg, dpre1, dh_prev);
    PMB_LAUNCH_CHECK("agent_step_bwd_kernel");
    return PMB_OK;
}

}  // namespace

int64_t agent_step_bwd_scratch(const pmb_dims* d, int64_t R) {
    DwProblems P;
    const int64_t part = dw_problems(d, R, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, AgentGrads{}, &P);
    const int sl = dw_slices(dw_tiles(P), R);
    return align_up(R * 4 * d->H * 4, 256) + align_up(R * d->H * 4, 256) + (sl > 1 ? align_up(sl * part * 4, 256) : 0);
}

int agent_step_bwd(const pmb_dims* d, const pmb_batch* b, int t, const float* inputs, int64_t R, const float* flat_agent,
                   const float* x, const float* h_stash, const float* gates, const float* dq, const float* dh,
                   float* dh_prev, float* flat_grad_agent, void* scratch, int64_t scratch_bytes, cudaStream_t s) {
    if (scratch_bytes < agent_step_bwd_scratch(d, R)) {
        set_error("agent_step_bwd: scratch too small (%lld < %lld)", (long long)scratch_bytes,
                  (long long)agent_step_bwd_scratch(d, R));
        return PMB_ERR_WORKSPACE;
    }
    const int H = d->H;
    const AgentParams ap = agent_params(d, flat_agent);
    float* dg = static_cast<float*>(scratch);
    float* dpre1 = reinterpret_cast<float*>(static_cast<char*>(scratch) + align_up(R * 4 * H * 4, 256));
    float* partial = reinterpret_cast<float*>(reinterpret_cast<char*>(dpre1) + align_up(R * H * 4, 256));
    const bool wide = ceil_div(R, 64) >= 2 * (int64_t)sm_count();      // 64-row tiles once they fill the machine twice
    int rc;
#define PMB_STEP(HH)                                                                                                      \
    rc = wide ? launch_step_bwd<HH, 4>(ap, d->A, R, x, h_stash, gates, dq, dh, dg, dpre1, dh_prev, s)                      \
              : launch_step_bwd<HH, 1>(ap, d->A, R, x, h_stash, gates, dq, dh, dg, dpre1, dh_prev, s);                     \
    break
    switch (H) {
        case 16: PMB_STEP(16);
        case 32: PMB_STEP(32);
        case 64: PMB_STEP(64);
        case 128: PMB_STEP(128);
        default: set_error("rnn_hidden_dim %d unsupported (16, 32, 64, 128)", H); return PMB_ERR_INVALID;
    }
#undef PMB_STEP
    if (rc) return rc;

    DwProblems P;
    const int64_t part = dw_problems(d, R, inputs, x, h_stash, dq, dg, dpre1, agent_grads(d, flat_grad_agent), &P);
    const int tiles = dw_tiles(P), sl = dw_slices(tiles, R);
    StepInput in{};
    if (b) {
        in.obs = static_cast<const float*>(b->obs); in.obs_sb = b->obs_sb;
        in.actions = b->actions; in.actions_sb = b->actions_sb;
        in.filled = b->filled; in.filled_sb = b->filled_sb;
    }
    in.t = t; in.N = b ? d->N : 1; in.O = d->O; in.A = d->A; in.use_act = d->obs_last_action; in.use_id = d->obs_agent_id;
    const int64_t rows_per_slice = align_up(ceil_div(R, sl), TM);
    step_dw_kernel<<<dim3((unsigned)tiles, (unsigned)sl), NT, 0, s>>>(P, in, R, rows_per_slice, partial, part);
    PMB_LAUNCH_CHECK("step_dw_kernel");
    if (sl == 1) return PMB_OK;
    step_dw_reduce_kernel<<<(unsigned)ceil_div(part, 256), 256, 0, s>>>(P, partial, sl, part);
    PMB_LAUNCH_CHECK("step_dw_reduce_kernel");
    return PMB_OK;
}

}  // namespace pmb
