/*
 * pymarl_b200.h - C ABI of libpymarl_b200.so: the PyMARL QMIX/VDN/IQL learner step and the
 * batched agent forward / epsilon-greedy action selection as hand-written sm_100a CUDA.
 *
 * The reference (nicholasburden/pymarl) has no FFI for this path: its boundary is Python
 * duck typing through four registries.  The Python mirror of that surface lives in
 * pymarl_b200/ (QLearner, BasicMAC, RNNAgent, QMixer, VDNMixer, EpsilonGreedyActionSelector)
 * and binds the entry points below with ctypes (pymarl_b200/_lib.py); INTEGRATION.md shows
 * the stub.  Each entry point names the reference code it replaces (paths relative to
 * /root/reference/src).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host
 *   - the library allocates nothing: workspaces are sized by pmb_*_workspace_bytes() and
 *     allocated by the caller (torch caching allocator), so calls are CUDA-graph capturable
 *   - calls are asynchronous on `stream`; return 0 on success, else a pmb_status (a message
 *     is available from pmb_last_error()); nothing is printed, nothing throws
 *   - not re-entrant on the same buffers; one learner per (process, device)
 *
 * Batch layout = the reference EpisodeBatch (components/episode_buffer.py:58-86,
 * run.py:122-135): batch major, time second, innermost dims contiguous; only the batch
 * stride is free (a `batch[:, :max_t]` slice keeps the full-T batch stride).
 *
 * Internal (workspace) activations are TIME major: x/h/q[t][p][.] with p = b*N + n.
 */
#ifndef PYMARL_B200_H
#define PYMARL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pmb_stream;            /* cudaStream_t */

enum pmb_status {
    PMB_OK = 0,
    PMB_ERR_INVALID = 1,             /* bad dims / null pointer / unsupported size */
    PMB_ERR_CUDA = 2,                /* a CUDA runtime call failed; see pmb_last_error() */
    PMB_ERR_WORKSPACE = 3            /* workspace too small */
};

enum pmb_mixer { PMB_MIXER_NONE = 0 /* IQL */, PMB_MIXER_VDN = 1, PMB_MIXER_QMIX = 2 };

/* precision tiers (BASELINE.json north_star): FP32 = CUDA-core FFMA, parity 1e-5;
 * BF16 = tcgen05 tensor cores with fp32 accumulate, parity 1e-2. */
enum pmb_precision { PMB_PREC_FP32 = 0, PMB_PREC_BF16 = 1 };

typedef struct pmb_dims {
    int32_t B;                 /* episodes in the batch                                   */
    int32_t T;                 /* batch.max_seq_length                                    */
    int32_t N;                 /* n_agents                                                */
    int32_t O;                 /* obs dim                                                 */
    int32_t S;                 /* state dim                                               */
    int32_t A;                 /* n_actions                                               */
    int32_t H;                 /* rnn_hidden_dim  (16, 32, 64 or 128)                     */
    int32_t E;                 /* mixing_embed_dim (8, 16, 32 or 64)                      */
    int32_t obs_last_action;   /* controllers/basic_controller.py:111                     */
    int32_t obs_agent_id;      /* controllers/basic_controller.py:118                     */
    int32_t mixer;             /* enum pmb_mixer (learners/q_learner.py:19-27)            */
    int32_t double_q;          /* learners/q_learner.py:71                                */
    int32_t precision;         /* enum pmb_precision                                      */
    int32_t reserved;          /* flags.  bit 0 (pmb_select_actions_step, tensor-core tier only): the packed weight
                                * images a previous call left in `scratch` are still current - same parameters, same
                                * scratch - so the step skips its two weight-pack launches.
                                * bit 1 (pmb_qlearner_train_step): skip the padded timesteps of a ragged batch.  The step
                                * sorts the episodes on the device by the forward steps they need (F_b = min(T, l_b + 2),
                                * l_b = last t with filled = 1; 0 for an empty episode), longest first and stable, and the
                                * agent kernels (fc1, both recurrences, fc2 + target selection, BPTT, fc1/fc2 weight
                                * gradients) run only the (t, 128-row tile) items some row of the tile still needs.  Loss
                                * sums and gradients are those of the unsorted step up to fp32 summation order.  Honoured
                                * where batch.ep_index is (bf16 tier, H = 64, A <= 64, QMIX with E = 32 or VDN / IQL,
                                * O <= 320, agent id folding into the K padding of obs); elsewhere ignored, and the step is
                                * bit-identical to the step without it.  pmb_learner_workspace_bytes counts the schedule
                                * area only where the bit is honoured.  0 is always safe.                             */
} pmb_dims;

/* Element type of pmb_batch.obs.  BF16 (a scheme with "obs": {..., "dtype": th.bfloat16}, stored with torch's
 * round-to-nearest-even) is read natively only where pmb_obs_bf16_supported() says so; every other entry point that reads
 * obs returns PMB_ERR_INVALID for it.  The bf16 tier rounds obs to bf16 before its first use, so there a bf16-stored batch
 * gives results bit-identical to an fp32-stored one holding the same (bf16-representable) values. */
enum pmb_dtype { PMB_DTYPE_F32 = 0, PMB_DTYPE_BF16 = 1, PMB_DTYPE_U8 = 2 };

/* The EpisodeBatch fields the path reads.  *_sb = batch stride in ELEMENTS (of the field's own type). */
typedef struct pmb_batch {
    const void*    obs;        int64_t obs_sb;          /* [B,T,N,O] f32, or bf16 (obs_dtype) */
    const void*    state;      int64_t state_sb;        /* [B,T,S]   f32, or bf16 (state_dtype) (QMIX only, else NULL) */
    const int64_t* actions;    int64_t actions_sb;      /* [B,T,N,1] i64 */
    const void*    avail;      int64_t avail_sb;        /* [B,T,N,A] i32, or u8 (avail_dtype) */
    const float*   reward;     int64_t reward_sb;       /* [B,T,1]   f32 */
    const uint8_t* terminated; int64_t terminated_sb;   /* [B,T,1]   u8  */
    const int64_t* filled;     int64_t filled_sb;       /* [B,T,1]   i64 */
    /* Optional (may be NULL): zero-copy replay sampling.  Batch row b is episode ep_index[b] of the fields above
     * (which then are the WHOLE replay buffer): ReplayBuffer.sample / EpisodeBatch.__getitem__(ids)
     * (components/episode_buffer.py:205-217,291-298) without the gather copy.  Device array of B ids.  Supported by
     * the tensor-core tier of pmb_qlearner_train_step only. */
    const int64_t* ep_index;
    int32_t obs_dtype;         /* enum pmb_dtype; 0 (fp32) is always accepted, any value but 0 and 1 is PMB_ERR_INVALID */
    /* Compact state / avail storage ("state": {..., "dtype": th.bfloat16}, "avail_actions": {..., "dtype": th.uint8} or
     * th.bool, passed as uint8).  Read natively only where pmb_field_dtype_supported() says so; elsewhere, and for any
     * other value, PMB_ERR_INVALID.  The tensor-core mixer rounds state to bf16 before its first use and avail holds 0 / 1,
     * so the results are bit-identical to fp32 / i32 storage of the same values.
     * The two fields take what was the struct's tail padding: sizeof(pmb_batch) stays 128 and a zero-initialised struct
     * laid out by an earlier header keeps its meaning. */
    int16_t state_dtype;       /* 0 = f32 (always accepted), PMB_DTYPE_BF16 */
    int16_t avail_dtype;       /* 0 = i32, the reference's th.int (always accepted), PMB_DTYPE_U8 */
} pmb_batch;

/* 1 where the kernels of `entry` read PMB_DTYPE_BF16 obs natively for these dims, else 0 (host only, no device call):
 *   PMB_ENTRY_TRAIN_STEP      pmb_qlearner_train_step on the fused tensor-core path (bf16 tier, H = 64, A <= 64, QMIX with
 *                             E = 32 or VDN / IQL, O <= 320, agent id folding into the K padding of obs) where the
 *                             streaming fc1 kernel runs (its staging ring fits shared memory)
 *   PMB_ENTRY_SELECT_ACTIONS  pmb_select_actions_step on the tensor-core tier where the streaming fc1 kernel runs
 * The fp32 tier, the generic tcgen05 fc1 GEMM, pmb_agent_fc1_fwd, pmb_agent_unroll_bwd and the COMA entry points read fp32
 * obs only: convert first. */
enum pmb_entry { PMB_ENTRY_TRAIN_STEP = 0, PMB_ENTRY_SELECT_ACTIONS = 1 };
int pmb_obs_bf16_supported(const pmb_dims* d, int32_t entry);

/* 1 where the kernels of `entry` accept `field` stored as `dtype` for these dims, else 0 (host only, no device call).
 * dtype 0 (the reference's type: f32 obs / state, i32 avail) is accepted everywhere.  Besides that:
 *   PMB_FIELD_OBS,   PMB_DTYPE_BF16  as pmb_obs_bf16_supported()
 *   PMB_FIELD_STATE, PMB_DTYPE_BF16  PMB_ENTRY_TRAIN_STEP where the tensor-core mixer runs (bf16 tier, QMIX with E = 32)
 *   PMB_FIELD_AVAIL, PMB_DTYPE_U8    PMB_ENTRY_TRAIN_STEP where the tensor-core agent runs (bf16 tier, H = 64, A <= 64);
 *                                    PMB_ENTRY_SELECT_ACTIONS on the tensor-core tier (bf16 tier, H = 64, A <= 64, O <= 320)
 * The fp32 tier, pmb_target_select, pmb_epsilon_greedy, pmb_mixer_* and the COMA entry points read f32 state and i32
 * avail only: convert first. */
enum pmb_field { PMB_FIELD_OBS = 0, PMB_FIELD_STATE = 1, PMB_FIELD_AVAIL = 2 };
int pmb_field_dtype_supported(const pmb_dims* d, int32_t entry, int32_t field, int32_t dtype);

/* Flat parameter layout.  Agent tensors keep the reference order (modules/agents/rnn_agent.py:19-21);
 * the mixer puts the four hypernet weight matrices first so they form ONE [ (N+3)E, S ]
 * matrix (hyper_w_1 | hyper_w_final | hyper_b_1 | V.0), then their biases in the same
 * order, then V.2.weight, V.2.bias (modules/mixers/qmix.py:17-26). */
enum pmb_param_id {
    PMB_P_FC1_W = 0, PMB_P_FC1_B, PMB_P_W_IH, PMB_P_W_HH, PMB_P_B_IH, PMB_P_B_HH, PMB_P_FC2_W, PMB_P_FC2_B,
    PMB_P_HW1_W, PMB_P_HWF_W, PMB_P_HB1_W, PMB_P_V0_W, PMB_P_HW1_B, PMB_P_HWF_B, PMB_P_HB1_B, PMB_P_V0_B,
    PMB_P_V2_W, PMB_P_V2_B, PMB_P_COUNT
};
typedef struct pmb_layout {
    int64_t offset[PMB_P_COUNT];     /* element offset of each tensor in the flat buffer  */
    int64_t numel[PMB_P_COUNT];
    int64_t n_agent;                 /* elements of the 8 agent tensors                   */
    int64_t n_total;                 /* agent + mixer (mixer part is 0 unless QMIX)       */
} pmb_layout;

/* hyper-parameters of one train step (learners/q_learner.py:30,86,102,105) */
typedef struct pmb_hparams {
    float gamma, lr, alpha, eps, grad_norm_clip;
    int32_t do_target_sync;          /* host decides: (episode_num - last)/interval >= 1  */
    int32_t skip_update;             /* 1: stop after the gradients (multi-GPU: all-reduce, then pmb_clip_rmsprop_update) */
    int32_t keep_q;                  /* debug bits (tests): 1 = bf16 tier also writes the Q tensors (mac_out) into the
                                      * workspace; 2 = stop after the forward pass and the loss sums (q_learner.py:39-97),
                                      * leaving every forward intermediate in the workspace.  With padded-step skipping
                                      * (pmb_dims.reserved bit 1) the Q tensors are unspecified on the skipped (t, tile)
                                      * items, and chosen / tmax are 0 there */
} pmb_hparams;

/* stats buffer: 16 doubles on the device, written by the step */
enum pmb_stat_id {
    PMB_S_MASK_SUM = 0,      /* sum(mask)                       q_learner.py:97  */
    PMB_S_TD2_SUM,           /* sum((td*mask)^2)                :97              */
    PMB_S_TDABS_SUM,         /* sum(|td*mask|)                  :113             */
    PMB_S_QTAKEN_SUM,        /* sum(chosen_q_tot*mask)          :114             */
    PMB_S_TARGET_SUM,        /* sum(targets*mask)               :115             */
    PMB_S_GRAD_NORM,         /* total grad norm before clipping :102             */
    PMB_S_LOSS,              /* TD2_SUM / MASK_SUM                                */
    PMB_S_CLIP_COEF,
    PMB_S_COUNT = 16
};

const char* pmb_last_error(void);
int  pmb_version(void);
/* sm count, compute capability and opt-in shared memory of the current device */
int  pmb_device_info(int32_t* sm_count, int32_t* cc_major, int32_t* cc_minor, int64_t* smem_optin_bytes);
int  pmb_flat_layout(const pmb_dims* d, pmb_layout* out);
/* bytes of scratch pmb_qlearner_train_step needs for these dims */
int64_t pmb_learner_workspace_bytes(const pmb_dims* d);

/* ---- K1: agent forward -------------------------------------------------------------- */
/* fc1 over nt timesteps starting at t0, inputs never concatenated:
 *   x = relu(W_obs obs + W_act[:, a_{t-1}] (0 at t == 0 or if step t-1 is padded) + W_id[:, n] + b)
 * replaces BasicMAC._build_inputs + RNNAgent.fc1 (basic_controller.py:100-135, rnn_agent.py:32).
 * x_out: [nt][B*N][H]. */
int pmb_agent_fc1_fwd(const pmb_dims* d, const pmb_batch* b, int32_t t0, int32_t nt,
                      const float* flat_agent, float* x_out, pmb_stream stream);
/* same for an already concatenated input matrix inputs[R][D_in] (RNNAgent.forward called
 * directly, rnn_agent.py:27-32). */
int pmb_agent_fc1_dense_fwd(const pmb_dims* d, int64_t rows, int32_t d_in, const float* inputs,
                            const float* flat_agent, float* x_out, pmb_stream stream);
/* GRUCell + fc2 unrolled over nt steps for R = rows (rnn_agent.py:33-36, the t loops of
 * q_learner.py:47-52,58-62).  h0 NULL = zeros (basic_controller.py:77-81).
 * h_stash [(nt+1)][R][H] (slot 0 = h0) and gates [nt][R][4H] (r,z,n,W_hn h+b_hn) are
 * written when non-NULL (needed by the backward); q [nt][R][A]; h_last [R][H] optional.
 * H = 128: gates is required (it first receives the input gates x W_ih^T + b_ih), and so is
 * h_stash unless nt == 1 and h_last is given (q is computed from the stashed hidden states). */
int pmb_agent_gru_unroll_fwd(const pmb_dims* d, int64_t rows, int32_t nt, const float* flat_agent,
                             const float* x, const float* h0, float* h_stash, float* gates,
                             float* q, float* h_last, pmb_stream stream);

/* ---- K2: chosen-action gather, avail masking, double-Q target (q_learner.py:55-78) ---- */
/* q_on, q_tg: [T][B*N][A] time major.  chosen, tmax: [B][T-1][N]; cur_max (int32, may be
 * NULL): the arg-max action index.  Ties -> lowest index; masked value -9999999. */
int pmb_target_select(const pmb_dims* d, const pmb_batch* b, const float* q_on, const float* q_tg,
                      float* chosen, float* tmax, int32_t* cur_max, pmb_stream stream);

/* ---- K3: mixers (modules/mixers/qmix.py:28-47, vdn.py:9-10) ---------------------------- */
/* agent_qs [B][T-1][N]; uses state[:, t_off : t_off+T-1] (0 online, 1 target).
 * QMIX: raw [B*(T-1)][(N+3)E] receives the hypernet outputs (kept for the backward).
 * q_tot [B*(T-1)] (VDN) ; for PMB_MIXER_NONE the call is an error (IQL has no mixer). */
int pmb_mixer_fwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs,
                  int32_t t_off, float* raw, float* q_tot, pmb_stream stream);

/* ---- K4: TD target, masked loss sums, dL/dq_tot (q_learner.py:39-44,86-97) ------------- */
/* q_tot / t_tot: [B][T-1][W], W = 1 (QMIX/VDN) or N (IQL).  g_out same shape =
 * 2 * td * mask * mask (NOT divided by sum(mask); the update kernel applies 1/sum(mask)).
 * stats[0..4] accumulate (zero them first with pmb_stats_reset). */
int pmb_td_loss(const pmb_dims* d, const pmb_batch* b, const float* q_tot, const float* t_tot, float gamma,
                float* g_out, double* stats, pmb_stream stream);
int pmb_stats_reset(double* stats, pmb_stream stream);

/* ---- K4b: mixer backward -------------------------------------------------------------- */
/* QMIX: raw (in) is overwritten by d_raw; writes d_agent_qs [B][T-1][N] and ACCUMULATES
 * nothing: flat_grad_mixer is overwritten.  scratch: pmb_mixer_bwd_workspace_bytes().
 * VDN: d_agent_qs[m][n] = g[m]. */
int64_t pmb_mixer_bwd_workspace_bytes(const pmb_dims* d);
int pmb_mixer_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_mixer, const float* agent_qs,
                  float* raw, const float* g, float* d_agent_qs, float* flat_grad_mixer,
                  void* scratch, int64_t scratch_bytes, pmb_stream stream);

/* ---- K5: agent backward (BPTT through q_learner.py:47-55) ------------------------------ */
/* d_chosen [B][T-1][N].  gates (in) is overwritten by the gate pre-activation gradients.
 * x_on: fc1 outputs [T][R][H]; dpre1: scratch [T][R][H].  flat_grad_agent is overwritten. */
int64_t pmb_agent_bwd_workspace_bytes(const pmb_dims* d);
int pmb_agent_unroll_bwd(const pmb_dims* d, const pmb_batch* b, const float* flat_agent, const float* x_on,
                         const float* h_stash, float* gates, const float* d_chosen, float* dpre1,
                         float* flat_grad_agent, void* scratch, int64_t scratch_bytes, pmb_stream stream);

/* ---- K5b: backward of ONE agent step, for autograd through RNNAgent / BasicMAC (a user's learner calling
 * loss.backward(); rnn_agent.py:27-36, basic_controller.py:40-49,100-135) ------------------------------------------------
 * The step is pmb_agent_fc1_fwd (batch at time t) or pmb_agent_fc1_dense_fwd (inputs [rows][O], d->O = D_in and both
 * one-hot flags 0), then pmb_agent_gru_unroll_fwd with nt = 1, which saved x [R][H] (fc1 output), h_stash [2][R][H]
 * (h_prev | h) and gates [R][4H].  fp32 kernels on every precision tier (pmb_dims.precision is ignored).
 * dq [R][A] = dL/dq and dh [R][H] = dL/dh may be NULL (no gradient reached them).  Writes dh_prev [R][H] = dL/dh_prev
 * (may be NULL) and OVERWRITES flat_grad_agent, an n_agent-float block in the flat agent layout, with the step's eight
 * parameter gradients: fc1.weight over the whole D_in (obs, last-action and agent-id columns), every other tensor
 * dense.  Pass exactly one of b (with t the batch time the forward read) and inputs.  2 launches (3 when the rows are
 * split into slices), no float atomics: identical calls give identical bits.  scratch >=
 * pmb_agent_step_bwd_workspace_bytes(d, rows). */
int64_t pmb_agent_step_bwd_workspace_bytes(const pmb_dims* d, int64_t rows);
int pmb_agent_step_bwd(const pmb_dims* d, const pmb_batch* b, int32_t t, const float* inputs, int64_t rows,
                       const float* flat_agent, const float* x, const float* h_stash, const float* gates, const float* dq,
                       const float* dh, float* dh_prev, float* flat_grad_agent, void* scratch, int64_t scratch_bytes,
                       pmb_stream stream);

/* ---- K6: grad-norm clip + RMSprop + optional hard target sync (q_learner.py:102-107) --- */
/* g is the un-normalised gradient; stats[PMB_S_MASK_SUM] supplies the 1/sum(mask) factor.
 * clip_grad_norm_: coef = min(1, clip / (norm + 1e-6)); RMSprop: v = a v + (1-a) g^2,
 * p -= lr g / (sqrt(v) + eps).  flat_target may be NULL.  scratch: 4096 floats. */
int pmb_clip_rmsprop_update(int64_t n, float* flat_p, float* flat_g, float* flat_sq, float* flat_target,
                            int32_t do_target_sync, double* stats, float lr, float alpha, float eps,
                            float grad_norm_clip, float* scratch, pmb_stream stream);

/* ---- K8: data-parallel exchange (SURVEY.md section 8e; no counterpart in the reference, which is single-process) ----
 * Episodes shard over ranks; every rank runs pmb_qlearner_train_step with skip_update = 1, then
 *   pmb_dp_pack(n, flat_g, stats)    : appends the five loss sums as (hi, lo) float pairs behind the n gradients (hi + lo
 *                                      = the double to 2^-48; mask_sum, a count, split at a multiple of 2^12 so that fp32
 *                                      sums of up to 8 ranks keep it exact below 2^36) and zeroes the other 6 tail floats
 *   ONE all-reduce(sum, fp32) over flat_g[0 .. n + PMB_DP_TAIL_FLOATS)   (NCCL, issued by the host plumbing)
 *   pmb_dp_unpack(n, flat_g, stats)  : restores the (now global) sums
 *   pmb_clip_rmsprop_update(...)     : identical update on every rank (replicated parameters / optimizer state)
 * flat_g must therefore hold n + PMB_DP_TAIL_FLOATS floats. */
#define PMB_DP_TAIL_FLOATS 16
int pmb_dp_pack(int64_t n, float* flat_g, const double* stats, pmb_stream stream);
int pmb_dp_unpack(int64_t n, const float* flat_g, double* stats, pmb_stream stream);

/* Fused exchange + update over NVLink peer memory (csrc/dp_peer.cu): ONE kernel per rank replaces pack -> all-reduce ->
 * unpack -> pmb_clip_rmsprop_update.  Every rank keeps its flat gradient in an exchange buffer of
 * pmb_dp_exchange_floats(n) floats ([n grads | 16 loss-sum floats | flags], zero-initialised once) that the other ranks of
 * the node map with CUDA IPC: pmb_ipc_export on the owner gives a 64-byte handle + byte offset (the pointer must come from
 * cudaMalloc, e.g. torch's caching allocator without expandable segments), the host plumbing exchanges them (any
 * all-gather), pmb_ipc_open maps a peer's buffer.  pmb_dp_fused_allreduce_update(world <= 8, rank, bufs[world] (own
 * buffer at index rank), n, step = 1, 2, 3, ... (consecutive), ...): one-shot all-reduce in rank order (bit-identical sums
 * on every rank), global grad norm, clip, RMSprop and optional hard target sync of the replicated parameters; afterwards the
 * own exchange buffer holds the global normalised / clipped gradient and stats the global sums.  scratch: 4 n + 2048 bytes,
 * zeroed ONCE and kept for the life of the exchange (it holds the grid barrier's counter).  All ranks must call it with the
 * same step id; a peer that does not show up within ~2 s raises the error word (scratch tail) instead of hanging. */
int pmb_ipc_export(const void* dev_ptr, void* handle_out_64_bytes, int64_t* offset_out);
int pmb_ipc_open(const void* handle_64_bytes, int64_t offset, void** ptr_out);
int pmb_ipc_close(void* mapped_ptr, int64_t offset);
int64_t pmb_dp_exchange_floats(int64_t n);
int pmb_dp_fused_allreduce_update(int32_t world, int32_t rank, void* const* bufs, int64_t n, int64_t step, float* flat_p,
                                  float* flat_sq, float* flat_target, int32_t do_target_sync, double* stats, float lr,
                                  float alpha, float eps, float grad_norm_clip, void* scratch, int64_t scratch_bytes,
                                  pmb_stream stream);

/* ---- K7: epsilon-greedy action selection (components/action_selectors.py:44-62) --------- */
/* q [rows_b][N][A] f32, avail [rows_b][N][A] i32.  Draw modes:
 *   u != NULL, expo != NULL : injected draws (u [b][N] uniform, expo [b][N][A] Exp(1)), the
 *                             reference's generator order -> bit-exact with the reference
 *   else                     : in-kernel Philox4x32-10 keyed by (seed, offset)
 * actions_out int64 [b][N]. */
int pmb_epsilon_greedy(int64_t rows, int32_t A, const float* q, const int32_t* avail, float epsilon,
                       const float* u, const float* expo, uint64_t seed, uint64_t offset,
                       int64_t* actions_out, pmb_stream stream);

/* one fused rollout step of BasicMAC.select_actions (basic_controller.py:30-38) for all B
 * envs at time t: fc1 + GRU + fc2 + masking + epsilon-greedy.  hidden [B*N][H] is updated
 * in place (NULL-initialise with zeros at t_ep == 0 yourself); q_out [B][N][A] optional. */
int64_t pmb_select_actions_workspace_bytes(const pmb_dims* d);
int pmb_select_actions_step(const pmb_dims* d, const pmb_batch* b, int32_t t, const float* flat_agent,
                            float* hidden, float epsilon, const float* u, const float* expo,
                            uint64_t seed, uint64_t offset, int64_t* actions_out, float* q_out,
                            void* scratch, int64_t scratch_bytes, pmb_stream stream);

/* ---- bf16 tensor-core GEMM (tcgen05, fp32 accumulate):  c[m][n] = sum_k a[m][k] w[n][k] + bias[n] ----
 * a [m][k], w [n][k], c [m][n] fp32 row major.  The building block of the bf16 tier, exported
 * for unit tests and diagnostics. */
int64_t pmb_gemm_bf16_workspace_bytes(int32_t n, int32_t k);
int pmb_gemm_bf16_tn(int64_t m, int32_t n, int32_t k, const float* a, const float* w, const float* bias, float* c,
                     void* scratch, int64_t scratch_bytes, pmb_stream stream);

/* out[c][k] = sum_m d[m][c] a[m][k] (weight-gradient form, reduction over rows), bias_out[c] = sum_m d[m][c].
 * d [m][ldd], a [m][lda] fp32; out [c][k] fp32. */
int64_t pmb_gemm_bf16_atb_workspace_bytes(int64_t m, int32_t c, int32_t k);
int pmb_gemm_bf16_atb(int64_t m, int32_t c, int32_t k, const float* d, int64_t ldd, const float* a, int64_t lda,
                      float* out, float* bias_out, void* scratch, int64_t scratch_bytes, pmb_stream stream);

/* ---- whole learner step (learners/q_learner.py:37-107) ---------------------------------- */
/* flat_p / flat_g / flat_sq: online params, grads, RMSprop square_avg (n_total floats);
 * flat_target: target params.  workspace >= pmb_learner_workspace_bytes().  stats: 16 doubles. */
int pmb_qlearner_train_step(const pmb_dims* d, const pmb_batch* b, const pmb_hparams* hp,
                            float* flat_p, float* flat_g, float* flat_sq, float* flat_target,
                            void* workspace, int64_t workspace_bytes, double* stats, pmb_stream stream);

/* Per-kernel timing of the calls issued between begin and end (CUDA events recorded on the
 * launch stream between the kernels; bench.py uses it for the roofline of the dominant
 * kernel).  ms_host[i] / names_host[i*names_stride] are HOST buffers. */
int64_t pmb_launch_count(void);      /* kernels launched by this library since it was loaded */
int pmb_profile_begin(void);
int pmb_profile_end(float* ms_host, char* names_host, int32_t names_stride, int32_t max_phases, int32_t* n_out);

/* ---- replay buffer in HBM (SURVEY.md section 8f) ---------------------------------------------------------------
 * pmb_gather_episodes: dst[f][j] = src[f][ep_ids[j]] for every field f, whole episodes (contiguous [T, ...] blocks of
 * bytes_per_episode bytes) - ReplayBuffer.sample / EpisodeBatch.__getitem__(ndarray) (components/episode_buffer.py:
 * 205-217, 291-298) in ONE launch.  `fields` is a HOST array; ep_ids is a device array of n_ids (< 65536) ids in
 * [0, n_src_episodes).
 * pmb_max_t_filled: out[0] = max_b sum_t filled[b, t]  (episode_buffer.py:255-256), device scalar. */
typedef struct pmb_gather_field {
    const void* src;
    void* dst;
    int64_t bytes_per_episode;
} pmb_gather_field;
int pmb_gather_episodes(const pmb_gather_field* fields_host, int32_t n_fields, const int64_t* ep_ids, int64_t n_ids,
                        int64_t n_src_episodes, pmb_stream stream);
int pmb_max_t_filled(const int64_t* filled, int64_t B, int32_t T, int64_t filled_sb, int64_t* out, pmb_stream stream);

/* pmb_gather_episode_steps: the first `steps` timesteps of episodes ep_ids[j] of every field, for a replay buffer in HBM or
 * in pinned host memory (then the GPU reads the sampled episodes over PCIe, nothing is staged on the host).
 * Field f: src is [n_src_episodes][T_src][cell_bytes], either device memory or page-locked host memory mapped into the
 * device's address space (cudaHostAlloc / pmb_host_alloc; the library uses its device alias).  Pageable host memory is
 * PMB_ERR_INVALID.  dst is device memory [n_ids][dst_stride_bytes], 16-byte aligned, dst_stride_bytes a multiple of 16
 * and >= steps * cell_bytes; row j receives steps * cell_bytes bytes, and the bytes of its last 16-byte word beyond them
 * are written as zero (row padding).  At most 8 fields; ep_ids is a device array of n_ids ids (any count).
 * trim != 0: episode j copies only its first F_j = min(steps, l_j + 2) timesteps, l_j = its last t < steps with
 * filled[id][t] != 0 (F_j = 0 when there is none; filled is the buffer's int64 [n_src_episodes][T_src] field, device or
 * mapped host memory, the same F as the padded-step skipping of the learner step), and the rest of its `steps` is
 * written as zeros without reading the source.  trim == 0 copies all `steps` (filled may be NULL).  Ids outside
 * [0, n_src_episodes) leave their row untouched. */
typedef struct pmb_step_field {
    const void* src;
    void* dst;
    int64_t cell_bytes;
    int64_t dst_stride_bytes;
} pmb_step_field;
int pmb_gather_episode_steps(const pmb_step_field* fields_host, int32_t n_fields, const int64_t* ep_ids, int64_t n_ids,
                             int64_t n_src_episodes, int32_t T_src, int32_t steps, const int64_t* filled, int32_t trim,
                             pmb_stream stream);

/* Page-locked host memory mapped into every device's address space (cudaHostAlloc, portable | mapped), for a replay
 * buffer that pmb_gather_episode_steps reads in place.  These two are the only calls of the library that allocate, and
 * only on request.  The memory is not zeroed. */
int pmb_host_alloc(int64_t bytes, void** out);
int pmb_host_free(void* p);

/* pmb_batch_update: EpisodeBatch.update(data, bs, ts, mark_filled) (components/episode_buffer.py:98-154) for a batch that
 * lives in HBM, every field of the call in ONE launch.  Source field f is a dense device array [nb][nt][cell_bytes]; cell
 * (i, j) is written to episode b(i) = b_index[i] (device array, may be NULL: b0 + i * b_step), timestep t0 + j of the
 * destination field (byte strides given).  onehot_dim > 0 fuses the OneHot preprocess (components/transforms.py:12-21,
 * `preprocess = {"actions": ("actions_onehot", [OneHot(n_actions)])}`, run.py:133-135): the source cell holds int64
 * indices [G] and the destination cell is float32 [G][onehot_dim].  filled (may be NULL): filled[b][t] = 1 for every
 * written cell (mark_filled).  `fields` is a HOST array of at most 12 entries; n_rows = episodes in the destination. */
typedef struct pmb_update_field {
    const void* src;
    void* dst;
    int64_t cell_bytes;
    int64_t dst_batch_stride_bytes;
    int64_t dst_time_stride_bytes;         /* 0 for episode-constant fields */
    int32_t onehot_dim;
    int32_t reserved;
} pmb_update_field;
int pmb_batch_update(const pmb_update_field* fields_host, int32_t n_fields, const int64_t* b_index, int64_t b0, int64_t b_step,
                     int64_t nb, int64_t n_rows, int64_t t0, int64_t nt, int64_t* filled, int64_t filled_sb, pmb_stream stream);

/* Strided host -> device copy of `rows` pieces of `row_bytes` (source pitch `src_pitch_bytes`, destination dense):
 * one cudaMemcpy2DAsync.  Replaces the per-timestep `.to(self.args.device)` of a host-resident runner batch
 * (controllers/basic_controller.py:32,105,113), which materialises a contiguous host copy of `batch[k][:, t]` first. */
int pmb_h2d_rows(void* dst_dev, const void* src_host, int64_t rows, int64_t row_bytes, int64_t src_pitch_bytes,
                 pmb_stream stream);

/* ---- COMA learner (SURVEY.md section 8f rank 4; learners/coma_learner.py:32-148, modules/critics/coma.py:22-59,
 * utils/rl_utils.py:4-15) - fp32 (CUDA-core) tier --------------------------------------------------------------------
 * pmb_dims: E = critic hidden width (128 in the reference), mixer ignored, S = state dim (required).
 * Flat critic layout = state_dict order: fc1.weight [E, D] | fc1.bias | fc2.weight [E, E] | fc2.bias | fc3.weight [A, E] |
 * fc3.bias with D = S + O + 2 N A + N (coma.py:52-59).  The critic's one-hot inputs are generated from actions / filled;
 * actions_onehot is never read.
 * pmb_coma_train_step: target critic over all T -> td-lambda targets -> for t = T-2 .. 0 one critic fwd / bwd / clip /
 * RMSprop step (skipped when nothing is unmasked at t) -> agent unroll over T-1 steps -> policy head (masked softmax,
 * epsilon floor, renormalisation) -> COMA loss -> BPTT with the dense d(loss)/d(logits) -> clip / RMSprop of the agent.
 * stats: (T-1) + 1 rows of 16 doubles, zeroed by the call.  Row t < T-1 (critic step t): [mask_sum, td2_sum, tdabs_sum,
 * qtaken_sum, target_sum, grad_norm, loss, clip_coef]; row T-1 (agent): [mask_sum (x N), sum(adv log_pi mask),
 * sum(adv mask), sum(pi_max mask), -, grad_norm, -, clip_coef].  The hard target-critic sync (:92-94) is the host's. */
typedef struct pmb_coma_hparams {
    float gamma, td_lambda, lr, critic_lr, alpha, eps, grad_norm_clip;
    float epsilon;                       /* mac.action_selector.epsilon: the epsilon floor of BasicMAC.forward */
} pmb_coma_hparams;
int64_t pmb_coma_critic_numel(const pmb_dims* d);
int64_t pmb_coma_workspace_bytes(const pmb_dims* d);
int pmb_coma_workspace_views(const pmb_dims* d, void* workspace, float** q_vals, float** targets, float** pi, float** logits);
int pmb_coma_train_step(const pmb_dims* d, const pmb_batch* b, const pmb_coma_hparams* hp, float* agent_p, float* agent_g,
                        float* agent_sq, float* critic_p, float* critic_g, float* critic_sq, const float* target_critic_p,
                        void* workspace, int64_t workspace_bytes, double* stats, pmb_stream stream);
/* COMACritic.forward(batch, t) alone (coma.py:22-27): q_out [B][nt][N][A] for batch timesteps t0 .. t0 + nt - 1;
 * workspace >= pmb_coma_workspace_bytes(d). */
int pmb_coma_critic_fwd(const pmb_dims* d, const pmb_batch* b, const float* critic_p, int32_t t0, int32_t nt, float* q_out,
                        void* workspace, int64_t workspace_bytes, pmb_stream stream);
/* ---- COMACritic.forward as one autograd node, for a user's actor-critic learner calling loss.backward() on the
 * critic's q (coma_learner.py:118-146) ------------------------------------------------------------------------------
 * pmb_coma_critic_step_fwd: pmb_coma_critic_fwd's launches, giving the same q_out bits, with the two hidden activations
 * x1 = relu(fc1(input)) and x2 = relu(fc2(x1)) written to x1_out / x2_out, [B * nt * N][E] each.  Row order: the nt
 * timesteps go in chunks of c = clamp((64 << 20) / (B N D), 1, T) timesteps (the last chunk may be shorter); chunk
 * after chunk, the rows of a chunk of cn timesteps are (b, tt, n), b-major.  With nt <= c that is [B][nt][N].
 * workspace >= pmb_coma_workspace_bytes(d).  Per chunk: 4 launches (input generation, three GEMMs) and one copy.
 * pmb_coma_critic_step_bwd: from dq [B][nt][N][A] = dL/dq (dense fp32) and the x1 / x2 of the forward over the same
 * (d, batch, t0, nt), OVERWRITES critic_g, a pmb_coma_critic_numel(d)-float block in the flat critic layout, with the
 * gradients of all six critic tensors.  fc1.weight gets every column of D: the state columns from dx1 summed over the
 * N agents of an (episode, step), the obs columns dense, the two one-hot action blocks and the agent-id block by index
 * from actions / filled as the forward generates them; the input matrix is not built.  No gradient reaches the batch.
 * fp32 kernels on every precision tier.  2 launches (3 when the rows are split into slices), no float atomics:
 * identical calls give identical bits.  scratch >= pmb_coma_critic_step_bwd_workspace_bytes(d, nt). */
int pmb_coma_critic_step_fwd(const pmb_dims* d, const pmb_batch* b, const float* critic_p, int32_t t0, int32_t nt,
                             float* q_out, float* x1_out, float* x2_out, void* workspace, int64_t workspace_bytes,
                             pmb_stream stream);
int64_t pmb_coma_critic_step_bwd_workspace_bytes(const pmb_dims* d, int32_t nt);
int pmb_coma_critic_step_bwd(const pmb_dims* d, const pmb_batch* b, const float* critic_p, int32_t t0, int32_t nt,
                             const float* dq, const float* x1, const float* x2, float* critic_g, void* scratch,
                             int64_t scratch_bytes, pmb_stream stream);
/* BasicMAC.forward's policy head for agent_output_type == "pi_logits" (controllers/basic_controller.py:51-73,
 * mask_before_softmax): probs [rows][A] from logits / avail [rows][A]; test_mode: plain masked softmax. */
int pmb_policy_head(int64_t rows, int32_t A, float epsilon, int32_t test_mode, const float* logits, const int32_t* avail,
                    float* probs, pmb_stream stream);
/* MultinomialActionSelector.select_action (components/action_selectors.py:19-31): Categorical(masked probs).sample() =
 * arg-max(p / Exp(1)); expo [rows][A] injects the draws (bit-exact with torch's generator order), else an in-kernel
 * counter-based generator keyed by (seed, offset); greedy != 0: arg-max of the masked probabilities (test mode). */
int pmb_multinomial(int64_t rows, int32_t A, const float* probs, const int32_t* avail, const float* expo, int32_t greedy,
                    uint64_t seed, uint64_t offset, int64_t* actions_out, pmb_stream stream);

/* views into the learner workspace, for tests and the Python mirror */
typedef struct pmb_ws_views {
    float *x_on, *x_tg, *h_stash, *gates, *q_on, *q_tg, *chosen, *tmax, *raw_on, *raw_tg,
          *q_tot, *t_tot, *g, *d_chosen, *scratch;
    int64_t scratch_bytes;
    float* obs_img;            /* bf16 tier: obs tile images written by the fc1 GEMM */
    float* state_img;          /* bf16 tier: state tile images shared by both mixers and the hypernet weight gradients */
    float* h_tg;               /* bf16 tier: h tile images of the target net */
    float* relu_mask;          /* bf16 tier: bit mask (x > 0) of the online fc1 output */
    /* padded-step skipping (pmb_dims.reserved bit 1), NULL where the bit is not honoured: written by the step */
    int64_t* ep_order;         /* [B] buffer episode of sorted batch row b (the incoming ep_index composed with the sort) */
    int32_t* tile_steps;       /* [ceil(B N / 128)] forward steps run for each 128-row tile of the sorted rows */
} pmb_ws_views;
int pmb_learner_workspace_views(const pmb_dims* d, void* workspace, int64_t workspace_bytes, pmb_ws_views* out);

#ifdef __cplusplus
}
#endif
#endif /* PYMARL_B200_H */
