// Parameter blocks and host launchers of the tcgen05 GRU kernels (gru_tc.cu).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/pymarl_b200.h"

namespace pmb {
namespace tc {

struct GruFwdParams {
    const __nv_bfloat16* w_ih_img;   // 192 rows x 128 B
    const __nv_bfloat16* w_hh_img;   // 192 rows x 128 B
    const __nv_bfloat16* w2_img;     // 64 rows x 128 B (rows >= A are zero)
    const float *b_ih, *b_hh, *b2;
    const uint8_t* x_ti;             // [nt][n_tiles][16 KB]
    const float* h0;                 // fp32 [R][64] or null (may alias h_last)
    uint8_t* h_ti;                   // [(nt+1)][n_tiles][16 KB] or null
    uint8_t* g_ti;                   // [nt][n_tiles][4][16 KB] (r, z, n, hn) or null
    float* q;                        // fp32 [nt][R][A]
    float* h_last;                   // fp32 [R][64] or null
    int64_t R;
    int nt, A, n_tiles;
    // optional fused epsilon-greedy selection on the q of the LAST step (components/action_selectors.py:44-62; same
    // arithmetic and Philox indexing as epsilon_greedy_kernel in select.cu): actions_out == nullptr disables it
    const void* avail;               // already offset to the step: row (b, n) at cell b*avail_sb + n*A of avail
    int64_t avail_sb;
    int avail_u8;                    // cells are u8 (else i32)
    int N;
    float epsilon;
    const float* u;                  // injected draws [R] / [R][A], or null -> Philox(seed, offset)
    const float* expo;
    uint64_t seed, offset;
    int64_t* actions_out;            // [R]
};


}  // namespace tc

int tc_gru_fwd(const tc::GruFwdParams& P, cudaStream_t s);
int64_t tc_agent_dw_scratch_bytes();
int tc_agent_dw(const pmb_dims* d, const pmb_batch* b, const uint8_t* dpre1_ti, const uint8_t* h_ti, const uint8_t* obs_ti,
                const float* d_chosen, int n_tiles, float* fc1_w, float* fc1_b, float* fc2_w, float* fc2_b, void* scratch,
                int64_t scratch_bytes, cudaStream_t s, const int32_t* live_items = nullptr, const int32_t* n_live = nullptr);
int tc_gru_fwd2(const __nv_bfloat16* w_ih_img, const __nv_bfloat16* w_hh_img, const float* b_ih, const float* b_hh,
                const uint8_t* x_ti, uint8_t* h_ti, uint8_t* g_ti, int64_t R, int nt, int n_tiles, cudaStream_t s, int tiles_per_cta = 2,
                const int32_t* tile_steps = nullptr);
int tc_q_select(const pmb_dims* d, const pmb_batch* b, const __nv_bfloat16* w2_on_img, const __nv_bfloat16* w2_tg_img,
                const float* b2_on, const float* b2_tg, const uint8_t* h_on_ti, const uint8_t* h_tg_ti, int n_tiles,
                float* chosen, float* tmax, float* q_on_out, float* q_tg_out, cudaStream_t s,
                const int32_t* live_items = nullptr, const int32_t* n_live = nullptr, const int32_t* tile_steps = nullptr);
int64_t tc_gru_bwd2_partial_bytes(int n_tiles);
int tc_gru_bwd2(const __nv_bfloat16* w_ih_img, const __nv_bfloat16* w_hh_img, const __nv_bfloat16* w2_img,
                const uint8_t* x_ti, const uint8_t* h_ti, const uint8_t* g_ti, uint8_t* dpre1_ti, const uint32_t* relu_mask,
                const float* d_chosen, const int64_t* actions, int64_t actions_sb, const int64_t* ep_index, int64_t R, int T,
                int N, int A, int n_tiles, float* partial, cudaStream_t s, const int32_t* tile_steps = nullptr);
int tc_gru_bwd2_reduce(const float* partial, int n_tiles, float* w_ih, float* w_hh, float* b_ih, float* b_hh, cudaStream_t s);
int tc_ti_zero_pad(uint8_t* buf, int n_t, int n_tiles, int64_t R, cudaStream_t s);

// Padded-step skipping (pmb_dims.reserved bit 1, skip_schedule.cu): the device-side schedule of one learner step.
// Episodes are sorted by the forward steps they need, longest first, so that the rows still live at step t are a prefix
// of the time-major row range: the live (t, tile) items are tiles [0, live_tiles(t)) of every t.
struct SkipSchedule {
    int64_t* ep_order;      // [B]        buffer episode of sorted batch row b (composed with the incoming ep_index)
    int32_t* tile_steps;    // [n_tiles]  forward steps of a tile = those of its first episode (0: only empty episodes)
    int32_t* items;         // [T * n_tiles] live items t * n_tiles + tile, t-major, tiles ascending; then -1
    int32_t* n_items;       // [1]
    int32_t* steps;         // [B]        forward steps F_b of batch row b (incoming order)
    int32_t* steps_sorted;  // [B]
};
int64_t skip_schedule_bytes(int B, int T, int n_tiles);
SkipSchedule skip_schedule_views(void* base, int B, int T, int n_tiles);
int tc_skip_schedule(const pmb_dims* d, const pmb_batch* b, const SkipSchedule& S, int n_tiles, cudaStream_t s);

}  // namespace pmb
