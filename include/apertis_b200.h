/*
 * apertis_b200 -- C ABI of the B200-native Apertis SSM + MoE block hot path.
 *
 * The reference (CuzImSlymi/Apertis-LLM) is pure Python/PyTorch and has no FFI of its own: its
 * seam for this path is the nn.Module contract of SelectiveLinearAttention
 * (src/model/core.py:295-401) and AdaptiveExpertSystem (src/model/core.py:403-607).  The entry
 * points below are what a ctypes binding for that seam binds; each one names the reference lines it
 * replaces.  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes, no torch / ATen types.
 *  - every function returns 0 (AB_OK) or an AB_ERR_* code; ab_last_error() gives the text.  Nothing
 *    throws, aborts or allocates device memory: the caller owns every buffer, including workspaces
 *    whose sizes come from the *_plan / *_workspace_bytes queries.
 *  - all pointers are device pointers unless the name starts with h_.  All work is enqueued on the
 *    cudaStream_t passed in (stream-ordered, re-entrant, no hidden global device state).
 *  - `dtype` selects the activation type of the big [tokens, channels] tensors: AB_F32 or AB_BF16.
 *    Parameters and reductions are always fp32.
 *  - strides are in ELEMENTS of the tensor's dtype; "rows" = tokens = B*L, row-major, channels last.
 */
#ifndef APERTIS_B200_H
#define APERTIS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define AB_OK 0
#define AB_ERR_INVALID 1     /* bad argument / unsupported shape */
#define AB_ERR_CUDA 2        /* a CUDA runtime / driver call failed */
#define AB_ERR_UNSUPPORTED 3 /* device is not sm_100 */

#define AB_F32 0
#define AB_BF16 1

#define AB_ACT_GELU 0 /* exact erf GELU (nn.GELU(), core.py:464) */
#define AB_ACT_RELU 1
#define AB_ACT_SILU 2

/* ---- library ------------------------------------------------------------------------------- */
int ab_version(void);
/* 0 iff `device` is a compute-capability 10.x part (B200); the kernels are sm_100a-only. */
int ab_device_check(int device);
/* copies the calling thread's last error text into buf (NUL-terminated); returns its length. */
int ab_last_error(char* buf, size_t n);

/* ---- SSM: causal depthwise conv1d + SiLU  (core.py:368-375) ----------------------------------
 * xa[b,t,c] = silu(bias[c] + sum_j w[c,j] * xp[b,t-(Kc-1)+j,c]), zero left padding.  2 <= Kc <= 8.
 * The backward workspace (ab_causal_conv1d_silu_bwd_workspace_bytes) is sized for Kc = 8, so it serves every Kc.
 * xp rows may be strided (xp_stride elements between tokens); xa is contiguous [B,L,Di]. */
int ab_causal_conv1d_silu_fwd(const void* xp, int64_t xp_stride, const float* w, const float* bias, void* xa,
                              int B, int L, int Di, int Kc, int dtype, cudaStream_t stream);
size_t ab_causal_conv1d_silu_bwd_workspace_bytes(int B, int L, int Di);
/* backward of the above with recompute of the pre-activation: dxp ([B,L,Di] rows, dxp_stride elements apart),
 * dw [Di,Kc] and dbias [Di] (fp32, overwritten).  Deterministic (two-stage reduction in ws). */
int ab_causal_conv1d_silu_bwd(const void* xp, int64_t xp_stride, const void* dxa, const float* w, const float* bias,
                              void* dxp, int64_t dxp_stride, float* dw, float* dbias, void* ws, size_t ws_bytes,
                              int B, int L, int Di, int Kc, int dtype, cudaStream_t stream);

/* ---- SSM: chunked selective scan  (core.py:324-353 scans, :383 softplus, :394-396 skip + gate) --
 * Per channel c = h*16 + n:   delta = softplus(dlog[b,t,h]);  abar = exp(-exp(A_log[c]) * delta);
 *   state_t = abar * state_{t-1} + Bm[b,t,c];   y_ssm = Cm[b,t,c] * state_t;
 *   y = (y_ssm + D[c] * xa[b,t,c]) * silu(z[b,t,c]).
 * This is the true recurrence of core.py:337-353; it equals the training-mode log-cumsum form
 * (core.py:324-335) wherever that form is finite.
 * The sequence is cut into tiles of `tile_rows` tokens x `slab` channels; a tile's incoming state is
 * resolved either in one pass (decoupled look-back over per-tile aggregates published through `ws`)
 * or in two passes (aggregate kernel, combine kernel, apply kernel).
 *
 * ab_selective_scan_plan: tiling the library will use for (L, Di, dtype) and the buffer sizes:
 *   n_chunks = ceil(L / tile_rows);  hstart is fp32 [B, n_chunks, Di];
 *   ws_bytes: workspace for fwd/bwd.  For the single-pass mode the workspace must be zero-filled
 *   once when allocated, must not be shared between streams, and every launch that uses it must
 *   pass a strictly larger `epoch` (1, 2, 3, ...) than the previous launch on that workspace. */
#define AB_SCAN_SINGLE_PASS 0
#define AB_SCAN_TWO_PASS 1
/* AB_SCAN_PIPELINED: persistent CTAs take super-tiles (4 consecutive tiles of a chain) from a ticket; a prepass running 8
 * tiles ahead publishes the aggregates, the main pass streams every tile once with its incoming state resolved.  The
 * forward saves, per batch, the state entering every run of 4 tokens and then delta = softplus(dt) as [L, Hp] rows
 * (hstart is [B, n_chunks, Di] with n_chunks = ceil(L/4) + ceil(L*Hp/Di), Hp = H rounded up to 4); the backward reads both
 * and returns d dlog final as fp32 [B,L,H].  The launch epoch lives in the workspace
 * (zero-filled once, one workspace per stream and per mode; the `epoch` argument is ignored), so replayed CUDA graphs
 * are valid.  No y_ssm / dyssm in this mode.  *mode is in/out: a request the schedule does not cover (too many
 * chains for scanner CTAs, odd widths) comes back as another mode together with that mode's sizes. */
#define AB_SCAN_PIPELINED 2
int ab_selective_scan_plan(int B, int L, int Di, int dtype, int* mode, int* tile_rows, int* slab, int* n_chunks,
                           size_t* ws_bytes);
/* y, y_ssm (optional), xa: contiguous [B,L,Di]; dlog contiguous [B,L,H]; Bm/Cm share bc_stride; z has
 * z_stride.  h0 [B,Di] optional initial state, h_last [B,Di] optional final state, hstart optional
 * (required for the backward): state entering every tile. */
int ab_selective_scan_fwd(const void* xa, const void* dlog, const void* Bm, const void* Cm, int64_t bc_stride,
                          const void* z, int64_t z_stride, const float* A_log, const float* D, const float* h0,
                          void* y, void* y_ssm, float* h_last, float* hstart, void* ws, size_t ws_bytes,
                          uint32_t epoch, int mode, int B, int L, int Di, int H, int dtype, cudaStream_t stream);
/* Backward with in-tile recompute of the states from hstart.  dout = grad of y; dyssm (optional)
 * = grad of y_ssm.  Outputs: dxa, dz contiguous [B,L,Di]; dBm, dCm with dbc_stride;
 * ddlog_parts fp32 [B,L,H*4] (the backward works on 4-channel vectors: 4 partial sums per head, already
 * multiplied by softplus'; the caller adds them; AB_SCAN_PIPELINED: [B,L,H], final); dA_log [Di] and dD [Di] fp32 (overwritten;
 * deterministic two-stage reduction through ws). */
int ab_selective_scan_bwd(const void* xa, const void* dlog, const void* Bm, const void* Cm, int64_t bc_stride,
                          const void* z, int64_t z_stride, const void* dout, const void* dyssm,
                          const float* A_log, const float* D, const float* hstart,
                          void* dxa, void* dBm, void* dCm, int64_t dbc_stride, void* dz, float* ddlog_parts,
                          float* dA_log, float* dD, void* ws, size_t ws_bytes, uint32_t epoch, int mode,
                          int B, int L, int Di, int H, int dtype, cudaStream_t stream);

/* ---- SSM: stacked weight of the fused parameter projection  (core.py:376-383) ------------------------------------
 * p = xa Wp^T is split into (dtf [R] | B | C) and dt = dtf Wdt^T + b; dtf feeds nothing else, so
 * dt = xa (Wdt Wp[0:R])^T + b.  Wcat [(Hp + 2 Di), Di] = [Wdt Wp[0:R] (H rows); 0 (Hp - H rows); Wp[R:R+2Di]] lets ONE
 * GEMM produce [dt (no bias) | pad | B | C] rows in the layout the scan reads.  fwd builds Wcat (out_dtype bf16 | f32)
 * from the fp32 parameters Wp [R+2Di, Di], Wdt [H, R]; bwd maps dWcat (fp32) back to dWp and dWdt (overwritten). */
int ab_dt_compose_fwd(const float* Wp, const float* Wdt, void* Wcat, int H, int Hp, int R, int Di, int out_dtype,
                      cudaStream_t stream);
int ab_dt_compose_bwd(const float* dWcat, const float* Wp, const float* Wdt, float* dWp, float* dWdt, int H, int Hp,
                      int R, int Di, cudaStream_t stream);

/* ---- SSM: selective scan, "rounds" schedule (csrc/ssm_scan_rounds.cu) ------------------------------------------
 * Same arithmetic as above (core.py:324-353, :383, :394-396) for channel c = h*N + n with ssm_d_state N = Di / H in
 * {16, 32, 64} (the older schedules above take N = 16 only), one persistent kernel per direction: warps walk chunks of
 * one 64-channel slab (4, 2 or 1 whole heads) serially (two channels per lane), every chunk is visited twice (aggregate pass, then the streaming
 * pass with the incoming state known), a round's chunk aggregates are prefixed by a two-level scan of whoever arrives
 * last.  Row strides are in elements; every activation may be a column slice of a wider row-major buffer, which is how
 * the fused projection outputs ([xp | z] and [dt | B | C]) are consumed and produced without copies.
 *   dlog [B,L,H] (row stride dlog_stride) holds the dt_proj_head output WITHOUT its bias when dt_bias != NULL
 *   (delta = softplus(dlog + dt_bias[h])), or with it when dt_bias == NULL.
 *   state: fp32 buffer of `state_floats` elements written by the forward and read by the backward
 *   (the scan state entering every group of 8 tokens, then delta of every (token, head)).
 *   ws: workspace of ws_bytes (ab_ssm_scan_plan), ZERO-FILLED ONCE by the caller when it is allocated; every launch
 *   leaves its counters zeroed for the next one, so the same workspace serves any number of launches (of any shape) on
 *   ONE stream and the launch sequence can be captured in a graph.
 * A wait that cannot complete (protocol error, preempted grid) traps: the launch fails with a CUDA error. */
int ab_ssm_scan_plan(int B, int L, int Di, int dtype, int64_t* state_floats, size_t* ws_bytes);
/* tuning knobs (0 = library default): chunk length of the forward / backward (multiple of 8 tokens), resident warps per SM,
 * stages (2 or 3) of a team's shared-memory ring in the forward / backward */
int ab_ssm_scan_tune(int tc_fwd, int tc_bwd, int warps_per_sm, int stages_fwd, int stages_bwd);
int ab_ssm_scan_fwd(const void* xa, int64_t xa_stride, const void* dlog, int64_t dlog_stride, const float* dt_bias,
                    const void* Bm, const void* Cm, int64_t bc_stride, const void* z, int64_t z_stride,
                    const float* A_log, const float* D, const float* h0, void* y, void* y_ssm, float* h_last,
                    float* state, void* ws, size_t ws_bytes, int B, int L, int Di, int H, int dtype,
                    cudaStream_t stream);
/* dout = grad of y (contiguous [B,L,Di]); dyssm (optional) = grad of y_ssm.  Outputs: dxa, dz, dBm / dCm (shared stride)
 * and ddlog (activation dtype, final: already multiplied by softplus'; columns [H, ddlog_cols) are written as zero),
 * ddt_bias [H] (optional), dA_log [Di], dD [Di] fp32, overwritten (fixed-order reductions: bitwise reproducible). */
int ab_ssm_scan_bwd(const void* xa, int64_t xa_stride, const void* Bm, const void* Cm, int64_t bc_stride,
                    const void* z, int64_t z_stride, const void* dout, const void* dyssm, const float* A_log,
                    const float* D, const float* state, void* dxa, int64_t dxa_stride, void* dBm, void* dCm,
                    int64_t dbc_stride, void* dz, int64_t dz_stride, void* ddlog, int64_t ddlog_stride, int ddlog_cols,
                    float* ddt_bias, float* dA_log, float* dD, void* ws, size_t ws_bytes, int B, int L, int Di, int H,
                    int dtype, cudaStream_t stream);

/* ---- MoE: router  (core.py:480-492 LN+Linear+noise+softmax+top-k, :499-505 lb, :524-526 rz, :529) --
 * Per token s: stats (mean, rstd) of x[s,:] (eps inside the sqrt, as nn.LayerNorm);
 *   logits = LN(x)*ln_w+ln_b @ Wr^T + br (+ noise[s,e]*noise_scale[e] when noise != NULL);
 *   gates = softmax(logits); (probs, idx) = top-K descending, ties -> lower expert index;
 *   w = probs / (sum probs + 1e-6); lse = logsumexp(logits).
 * stats_out [S,2] fp32 is reused by every expert's LayerNorm (same row, same eps).
 * aux [2E+1] fp32: sum_s gates[s,e], count of tokens with e in their top-K, sum_s lse^2
 * (deterministic two-stage reduction through ws). */
size_t ab_moe_router_workspace_bytes(int S, int Dm, int E);
/* quant: how the clean logits are formed.  AB_ROUTER_EXACT: fp32 throughout (the reference without autocast).
 * AB_ROUTER_BF16 / AB_ROUTER_FP16: what the reference computes under torch.autocast of that dtype (core.py:482 is an
 * autocast nn.Linear followed by .float()): LayerNorm output, router weight and bias rounded to the dtype, fp32
 * accumulation, the sum rounded once -- so that top-k picks the experts the reference picks in that mode. */
#define AB_ROUTER_EXACT 0
#define AB_ROUTER_BF16 1
#define AB_ROUTER_FP16 2
/* lclean [S,E] (optional unless the backward is needed) = logits before the noise term; logits [S,E]
 * (optional) = the noisy logits that were soft-maxed. */
int ab_moe_router_fwd(const void* x, const float* ln_w, const float* ln_b, float eps, const float* Wr, const float* br,
                      const float* noise, const float* noise_scale, float* lclean, float* logits, float* gates,
                      int32_t* idx, float* probs, float* w, float* lse, float* stats_out, float* aux, void* ws,
                      size_t ws_bytes, int S, int Dm, int E, int K, int dtype, int quant,
                      cudaStream_t stream);
/* selection only, from given logits (the bit-exact test boundary of SURVEY.md section 7 hard part 3) */
int ab_moe_topk_from_logits(const float* logits, float* gates, int32_t* idx, float* probs, float* w, float* lse,
                            int S, int E, int K, cudaStream_t stream);

/* ---- MoE: capacity plan  (core.py:508-511 capacity, :547-590 dispatch rule) ---------------------
 * Slot-major then expert order; an expert keeps at most `cap` rows over all slots; on overflow of a
 * (slot, expert) group the rows with the largest w[:,slot] stay (ties -> lower token id).  `active`
 * [E] int32 (NULL = all) is the whole-expert dropout mask of core.py:514-521.
 * Outputs (all int32): counts[E]; seg_off[E+1] = start row of each expert's segment in the permuted
 * layout, segments padded to multiples of `row_align` (AB_GEMM_ROW_TILE, the GEMM's row tile); row_of[S,K] = permuted row
 * of a kept (token, slot) or -1; tok_of_row[max_rows], slot_of_row[max_rows] (-1 for padding rows);
 * tile_expert[max_rows/row_align] expert of each row tile (-1 beyond the end); n_rows[2] = {padded
 * total rows, kept rows}.  max_rows = ab_moe_max_rows(S,K,E,cap,row_align).  No host synchronisation.
 * fixed_seg > 0 (expert-parallel exchange layout): every expert segment is exactly fixed_seg rows
 * (a multiple of row_align; >= cap when cap < S, otherwise at least the largest count - the kernel traps if a segment
 * would overflow) at offset e*fixed_seg and max_rows must equal E*fixed_seg. */
int64_t ab_moe_max_rows(int S, int K, int E, int cap, int row_align);
size_t ab_moe_plan_workspace_bytes(int S, int K, int E);
int ab_moe_plan(const int32_t* idx, const float* w, const int32_t* active, int cap, int32_t* counts, int32_t* seg_off,
                int32_t* row_of, int32_t* tok_of_row, int32_t* slot_of_row, int32_t* tile_expert, int32_t* n_rows,
                void* ws, size_t ws_bytes, int S, int K, int E, int row_align, int64_t max_rows, int fixed_seg,
                cudaStream_t stream);

/* ---- MoE: permute (+ per-expert LayerNorm) and weighted unpermute  (core.py:593, :436, :605) -----
 * permute_ln: for every row r < padded total: xn[r,:] = bf16|f32( (x[tok,:]-mean)*rstd*ln_w[e,:]+ln_b[e,:] ),
 * zeros for padding rows.  ln_w/ln_b are stacked [E,Dm].  out_dtype selects the GEMM operand type. */
int ab_moe_permute_ln(const void* x, const float* stats, const float* ln_w, const float* ln_b,
                      const int32_t* tok_of_row, const int32_t* tile_expert, const int32_t* n_rows, void* xn,
                      int Dm, int row_align, int64_t max_rows, int dtype, int out_dtype, cudaStream_t stream);
/* unpermute: m[s,:] = sum_k (row_of[s,k] >= 0) * w[s,k] * y[row_of[s,k],:]  in fixed slot order;
 * out = res + dropout_p(m): the caller's output dropout and residual add (core.py:918-919) in the same pass
 * (res NULL: no residual; drop_p 0: no dropout; drop_seed: device uint32[2]). */
int ab_moe_unpermute(const void* y, const int32_t* row_of, const float* w, const float* res, void* out, float drop_p,
                     const uint32_t* drop_seed, int S, int K, int Dm, int y_dtype, int out_dtype, cudaStream_t stream);
/* backward of unpermute: dy[r,:] = w[r]*dout[tok,:] (dy_dtype), dw_row[r] = <dout[tok,:], y[r,:]>; padding rows -> 0 */
int ab_moe_unpermute_bwd(const void* dout, const void* y, const float* w, const int32_t* tok_of_row,
                         const int32_t* slot_of_row, const int32_t* n_rows, void* dy, float* dw_row, float drop_p,
                         const uint32_t* drop_seed, int K, int Dm,
                         int64_t max_rows, int dout_dtype, int y_dtype, int dy_dtype, cudaStream_t stream);
/* backward of permute_ln per row: dxrow[r,:] = LayerNorm-backward(dxn[r,:]) (fp32), and the per-expert
 * affine grads dln_w/dln_b [E,Dm] (deterministic two-stage reduction through ws). */
size_t ab_moe_permute_ln_bwd_workspace_bytes(int Dm, int row_align, int64_t max_rows);
int ab_moe_permute_ln_bwd(const void* dxn, const void* x, const float* stats, const float* ln_w,
                          const int32_t* tok_of_row, const int32_t* tile_expert, const int32_t* n_rows,
                          float* dxrow, float* dln_w, float* dln_b, void* ws, size_t ws_bytes, int Dm, int E,
                          int row_align, int64_t max_rows, int dtype, int dxn_dtype, cudaStream_t stream);
/* per-expert column sums of a permuted [rows, C] matrix (bias gradients): out[E,C] fp32 */
size_t ab_moe_segment_colsum_workspace_bytes(int C, int row_align, int64_t max_rows);
int ab_moe_segment_colsum(const void* a, const int32_t* tile_expert, const int32_t* n_rows, float* out, void* ws,
                          size_t ws_bytes, int C, int E, int row_align, int64_t max_rows, int dtype, cudaStream_t stream);

/* ---- MoE: router backward  (autograd of core.py:480-505, 524-529) ----------------------------
 * Per token: dw[s,k] = dw_row[row_of[s,k]] (0 if dropped) -> d probs -> d gates (+ lb term
 * g_lb*f[e]) -> softmax backward (+ rz term g_rz*2*lse*gates) -> d logits -> router Linear and
 * LayerNorm backward; adds the expert path  sum_k dxrow[row_of[s,k],:]  and writes dx [S,Dm].
 * scal (device, fp32 [2]) = {g_lb, g_rz} = upstream grads times coef*E/S and coef/S.
 * f [E] = count_e / S (the no-grad fraction of core.py:504).  Param grads (fp32, overwritten):
 * dWr [E,Dm], dbr [E], dln_w [Dm], dln_b [Dm], dnoise_scale [E]. */
size_t ab_moe_router_bwd_workspace_bytes(int S, int Dm, int E);
int ab_moe_router_bwd(const void* x, const float* stats, const float* ln_w, const float* ln_b, const float* Wr,
                      const float* br, const float* gates, const int32_t* idx, const float* probs, const float* lse,
                      const float* lclean, const float* noise, const float* f, const float* scal, const float* dw_row,
                      const float* dxrow, const int32_t* row_of, void* dx, float* dWr, float* dbr, float* dln_w,
                      float* dln_b, float* dnoise_scale, void* ws, size_t ws_bytes, int S, int Dm, int E, int K,
                      int dtype, cudaStream_t stream);

/* ---- expert parallelism over peer memory (NVLink 5 / NVSwitch)  (SURVEY.md 8(e); no reference counterpart: the reference
 * is DDP only, pipeline.py:435-466) ------------------------------------------------------------------------------------
 * The four row exchanges of the expert-parallel MoE fused into the kernels that produce the rows: instead of writing them
 * locally and handing them to an all-to-all, the producer stores every row straight into the consuming rank's buffer
 * through peer-mapped pointers, so the transfer overlaps the producing kernel and no exchange kernel exists.
 * Layouts: a SOURCE rank (owner of tokens) keeps the permuted layout [W owners][rows_per_peer] (fixed expert segments,
 * ab_moe_plan fixed_seg); an OWNER rank (owner of experts) works on [W sources][rows_per_peer].  Row (d, j) of a source
 * rank s is row (s, j) of owner d and vice versa; `peer_*` is a HOST array of the W peer-mapped device addresses of the
 * destination buffer on every rank (entry `rank` = the local one).  The caller orders the ranks with its own barriers (the
 * host side uses torch symmetric memory): all producers -> barrier -> consumers.
 *   ab_ep_permute_ln       ab_moe_permute_ln, each normalised row stored into its owner's receive buffer        (dispatch)
 *   ab_ep_grouped_gemm_nt  ab_grouped_gemm_nt, each result row stored into its source rank's buffer            (combine)
 *   ab_ep_unpermute_bwd    ab_moe_unpermute_bwd, each dY row stored into its owner's receive buffer         (dY dispatch)
 *   ab_ep_grouped_gemm_nn  ab_grouped_gemm_nn, each input-gradient row stored into its source rank's buffer (dXn return)
 * The GEMM variants take epi = AB_EPI_NONE | AB_EPI_BIAS | AB_EPI_DACT | AB_EPI_ADD (one output) and no dropout. */
int ab_ep_permute_ln(const void* x, const float* stats, const float* ln_w, const float* ln_b, const int32_t* tok_of_row,
                     const int32_t* tile_expert, const int32_t* n_rows, const uint64_t* peer_xn, int W, int rank,
                     int64_t rows_per_peer, int Dm, int row_align, int64_t max_rows, int dtype, int out_dtype, cudaStream_t stream);
int ab_ep_unpermute_bwd(const void* dout, const void* y, const float* w, const int32_t* tok_of_row, const int32_t* slot_of_row,
                        const int32_t* n_rows, const uint64_t* peer_dy, int W, int rank, int64_t rows_per_peer, float* dw_row,
                        float drop_p, const uint32_t* drop_seed, int K, int Dm, int64_t max_rows, int dout_dtype, int y_dtype,
                        int dy_dtype, cudaStream_t stream);
int ab_ep_grouped_gemm_nt(const void* A, const void* W, const float* bias, const void* aux, const uint64_t* peer_c, int peer_w,
                          int rank, int64_t rows_per_peer, const int32_t* tile_expert, const int32_t* n_rows, int64_t max_rows,
                          int N, int K, int E, int epi, int act, int c_dtype, cudaStream_t stream);
int ab_ep_grouped_gemm_nn(const void* A, const void* W, const float* bias, const void* aux, const uint64_t* peer_c, int peer_w,
                          int rank, int64_t rows_per_peer, const int32_t* tile_expert, const int32_t* n_rows, int64_t max_rows,
                          int N, int K, int E, int epi, int act, int c_dtype, cudaStream_t stream);

/* ---- MoE: grouped expert GEMM on tcgen05 / TMEM, operands staged by TMA  (core.py:596 = :437-440) --
 * bf16 operands, fp32 accumulation in tensor memory.  The kernel runs on CTA pairs (tcgen05 cta_group::2): a row tile is
 * AB_GEMM_ROW_TILE = 256 permuted rows (128 per CTA) and belongs to one expert (tile_expert[max_rows / 256]); tiles
 * past n_rows[0] are skipped on the device (no host sync).  max_rows must be a multiple of AB_GEMM_ROW_TILE.
 *
 * ab_grouped_gemm_nt :  C[r, n] = epi( sum_k A[r,k] * W[e, n, k] )         (forward: W = nn.Linear weight)
 *    A [max_rows, K] bf16 row-major, W stacked [E, N, K] bf16.
 * ab_grouped_gemm_nn :  C[r, n] = epi( sum_k A[r,k] * W[e, k, n] )         (dgrad: same W tensor, no transpose copy)
 *    W stacked [E, K, N] bf16.
 * epilogue `epi`:
 *    AB_EPI_BIAS        C = acc + bias[e,n]                                  -> c (c_dtype)
 *    AB_EPI_BIAS_ACT    pre = acc + bias[e,n]; c2 = pre; c = act(pre)        -> c, c2 (both bf16|f32 as c_dtype)
 *    AB_EPI_DACT        C = acc * act'(aux[r,n])   (aux = saved pre-activation, c_dtype)
 *    AB_EPI_NONE        C = acc
 * ab_grouped_gemm_tn :  Cw[e, m, n] = sum_{r in expert e} A[r,m] * Bm[r,n]   (wgrad; fp32 out [E,M,N])
 */
#define AB_GEMM_ROW_TILE 256
int ab_gemm_row_tile(void);   /* = AB_GEMM_ROW_TILE: the `row_align` to plan the permuted layout with */
#define AB_EPI_NONE 0
#define AB_EPI_BIAS 1
#define AB_EPI_BIAS_ACT 2
#define AB_EPI_DACT 3
#define AB_EPI_ADD 4    /* C = acc + aux[r,n]  (aux has C's shape and dtype; dense GEMMs) */
/* drop_p > 0 fuses the expert-internal nn.Dropout (core.py:439) into the epilogue: AB_EPI_BIAS_ACT scales
 * act(pre) by mask/(1-p), AB_EPI_DACT applies the same mask to the incoming gradient.  The keep-mask is a
 * counter-based hash of (row, column, drop_seed[0..1]) (drop_seed: device uint32[2]), regenerated, not stored. */
int ab_grouped_gemm_nt(const void* A, const void* W, const float* bias, const void* aux, void* c, void* c2,
                       const int32_t* tile_expert, const int32_t* n_rows, int64_t max_rows, int N, int K, int E,
                       int epi, int act, int c_dtype, float drop_p, const uint32_t* drop_seed, cudaStream_t stream);
int ab_grouped_gemm_nn(const void* A, const void* W, const float* bias, const void* aux, void* c, void* c2,
                       const int32_t* tile_expert, const int32_t* n_rows, int64_t max_rows, int N, int K, int E,
                       int epi, int act, int c_dtype, float drop_p, const uint32_t* drop_seed, cudaStream_t stream);
/* nsrc > 1 (expert-parallel receive layout): expert e's rows are the nsrc blocks
 * [s*src_stride + seg_off[e], s*src_stride + seg_off[e+1]), s = 0..nsrc-1.  With few local experts the output has fewer
 * tiles than the chip has CTA pairs: given a workspace of ab_grouped_gemm_tn_workspace_bytes (may be 0) the contraction is
 * cut over the source blocks and the partial products are summed in a fixed order.  ws may be NULL (never split). */
size_t ab_grouped_gemm_tn_workspace_bytes(int M, int N, int E, int nsrc);
int ab_grouped_gemm_tn(const void* A, const void* Bm, float* Cw, const int32_t* seg_off, int64_t max_rows, int M,
                       int N, int E, int nsrc, int64_t src_stride, void* ws, size_t ws_bytes, cudaStream_t stream);

/* ---- dense GEMMs on the same tcgen05 kernel: the SSM layer's projections (core.py:366-367 in_proj_x | in_proj_z,
 * :376-383 x_param_proj with dt_proj_head folded in, :397 out_proj) and their autograd.  Row-major bf16 operands,
 * fp32 accumulation; S need not be a multiple of the row tile.  epi = AB_EPI_NONE | AB_EPI_BIAS (bias [N] fp32) |
 * AB_EPI_ADD (aux [S,N] of c_dtype is added: a second gradient contribution accumulated in the epilogue).
 *   ab_dense_gemm_nt:  C[S,N] = epi(A[S,K] * W[N,K]^T)        (forward of nn.Linear)
 *   ab_dense_gemm_nn:  C[S,N] = epi(A[S,K] * W[K,N])          (input gradient: same weight tensor, no transpose copy)
 *   ab_dense_gemm_tn:  Cw[M,N] = A[S,M]^T * Bm[S,N]  (fp32)   (weight gradient; the contraction over S is cut into slices
 *                      whose partial products go to ws (ab_dense_gemm_tn_workspace_bytes, may be 0) and are summed in a
 *                      fixed order) */
int ab_dense_gemm_nt(const void* A, const void* W, const float* bias, const void* aux, void* C, int64_t S, int N, int K,
                     int epi, int c_dtype, cudaStream_t stream);
int ab_dense_gemm_nn(const void* A, const void* W, const float* bias, const void* aux, void* C, int64_t S, int N, int K,
                     int epi, int c_dtype, cudaStream_t stream);
size_t ab_dense_gemm_tn_workspace_bytes(int64_t S, int M, int N);
int ab_dense_gemm_tn(const void* A, const void* Bm, float* Cw, void* ws, size_t ws_bytes, int64_t S, int M, int N,
                     cudaStream_t stream);

/* ---- language-model head: shifted cross-entropy  (core.py:1412-1460; SURVEY.md 8(f) row 4) -----------------------------
 * loss = mean over the counted positions of CE(logits[b, l, :], labels[b, l+1]), l < L-1, labels == ignore_index not counted
 * (nn.CrossEntropyLoss(ignore_index=-100) on logits[..., :-1, :] / labels[..., 1:]).  The logits [B, L, V] come from
 * ab_dense_gemm_nt of the hidden states with the (tied) embedding matrix, in c_dtype; V*sizeof must be a multiple of 16.
 *   fwd: lse[B*(L-1)] = log-sum-exp per row, row_loss / row_valid [B*(L-1)], sums[2] = {sum of row losses, counted rows}
 *        (fixed-order reduction); the loss is sums[0] / sums[1].  One read of the logits.
 *   bwd: dlogits[B, L, V] = (softmax - onehot) * scale[0] on the counted positions, 0 elsewhere (scale: device float =
 *        upstream gradient / sums[1]); feeds ab_dense_gemm_nn / _tn for the hidden-state and embedding gradients.
 * An out-of-range label traps (torch raises a device assert). */
int ab_shifted_ce_fwd(const void* logits, const int64_t* labels, float* lse, float* row_loss, float* row_valid, float* sums,
                      int B, int L, int V, int64_t ignore_index, int dtype, cudaStream_t stream);
int ab_shifted_ce_bwd(const void* logits, const int64_t* labels, const float* lse, const float* scale, void* dlogits, int B,
                      int L, int V, int64_t ignore_index, int dtype, cudaStream_t stream);

/* ---- block wrappers: pre-norm LayerNorm  (core.py:694-695, 887-888; SURVEY.md 8(f) row 1) ------------
 * y = (x - mean) * rstd * w + b per row, eps inside the sqrt; stats [S,2] = (mean, rstd) saved for the backward.
 * backward: dx = LayerNorm-backward(dy) (+ dres when given: the residual branch's gradient, fused add),
 * dw/db [Dm] fp32 (overwritten, deterministic two-stage reduction through ws). */
int ab_layernorm_fwd(const void* x, const float* w, const float* b, float eps, void* y, float* stats, int S, int Dm,
                     int x_dtype, int y_dtype, cudaStream_t stream);
size_t ab_layernorm_bwd_workspace_bytes(int S, int Dm);
int ab_layernorm_bwd(const void* dy, const void* x, const float* stats, const float* w, const void* dres, void* dx,
                     float* dw, float* db, void* ws, size_t ws_bytes, int S, int Dm, int x_dtype, int dy_dtype,
                     cudaStream_t stream);

/* output Dropout + residual add of the wrappers (core.py:836-837, 918-919): out = dropout_p(sub) + res.
 * res may be NULL (then it is the dropout alone: used for the backward, dsub = dropout-mask(dout)).  The mask is
 * a counter-based hash of (element index, seed[0..1]); seed is a device uint32[2], ignored when p == 0. */
int ab_dropout_add(const void* sub, const void* res, void* out, float p, const uint32_t* seed, int64_t n, int sub_dtype,
                   int out_dtype, cudaStream_t stream);

/* ---- helpers ----------------------------------------------------------------------------------- */
/* fp32 -> bf16 cast of n elements (weight shadows for the tensor-core path) */
int ab_cast_f32_to_bf16(const float* src, void* dst, int64_t n, cudaStream_t stream);
/* splits fp32 into bf16 hi + bf16 lo (x ~= hi + lo) and lays them out for the 3-product fp32-accurate
 * GEMM mode: dst [rows, 3*cols] bf16 = which==0 ? [hi | hi | lo] : [hi | lo | hi] per row. */
int ab_split_f32_to_bf16x3(const float* src, void* dst, int64_t rows, int64_t cols, int which, cudaStream_t stream);
/* row-stacked variant for operands whose contraction index is the row: group g = src rows
 * [seg_off[g], seg_off[g+1]) (or uniform groups of rows_per_group when seg_off == NULL) becomes dst rows
 * [3*seg_off[g], 3*seg_off[g+1]) = which==0 ? [hi; hi; lo] : [hi; lo; hi]. */
int ab_split_f32_to_bf16x3_rows(const float* src, void* dst, const int32_t* seg_off, int G, int64_t rows_per_group,
                                int64_t cols, int which, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* APERTIS_B200_H */
