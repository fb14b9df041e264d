/*
 * rorl_b200 -- C ABI of the B200-native kernels behind the recurrent off-policy update hot path
 * of FanmingL/Recurrent-Offpolicy-RL (SURVEY.md section 8b).
 *
 * The reference has no C ABI of its own: at this boundary it binds third-party pybind modules
 * (selective_scan_cuda, causal_conv1d_cuda, flash_attn_2_cuda), in-tree Triton kernels and ATen.
 * Every entry point below names the reference interface it replaces (file:line under
 * /root/reference).  INTEGRATION.md shows the ctypes stub a maintainer of the reference would add.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless stated otherwise;
 *   - fp32, contiguous innermost dimension, 16-byte aligned bases; "ld_x" = row stride in floats;
 *   - the caller owns every buffer (inputs, outputs, partial/workspace buffers) and keeps it alive
 *     until `stream` has passed the call; the library allocates nothing, never synchronises and
 *     never touches the host: every call is CUDA-graph capturable;
 *   - return 0 on success; negative = argument error (-1 shape, -2 alignment, -3 null/inconsistent
 *     argument, -4 workspace too small); 1000 + cudaError_t = launch error;
 *   - re-entrant; all work is enqueued on `stream`;
 *   - sm_100a only. There is no CPU implementation behind this ABI.
 */
#ifndef RORL_B200_H
#define RORL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

/* ABI version, bumped on any signature change. */
int rorl_abi_version(void);

/* ------------------------------------------------------------------------------------------------
 * GILR real gated linear recurrence: h_t = f_t h_{t-1} + (1 - f_t) v_t, h_{-1} = 0.  [B, L, C].
 * Replaces TritonSequentialScan.forward/backward = real_scan_tie_input_gate(v, f)
 * (ref: offpolicy_rnn/models/gilr/scan_triton/real_rnn_tie_input_gate.py:170-214,264; kernels :9-33,
 * :67-116).  Unlike the reference, v/f are NOT overwritten by the backward; C % 4 == 0 (the
 * reference requires C % 256 == 0).
 * The fused variants take the raw in_proj outputs and the reset flag start[B, L] (may be NULL) and
 * apply v = tanh(u_v), f = sigmoid(u_f) * (1 - start) in-kernel (ref: gilr/gilr.py:52-56).
 * ---------------------------------------------------------------------------------------------- */
int rorl_gilr_scan_fwd(const float* v, const float* f, float* h, int64_t B, int64_t L, int64_t C,
                       cudaStream_t stream);
int rorl_gilr_scan_bwd(const float* dh, const float* v, const float* f, const float* h, float* dv, float* df,
                       int64_t B, int64_t L, int64_t C, cudaStream_t stream);
int rorl_gilr_fused_fwd(const float* u_v, const float* u_f, const float* start, float* h, int64_t B, int64_t L,
                        int64_t C, cudaStream_t stream);
int rorl_gilr_fused_bwd(const float* dh, const float* u_v, const float* u_f, const float* h, const float* start,
                        float* du_v, float* du_f, int64_t B, int64_t L, int64_t C, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * LRU complex linear recurrence: h_t = f_t h_{t-1} + v_t (complex, per-step decay), h_{-1} = h0
 * ([B, C], may be NULL = 0).  Replaces TritonSequentialScan_Complex = complex_scan(v_re, v_im,
 * f_re, f_im, h0_re, h0_im, grad_detach) (ref: offpolicy_rnn/models/lru/scan_triton/
 * complex_rnn.py:174-244; kernels :43-87, :90-170).  grad_detach is [B, L] (may be NULL = 0).
 * No gradient is produced for h0 (ref :242).
 * ---------------------------------------------------------------------------------------------- */
int rorl_lru_scan_fwd(const float* v_re, const float* v_im, const float* f_re, const float* f_im,
                      const float* h0_re, const float* h0_im, float* h_re, float* h_im, int64_t B, int64_t L,
                      int64_t C, cudaStream_t stream);
int rorl_lru_scan_bwd(const float* g_re, const float* g_im, const float* f_re, const float* f_im,
                      const float* h_re, const float* h_im, const float* h0_re, const float* h0_im,
                      const float* grad_detach, float* dv_re, float* dv_im, float* df_re, float* df_im,
                      int64_t B, int64_t L, int64_t C, cudaStream_t stream);

/* LRU scan with the layer's own parameterisation fused in (ref: offpolicy_rnn/models/lru/lru.py:95-117 materialises
 * gamma * u and lambda * (1 - start) as four [B, L, C] tensors before calling complex_scan):
 *   h_t = lambda (1 - start_t) h_{t-1} + gamma u_t.   u_re, u_im: [B, L, C]; lam_re, lam_im, gamma: [C];
 * start: [B, L] or NULL.  16 B per element forward, 24 B backward (SURVEY.md 8d).  Backward: du [B, L, C] and the
 * per-row partial sums dlam_re / dlam_im / dgamma [B, C] the caller reduces over axis 0.  No grad_detach here. */
int rorl_lru_fused_fwd(const float* u_re, const float* u_im, const float* lam_re, const float* lam_im, const float* gamma,
                       const float* start, const float* h0_re, const float* h0_im, float* h_re, float* h_im, int64_t B,
                       int64_t L, int64_t C, cudaStream_t stream);
int rorl_lru_fused_bwd(const float* g_re, const float* g_im, const float* lam_re, const float* lam_im, const float* gamma,
                       const float* start, const float* h_re, const float* h_im, const float* h0_re, const float* h0_im,
                       float* du_re, float* du_im, float* dlam_re_part, float* dlam_im_part, float* dgamma_part,
                       int64_t B, int64_t L, int64_t C, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Mamba selective scan with reset flag.  Replaces selective_scan_cuda.fwd / .bwd as called by
 * SelectiveScanFn (ref: offpolicy_rnn/models/smamba/mamba_ssm/ops/selective_scan_interface_new.py:
 * 19-84; semantics = selective_scan_ref :96-166) and the s6 Triton pair fwd_recurrence /
 * bwd_recurrence (ref: offpolicy_rnn/models/s6/selective_scan/triton_scan.py:19-72,75-182).
 *
 * Token-major layout: u, delta, z, y: [B, L, D] with row strides ld_*; Bm, Cm: [B, L, N] with row
 * strides ld_B, ld_C; A: [D, N] (-exp(A_log), or A_log itself with flag bit 1); Dskip, delta_bias: [D] or NULL; z may be NULL;
 * start: [B, L] (1 = reset the state before this step) or NULL.  N in {16, 32, 64}; D % 4 == 0.
 * h0 (may be NULL = 0): [B, D, N] state carried into the call (the s6 layer's `initial_state`,
 * ref: offpolicy_rnn/models/s6/selective_scan/cpu_scan.py:52-53); a constant: no gradient is produced for it.
 * ckpt (may be NULL when no backward follows): [B, L / rorl_selscan_ckpt_every(), D, N] state
 * checkpoints the backward consumes; last_state (may be NULL): [B, D, N].
 *
 * Backward outputs: du, ddelta (w.r.t. the raw delta), dz: [B, L, D]; plus partial sums the caller
 * reduces (deterministic; no atomics):
 *   dBC_part  [ceil(D / rorl_selscan_dtile(N)), B, L, 2N]  sum over axis 0 -> dB = [..., :N], dC = [..., N:]
 *   dA_part   [B, D, N]   sum over axis 0 -> dA
 *   dD_part   [B, D], dbias_part [B, D]   sum over axis 0 -> dD, d(delta_bias)
 * `delta_softplus` is a flag word: bit 0 = delta = softplus(delta_raw + delta_bias) (else delta_raw + delta_bias);
 * bit 1 = `A` points at the PARAMETER A_log and the kernels form A = -exp(A_log) themselves (ref: smamba/mamba.py:215),
 * in which case dA_part holds partials of d A_log (= dA * A), so that no exp / neg / mul launches surround the scan.
 * ---------------------------------------------------------------------------------------------- */
int rorl_selscan_dtile(int64_t N);
int rorl_selscan_ckpt_every(void);
int rorl_selscan_fwd(const float* u, const float* delta, const float* A, const float* Bm, const float* Cm,
                     const float* Dskip, const float* z, const float* delta_bias, const float* start, const float* h0,
                     float* y, float* ckpt, float* last_state, int64_t B, int64_t L, int64_t D, int64_t N, int64_t ld_u,
                     int64_t ld_delta, int64_t ld_z, int64_t ld_B, int64_t ld_C, int64_t ld_y, int delta_softplus,
                     cudaStream_t stream);
int rorl_selscan_bwd(const float* u, const float* delta, const float* A, const float* Bm, const float* Cm,
                     const float* Dskip, const float* z, const float* delta_bias, const float* start, const float* h0,
                     const float* dy, const float* ckpt, float* du, float* ddelta, float* dz, float* dBC_part,
                     float* dA_part, float* dD_part, float* dbias_part, int64_t B, int64_t L, int64_t D, int64_t N,
                     int64_t ld_u, int64_t ld_delta, int64_t ld_z, int64_t ld_B, int64_t ld_C, int64_t ld_dy,
                     int64_t ld_du, int64_t ld_ddelta, int64_t ld_dz, int delta_softplus, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Depthwise causal conv1d over time + SiLU, with the valid-step mask applied to the conv INPUT.
 * Replaces `x = mask * x; x = act(conv1d(x)[..., :L])` on the d_conv > 4 path
 * (ref: offpolicy_rnn/models/smamba/mamba.py:207-212; nn.Conv1d construction :75-83).
 * x, y: [B, L, D] token-major with row strides; w: [D, K] (= conv1d.weight[:, 0, :]); bias: [D] or
 * NULL; mask: [B, L] or NULL.  K in {2, 3, 4, 8, 16}.  Backward: dx [B, L, D]; dw_part [P, D, K],
 * dbias_part [P, D] with P = B * rorl_conv1d_nseg(L) are per-segment partial sums the caller reduces
 * over axis 0.
 * ---------------------------------------------------------------------------------------------- */
int rorl_conv1d_nseg(int64_t L);
/* the same depthwise causal conv with the activation selectable: act = 1 SiLU (the two entry points below), act = 0 none
 * (the `conv1d_*` encoder layer, ref: offpolicy_rnn/models/conv1d/conv1d.py:26-35) */
int rorl_conv1d_fwd(const float* x, const float* w, const float* bias, const float* mask, float* y, int64_t B, int64_t L,
                    int64_t D, int64_t K, int64_t ld_x, int64_t ld_y, int act, cudaStream_t stream);
int rorl_conv1d_bwd(const float* x, const float* w, const float* bias, const float* mask, const float* dy, float* dx,
                    float* dw_part, float* dbias_part, int64_t B, int64_t L, int64_t D, int64_t K, int64_t ld_x,
                    int64_t ld_dy, int64_t ld_dx, int act, cudaStream_t stream);
int rorl_conv1d_silu_fwd(const float* x, const float* w, const float* bias, const float* mask, float* y,
                         int64_t B, int64_t L, int64_t D, int64_t K, int64_t ld_x, int64_t ld_y,
                         cudaStream_t stream);
int rorl_conv1d_silu_bwd(const float* x, const float* w, const float* bias, const float* mask, const float* dy,
                         float* dx, float* dw_part, float* dbias_part, int64_t B, int64_t L, int64_t D, int64_t K,
                         int64_t ld_x, int64_t ld_dy, int64_t ld_dx, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Fused residual-add + LayerNorm / RMSNorm over the last dimension (rows = B*L tokens).
 * Replaces layer_norm_fn / rms_norm_fn (ref: offpolicy_rnn/models/smamba/mamba_ssm/ops/triton/
 * layernorm.py:464-478, kernels :65-120,196-290; semantics layernorm_cpu.py:6-35):
 *   r = x + residual (residual may be NULL); y = norm(r) * w + b; residual_out = r (may be NULL).
 * rstd/mean: [rows] saved for the backward (mean unused for RMS).
 * Backward: dy [rows, C] and dres_out [rows, C] (gradient arriving at residual_out, may be NULL)
 * -> dx [rows, C] (= gradient w.r.t. both x and residual); dw_part/db_part [nparts, C] with
 * nparts = rorl_addnorm_nparts(rows), reduced over axis 0 by the caller.
 * ---------------------------------------------------------------------------------------------- */
int rorl_addnorm_nparts(int64_t rows);
int rorl_addnorm_fwd(const float* x, const float* residual, const float* w, const float* b, float* y,
                     float* residual_out, float* mean, float* rstd, int64_t rows, int64_t C, float eps, int is_rms,
                     cudaStream_t stream);
int rorl_addnorm_bwd(const float* dy, const float* dres_out, const float* r, const float* w, const float* mean,
                     const float* rstd, float* dx, float* dw_part, float* db_part, int64_t rows, int64_t C,
                     int is_rms, int has_bias, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Fused target-Q / masked-TD / actor / entropy reductions over the valid-step mask.
 * Replaces the ATen chains in _target_Q, QValueGuard.clamp/update, _Q_loss, _policy_loss,
 * _alpha_loss, _mask_mean (ref: offpolicy_rnn/algorithm/sac_full_length_rnn_ensembleQ.py:80-132,
 * sac_full_length_rnn_redq.py:16-47, td3_full_length_rnn_ensembleQ.py:23-71,
 * offpolicy_rnn/utility/q_value_guard.py:22-38).
 *
 * guard: device double[4] = {min, max, initialised(0/1), decay} (the reference keeps these as Python
 * floats, i.e. doubles); work: device scratch of rorl_loss_work_floats() floats, zero-initialised
 * once by the caller.  All kernels are single-launch, deterministic two-level reductions.
 * ---------------------------------------------------------------------------------------------- */
/* m[i] = min over the selected ensemble members of q[e, i] - alpha * logp[i] (logp may be NULL);
 * on the first call (guard[2] == 0) also initialises guard min/max from m (ref q_value_guard.py:22-27). */
int rorl_target_minq(const float* q, const int32_t* sel, int64_t nsel, int64_t E, int64_t M, const float* logp,
                     const float* log_alpha, float* m, double* guard, float* work, cudaStream_t stream);
/* y[i] = reward + (1 - done') * gamma * clamp(m, guard.min, guard.max) with done' = done zeroed where
 * timeout > 0; then guard.update(y * mask) with EMA decay (ref q_value_guard.py:29-38);
 * stats[0] = max |y|, stats[1] = sum(mask). */
int rorl_target_finish(const float* m, const float* reward, const float* done, const float* timeout,
                       const float* mask, float gamma, float* y, double* guard, float* stats, float* work,
                       int64_t M, cudaStream_t stream);
int64_t rorl_loss_work_floats(int64_t M);
/* loss = sum_i mask_i sum_e (q[e,i] - y[i])^2 / nvalid; dq[e,i] = 2 mask_i (q - y) / nvalid. */
int rorl_q_loss_fwd_bwd(const float* q, const float* y, const float* mask, const float* nvalid, float* loss,
                        float* dq, float* work, int64_t E, int64_t M, cudaStream_t stream);
/* actor: loss = sum_i mask_i (alpha logp_i - agg_e q[e,i]) / nvalid, agg = min (mode 0) or mean (mode 1);
 * logp may be NULL (TD3).  Outputs dq [E, M], dlogp [M] (if logp), and the entropy side results
 * out[0] = actor loss, out[1] = masked mean logp, out[2] = alpha loss = -log_alpha * mean(logp + H),
 * out[3] = d alpha_loss / d log_alpha. */
int rorl_actor_loss_fwd_bwd(const float* q, const float* logp, const float* mask, const float* nvalid,
                            const float* log_alpha, float target_entropy, int mode, float* out, float* dq,
                            float* dlogp, float* work, int64_t E, int64_t M, cudaStream_t stream);
/* Discrete actions (ref: sac_full_length_rnn_ensembleQ.py:134-185, sac_full_length_rnn_redq.py:52-88): q [E, M, A] holds one
 * Q per action, logp [M, A] the policy's log-probabilities; 1 <= A <= 256.
 * rorl_discrete_target_expect: m[i] = sum_a exp(logp[i, a]) (min over the selected members of q[e, i, a] - alpha logp[i, a]),
 * alpha = exp(log_alpha[0]); like rorl_target_minq it initialises guard min/max from m on the first call, and m feeds
 * rorl_target_finish unchanged.
 * rorl_discrete_actor_loss_fwd_bwd: agg = min over members (mode 0) or mean (mode 1), p = exp(logp);
 *   out[0] = sum_i mask_i sum_a p (alpha logp - agg) / nvalid (actor loss), out[1] = sum_i mask_i sum_a p logp / nvalid;
 *   dlogp[i, a] = mask_i / nvalid * p (alpha logp - agg + alpha).  q receives no gradient (the discrete value ignores its
 *   action argument and its weights are frozen under the actor). */
int rorl_discrete_target_expect(const float* q, const int32_t* sel, int64_t nsel, int64_t E, int64_t M, int64_t A,
                                const float* logp, const float* log_alpha, float* m, double* guard, float* work,
                                cudaStream_t stream);
int rorl_discrete_actor_loss_fwd_bwd(const float* q, const float* logp, const float* mask, const float* nvalid,
                                     const float* log_alpha, int mode, float* out, float* dlogp, float* work, int64_t E,
                                     int64_t M, int64_t A, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Multi-tensor AdamW step (+ optional Polyak target update) over a flat parameter arena.
 * Replaces torch.optim.AdamW over param groups (ref: offpolicy_rnn/algorithm/sac.py:61,81-90;
 * group construction sac_full_length_rnn_redq_sep_optim.py:37-102) and the per-parameter
 * soft-update loop (ref: offpolicy_rnn/models/rnn_base.py:475-491).
 * p, g, m, v (and target, may be NULL): flat fp32 arrays of n elements; seg_end[nseg] (int64, device)
 * and seg_lr / seg_wd [nseg] (double, device) describe contiguous LR / weight-decay groups (nseg <= 64);
 * step_ptr: device int32 count of completed steps (incremented on the stream after the update).
 * Gradient clipping (ref: sac_full_length_rnn_ensembleQ.py:239-250,274-287), applied to g IN PLACE before the step:
 *   gnorm_sq != NULL: clip_grad_norm_ -- g *= min(1, max_norm / (sqrt(gnorm_sq[0]) + 1e-6)), gnorm_sq[0] = sum(g^2)
 *                     over the model (device scalar, e.g. from rorl_sumsq);
 *   seg_clip != NULL: clip_grad_value_ -- per-segment bound (double[nseg], <= 0 = off).
 * target <- tau * target + (1 - tau) * p_new when target != NULL.
 * ---------------------------------------------------------------------------------------------- */
int rorl_adamw_polyak(float* p, float* g, float* m, float* v, float* target, const int64_t* seg_end,
                      const double* seg_lr, const double* seg_wd, const double* seg_clip, int64_t nseg, int64_t n,
                      float beta1, float beta2, float eps, float tau, int32_t* step_ptr, const float* gnorm_sq,
                      float max_norm, cudaStream_t stream);
/* out[0] = sum(p^2) (l2_norm_square, ref rnn_base.py:531-532) */
int rorl_sumsq(const float* p, int64_t n, float* out, float* work, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * tcgen05 tensor-core GEMM with fp32 parity: every fp32 operand is split into bf16 hi + lo and the product is
 * accumulated as lo*hi + hi*lo + hi*hi in the fp32 TMEM accumulator.
 * Replaces the cuBLAS fp32 SGEMMs behind nn.Linear / EnsembleLinear (ref: offpolicy_rnn/models/
 * ensemble_linear_model.py:36-49; smamba projections, ref: offpolicy_rnn/models/smamba/mamba.py:176,231-233,252).
 *   D[g][M, N] = act(A[g][M, K] * B[g][N, K]^T + bias[g][N]),  g = 0..G-1
 * Both operands K-major (reduction dimension contiguous).  strideA / strideB == 0: operand shared by all g.
 * act: flag word -- bits 0-1: 1 = ELU, 2 = exact (erf) GELU (the cgpt FFN, ref TransformerFlashAttention.py:43-57);
 * Dpre, may be NULL, receives the pre-activation in D's layout (the GELU backward needs it, rorl_gelu_bwd_colsum);
 * bit 2 (4) ACCUMULATE: D += result, so that a gradient with two producers (the scan's du and x_proj's input
 * gradient, ref: smamba/mamba.py:213-233) needs no separate add pass.
 * passes: 2 = the two-term bf16 split, 3 bf16 MMAs (fp32 parity to ~2^-17); 4 = its hi * hi term alone (one bf16 MMA
 * per k-step: what a layer the reference runs under bf16 autocast computes, ref TransformerFlashAttention.py:80-81).
 * Any other value: RORL_ERR_ARG.  reduce_g != 0: the G products are summed into one D[M, N] (data-gradient of an
 * ensemble layer with shared input).
 * K, N, ld*, stride* multiples of 4; bases 16-byte aligned.
 * work: device scratch of rorl_gemm_tn_work_bytes(...) bytes, 16-byte aligned: the kernel pre-splits the B operand --
 * the weights, re-read by every row tile -- into its bf16 copy there: hi [GB][N][Kp] followed by lo [GB][N][Kp], with
 * GB = G if B is batched (strideB != 0), else 1, and Kp = K rounded up to a multiple of 8 (columns K..Kp-1 are neither
 * written nor read).
 * transb is a flag word.  Bit 1 (2): `work` ALREADY holds B's split copy -- the caller keeps it up to date with
 * rorl_split_bf16_multi after every change of the weights -- and the per-call pre-split launch is skipped (an update
 * issues ~110 GEMMs on weights that change three times).  Bit 0 (1): B is stored [K, N] with row stride ldb --
 * nn.Linear's weight as its input-gradient GEMM needs it, EnsembleLinear's [E, in, out] weight as its forward needs
 * it -- and the pre-split transposes it.
 * ---------------------------------------------------------------------------------------------- */
/* bytes of `work` for rorl_gemm_tn: 2 * GB * N * Kp bf16; RORL_ERR_ARG for passes other than 2 / 4 */
int64_t rorl_gemm_tn_work_bytes(int64_t N, int64_t K, int64_t G, int64_t strideB, int passes);
/* (Re)build the split copies of many B operands in one launch.  jobs: DEVICE array of njobs records
 *   struct { const float* src; void* dst; int32_t N, K, G, transposed; int64_t ld, gs; }      (48 bytes each)
 * src: G groups (group stride gs floats) of [N, K] rows with row stride ld, or -- transposed != 0 -- of [K, N] rows;
 * dst: rorl_gemm_tn_work_bytes(N, K, G, gs, 2) bytes, receives hi [G][N][Kp] then lo [G][N][Kp] (Kp = K rounded up
 * to 8): the buffer to hand to rorl_gemm_tn as `work` with transb bit 1. */
int rorl_split_bf16_multi(const void* jobs, int64_t njobs, cudaStream_t stream);
int rorl_gemm_tn(const float* A, const float* B, const float* bias, float* D, float* Dpre, int64_t M, int64_t N, int64_t K, int64_t G,
                 int64_t lda, int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD,
                 int64_t strideBias, int act, int passes, int reduce_g, int transb, void* work, cudaStream_t stream);
/* Weight-gradient form: D[s][g][M, N] = sum over the s-th slice of rows r of A[g][r, M]^T B[g][r, N] (both operands
 * row-major with the REDUCTION over rows, i.e. MN-major for the tensor core; no transposed copies).  Split-K over
 * the R rows: splits = rorl_gemm_nt_splits(M, N, R, G); partial s lands at D + s * strideSplit and the caller sums
 * the partials (deterministic).  M, N, ld*, stride* multiples of 4; passes 2 or 4 as for rorl_gemm_tn. */
int rorl_gemm_nt_splits(int64_t M, int64_t N, int64_t R, int64_t G);
int rorl_gemm_nt(const float* A, const float* B, float* D, int64_t M, int64_t N, int64_t R, int64_t G, int64_t lda,
                 int64_t ldb, int64_t ldd, int64_t strideA, int64_t strideB, int64_t strideD, int64_t splits,
                 int64_t strideSplit, int passes, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Output layer of the ensemble-Q head (`efc-E` with out_dim = 1) and its backward fused with the ELU backward and
 * bias gradient of the layer below.  Replaces EnsembleLinear's bmm [E, M, K] x [E, K, 1] and, in the backward, the
 * outer-product bmm + elu_backward + reductions (ref: offpolicy_rnn/models/ensemble_linear_model.py:36-49,
 * contextual_model.py:97-116).  K in {128, 256, 384, 512}; y, g [E, M, K] contiguous; w [E, K]; b [E] or NULL.
 *   rorl_efc_dot_fwd : q[e, m] = sum_k y[e, m, k] w[e, k] + b[e]
 *   rorl_efc_head_bwd: g = dq w elu'(y) (elu != 0: y is an ELU OUTPUT; else g = dq w);
 *                      part [E][nblk][2K + 4] = per-CTA partials of (dw[e, k] = sum_m dq y | sum_m g[e, m, k] |
 *                      db[e] = sum_m dq, 0, 0, 0), nblk = rorl_efc_head_nblk(); the caller sums over nblk.
 * ---------------------------------------------------------------------------------------------- */
int rorl_efc_head_nblk(void);
int rorl_efc_dot_fwd(const float* y, const float* w, const float* b, float* q, int64_t E, int64_t M, int64_t K, cudaStream_t stream);
int rorl_efc_head_bwd(const float* dq, const float* y, const float* w, float* g, float* part, int64_t E, int64_t M, int64_t K,
                      int elu, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Tanh-Gaussian policy head (csrc/head.cu), forward and backward in one kernel each.  Replaces the elementwise graph
 * of ContextualSACPolicySingleHead.forward after the universal network
 * (ref: offpolicy_rnn/policy_value_models/contextual_sac_policy_single_head.py:105-123):
 *   out [M, 2A] (row stride ld_out) = [logstd | mean];  noise [M, A] standard normal draws
 *   logstd clamped to [min_logstd, max_logstd]; sample = mean + noise * exp(logstd)
 *   action_mean = tanh(mean), action_sample = tanh(sample)            [M, A]
 *   log_prob [M] = sum_a N(sample; mean, std) log-density - 2 (log 2 - sample - softplus(-2 sample))
 * bwd: d_mean / d_sample / d_log_prob may be NULL (treated as zero); d_out [M, 2A] contiguous.
 * ---------------------------------------------------------------------------------------------- */
int rorl_tanh_gaussian_fwd(const float* out, const float* noise, float* action_mean, float* action_sample, float* log_prob,
                           int64_t M, int64_t A, int64_t ld_out, float min_logstd, float max_logstd, cudaStream_t stream);
int rorl_tanh_gaussian_bwd(const float* out, const float* noise, const float* d_mean, const float* d_sample, const float* d_log_prob,
                           float* d_out, int64_t M, int64_t A, int64_t ld_out, float min_logstd, float max_logstd,
                           cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Categorical policy head (csrc/categorical.cu), forward and backward in one kernel each.  Replaces the elementwise graph
 * of ContextualSACDiscretePolicy.process_model_out (ref: offpolicy_rnn/policy_value_models/contextual_sac_discrete_policy.py:
 * 106-111).  logits [M, A] with row stride ld (>= A); 1 <= A <= 256; M == 0 is a no-op.
 *   s = softmax(logits); probs = (s + 0.01) / sum(s + 0.01); logp = log(probs)          [M, A] contiguous
 *   mode[i] = argmax_a probs (first index on ties), written as float                    [M]
 *   sample[i] = first a with cumsum(probs)[a] > u[i] * sum(probs), as float             [M]; u [M] uniform draws, or NULL
 *               (no sample drawn; sample may then be NULL too)
 * bwd: d_logits [M, A] contiguous = s * (v - sum_a s v), v = d_logp / probs / sum(s + 0.01): autograd through the ops above
 * in closed form (the renormalising sum's gradient is uniform over a and the softmax Jacobian removes it).  Recomputes
 * everything from the logits.
 * ---------------------------------------------------------------------------------------------- */
int rorl_categorical_fwd(const float* logits, int64_t ld, const float* u, float* probs, float* logp, float* mode,
                         float* sample, int64_t M, int64_t A, cudaStream_t stream);
int rorl_categorical_bwd(const float* logits, int64_t ld, const float* d_logp, float* d_logits, int64_t M, int64_t A,
                         cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GRU recurrence as a persistent thread-block-cluster kernel (W_hh resident in registers across a
 * cluster of H / 64 CTAs, h_t exchanged through distributed shared memory each step).
 * Replaces the recurrent part of torch.nn.GRU(input, H, batch_first=True) on the `gru` encoder path
 * (ref: offpolicy_rnn/models/rnn_base.py:59,245-247,454; gate order r, z, n as in torch.nn.GRU).
 * gi [B, L, 3H] = x W_ih^T + b_ih is computed by the caller (one GEMM); w_hh [3H, H]; b_hh [3H] or
 * NULL; h0 [B, H] or NULL (= 0).  out [B, L, H] = h_t for every step; h_last [B, H] (may be NULL);
 * save [B, L, 4H] = (r, z, n, W_hn h + b_hn) for the backward (NULL when no backward follows).
 * H in {128, 256}.
 * Backward: dout [B, L, H] (gradient w.r.t. out), dh_last [B, H] or NULL -> dgi [B, L, 3H] (gradient
 * w.r.t. gi = gradient w.r.t. the r and z rows of gh as well), dghn [B, L, H] (gradient w.r.t.
 * W_hn h + b_hn), dh0 [B, H] (may be NULL).  Weight gradients are GEMMs over all steps, left to the
 * caller: dW_hh = [dgi_r, dgi_z, dghn]^T h_{t-1}.
 * ---------------------------------------------------------------------------------------------- */
int rorl_gru_save_floats_per_step(int64_t H);
/* Tuning knob (process-wide, read at launch time): SMs the forward recurrence may occupy, default 148.  A caller that
 * runs two independent recurrences on two streams sets about half for the duration of those launches. Returns the value set. */
int rorl_gru_set_fwd_sms(int sms);
int rorl_gru_fwd(const float* gi, const float* w_hh, const float* b_hh, const float* h0, float* out, float* save,
                 float* h_last, int64_t B, int64_t L, int64_t H, cudaStream_t stream);
int rorl_gru_bwd(const float* dout, const float* dh_last, const float* w_hh, const float* save, const float* out,
                 const float* h0, float* dgi, float* dghn, float* dh0, int64_t B, int64_t L, int64_t H,
                 cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * LSTM recurrence as a persistent thread-block-cluster kernel (W_hh resident in registers across a
 * cluster of H / 32 CTAs, h_t exchanged through distributed shared memory each step; csrc/lstm.cu).
 * Replaces the recurrent part of torch.nn.LSTM(input, H, batch_first=True) on the `lstm` encoder path
 * (ref: offpolicy_rnn/models/rnn_base.py layer table 'lstm' -> nn.LSTM; gate order i, f, g, o as in torch.nn.LSTM:
 * gates = gi + h W_hh^T + b_hh, c' = sigmoid(f) c + sigmoid(i) tanh(g), h' = sigmoid(o) tanh(c')).
 * gi [B, L, 4H] = x W_ih^T + b_ih is computed by the caller (one GEMM); w_hh [4H, H] (16-byte aligned); b_hh [4H]
 * or NULL; h0, c0 [B, H] or NULL (= 0).  out [B, L, H] = h_t for every step; h_last, c_last [B, H] (may be NULL);
 * save [B, L, 5H] = (sigmoid(i), sigmoid(f), tanh(g), sigmoid(o), c_t) per step for the backward (NULL when no
 * backward follows; rorl_lstm_save_floats_per_step(H) = 5H).  H in {16, 32, 64, 128, 256}.
 * Backward: dout [B, L, H] (gradient w.r.t. out), dh_last, dc_last [B, H] or NULL (= 0), the forward's save and c0
 * -> dgates [B, L, 4H] (gradient w.r.t. the pre-activation gates = w.r.t. gi = w.r.t. b_hh per step), dh0, dc0
 * [B, H] (may be NULL).  Weight gradients are GEMMs over all steps, left to the caller: dW_hh = dgates^T h_{t-1}.
 * Deterministic (no atomics), no host synchronisation or allocation: both launches can be graph-captured.
 * ---------------------------------------------------------------------------------------------- */
int rorl_lstm_save_floats_per_step(int64_t H);
int rorl_lstm_fwd(const float* gi, const float* w_hh, const float* b_hh, const float* h0, const float* c0, float* out,
                  float* save, float* h_last, float* c_last, int64_t B, int64_t L, int64_t H, cudaStream_t stream);
int rorl_lstm_bwd(const float* dout, const float* dh_last, const float* dc_last, const float* w_hh, const float* save,
                  const float* c0, float* dgates, float* dh0, float* dc0, int64_t B, int64_t L, int64_t H,
                  cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Causal variable-length attention with ALiBi on tcgen05 tensor cores (bf16 operands, fp32 accumulate), head
 * dimension hd = any multiple of 8 from 8 to 128 (the _hd entry points; the entry points without the suffix are those
 * with hd = 64).  Replaces flash_attn_varlen_qkvpacked_func(qkv[T, 3, H, hd], cu_seqlens, max_seqlen, p = 0,
 * softmax_scale, causal = True, alibi_slopes) as used by flash_attn's MHA in the cgpt encoder layer
 * (ref: offpolicy_rnn/models/flash_attention/TransformerFlashAttention.py:65-85,104-121).
 *
 * Token spaces.  TMA needs 16-byte aligned inner coordinates, so inside the attention kernels every sequence starts
 * on an 8-token boundary of an ATTENTION TOKEN SPACE of T tokens (Tp = T rounded up to a multiple of 64); gmap
 * (device int32[T], or NULL = identity) gives the source row of each attention-space token (-1 = padding slot).
 * rorl_attn_prep gathers an fp32 source [rows, nsec, H, hd] (row stride ld_tok floats) into bf16 copies in that
 * space, padded along d to DP = 64 (hd <= 64) or DP = 128 (hd > 64) with zero columns: row-major rm [nsec][T, H, DP]
 * and token-contiguous tr [nsec][H, DP, Tp] (either may be NULL); with o != NULL (nsec == 1, o [rows, H, hd] in
 * SOURCE rows, row stride ld_o) it also writes D[H, Tp] = sum_d src * o (the backward's row statistic).
 * bf16 buffers are passed as void*.  The forward and backward take these DP-padded copies.
 * tiles: device int32[ntiles][4] = (first attention-space token of the sequence, sequence length, 128-row tile
 * index, first OUTPUT row of the sequence), one entry per 128-row tile of every sequence.
 * Forward: O fp32 with row stride ld_o, written at OUTPUT rows (columns h*hd .. h*hd+hd-1 of head h; other rows
 * and columns are not touched), lse [H, Tp] (log2 domain, attention space) for the backward (may be NULL).
 * Backward: dq, dk, dv fp32 with row stride ld_d, written at OUTPUT rows, columns h*hd .. h*hd+hd-1.
 * An unsupported head_dim returns RORL_ERR_SHAPE.
 * dropout_p > 0: attention-probability dropout (flash-attn's dropout_p; ref TransformerFlashAttention.py:65-70):
 * keep bits come from a counter hash of (seed[0] (device int64), salt, head, query token, key token); the backward
 * must be given the same (dropout_p, seed value, salt) as its forward.  dropout_p == 0: seed may be NULL.
 * ---------------------------------------------------------------------------------------------- */
int rorl_attn_prep(const float* src, int64_t ld_tok, int64_t nsec, int64_t H, int64_t T, int64_t Tp, const int32_t* gmap,
                   void* rm_bf16, void* tr_bf16, const float* o, int64_t ld_o, float* Dout, cudaStream_t stream);
int rorl_attn_fwd(const void* q_rm, const void* k_rm, const void* v_tr, const int32_t* tiles, int64_t ntiles,
                  const float* slopes, float softmax_scale, float* O, int64_t ld_o, float* lse, int64_t H, int64_t T,
                  int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt, cudaStream_t stream);
int rorl_attn_bwd(const void* q_rm, const void* k_rm, const void* v_rm, const void* do_rm, const void* q_tr,
                  const void* k_tr, const void* do_tr, const float* lse, const float* D, const int32_t* tiles,
                  int64_t ntiles, const float* slopes, float softmax_scale, float* dq, float* dk, float* dv,
                  int64_t ld_d, int64_t H, int64_t T, int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt,
                  cudaStream_t stream);
int rorl_attn_prep_hd(const float* src, int64_t ld_tok, int64_t nsec, int64_t H, int64_t T, int64_t Tp, const int32_t* gmap,
                      void* rm_bf16, void* tr_bf16, const float* o, int64_t ld_o, float* Dout, int64_t head_dim,
                      cudaStream_t stream);
int rorl_attn_fwd_hd(const void* q_rm, const void* k_rm, const void* v_tr, const int32_t* tiles, int64_t ntiles,
                     const float* slopes, float softmax_scale, float* O, int64_t ld_o, float* lse, int64_t H, int64_t T,
                     int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt, int64_t head_dim, cudaStream_t stream);
int rorl_attn_bwd_hd(const void* q_rm, const void* k_rm, const void* v_rm, const void* do_rm, const void* q_tr,
                     const void* k_tr, const void* do_tr, const float* lse, const float* D, const int32_t* tiles,
                     int64_t ntiles, const float* slopes, float softmax_scale, float* dq, float* dk, float* dv,
                     int64_t ld_d, int64_t H, int64_t T, int64_t Tp, float dropout_p, const int64_t* seed, int64_t salt,
                     int64_t head_dim, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Trajectory gather: builds the padded, nest-stacked [rows, Lmax, F] fp32 batch of
 * NestedMemoryArray.sample_trajs directly from a device-resident fp32 ring buffer, following a
 * host-computed plan (ref: offpolicy_rnn/buffers/transition_buffer/nested_replay_memory.py:103-185;
 * layout SURVEY.md App. A).  plan: device int64[4*ntraj + rows] = (src_start, row, ptr, len) per placed
 * trajectory (src_start = first ring row, ptr = first step of its blank prefix in the batch row, len =
 * stored steps), followed by row_end[rows] (first step of each row's tail).  colmap: device
 * int32[3 + 2*npairs] = {start_col, mask_col, npairs, (dst_col, src_col)...} (pre-step target <- first
 * transition's source columns); start_col is passed again by value.  batch [rows, Lmax, F] and valid
 * [rows, Lmax] are fully written (zero-filled first).  max_len = longest `len` in the plan.
 * ---------------------------------------------------------------------------------------------- */
int rorl_traj_gather(const float* ring, int64_t F, const int64_t* plan, int64_t ntraj, const int32_t* colmap,
                     int64_t start_col, float* batch, float* valid, int64_t rows, int64_t Lmax, int64_t skip,
                     int64_t max_len, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Deterministic row reductions of the backward pass (csrc/reduce.cu): no atomics, per-CTA partials in `work`.
 * Replace ATen `sum(0)` / `mm` launches autograd issues for the reference's nn.Linear / EnsembleLinear biases and
 * narrow-input weights (ref: offpolicy_rnn/models/ensemble_linear_model.py:29-60; torch.nn.Linear backward).
 *   rorl_colsum          out[g, n] = sum_m x[g, m, n]      x: G groups of [M, N], row stride ldx, group stride gsx
 *   rorl_elu_bwd_colsum  gout = dy * (y > 0 ? 1 : y + 1)   ELU backward from the layer OUTPUT y, fused with the
 *                        out[g, n] = sum_m gout[g, m, n]   bias gradient of that layer
 *   rorl_skinny_wgrad    dW[n, k] = sum_m g[m, n] x[m, k]  K <= 16 (obs / action encoders, dt_proj); dW is [N, KP],
 *                        KP = K rounded up to a multiple of 4, columns >= K are zero
 * N % 4 == 0 and 16-byte aligned rows for the column sums; `work` holds rorl_*_work_floats() floats.
 * ---------------------------------------------------------------------------------------------- */
int64_t rorl_colsum_work_floats(int64_t G, int64_t M, int64_t N);
/* tickets: device int32[rorl_colsum_tickets()] zero-initialised ONCE by the caller (the kernels re-arm them): with it the
 * per-CTA partial rows are folded by the last CTA to finish, in a fixed order (deterministic), in the SAME launch; NULL:
 * a second tiny launch does the fold.  One ticket array must not be shared by launches that can run concurrently. */
int rorl_colsum_tickets(void);
int rorl_colsum(const float* x, float* out, float* work, int64_t G, int64_t M, int64_t N, int64_t ldx, int64_t gsx,
                int32_t* tickets, cudaStream_t stream);
int rorl_elu_bwd_colsum(const float* dy, const float* y, float* g, float* out, float* work, int64_t G, int64_t M,
                        int64_t N, int64_t ld_dy, int64_t ld_y, int64_t ld_g, int64_t gs_dy, int64_t gs_y, int64_t gs_g,
                        int32_t* tickets, cudaStream_t stream);
/* the same for the exact GELU, from the PRE-activation: gout = dy * (Phi(pre) + pre phi(pre)), out = column sums of gout */
int rorl_gelu_bwd_colsum(const float* dy, const float* pre, float* g, float* out, float* work, int64_t G, int64_t M,
                         int64_t N, int64_t ld_dy, int64_t ld_pre, int64_t ld_g, int64_t gs_dy, int64_t gs_pre, int64_t gs_g,
                         int32_t* tickets, cudaStream_t stream);
/* out[r * out_ld + c] = sum_p part[p][r * C + c]  (part: P planes of contiguous [rows, C]; C, out_ld % 4 == 0): per-tile
 * partial rows summed straight into a column block of a wider buffer -- the selective scan's dB | dC partials into
 * their columns of d(x_dbl) (ref: the column slices of smamba/mamba.py:214-222). */
int rorl_sum_leading_rows(const float* part, float* out, int64_t P, int64_t rows, int64_t C, int64_t out_ld, cudaStream_t stream);
/* y[m, n] = act(bias[n] + sum_k x[m, k] W[n, k]) for K <= 16, N % 4 == 0 (bias may be NULL; elu != 0: ELU): forward of
 * the same projections; ldy lets several of them write side by side into one [M, sum N] buffer (no concatenation).
 * Row m of x is read at x + (m / seg_rows) * seg_stride + (m % seg_rows) * ldx, so that a [B, L, K] slice of the
 * sampled batch tensor (ref: the column / time slices of sac_full_length_rnn_ensembleQ.py:318-343) is used in place;
 * seg_rows = M, seg_stride = 0 for a plain [M, K] operand.  rorl_skinny_wgrad addresses x the same way.
 * rorl_skinny_dgrad: dx[m, k] = sum_n g[m, n] W[n, k] (dx contiguous [M, K]; N <= 1024). */
int rorl_skinny_linear(const float* x, const float* W, const float* bias, float* y, int64_t M, int64_t N, int64_t K,
                       int64_t ldx, int64_t seg_rows, int64_t seg_stride, int64_t ldy, int elu, cudaStream_t stream);
int64_t rorl_skinny_wgrad_work_floats(int64_t M, int64_t N, int64_t K);
int rorl_skinny_wgrad(const float* g, const float* x, float* dW, float* work, int64_t M, int64_t N, int64_t K,
                      int64_t ldg, int64_t ldx, int64_t seg_rows, int64_t seg_stride, cudaStream_t stream);
int rorl_skinny_dgrad(const float* g, const float* W, float* dx, int64_t M, int64_t N, int64_t K, int64_t ldg, cudaStream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Decode step (csrc/step.cu): what one environment step of the policy (L = 1) runs.
 *
 * rorl_small_linear: y[g][m, n] = act(bias[g][n] + sum_k x[g][m, k] W[g](n, k)) for 1 <= M <= 64 rows, any K >= 1, any N,
 * in fp32 on the FMA pipe (the rollout's projections; a tensor-core tile would compute one to a few real rows).
 *   layout 0: W [N, K] (nn.Linear), G = 1, x_gstride = 0, bias [N];
 *   layout 1: W [G, K, N] (EnsembleLinear), bias [G, N]; x of member g at x + g * x_gstride (0 = one input shared by
 *             all G members); y of member g at y + g * M * ldy.
 * Row m of x is at x + m * ldx (ldx >= K), row m of y at y + m * ldy (ldy >= N).  bias may be NULL; elu != 0 applies ELU.
 * The summation order along K is fixed by the block shape, not the grid: repeated calls are bit-identical.
 *
 * rorl_mamba_step_conv: one step of the smamba mixer's depthwise conv (ref: smamba/mamba.py Mamba.step): the window
 * [B, D, Kc] (row b at win + b * ld_win) is rolled left by one and the new column xs = xz[b, :D] appended, then
 * u[b, d] = silu(sum_j window[b, d, j] conv_w[d, j] + conv_b[d]) into u [B, D] contiguous.  conv_b may be NULL.
 * rorl_mamba_step_ssm: one step of the selective SSM with the carried state h [B, D, Ns] (row b at h + b * ld_h):
 *   delta = softplus(x_dbl[b, :R] . dt_w[d, :] + dt_b[d]);  A = -exp(A_log[d, n]);
 *   h <- exp(delta A) h + delta u B (B = x_dbl[b, R:R+Ns]);  y[b, d] = (C . h + Dskip[d] u) silu(z[b, d])
 * with C = x_dbl[b, R+Ns:R+2Ns]; y [B, D] contiguous; Dskip may be NULL.  For both, win_in / h_in may equal win_out /
 * h_out (update in place).  As in the reference's step, no reset flag or mask is read.
 * ---------------------------------------------------------------------------------------------- */
int rorl_small_linear(const float* x, int64_t ldx, int64_t x_gstride, const float* W, const float* bias, float* y, int64_t ldy,
                      int64_t M, int64_t N, int64_t K, int64_t G, int layout, int elu, cudaStream_t stream);
int rorl_mamba_step_conv(const float* xz, int64_t ld_xz, const float* conv_w, const float* conv_b, const float* win_in,
                         int64_t ld_win_in, float* win_out, int64_t ld_win_out, float* u, int64_t B, int64_t D, int64_t Kc,
                         cudaStream_t stream);
int rorl_mamba_step_ssm(const float* u, const float* x_dbl, int64_t ld_xdbl, const float* z, int64_t ld_z, const float* dt_w,
                        const float* dt_b, const float* A_log, const float* Dskip, const float* h_in, int64_t ld_h_in, float* h_out,
                        int64_t ld_h_out, float* y, int64_t B, int64_t D, int64_t R, int64_t Ns, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RORL_B200_H */
