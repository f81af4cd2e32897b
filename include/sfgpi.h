/*
 * sfgpi.h -- C ABI of the B200-native SF/GPI hot path (libsfgpi.so, sm_100a only).
 *
 * Drop-in boundary for the data-parallel hot path of okgarces/deep-successor-features-for-transfer.  The reference
 * is pure Python/PyTorch; each entry point below replaces the eager-op sequence of the reference function it cites.
 * A reference-side binding is a ctypes stub (see INTEGRATION.md).  Conventions:
 *   - every pointer is a DEVICE pointer unless named host_*; tensors are dense, row-major, fp32 unless noted;
 *   - `stream` is a cudaStream_t passed as void*; all work is stream-ordered, nothing synchronises;
 *   - buffers are borrowed for the call, never owned; outputs are caller-allocated;
 *   - return value: 0 = ok, negative = SFGPI_E_* (sfgpi_last_error() gives the text).  No CPU fallback exists.
 *
 * Packed parameter storage ("library"): one row of `row_stride` floats per policy,
 *   row = [ W_0 | b_0 | W_1 | b_1 | ... | W_{L-1} | b_{L-1} | (pad) ],  W_l is [dims[l+1]][dims[l]] (nn.Linear layout),
 * every tensor offset a multiple of 4 floats.  Online nets, target nets, Adam exp_avg and exp_avg_sq are four
 * buffers [N][row_stride] of identical layout.
 */
#ifndef SFGPI_H
#define SFGPI_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SFGPI_MAX_LAYERS 8
#define SFGPI_MAX_SEGMENTS 8

#define SFGPI_ACT_NONE 0
#define SFGPI_ACT_RELU 1
#define SFGPI_ACT_TANH 2

#define SFGPI_OK 0
#define SFGPI_E_INVALID (-1)   /* bad argument / unsupported shape */
#define SFGPI_E_SMEM (-2)      /* shape needs more shared memory than an SM has */
#define SFGPI_E_CUDA (-3)      /* CUDA runtime error at launch */

/* psi network shape = product of the mains' sf_model_lambda (main_tsfdqn_sequential_torch.py:44-75). */
typedef struct {
    int32_t n_layers;                      /* number of Linear layers L (>= 1) */
    int32_t dims[SFGPI_MAX_LAYERS + 1];    /* dims[0] = S ... dims[L] = A*D */
    int32_t acts[SFGPI_MAX_LAYERS];        /* SFGPI_ACT_* applied after layer l */
    int32_t w_off[SFGPI_MAX_LAYERS];       /* float offset of W_l inside a policy row */
    int32_t b_off[SFGPI_MAX_LAYERS];       /* float offset of b_l inside a policy row */
    int32_t row_stride;                    /* floats per policy row */
    int32_t n_actions;                     /* A */
    int32_t n_features;                    /* D;  dims[L] == A*D */
} sfgpi_net_desc;

/*
 * Fused ensemble psi forward (A1/A2/A3 + the epilogues of A4/A6).  For every policy j in [policy_lo, policy_lo+n_pol)
 * and every state b: psi_j(x_b) through the whole MLP in one kernel (activations never leave the SM), then any of:
 *   psi_out   [B][n_pol][A*D]        get_successor(s) / get_next_successors      (sfdqn.py:290-301, tsfdqn.py:283-307)
 *   acts_out  [l][n_pol][B][dims[l+1]] post-activation outputs of layers 0..L-2, saved for the backward pass
 *   sel_out   [n_pol][B][D]          psi_j(x_b)[a_b,:] with a_b = sel_actions[b] (int64, shared by all policies)
 *                                    or decoded from packed GPI keys sel_keys[(j_local)*sel_key_stride + b]
 *                                    (sfdqn.py:331 `target_psi_model(next_states)[indices, next_actions,:]`)
 *   GPI       q = psi . w  for n_w reward vectors w [n_w][D]; q_out [B][n_pol][A] (first vector only);
 *             key_action[wi][b] = max over (j,a) of pack(q, a), key_task[wi][b] = max of pack(q, task_base+j)
 *             (atomicMax on int64; keys must be pre-filled with INT64_MIN; see sfgpi_pack semantics below)
 *             = GPI_w of sfdqn.py:215-240 without materialising psi[B,N,A,D].
 * Any output pointer may be NULL.  `params` is the [N][row_stride] buffer to read (online or target).
 * mode: 0 = fp32 CUDA-core path (1e-5 parity mode).
 */
typedef struct {
    sfgpi_net_desc net;
    const float *params;
    int32_t policy_lo, n_pol;
    const float *x;                 /* [B][S] */
    int32_t B;
    float *psi_out;
    float *acts_out[SFGPI_MAX_LAYERS];
    const int64_t *sel_actions;
    const int64_t *sel_keys;
    int32_t sel_key_stride;
    float *sel_out;
    const float *w;
    int32_t n_w;
    int32_t w_diag;                 /* 1: policy slot p is scored with w[p] only (keys [n_pol][B]); 0: all n_w vectors */
    int64_t *key_action;
    int64_t *key_task;
    int32_t task_base;
    float *q_out;
    int32_t mode;
    void *acts_bf16_out;            /* tensor-core mode only: [L-1][n_pol][B][256] bf16 post-activation outputs (row-major),
                                       the operands of sfgpi_mlp_backward_tc */
    void *relu_mask_out;            /* tensor-core mode only: [L-1][n_pol][B][8] uint32, bit c%32 of word c/32 = (activation c > 0)
                                       for ReLU layers: all the dgrad chain needs of them */
} sfgpi_forward_args;

int sfgpi_mlp_forward(const sfgpi_forward_args *args, void *stream);

/*
 * Packed (value,index) keys: key = (orderable_i32(q) << 32) | (0xFFFFFFFF - index); signed int64 max == max q, ties
 * -> smallest index (torch.argmax first-index rule, sfdqn.py:239,316), -0 == +0.  A NaN q is never selected; when every
 * q of a (state, reward vector) is NaN or -inf the key decodes to index 0 (action 0, task task_base) with value -inf --
 * torch.argmax would pick the first NaN of a row that mixes NaN with numbers.  Every GPI entry point writes a key for every
 * valid state.  Signed so that the cross-GPU reduction is a plain NCCL/gloo MAX all-reduce on int64.  Decode: action/task
 * as int64 (torch index dtype), value as fp32.
 */
int sfgpi_keys_fill(int64_t *keys, int64_t n, void *stream);
int sfgpi_keys_decode(const int64_t *keys, int64_t n, int64_t *index_out, float *value_out, void *stream);

/*
 * Unfused GPI epilogue on a materialised psi [B][N][A][D] (GPI_w, sfdqn.py:236-239): q_out [B][N][A] (nullable),
 * key_action/key_task [B] written directly (no pre-fill needed).
 */
int sfgpi_gpi_from_psi(const float *psi, const float *w, int32_t B, int32_t N, int32_t A, int32_t D, int32_t task_base,
                       float *q_out, int64_t *key_action, int64_t *key_task, void *stream);

/*
 * TD target, losses and their gradients (sfdqn.py:330-345; tsfdqn.py:621-645; features/deep.py:112-121), batched over
 * n_pol policies that all see the same replay batch.
 *   variant 0 (G1): loss = l1                        (no reward head)
 *   variant 1 (G2): loss = l1 + l2,  l2 = MSE(w.phi, r)
 *   variant 2 (G3): phi~ = phi * (h(g(s)) + h(g(s'))), targets carry grad into g,h; loss = l1 + beta*l2
 * Inputs per policy p: cur_sel/next_sel [n_pol][B][D].  Outputs: d_out [n_pol][B][D] = dLoss/dpsi(s)[a_b,:];
 * loss_part [n_pol][n_blocks][2] partial sums of (diff^2, e^2); aux_grad_part [n_pol][n_blocks][aux_len] partial
 * gradients of [w (D) | g.W (G*S) | g.b (G) | h.W (D*G) | h.b (D)] (variant 1: only w).  n_blocks = sfgpi_td_partials(B)
 * (one partial per 8-CTA thread-block cluster = 256 transitions).
 */
typedef struct {
    int32_t variant, n_pol, B, S, A, D, G;
    float beta;
    const float *cur_sel, *next_sel;
    const float *phis;              /* [B][D] */
    const float *rs;                /* [B] */
    const float *gammas;            /* [B] */
    const float *states, *next_states;   /* [B][S] (variant 2) */
    const float *w;                 /* [n_pol][w_stride] */
    const float *g;                 /* [n_pol][g_stride]: W[G][S] | b[G] */
    const float *h;                 /* W[D][G] | b[D], shared */
    int32_t w_stride, g_stride;
    float *d_out;
    float *loss_part;
    float *aux_grad_part;
    int32_t aux_len;
    /* optional: instead of next_sel, gather psi^-(s')[a*_b,:] here from the target nets' full output next_psi [B][n_pol][A*D]
       with a*_b decoded from the packed GPI keys next_keys[p * next_key_stride + b] (sfdqn.py:331) */
    const float *next_psi;
    const int64_t *next_keys;
    int32_t next_key_stride;
    /* variant 2 scratch: [n_pol][n_blocks][2*D + D*S] partial sums (dw | T | t), see csrc/td.cu.  In variant 2 the g / h
       gradients are linear images of T and t; sfgpi_td_step reduces those and writes ONE complete gradient row per policy into
       partial slot 0 of aux_grad_part (read it with n_part = 1); loss_part keeps n_blocks partials */
    float *tsf_part;
    const void *peer_keys;          /* optional sfgpi_peer_keys_args (policy sharding over peer memory): the kernel signals, waits
                                       and pulls the MAX over ranks of the keys of its own rows itself (next_keys is not read) --
                                       the MAX reduce-scatter of the GPI keys fused into the TD step */
    int32_t defer_expand;           /* variant 2, nonzero: skip the expand launch here; the caller hands this struct to
                                       sfgpi_mlp_backward_tc (expand_td), whose dgrad launch runs it on otherwise idle SMs */
    const float *tsf_mc;            /* variant 2, optional [n_pol][D*S + D]: M = Wh Wg (row-major [D][S]) then c = 2 (Wh bg + bh) of
                                       every policy, e.g. from sfgpi_step_prep (tsf_* fields); NULL: every CTA derives them itself */
    int32_t n_flows;                /* variant 2: K planar flows z <- z + scale_k * tanh(z . weight_k + bias_k) applied to s and s' ahead
                                       of g's Linear (normalising-flow g, tsfdqn_nf.py:331-358, 569-571).  The flows' parameters follow
                                       the Linear in every g row: W[G][S] | b[G] | K x (weight[S] | bias | scale[S]); g_stride, aux_len and
                                       the gradient row [w | dW | db | K x (dweight | dbias | dscale) | dWh | dbh] grow by K*(2S+1), and
                                       tsf_part by the same per block.  0: g is the plain Linear of tsfdqn.py:537-539 */
} sfgpi_td_args;

int sfgpi_td_partials(int32_t B);
int sfgpi_td_step(const sfgpi_td_args *args, void *stream);

/*
 * Backward of the psi MLP for n_pol policies: fused dgrad chain (dZ_l for every layer, activations' derivative from the
 * saved outputs) followed by split-K wgrad + bias grad.  The last layer's dZ is the sparse d_out (only the taken
 * action's D columns are non-zero, sfdqn.py:334-335).
 * actions == NULL: d_out is DENSE, dL/dpsi of a general loss in the layout of the forward's psi_out, [B][n_pol][A*D] fp32
 * (the same rule holds for sfgpi_mlp_backward_tc and sfgpi_mlp_backward_stream).
 *   dz [l][n_pol][B][dims[l+1]] for l = 0..L-2 (scratch, caller-allocated);
 *   grad_part [n_pol][n_split][row_stride]: split-K partial gradients in library row layout.
 */
typedef struct {
    sfgpi_net_desc net;
    const float *params;
    int32_t policy_lo, n_pol;
    const float *x;                 /* [B][S] */
    int32_t B;
    const float *acts[SFGPI_MAX_LAYERS];
    const int64_t *actions;         /* [B]; NULL: d_out is dense */
    const float *d_out;             /* [n_pol][B][D]; dense: [B][n_pol][A*D] */
    float *dz[SFGPI_MAX_LAYERS];
    float *grad_part;
    int32_t n_split;
} sfgpi_backward_args;

int sfgpi_mlp_backward(const sfgpi_backward_args *args, void *stream);

/*
 * Fused multi-tensor Adam (torch/optim/adam.py::_single_tensor_adam order; sfdqn.py:282-286, tsfdqn.py:255-270) for
 * n_pol optimizers; every call is exactly one kernel launch.  A segment is a contiguous parameter range with its own
 * lr / weight decay and its own gradient source (sum of n_part partials).  Per-policy strides select optimizer p's
 * slice; param_stride 0 with n_pol > 1 = shared tensor (TSF's h, whose moments are nevertheless per optimizer).  A
 * shared tensor follows the frozen-snapshot rule: every optimizer steps it from the same pre-step value, and the
 * n_pol deltas are summed in a fixed order.  `step` [n_pol] int32 is incremented on device.  Also reduces
 * loss_part -> losses [n_pol][3] = (loss, l1, l2) when loss_part != NULL.
 */
typedef struct {
    float *param;  int64_t param_stride;
    float *m;      int64_t m_stride;
    float *v;      int64_t v_stride;
    const float *grad_part; int64_t grad_pol_stride; int64_t grad_part_stride; int32_t n_part;
    int32_t len;
    float lr, weight_decay;
    float clamp_min, clamp_max;     /* applied to the stepped parameter when clamp_min < clamp_max (e.g. the G4 loss coefficient,
                                       features/deep_phi.py:212-215; the target task's omegas, tsfdqn.py:977-979); 0, 0: no clamp */
} sfgpi_adam_segment;

typedef struct {
    int32_t n_seg, n_pol;
    sfgpi_adam_segment seg[SFGPI_MAX_SEGMENTS];
    int32_t *step;                  /* [n_pol] */
    double beta1, beta2, eps;       /* doubles: torch derives 1-beta and beta**t in double before the fp32 cast */
    const float *loss_part; int32_t n_loss_part; float l1_scale, l2_scale, beta_loss;
    float *losses;
    double *consts;                 /* [n_pol][2]: {1 - beta1^t, sqrt(1 - beta2^t)} for t = step + 1, consistent with `step` on
                                       entry; read, not written */
    double *consts_next;            /* a second [n_pol][2] buffer, distinct from consts: the launch advances `step` and writes
                                       the NEXT step's corrections here (nothing reads this buffer or `step` during the launch);
                                       the caller swaps the two buffers for the next call.  A call that is not fresh needs
                                       step, consts and consts_next, else SFGPI_E_INVALID */
    int32_t fresh;                  /* nonzero: every call is the FIRST step of a brand-new optimizer (features/deep_phi.py:170 builds a
                                       new torch.optim.Adam per update): moments start at 0 and are not stored, t = 1, `step`, consts and
                                       consts_next are neither read nor written; m / v pointers of the segments may be NULL */
    float *losses_host;             /* optional: PINNED host buffer [n_pol][3]; the block that reduces the losses also stores them
                                       there (a zero-copy store over PCIe: the step's result reaches the host without a copy
                                       command between two kernels of the launch chain).  Valid once the launch has completed.
                                       Pageable memory is refused (SFGPI_E_INVALID): use a stream-ordered copy of `losses` */
} sfgpi_adam_args;

int sfgpi_adam_step(const sfgpi_adam_args *args, void *stream);
/* consts_a[i] = consts_b[i] = {1 - beta1^(step[i]+1), sqrt(1 - beta2^(step[i]+1))}, i < n: re-derives both correction buffers
 * from the step counters (used when optimizers whose buffers are out of phase are stepped together) */
int sfgpi_adam_refresh(const int32_t *step, double *consts_a, double *consts_b, int32_t n, double beta1, double beta2, void *stream);

/*
 * Tensor-core mode (mode 1): bf16 operands on tcgen05 with fp32 accumulation in TMEM, weights streamed by TMA.  Same
 * arguments and epilogues as sfgpi_mlp_forward; needs the bf16 shadow of the library produced by sfgpi_pack_bf16
 * ([n_policies_total][sfgpi_bf16_rows_per_policy()][256] bf16: the hidden 256x256 matrices, then the output matrix padded to
 * a multiple of 16 rows, preceded by the input matrix zero-padded to 256 columns).  Shapes: hidden widths == 256, S <= 63.  Stated tolerance vs fp32: 2e-2 scale-relative on
 * psi / q (SURVEY section 7: bf16 inputs, fp32 accumulate), GPI argmax equal wherever the fp32 top-1/top-2 gap exceeds it.
 */
int sfgpi_bf16_rows_per_policy(const sfgpi_net_desc *net);
int sfgpi_pack_bf16(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, void *out_bf16, void *stream);
/*
 * GPI form of the tensor-core forward: q = psi . w is folded into the output layer,
 *   Wq[p][row(wi, a)][:] = sum_d w[wi][d] * W_out[p][a*D + d][:],  bq likewise from b_out   (fp32 accumulate, bf16 Wq),
 * so the last GEMM has ~n_w*A columns instead of A*D and psi[B,N,A,D] is never formed (GPI_w, sfdqn.py:215-240).
 * Row order (an internal contract between sfgpi_fold_gpi / sfgpi_step_prep and sfgpi_mlp_forward_tc; treat wq / bq as opaque):
 * reward vectors are interleaved in blocks of WB = 8 (4 when 4 <= n_w < 8, 1 below): row = (block*A + a)*WB + (wi mod WB), vectors
 * padded to a multiple of WB with zero rows, so that the epilogue's per-state scan runs WB independent max/argmax chains.
 * wq_out: bf16 [n_pol][sfgpi_gpi_fold_rows()][256]; bq_out: fp32 [n_pol][sfgpi_gpi_fold_rows()].
 */
int sfgpi_gpi_fold_rows(const sfgpi_net_desc *net, int32_t n_w);
int sfgpi_fold_gpi(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, const float *w, int32_t n_w,
                   int32_t w_diag, void *wq_out, float *bq_out, void *stream);
int sfgpi_mlp_forward_tc(const sfgpi_forward_args *args, const void *params_bf16, int32_t n_policies_total, const void *wq,
                         const float *bq, void *stream);
/*
 * Up to 3 independent tensor-core forwards in ONE launch (the train step's online psi(s), GPI on s' and target psi(s') are
 * each a fraction of a wave at the shipped sizes; together they fill the machine).  Same semantics per job as
 * sfgpi_mlp_forward_tc.
 */
typedef struct {
    sfgpi_forward_args args;
    const void *params_bf16;
    int32_t n_policies_total;
    const void *wq;
    const float *bq;
} sfgpi_forward_tc_job;
int sfgpi_mlp_forward_tc_jobs(const sfgpi_forward_tc_job *jobs, int32_t n_jobs, void *stream);

/*
 * Tensor-core backward (bf16 operands, fp32 accumulate), the mode-1 twin of sfgpi_mlp_backward: dgrad chain + split-K wgrad of
 * autograd's backward through psi (sfdqn.py:345, tsfdqn.py:645).  Reads the online rows' bf16 shadow (sfgpi_pack_bf16), the
 * bf16 activations saved by sfgpi_mlp_forward_tc (acts_bf16_out) and the sparse d_out of sfgpi_td_step (or, actions == NULL, a
 * dense d_out [B][n_pol][A*D] fp32, rounded to bf16 like every other operand); writes fp32 split
 * partials in library row layout for sfgpi_adam_step.  Scratch (caller-allocated, bf16): dz_bf16 [L-1][n_pol][B][256],
 * dzo_bf16 [n_pol][B][sfgpi_bwd_tc_out_pad()], xo_bf16 [B][64].  n_split must equal sfgpi_bwd_tc_splits(B, wanted).
 * Same shape limits and stated tolerance as sfgpi_mlp_forward_tc, and S <= 63.
 */
typedef struct {
    sfgpi_net_desc net;
    const void *params_bf16;
    int32_t n_policies_total;
    int32_t policy_lo, n_pol;
    const float *x;                 /* [B][S] */
    int32_t B;
    const void *acts_bf16;          /* [L-1][n_pol][B][256] */
    const void *relu_masks;         /* [L-1][n_pol][B][8] uint32 from sfgpi_mlp_forward_tc (relu_mask_out); NULL: signs from acts */
    const int64_t *actions;         /* [B]; NULL: d_out is dense */
    const float *d_out;             /* [n_pol][B][D]; dense: [B][n_pol][A*D] */
    void *dz_bf16;
    void *dzo_bf16;
    void *xo_bf16;
    float *grad_part;               /* [n_pol][n_split][row_stride] */
    int32_t n_split;
    int32_t xo_ready;               /* nonzero: xo_bf16 already holds [x | 1 | 0] (sfgpi_step_prep built it) -> one launch fewer */
    const void *expand_td;          /* optional sfgpi_td_args of the preceding variant-2 TD step run with defer_expand: its TSF
                                       expand (independent of the psi backward, consumed only by Adam) rides in the dgrad launch */
} sfgpi_backward_tc_args;

int sfgpi_bwd_tc_out_pad(const sfgpi_net_desc *net);
int sfgpi_bwd_tc_splits(int32_t B, int32_t want);
int sfgpi_mlp_backward_tc(const sfgpi_backward_tc_args *args, void *stream);

/*
 * Tensor-core modes at the REFERENCE's precision: tcgen05.mma kind::tf32 on fp32 operands (csrc/mlp_stream_tc.cu).
 *   SFGPI_PREC_TF32    one pass, operands rounded to nearest tf32 (stated tolerance 2e-3 on psi / q)
 *   SFGPI_PREC_TF32X3  3-pass split a_hi.b_hi + a_hi.b_lo + a_lo.b_hi, fp32 accumulation in TMEM: meets the fp32 mode's 1e-5
 * Both read hi (/ lo) fp32 operand shadows of the library rows produced by sfgpi_pack_f32 (parts = 1 for TF32, 2 for TF32X3):
 *   shadow   [parts][n_policies_total][sfgpi_bf16_rows_per_policy()][256]   W_0 | hidden W_l | W_out padded: the forward's operands
 *   shadow_t [parts][n_policies_total][L-2][256][256]  W_l^T, l = 1..L-2   (optional: the dgrad chain's operands)
 *   wout_t   [parts][n_policies_total][256][sfgpi_f32_out_pad()]  W_{L-1}^T (optional)
 * (buffers must be zero-initialised once by the caller: padding columns are never written).  Shapes: hidden widths == 256, S <= 31.
 * sfgpi_mlp_forward_stream takes the same jobs as sfgpi_mlp_forward_tc_jobs with params_bf16 -> shadow, wq / bq -> the output of
 * sfgpi_fold_gpi_f32 (wq fp32 [parts][n_pol][sfgpi_gpi_fold_rows()][256]), args.acts_bf16_out -> fp32 [parts][L-1][n_pol][B][256].
 */
#define SFGPI_PREC_FP32 0
#define SFGPI_PREC_BF16 1
#define SFGPI_PREC_TF32 2
#define SFGPI_PREC_TF32X3 3
int sfgpi_f32_out_pad(const sfgpi_net_desc *net);
int sfgpi_pack_f32(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, int32_t n_policies_total,
                   int32_t precision, float *shadow, float *shadow_t, float *wout_t, void *stream);
int sfgpi_fold_gpi_f32(const sfgpi_net_desc *net, const float *params, int32_t policy_lo, int32_t n_pol, const float *w, int32_t n_w,
                       int32_t w_diag, int32_t precision, float *wq_out, float *bq_out, void *stream);
int sfgpi_mlp_forward_stream(const sfgpi_forward_tc_job *jobs, int32_t n_jobs, int32_t precision, void *stream);
/*
 * Backward of the psi MLP in the tf32 modes (the twin of sfgpi_mlp_backward_tc): streaming dgrad chain on the transposed operand
 * shadows + split-K wgrad with MN-major fp32 operands (csrc/mlp_stream_tc.cu, csrc/mlp_wgrad_tf32.cu).  Scratch (caller-allocated
 * fp32, parts = 1 / 2): dz [parts][L-1][n_pol][B][256], dzo [parts][n_pol][B][sfgpi_f32_out_pad()], xo [parts][B][32].
 * actions == NULL: d_out is dense, [B][n_pol][A*D] fp32 (split into hi / lo like the sparse one).
 */
typedef struct {
    sfgpi_net_desc net;
    int32_t precision;              /* SFGPI_PREC_TF32 / SFGPI_PREC_TF32X3 */
    const float *shadow_t;          /* sfgpi_pack_f32 outputs for the ONLINE rows */
    const float *wout_t;
    int32_t n_policies_total, policy_lo, n_pol;
    const float *x;                 /* [B][S] */
    int32_t B;
    const float *acts;              /* [parts][L-1][n_pol][B][256] from sfgpi_mlp_forward_stream (acts_bf16_out) */
    const void *relu_masks;         /* [L-1][n_pol][B][8] uint32 from the forward (required for ReLU layers) */
    const int64_t *actions;         /* [B]; NULL: d_out is dense */
    const float *d_out;             /* [n_pol][B][D]; dense: [B][n_pol][A*D] */
    float *dz, *dzo, *xo;
    float *grad_part;               /* [n_pol][n_split][row_stride] */
    int32_t n_split;                /* == sfgpi_bwd_tc_splits(B, wanted) */
} sfgpi_backward_stream_args;
int sfgpi_mlp_backward_stream(const sfgpi_backward_stream_args *args, void *stream);

/*
 * Gradient of a loss with respect to the psi MLP's INPUT states (csrc/input_grad.cu), from the layer-0 pre-activation gradient dZ_0
 * that the backward entry points above leave in their scratch.  One state tensor feeds all n_pol nets, so the policies' terms add:
 *   dx[b][s] = sum_{p < n_pol} sum_{k < dims[1]} dZ0[p][b][k] * W0_{policy_lo+p}[k][s]        dx [B][S] fp32, overwritten
 * dz0 by precision (the backward's own scratch, read as it is):
 *   SFGPI_PREC_FP32    fp32 [n_pol][B][dims[1]]   sfgpi_backward_args.dz[0]; any hidden width and S
 *   SFGPI_PREC_BF16    bf16 [n_pol][B][256]       slab 0 of sfgpi_backward_tc_args.dz_bf16; S <= 63
 *   SFGPI_PREC_TF32    fp32 [n_pol][B][256]       hi, slab 0 of sfgpi_backward_stream_args.dz; S <= 31
 *   SFGPI_PREC_TF32X3  as TF32, plus lo at dz0 + dz0_part_stride floats (that scratch's part stride, (L-1)*n_pol*B*256); dZ0 = hi + lo
 * W_0 is read from the fp32 library rows and used as the mode's forward used it: rounded to bf16 (the sfgpi_pack_bf16 value) in
 * BF16, to tf32 (the sfgpi_pack_f32 hi value) in TF32, as stored in FP32 / TF32X3.  FFMA with fp32 accumulation; the policies are
 * summed in a fixed order without atomics, so two calls give the same bits.  One launch; B == 0 or n_pol == 0: none.  Needs
 * n_layers >= 2 (tensor-core modes: first hidden width 256).
 */
typedef struct {
    sfgpi_net_desc net;
    int32_t precision;              /* SFGPI_PREC_*: the mode of the backward that wrote dz0 */
    const float *params;            /* [N][row_stride] fp32 library rows (W_0 at net.w_off[0]) */
    int32_t policy_lo, n_pol;
    int32_t B;
    const void *dz0;                /* layouts above */
    int64_t dz0_part_stride;        /* SFGPI_PREC_TF32X3: floats from the hi to the lo part; ignored otherwise */
    float *dx;                      /* [B][S] */
} sfgpi_input_grad_args;
int sfgpi_mlp_input_grad(const sfgpi_input_grad_args *args, void *stream);

/*
 * Learned features (phi), SURVEY 8f N3: the reward-regression head of SFDQN.pre_train (sfdqn_phi.py:850-862).
 *   phi [B][D] = output of the PhiFunction MLP (sfdqn_phi.py:90-123; run it with sfgpi_mlp_forward, n_actions = 1),
 *   e_b = w . phi_b - r_b ;  loss = mean_b e_b^2 (= mse_loss(reward_batch, fit_w(phis)))
 *   d_out [B][D] = dLoss/dphi = (2/B) e_b w   -> feed to sfgpi_mlp_backward (actions all 0)
 *   dw_part [n_blocks][D] = per-CTA partials of dLoss/dw, loss_part [n_blocks][2] = {0, sum e^2} -> sfgpi_adam_step (segment
 *   with n_part = n_blocks; l2_scale = 1/B, beta_loss = 1 reduces the loss).  n_blocks = sfgpi_phi_head_partials(B).
 */
int sfgpi_phi_head_partials(int32_t B);
int sfgpi_phi_head(const float *phi, const float *w, const float *r, int32_t B, int32_t D, float *d_out, float *dw_part,
                   float *loss_part, void *stream);

/*
 * G4 joint psi / phi step (features/deep_phi.py:95-224 with the loss coefficient of agents/sfdqn_phi.py:152-165), the part between
 * the forwards and the backwards: with phi = phi_theta(cat[s, a, s']) [B][D] (carries gradient), cur = psi_i(s)[a], nxt =
 * psi^-_i(s')[a*], reward map fit_w = Linear(D, 1) WITH bias, loss coefficient c:
 *   targets = phi + gamma * nxt ;  psi_loss = sum (cur - targets)^2 / (B*A*D) ;  phi_loss = sum (w.phi + b - r)^2 / B
 *   loss = phi_loss + c * psi_loss                                                           (deep_phi.py:136-185)
 * Outputs: d_psi [B][D] = dLoss/dpsi(s)[a,:], d_phi [B][D] = dLoss/dphi (both losses), grad_small [D + 2] = (dLoss/dw | dLoss/db |
 * -dLoss/dc: the coefficient's Adam group has maximize=True), losses [4] = (loss, psi_loss, phi_loss, c before the step).
 * One CTA, deterministic reductions; B <= 4096 (the phi agents run at batch 32).
 */
typedef struct {
    int32_t B, A, D;
    const float *cur_sel, *next_sel, *phi;  /* [B][D] */
    const float *rs, *gammas;               /* [B] */
    const float *w, *bias, *coef;           /* [D], [1], [1] */
    float *d_psi, *d_phi;                   /* [B][D] */
    float *grad_small;                      /* [D + 2] */
    float *losses;                          /* [4] */
} sfgpi_g4_args;
int sfgpi_g4_head(const sfgpi_g4_args *args, void *stream);

/*
 * Target-task adaptation of the TSF agent, batch 1 (SURVEY 8f N1; tsfdqn.py:859-997).  psi / next_psi: [N][A][D] = get_successors(s)
 * / get_next_successors(s') of sfgpi_mlp_forward* for ONE state.
 *   sfgpi_target_q     q[a] = w . sum_j (omega_j / sum omega) psi_j[a,:]  (get_test_action's greedy branch, :864-871), q_out [A]
 *                      and / or action_out [1] = argmax (first maximal index; the packed keys' NaN rule); A <= 256
 *   sfgpi_target_adapt update_test_reward_mapper (:917-997) + scheduler.step() (:895) in one kernel: loss = MSE(tsf(s,a),
 *                      phi~ + gamma tsf^-(s',a')) + beta (w.phi~ - r)^2 + l1_coef |omega|_1 with phi~ = phi * (h(sum_j omega^_j g_j(s))
 *                      + h(sum_j omega^_j g_j(s'))); Adam (betas 0.9 / 0.999, eps 1e-8, torch op order) on w (lr_w, wd_w) and omega
 *                      (lr_omega * (1 - lr_omega_decay)^epoch, wd_omega); omega clamped to >= 1e-7; step and epoch advance on the
 *                      device.  losses [3] = (loss, reward loss, psi loss) as the reference returns them.
 */
typedef struct {
    int32_t N, A, D, G, S;
    const float *psi, *next_psi;            /* [N][A][D] */
    const float *g; int32_t g_stride;       /* [N][g_stride]: W[G][S] | b[G] */
    const float *h;                         /* W[D][G] | b[D] */
    const float *s, *s1;                    /* [S] */
    const float *phi;                       /* [D] */
    float r, gamma;
    int32_t a, a1;
    float beta, l1_coef, lr_w, wd_w, lr_omega, wd_omega, lr_omega_decay;
    float *w, *omegas;                      /* [D], [N]: updated in place */
    float *w_m, *w_v, *o_m, *o_v;           /* Adam moments */
    int32_t *step, *epoch;                  /* [1] each, device */
    float *losses;                          /* [3] */
} sfgpi_target_args;
int sfgpi_target_q(const float *psi, int32_t N, int32_t A, int32_t D, const float *omegas, const float *w, float *q_out,
                   int64_t *action_out, void *stream);
int sfgpi_target_adapt(const sfgpi_target_args *args, void *stream);

/*
 * G1's per-environment-step LMS rule on the raw reward vector (features/successor.py:146-167): w += alpha (r - phi . w) phi,
 * one tiny kernel instead of 4 - 5 eager launches; phi [D], r [1] device pointers.
 */
int sfgpi_lms_update(float *w, const float *phi, const float *r, int32_t D, float alpha, void *stream);

/*
 * Step prologue of a tensor-core train step in ONE launch: sfgpi_pack_bf16 for up to two row sets (online, target),
 * sfgpi_keys_fill, sfgpi_fold_gpi and the backward pass's xo = [x | 1 | 0] operand (bf16 [B][64]) -- five independent
 * elementwise passes that would otherwise be five launches on the step's dependent chain -- plus, optionally, the staging of the
 * step's host-resident inputs.  A part is skipped when its count is 0 / its pointer NULL.  Outputs are bit-identical to the
 * separate entry points.
 */
#define SFGPI_PREP_COPIES 6
typedef struct {
    sfgpi_net_desc net;
    const float *pack_params[2];    /* library rows to pack ...                  */
    void *pack_out[2];              /* ... into these bf16 shadows               */
    int32_t pack_lo[2], pack_n[2];  /* policy range of each pack (n = 0: skip)   */
    int64_t *keys;                  /* GPI keys to reset to INT64_MIN (NULL: skip) */
    int64_t n_keys;
    const float *fold_params;       /* sfgpi_fold_gpi arguments (fold_n = 0: skip) */
    int32_t fold_lo, fold_n;
    const float *w;
    int32_t n_w, w_diag;
    void *wq;
    float *bq;
    const float *x;                 /* [B][S] states of the online forward (NULL: skip); may be a pinned host address */
    int32_t B;
    void *xo_bf16;                  /* [B][64] */
    /* input staging: up to 6 plain copies src -> dst run as the first blocks of the same grid.  src may be PINNED HOST memory
     * (the kernel reads it over PCIe: a replay batch arriving from the host costs no cudaMemcpyAsync calls) or pageable host
     * memory (copied with cudaMemcpyAsync ahead of the launch); `x` may alias a copy_src; bytes = 0: skip */
    const void *copy_src[SFGPI_PREP_COPIES];
    void *copy_dst[SFGPI_PREP_COPIES];
    int64_t copy_bytes[SFGPI_PREP_COPIES];
    /* optional (TSF): M = Wh Wg, c = 2 (Wh bg + bh) of tsf_n policies from tsf_lo on, once per step instead of once per CTA of the
       TD kernel (h(g(s)) + h(g(s')) = M (s + s') + c, tsfdqn.py:621-623): tsf_g [.][tsf_g_stride] = W[G][S] | b[G] per policy,
       tsf_h = W[D][G] | b[D] (shared), tsf_mc out [tsf_n][D*S + D].  tsf_n = 0: skipped */
    const float *tsf_g;
    const float *tsf_h;
    float *tsf_mc;
    int32_t tsf_g_stride, tsf_G, tsf_lo, tsf_n;
} sfgpi_step_prep_args;
int sfgpi_step_prep(const sfgpi_step_prep_args *args, void *stream);
/* Kernels one sfgpi_step_prep call launches: 2 when the GPI fold is large (>= 4096 folded rows: it runs as its own launch), else 1. */
int sfgpi_step_prep_launches(const sfgpi_step_prep_args *args);

/*
 * Device-resident replay ring (ReplayBuffer.replay, sfdqn.py:54-80): gathers B picked transitions out of the packed ring
 *   ring [capacity][row_stride] fp32, row = [ s (S) | s' (S) | phi (D) | r | gamma | action ]
 * into the six tensors of a replay batch: states [B][S], actions [B] int64, rewards [B], phis [B][D], next_states [B][S],
 * gammas [B].  picks [B] int64 (device) are ring indices.
 */
typedef struct {
    const float *ring;
    int64_t row_stride;
    int32_t S, D, B;
    const int64_t *picks;
    float *states;
    int64_t *actions;
    float *rewards;
    float *phis;
    float *next_states;
    float *gammas;
} sfgpi_replay_args;
int sfgpi_replay_gather(const sfgpi_replay_args *args, void *stream);

/*
 * Command list: one foreign call runs a whole train step (or any other fixed sequence of the entry points above plus plain
 * copies) back to back on `stream`.  p[] / i[] carry the operands of op (see csrc/run.cu); argument structs are referenced,
 * not copied, so the caller patches input pointers in place between replays.
 */
#define SFGPI_OP_NOP 0
#define SFGPI_OP_H2D 1              /* p0 = dst (device), p1 = src (pinned host), i0 = bytes */
#define SFGPI_OP_D2H 2              /* p0 = dst (host), p1 = src (device), i0 = bytes */
#define SFGPI_OP_D2D 3
#define SFGPI_OP_KEYS_FILL 4        /* p0 = keys, i0 = n */
#define SFGPI_OP_PACK_BF16 5        /* p0 = net desc, p1 = params, p2 = out, i0 = policy_lo, i1 = n_pol */
#define SFGPI_OP_FOLD_GPI 6         /* p0 = net desc, p1 = params, p2 = w, p3 = wq, p4 = bq, i0 = policy_lo, i1 = n_pol, i2 = n_w, i3 = w_diag */
#define SFGPI_OP_FORWARD 7          /* p0 = sfgpi_forward_args */
#define SFGPI_OP_FORWARD_TC_JOBS 8  /* p0 = sfgpi_forward_tc_job[], i0 = n_jobs */
#define SFGPI_OP_TD 9               /* p0 = sfgpi_td_args */
#define SFGPI_OP_BACKWARD 10        /* p0 = sfgpi_backward_args */
#define SFGPI_OP_BACKWARD_TC 11     /* p0 = sfgpi_backward_tc_args */
#define SFGPI_OP_ADAM 12            /* p0 = sfgpi_adam_args */
#define SFGPI_OP_EVENT 13           /* p0 = cudaEvent_t: cudaEventRecord on the stream (timing probes around a command) */
#define SFGPI_OP_PEER_KEYS 14       /* p0 = sfgpi_peer_keys_args */
#define SFGPI_OP_SHARD_PACK 15      /* p0 = w, p1 = h, p2 = h_prev, p3 = x_local, i0 = nw, i1 = nh */
#define SFGPI_OP_PEER_UNPACK 16     /* p0 = sfgpi_peer_unpack_args */
#define SFGPI_OP_STEP_PREP 17       /* p0 = sfgpi_step_prep_args */
#define SFGPI_OP_PACK_F32 19        /* p0 = net desc, p1 = params, p2 = shadow, p3 = shadow_t, p4 = wout_t, i0 = policy_lo, i1 = n_pol, i2 = n_policies_total, i3 = precision */
#define SFGPI_OP_FOLD_GPI_F32 20    /* p0 = net desc, p1 = params, p2 = w, p3 = wq, p4 = bq, i0 = policy_lo, i1 = n_pol, i2 = n_w | w_diag << 31, i3 = precision */
#define SFGPI_OP_FORWARD_STREAM 21  /* p0 = sfgpi_forward_tc_job[], i0 = n_jobs, i1 = precision */
#define SFGPI_OP_BACKWARD_STREAM 22 /* p0 = sfgpi_backward_stream_args */
#define SFGPI_OP_KEYS_DECODE 23     /* p0 = keys, p1 = index_out, p2 = value_out, i0 = n */
typedef struct {
    int32_t op;
    void *p[5];
    int64_t i[4];
} sfgpi_cmd;
int sfgpi_run(const sfgpi_cmd *cmds, int32_t n, void *stream);

/*
 * Policy sharding (one process per GPU): everything the ranks exchange per train step besides the GPI keys travels in ONE
 * all-gather of x_local = [ w of the local policies (nw) | delta of the shared TSF h applied by the local optimizers (nh) ].
 * pack builds x_local (delta = h - h_prev); unpack turns the gathered x_all [world][nw + nh] into w_all [world * nw] (global
 * policy order), h = h_prev + sum_r delta_r (rank order, identical everywhere) and h_prev = h.  nh = 0 without TSF.
 */
int sfgpi_shard_pack(const float *w, int32_t nw, const float *h, const float *h_prev, int32_t nh, float *x_local, void *stream);
int sfgpi_shard_unpack(const float *x_all, int32_t world, int32_t nw, int32_t nh, float *w_all, float *h, float *h_prev,
                       void *stream);

/*
 * Peer-memory exchange (policy sharding on one NVSwitch node, one process per GPU): the two per-step exchanges of the sharded
 * train step -- the MAX reduce-scatter of the packed GPI keys (replaces dist.all_reduce(keys, MAX), SURVEY 8e "Collective --
 * training with GPI") and the all-gather of x_local = [w | delta h] (sfgpi_shard_pack / _unpack above) -- as kernels inside the
 * step's launch chain that signal, wait and PULL over NVLink from arenas every rank has mapped with CUDA IPC.
 *   sfgpi_peer_alloc   cudaMalloc + zero + cudaIpcGetMemHandle: the 64-byte handle is what ranks exchange (any transport)
 *   sfgpi_peer_open    cudaIpcOpenMemHandle with lazy peer access; sfgpi_peer_close / sfgpi_peer_free undo the two
 * flags[r] = rank r's flag block, uint64 [SFGPI_PEER_CHANNELS][SFGPI_MAX_PEERS], zero-initialised; flags[r][ch][q] is written by
 * rank q only (q = r: by the rank itself, ordering its own CTAs).  `epoch` must be > 0, identical on every rank for the same exchange and strictly increasing per channel; data
 * buffers are double-buffered by the caller on epoch parity.  A rank that waits 20 s for a peer traps (the CUDA context fails
 * loudly instead of hanging).
 */
#define SFGPI_MAX_PEERS 16
#define SFGPI_PEER_CHANNELS 4
#define SFGPI_PEER_CH_KEYS 0
#define SFGPI_PEER_CH_X 1
#define SFGPI_IPC_HANDLE_BYTES 64
typedef struct {
    int32_t world, rank;
    void *flags[SFGPI_MAX_PEERS];
} sfgpi_peer_ctx;
typedef struct {
    sfgpi_peer_ctx ctx;
    int64_t epoch;
    const int64_t *keys_all[SFGPI_MAX_PEERS];   /* rank r's keys [n_total][B] of this epoch (keys_all[rank] is local) */
    int32_t row_lo, n_rows, B;                  /* this rank's rows: keys_out[row][b] = max_r keys_all[r][row_lo + row][b] */
    int64_t *keys_out;                          /* [n_rows][B], local */
} sfgpi_peer_keys_args;
typedef struct {
    sfgpi_peer_ctx ctx;
    int64_t epoch;
    const float *x[SFGPI_MAX_PEERS];            /* rank r's x_local [nw + nh] of this epoch */
    int32_t nw, nh;
    float *w_all, *h, *h_prev;                  /* as sfgpi_shard_unpack */
    const float *pack_w;                        /* optional [nw]: fused sfgpi_shard_pack -- x[rank] = [pack_w | h - h_prev] is
                                                   written by this launch itself before it signals */
} sfgpi_peer_unpack_args;
int sfgpi_peer_alloc(int64_t bytes, void **dptr, void *ipc_handle_out);
int sfgpi_peer_open(const void *ipc_handle, void **dptr);
int sfgpi_peer_close(void *dptr);
int sfgpi_peer_free(void *dptr);
int sfgpi_peer_reduce_keys(const sfgpi_peer_keys_args *args, void *stream);
int sfgpi_peer_unpack(const sfgpi_peer_unpack_args *args, void *stream);

/* Runtime options.  Returns the previous value or -1 (unknown option).  Both move a choice the library otherwise makes
 * from the launch size between two code paths that compute the same bits; the tests set them to run the other path and
 * compare the two.
 *   "forward_chain"   which bf16 forward kernel runs: 0 = ping-pong tile pairs always (csrc/mlp_forward_tc.cu), 1 (default) =
 *                     the layer-pipelined single-tile kernel (csrc/mlp_chain_tc.cu) for launches of <= 148 tiles, 2 = always.
 *   "gpi_wide_min"    folded GPI output layers (n_w * A columns, n_w >= 8) of at least this many columns are scanned by the
 *                     32-column-window variant (gpi_scan_wide8, csrc/forward_tc.cuh) in the pair kernel; default 256. */
int sfgpi_set_option(const char *name, int32_t value);

/* Developer aid: the kernel-window trace.  While it is on (SFGPI_TRACE=1 in the environment, or sfgpi_trace_enable(1)) every
 * kernel of a train step records the %globaltimer of its first CTA entry, of the first CTA past its dependency wait and of its
 * last CTA exit -- the gaps BETWEEN the kernels of a step, which per-kernel timers do not show.  Slots: 0 prologue, 1 forward,
 * 2 TD, 3 dgrad, 4 wgrad, 5 Adam.  sfgpi_trace_read synchronises the device, copies [n_slots][3] uint64 ns (entry = all ones
 * for a kernel that did not run) into `out`, resets the windows and returns the slots written (0: tracing is off);
 * sfgpi_trace_dump prints the same to stderr. */
void sfgpi_trace_enable(int32_t on);
int sfgpi_trace_read(uint64_t *out, int32_t n_slots);
void sfgpi_trace_dump(void);

const char *sfgpi_last_error(void);
int sfgpi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SFGPI_H */
