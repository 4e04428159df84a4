/* libnfk — C-ABI of the B200 (sm_100a) normalizing-flow kernels.
 *
 * Drop-in boundary for the flow hot path of vklyukin/nf_distillation (pure-Python/PyTorch reference):
 *   models/layers.py  (ActNorm, InvertibleConv1x1, Conv2d, Conv2dZeros, Split2d, gaussian_*)
 *   models/flows.py   (FlowStep.normal_flow / reverse_flow, get_block_2d / get_block_1d)
 *   pl_module.py      (NFModel.loss: multi-level latent MSE KD)
 * Each entry point names the reference lines whose arithmetic it replaces.
 *
 * Conventions
 *   - plain C: raw DEVICE pointers + sizes, `void* stream` is a cudaStream_t; no torch types.
 *   - the caller owns and allocates every buffer; nothing here allocates, synchronises or keeps global state.
 *   - every function returns NFK_OK (0) or a negative NFK_ERR_* code; kernels are stream-ordered and re-entrant.
 *   - fp32 tensors are contiguous NCHW ("z path"); coupling-network activations are pixel-major bf16
 *     matrices [pixels, channels] ("h path"), pixels = B*H*W in (b, y, x) order.
 */
#ifndef NFK_H_
#define NFK_H_

#ifdef __cplusplus
extern "C" {
#endif

#define NFK_OK 0
#define NFK_ERR_SHAPE (-1)  /* unsupported / inconsistent sizes */
#define NFK_ERR_ALIGN (-2)  /* pointer or leading dimension not 16-byte aligned */
#define NFK_ERR_ARG (-3)    /* missing / invalid argument */
#define NFK_ERR_LAUNCH (-4) /* CUDA launch failure */
#define NFK_ERR_DRIVER (-5) /* tensor-map encode / driver entry point failure */

/* Epilogues of nfk_gemm_nt_bf16 */
#define NFK_EPI_F32 0            /* out fp32  = acc (+ bias[col])                                   */
#define NFK_EPI_BIAS_RELU_BF16 1 /* out bf16  = relu(acc + bias[col])   (Conv2d+ActNorm+ReLU, folded);
                                    aux (optional) <- 1-bit mask (out > 0), word-major [N/32][ldaux >= M] words */
#define NFK_EPI_MASK_BF16 2      /* out bf16  = acc * mask(aux);  colsum[col] += column sums   (ReLU backward) */

int nfk_version(void);

/* ---- tensor-core GEMM tiles (tcgen05 + TMEM + TMA) --------------------------------------------------------
 * out[M,N] = A[M,K] * B[N,K]^T, A/B bf16 row-major (K contiguous), fp32 accumulate in TMEM.
 * Replaces the cuDNN/cuBLAS calls behind nn.Conv2d in models/layers.py:209,226 (Conv2d) and :249,259
 * (Conv2dZeros) — 3x3 convs arrive here as im2col / col2im GEMMs, 1x1 convs directly — and their dgrads.
 * K % 64 == 0, N % 16 == 0, lda/ldb/ldo % 8 == 0. */
int nfk_gemm_nt_bf16(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K, int epi,
                     void* out, long long ldo, const float* bias, const void* aux, long long ldaux, float* colsum,
                     void* stream);

/* Diagnostics: when buf != NULL ([grid][8] int64 on the device) the NT GEMM records, per CTA, cycles of the MMA
 * issuer {total, waiting for a free accumulator, waiting for operands, tiles} and of epilogue warp 0 {waiting for the
 * accumulator, draining it}. NULL switches it off. */
int nfk_gemm_set_prof(void* buf);

/* out[Mo,No] (fp32, caller-zeroed) += sum_k A[k,Mo] * B[k,No]; A/B bf16 row-major [Kpix, ld]. Weight gradients
 * of the coupling convs (autograd of nn.Conv2d in models/layers.py:209,249), split-K over pixels with
 * red.global.add. No % 64 == 0. */
int nfk_gemm_tn_bf16(const void* A, long long lda, const void* B, long long ldb, int Mo, int No, int Kpix,
                     float* out, long long ldo, int sm_count, void* stream);

/* ---- parameter-space prep ("K0"): every FlowStep of a model in one launch -----------------------------------
 * Items are read on the host at launch time (they travel in the kernel parameter block), so the arrays may be
 * temporaries; the device pointers inside them must stay valid until the stream reaches the kernel.
 *
 * nfk_invconv_prep_batch: one CTA per item builds the fused ActNorm o InvertibleConv1x1 matrix of one FlowStep
 * (models/layers.py:376-397 get_weight + :101-142), C <= 104:
 *   forward (reverse=0):  outW = W diag(exp(logs)), outb = outW * an_bias, W = P (L o tril + I)(U o triu + diag(s))
 *   inverse (reverse=1):  outW = diag(exp(-logs)) W^-1 (triangular solves in shared memory), outb = -an_bias
 *   out_sl[0] = +-(sum(an_logs) + sum(log_s))   (multiply by H*W for the per-sample log-det)
 *   transpose=1 selects the 1-D convention z = x @ W (models/layers.py:410-411).
 *   weight != NULL selects the non-LU branch (models/layers.py:366-375): in-kernel Gauss-Jordan slogdet/inverse;
 *   lower, upper, log_s, p, sign_s are then unused.
 * nfk_invconv_prep_bwd_batch: chain rule of that prep in either direction, (dWf, dbf, g_ld[B] or NULL) -> gradients
 * of actnorm.{bias,logs} and invconv.{lower,upper,log_s} (or invconv.weight); the inverse direction goes through
 * dW = -W^-T dW^-1 W^-T. dWf has row stride dWf_ld >= C, fwd.outW must hold the forward's outW, `pixels` = H*W (1 in
 * 1-D) scales the log-det gradient. Outputs are overwritten. */
typedef struct nfk_invconv_item {
  const float *an_bias, *an_logs, *lower, *upper, *log_s, *p, *sign_s, *weight;
  int C, reverse, transpose;
  float *outW, *outb, *out_sl;
} nfk_invconv_item;
typedef struct nfk_invconv_bwd_item {
  nfk_invconv_item fwd;
  const float* dWf;
  int dWf_ld;
  const float* dbf;
  const float* g_ld; /* [B] or NULL */
  int B;
  float pixels;
  float *d_bias, *d_logs, *d_lower, *d_upper, *d_log_s, *d_weight;
} nfk_invconv_bwd_item;
int nfk_invconv_prep_batch(int n, const nfk_invconv_item* items, void* stream);
int nfk_invconv_prep_bwd_batch(int n, const nfk_invconv_bwd_item* items, void* stream);

/* nfk_coupling_prep_batch: one grid row of CTAs per item turns the coupling-network weights of one FlowStep into bf16
 * GEMM operands with the ActNorm affine (models/layers.py:223-228) and the Conv2dZeros exp(3*logs) scale (:257-260)
 * folded in. K1p / K3p = 9*cin / 9*cout rounded up to 64.
 *   B1 [hid,K1p] (k = tap*cin+ci), B2 [hid,hid], B3 [K3p,hid] (row = tap*cout+co), bias1..3 the folded biases;
 *   with_transposed = 1 also writes B1T, B2T, B3T (the transposes the dgrads read).
 * nfk_coupling_prep_bwd_batch maps the gradients of those operands back to the reference parameters. */
typedef struct nfk_coupling_item {
  const float *w1, *b1, *l1, *w2, *b2, *l2, *w3, *b3, *l3;
  int cin, hid, cout, K1p, K3p, with_transposed;
  void *B1, *B1T, *B2, *B2T, *B3, *B3T;
  float *bias1, *bias2, *bias3;
} nfk_coupling_item;
typedef struct nfk_coupling_bwd_item {
  nfk_coupling_item fwd; /* parameters and sizes; the operand / bias outputs are not read */
  const float *dB1, *dbias1, *dB2, *dbias2, *dB3, *dbias3;
  float *dw1, *db1, *dl1, *dw2, *db2, *dl2, *dw3, *db3, *dl3;
} nfk_coupling_bwd_item;
int nfk_coupling_prep_batch(int n, const nfk_coupling_item* items, void* stream);
int nfk_coupling_prep_bwd_batch(int n, const nfk_coupling_bwd_item* items, void* stream);

/* ---- fp32 z path of a 2-D FlowStep (models/flows.py:142-202) ------------------------------------------------
 * y = Wf x + bf per pixel (ActNorm + invconv, models/layers.py:129-142,404-421); ld_out = ld_in + H*W*sl[0];
 * col = bf16 im2col (3x3, pad 1) of y[:, :C/2] -> [B*H*W, K1p] for the first coupling conv.
 * Wf == NULL: im2col of x only (inverse pass). C in {12,24,48,96}. */
int nfk_affine1x1_fwd(const float* x, const float* Wf, const float* bf, const float* sl, float* y, void* col,
                      int K1p, const float* ld_in, float* ld_out, int B, int C, int H, int W, void* stream);

/* h = col2im(P) + bias3 (last conv of the coupling net as per-tap products P [B*H*W, K3p], column = tap*C+co);
 * shift = h[0::2], s = sigmoid(h[1::2] + 2); forward y2 = (y2 + shift) * s, ld += sum log s
 * (models/flows.py:160-168); reverse y2 = y2 / s - shift, ld -= sum log s (:185-193). y updated in place. */
int nfk_coupling_fwd(const float* P, int K3p, const float* bias3, float* y, float* hsave, float* ld, int B, int C,
                     int H, int W, int reverse, void* stream);

int nfk_coupling_bwd(const float* g_out, const float* g_ld, const float* z_out, const float* hsave, float* dy,
                     void* dhcol, int K3p, float* dbias3, int B, int C, int H, int W, void* stream);

int nfk_affine1x1_bwd(const float* dy, const float* dcol, int K1p, const float* x, const float* Wf, float* dx,
                      float* dWf, float* dbf, int B, int C, int H, int W, void* stream);

/* Backward of the INVERSE coupling (models/flows.py:185-193: zc2 = z2 / s - shift, ld -= sum log s), same layout and
 * shape limits as nfk_coupling_bwd: g_zc = dL/dzc [B,C,H,W] (zc = the post-coupling tensor, z_out of the forward kernel
 * run with reverse = 1), hsave its saved (shift, logit) pairs, g_ld [B]. Writes dz (z2 half dL/dz2 = g_zc2 / s, z1 half
 * = g_zc1 -- the coupling net's share is added by nfk_col2im_add), the bf16 im2col of dh = (-g_zc2,
 * -(g_zc2 * (zc2 + shift) + g_ld) * (1 - s)) [B*H*W, K3p] and dbias3 += sum dh (dbias3 zeroed by the caller). */
int nfk_coupling_inv_bwd(const float* g_zc, const float* g_ld, const float* zc, const float* hsave, float* dz,
                         void* dhcol, int K3p, float* dbias3, int B, int C, int H, int W, void* stream);

/* dz[:, :C/2] += col2im(dcol) in place: the input gradient of the coupling net's first conv (3x3, pad 1) from the dgrad
 * GEMM's output dcol [B*H*W, K1p] fp32 (column = tap*(C/2) + ci), for the inverse pass whose conv reads z1 directly. */
int nfk_col2im_add(const float* dcol, int K1p, float* dz, int B, int C, int H, int W, void* stream);

/* ---- Split2d (models/layers.py:293-313), prior / bpd (models/kd_flows.py:134-150), KD MSE (pl_module.py:266-282) */
int nfk_split2d_fwd(const float* x, const float* w, const float* bias, const float* logs, float* z1_out, float* ld,
                    int B, int C, int H, int W, void* stream);
int nfk_split2d_rev(const float* z1, const float* w, const float* bias, const float* logs, const float* eps,
                    float temperature, float* out, int B, int C, int H, int W, void* stream);
int nfk_split2d_bwd(const float* x, const float* w, const float* bias, const float* logs, const float* g_z1,
                    const float* g_ld, float* dx, float* dw, float* dbias, float* dlogs, int B, int C, int H, int W,
                    void* stream);
/* Split2d with the following SqueezeLayer folded in (models/layers.py:32-44,316-327): z1_sq_out (optional,
 * [B, 4*C/2, H/2, W/2]) receives the space-to-depth copy of z1 in the same pass; the backward reads the gradient of
 * that squeezed tensor (g_z1_sq, optional) through the same index map and adds it to g_z1's. */
int nfk_split2d_squeeze_fwd(const float* x, const float* w, const float* bias, const float* logs, float* z1_out,
                            float* z1_sq_out, float* ld, int B, int C, int H, int W, void* stream);
int nfk_split2d_squeeze_bwd(const float* x, const float* w, const float* bias, const float* logs, const float* g_z1,
                            const float* g_z1_sq, const float* g_ld, float* dx, float* dw, float* dbias, float* dlogs,
                            int B, int C, int H, int W, void* stream);
/* First kernel of the 2-D flow (csrc/preproc.cu): data/src/utils.py:7-18 preprocess (when src is raw uint8 pixels:
 * floor(u8 / 2^(8-n_bits)) / 2^n_bits - 0.5; src_is_u8 == 0: src is fp32 and already preprocessed) + the dequantisation
 * noise of models/utils.py:26-41 (noise: U(0, 1/2^n_bits) drawn by the caller, optional) + the first SqueezeLayer
 * (models/layers.py:32-44): x_out [B,C,H,W] = v + noise (optional; may alias an fp32 src: in-place like the reference),
 * sq_out [B,4C,H/2,W/2] = its space-to-depth copy (optional). W % 4 == 0, H even. */
int nfk_dequant_squeeze(const void* src, int src_is_u8, int n_bits, const float* noise, float* x_out, float* sq_out,
                        int B, int C, int H, int W, void* stream);
int nfk_prior_bpd_fwd(const float* z, const float* mean, const float* logs, const float* logdet, int B, int n,
                      float scale, float* out, void* stream);
int nfk_prior_bpd_bwd(const float* z, const float* mean, const float* logs, const float* g_bpd, int B, int n,
                      float scale, float* dz, float* dlogdet, void* stream);
int nfk_kd_mse_fwd(const float* s, const float* t, int B, int n, float scale, float* acc, void* stream);
int nfk_kd_mse_bwd(const float* s, const float* t, const float* g, int B, int n, float scale, float* ds,
                   int accumulate, void* stream);

/* ---- last conv of the coupling net fused with the coupling (models/layers.py:231-260 Conv2dZeros +
 * models/flows.py:150-171 / :173-190): P^T = B3 * h2^T on tcgen05 with whole images as the N tile, col2im over the nine
 * taps, bias, then z2 <- (z2 + shift) * sigmoid(logit + 2) (reverse: z2 / sigmoid - shift) in place on y's upper C/2
 * channels, ld[b] += (-)sum log sigmoid. h2 [B*H*W, hid] bf16, B3 [K3p, hid] bf16 (rows tap*C + c, as built by
 * nfk_coupling_prep_batch), hsave (optional, [B*H*W, C] fp32) keeps the conv output for nfk_coupling_bwd.
 * Supported shapes (nfk_pconv_coupling_supported): C = 12 with maps of 256 pixels (W <= 16) or <= 128 pixels, C = 24
 * with <= 64 pixels, C = 48 with <= 32 pixels; H, W powers of two; hid % 64 == 0. */
int nfk_pconv_coupling_supported(int C, int H, int W, int hid);
int nfk_pconv_coupling_fwd(const void* h2, const void* B3, int K3p, const float* bias3, float* y, float* hsave,
                           float* ld, int B, int C, int H, int W, int hid, int reverse, void* stream);

/* ---- first conv of the coupling net, input gradient, fused with its col2im and nfk_affine1x1_bwd
 * (csrc/dgrad_col2im.cu): P^T = B1T * dpre1^T on tcgen05 with whole images as the N tile, then per pixel
 * dys = dy + col2im(P) on the y1 half (dy on the y2 half), dx = W'^T dys, dWf += dys x^T, dbf += sum dys.
 * dpre1 [B*H*W, hid] bf16 (the masked gradient at the first conv's output), B1T [K1p, hid] bf16 (rows tap*(C/2) + ci,
 * as built by nfk_coupling_prep_batch), K1p = round_up(9*C/2, 64); dy, x, dx [B,C,H,W] fp32, Wf [C,C]; dWf, dbf
 * are accumulated (zeroed by the caller). dx is bit-identical to nfk_gemm_nt_bf16 (NFK_EPI_F32) + nfk_affine1x1_bwd.
 * Supported shapes (nfk_conv1_dgrad_affine_bwd_supported): C = 12 with maps of <= 256 pixels, C = 24 with <= 128,
 * C = 48 with <= 64; H, W powers of two; hid % 64 == 0. */
int nfk_conv1_dgrad_affine_bwd_supported(int C, int H, int W, int hid);
int nfk_conv1_dgrad_affine_bwd(const void* dpre1, const void* B1T, int K1p, const float* dy, const float* x,
                               const float* Wf, float* dx, float* dWf, float* dbf, int B, int C, int H, int W, int hid,
                               void* stream);

/* ---- 1-D (tabular) FlowStep, fused (is_1d branches of models/flows.py:37-52,142-202, models/layers.py:410-411) --
 * Weights are packed once per optimiser step by nfk_flow1d_pack from the fused affine (nfk_invconv_prep_batch
 * with transpose=1, forward or inverse direction) and the six nn.Linear layers of get_block_1d:
 *   PF: per layer WT [nin][nout8] + bias [nout8] (forward), PB: per layer W [nout][nin8] (backward).
 * nfk_flow1d_sizes reports the block sizes and the per-layer offsets of the gradient block G
 * (dW_l [nout][nin8] at offG, db_l at offGB). x / y / dx are [B, D] row-major, cond is [B, Cc] (y_onehot). */
/* 1 when the step's weights (six Linear layers + the fused affine) and a sample tile fit in shared memory: for the
 * inference kernel (hidden widths up to 88 at D = 63), and with training != 0 also for the activation-saving
 * forward and the backward (which holds the weights and their gradient block: widths up to 48), else 0. */
int nfk_flow1d_supported(int D, int Cc, int hid, int training);
int nfk_flow1d_sizes(int D, int Cc, int hid, int* total_fwd, int* total_bwd, int* total_grad, int* n_act,
                     int* offsets);
int nfk_flow1d_pack(const float* Wf, const float* bf, const float* const* w, const float* const* b, int D, int Cc,
                    int hid, float* PF, float* PB, void* stream);
/* reverse=0: y = coupling(affine(x)), ld_out = ld_in + sl + sum log s;  reverse=1: y = affine_inv(coupling^-1(x)),
 * ld_out = ld_in + sl - sum log s (PF / sl built with reverse=1). acts (optional, [B, 5*hid + 2*D2]) keeps the MLP
 * activations for nfk_flow1d_bwd. */
int nfk_flow1d_fwd(const float* x, const float* cond, const float* PF, const float* sl, float* y, const float* ld_in,
                   float* ld_out, float* acts, int B, int D, int Cc, int hid, int reverse, void* stream);
/* Backward of nfk_flow1d_fwd. x_in = the step's input, y_out = the step's output (read when reverse=0: its first
 * D//2 features are the coupling MLP's input, its last features the coupled values), acts as saved by the forward.
 * dx [B, D]; G (pre-zeroed, nfk_flow1d_sizes layout) accumulates the parameter gradients. */
int nfk_flow1d_bwd(const float* x_in, const float* cond, const float* acts, const float* PB, const float* y_out,
                   const float* g_out, const float* g_ld, float* dx, float* G, int B, int D, int Cc, int hid,
                   int reverse, void* stream);
/* y = W x + b on [B, D] rows (stand-alone ActNorm1d / InvertibleConv1x1, models/layers.py:129-142,404-421). */
int nfk_affine_rows(const float* x, const float* Wf, const float* bf, const float* sl, float* y, const float* ld_in,
                    float* ld_out, int B, int D, float pixels, void* stream);

/* Same GEMM with an explicit tile width and, per n-tile, the k-block range [kb_begin, kb_end) (64 columns each)
 * that is not structurally zero — MADE's degree-sorted masks make the hidden weight block-triangular. */
int nfk_gemm_nt_bf16_ranged(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K, int epi,
                            void* out, long long ldo, const float* bias, const void* aux, long long ldaux,
                            float* colsum, int bn, const int* kb_begin, const int* kb_end, void* stream);

/* ---- MAF / MADE (no reference code exists — README.md:7 only; Papamakarios et al. 2017) ----------------------
 * masks from degrees: m1[o][i] = deg1[o] >= i+1, m2[o][k] = deg2[o] >= deg1[k], m3[r][k] = (r % D)+1 > deg2[k];
 * weights w1 [H,D], w2 [H,H], w3 [2D,H] (rows: mu then alpha) -> masked bf16 operands (and transposes). */
int nfk_made_prep(const float* w1, const float* w2, const float* w3, const int* deg1, const int* deg2, int D, int H,
                  int Dp, int N3p, void* B1, void* B1T, void* B2, void* B2T, void* B3, void* B3T, int with_t,
                  void* stream);
int nfk_made_prep_bwd(const float* dB1, const float* dB2, const float* dB3, const int* deg1, const int* deg2, int D,
                      int H, int Dp, float* dw1, float* dw2, float* dw3, void* stream);
int nfk_rows_to_bf16(const float* x, int B, int D, int Dp, void* xb, void* stream);
/* u = (x - mu) exp(-alpha), ld_out = ld_in - sum alpha; u is written in reversed feature order when flip != 0. */
int nfk_made_affine_fwd(const float* x, const float* out, int N3p, float* u, void* ub, int Dp, const float* ld_in,
                        float* ld_out, int B, int D, int flip, void* stream);
int nfk_made_affine_bwd(const float* x, const float* out, int N3p, const float* g_u, const float* g_ld, float* dx,
                        void* dout, float* db3, int B, int D, int flip, void* stream);
/* pass i of the sequential inverse: x[:, i] = u[:, i] exp(alpha_i) + mu_i */
int nfk_made_inv_update(float* x, void* xb, int Dp, const float* u_in, const float* out, int N3p, const float* ld_in,
                        float* ld_out, int B, int D, int i, int flip, int last, void* stream);
/* The whole D-step inverse of one MADE layer in ONE launch (csrc/maf_inverse.cu): a warp keeps x and the hidden
 * activations of its 16 samples in shared memory and finalises every hidden unit once, in degree order (~ one forward
 * pass of work, not D); a producer warp streams each job's weights through a shared-memory byte ring (one
 * cp.async.bulk per job). Three steps:
 *  1. nfk_made_inverse_jobs — HOST code (host pointers, no GPU): cnt1/cnt2 [D+1] = number of layer-1 / layer-2 hidden
 *     units with degree <= d (degrees sorted ascending). Returns the number of jobs of one sample tile and, when
 *     cap >= that number, writes 8 int32 per job: {phase (0: layer-1 tile pair, 1: layer-2 tile pair, 2: (mu, alpha))
 *     | second 8-row tile present << 2 | 16-wide k-chunks << 3, first row (phase 2: d), byte offset in the kernel's
 *     weight ring, jobs back to the latest job occupying any of those bytes, offset / 16 in the packed weight
 *     stream, bytes / 16, (push) bit mask of the 8-row output tiles the job's units feed, (push) d + 1 when x_d is
 *     finished right after this job (such a step has no (mu, alpha) job of its own)}. Call with cap = 0 to size.
 *     Depends on the degrees only.
 *     push = 1 (needs nfk_made_inverse_push_supported and degrees that change only on multiples of 8 units, else
 *     NFK_ERR_SHAPE): the PUSH kernel — layer-2 activations never reach shared memory, each finished 16-unit tile
 *     pair is multiplied straight into running (mu | alpha) sums kept in registers.
 *  2. nfk_made_inverse_pack — packs the masked bf16 operands of nfk_made_prep (B1 [H,Dp], B2 [H,H], B3 [N3p,H]) into
 *     the weight stream (sum of the jobs' bytes, 128-byte aligned, zero-initialised by the caller), job after job in
 *     shared-memory layout. jobs = the DEVICE copy of the table (16-byte aligned). Redo when the weights change.
 *  3. nfk_made_inverse_resident — u_in is in the layer's output order (reversed when flip != 0); x [B,D];
 *     ld_out = ld_in + sum alpha (either may be NULL); b1/b2 [H], b3 [>= 2D] fp32; mtiles: 16-sample tiles per warp
 *     of the pull kernel (1 or 2; 0 = choose). _supported: 1 if the shapes fit (H, Dp multiples of 64). */
int nfk_made_inverse_resident_supported(int D, int H, int Dp);
int nfk_made_inverse_push_supported(int D, int H, int Dp, int N3p);
int nfk_made_inverse_jobs(const int* cnt1, const int* cnt2, int D, int H, int Dp, int N3p, int push, int* jobs,
                          int cap);
int nfk_made_inverse_pack(const int* jobs, int njobs, const void* B1, const void* B2, const void* B3, int N3p, int D,
                          int H, int Dp, int push, void* wstream, void* stream);
int nfk_made_inverse_resident(const float* u_in, const void* wstream, const float* b1, const float* b2,
                              const float* b3, const int* jobs, int njobs, int push, int N3p, float* x,
                              const float* ld_in, float* ld_out, int B, int D, int H, int Dp, int flip, int mtiles,
                              void* stream);
/* Gradients of the inverse: given g_x [B,D] (input order) and g_ld [B] (NULL = 0) for x, ld_out = inverse(u_in, ld_in),
 * ONE reverse sweep d = D-1 .. 0 gives g_u [B,D] (output order), g_ld_in = g_ld, and dout [B,N3p] bf16 =
 * [mubar | alphabar | 0] with db3 += its column sums; dout is the upstream of the forward's parameter chain at x
 * (the dgrad / wgrad GEMMs of nfk_made_affine_bwd's dout). out [B,N3p] fp32 and the ReLU masks m1, m2 (word-major
 * [H/32][B], the EPI_BIAS_RELU_BF16 aux output) come from the forward recomputed at x. db3 must be zeroed.
 *  nfk_made_inv_bwd_update — pass d of the D-pass form: c [B, ldc] fp32 = the network's input gradient for the dout
 *     rows finished so far (NULL at d = D-1); writes g_u[:, d], dout[:, d], dout[:, D+d] and adds to db3. dout must be
 *     zero-initialised before pass D-1.
 *  nfk_made_inverse_bwd_jobs / _pack / _resident — the one-launch form (csrc/maf_inverse.cu), the mirror of the pull
 *     kernel with the same three steps: the HOST planner (same cnt1/cnt2 as nfk_made_inverse_jobs, same 8 int32 per
 *     job; [6] = the job's first 16-wide k-chunk; push form does not exist), the pack of the transposed operands
 *     B1T [Dp,H], B2T [H,H], B3T [H,N3p] of nfk_made_prep (with_t = 1), and the launch (mtiles as above).
 *     _supported: 1 if the shapes fit (H, N3p multiples of 64). */
int nfk_made_inv_bwd_update(const float* c, int ldc, const float* g_x, const float* g_ld, const float* out, int N3p,
                            const float* u_in, float* g_u, void* dout, float* db3, int B, int D, int d, int flip,
                            void* stream);
int nfk_made_inverse_bwd_supported(int D, int H, int N3p);
int nfk_made_inverse_bwd_jobs(const int* cnt1, const int* cnt2, int D, int H, int N3p, int* jobs, int cap);
int nfk_made_inverse_bwd_pack(const int* jobs, int njobs, const void* B1T, const void* B2T, const void* B3T, int D,
                              int H, int N3p, void* wstream, void* stream);
int nfk_made_inverse_bwd_resident(const float* g_x, const float* g_ld, const float* out, const void* m1,
                                  const void* m2, const float* u_in, const void* wstream, const int* jobs, int njobs,
                                  float* g_u, void* dout, float* db3, int B, int D, int H, int N3p, int flip,
                                  int mtiles, void* stream);

/* Fused conv#1 -> conv#2 of the coupling network: h2 = relu(relu(col*B1^T + b1)*B2^T + b2) in ONE kernel (CTA
 * pairs; h1 stays in tensor memory as the tcgen05 A operand of conv#2; csrc/cnet_ts.cu). col [M,K1p] bf16, B1 [512,K1p],
 * B2 [512,512] bf16 (nfk_coupling_prep_batch), h2 [M,512] bf16. Training additionally passes h1 [M,512] and the two
 * 1-bit ReLU mask buffers (word-major, [16][ldmask >= M]); inference passes NULL for them.
 * nfk_cnet_fused_supported: 1 if the kernels take hidden width hid and first-GEMM depth K (K1p / K3p): hid = 512 and
 * K a multiple of 64 up to 448 (the GEMM-1 A tile must leave shared memory for a weight ring of two slots). The entry
 * points return NFK_ERR_SHAPE otherwise; callers run the two nfk_gemm_nt_bf16 GEMMs instead. */
int nfk_cnet_fused_supported(int hid, int K);
int nfk_cnet_set_prof(void* buf); /* diagnostics: per-CTA cycle counters of the MMA issuer ([grid][8] int64) or NULL */
int nfk_cnet_fwd_fused(const void* col, int K1p, const void* B1, const void* B2, const float* bias1,
                       const float* bias2, void* h1, void* h2, void* mask1, void* mask2, long long ldmask, int M,
                       int hid, void* stream);
/* The same pipeline for the BACKWARD chain of the coupling net (student training): d2 = relu'(h2) .* (dhcol B3T^T) —
 * the Conv2dZeros input gradient through the ReLU mask of h2 — stays in tensor memory as the A operand of
 * d1 = relu'(h1) .* (d2 B2T^T); both are written out as bf16 [M, 512] (the weight-gradient GEMMs read them) and their
 * column sums are added into dbias2 / dbias1 (fp32 [512], caller-zeroed; NULL = not needed). dhcol [M, K3p] bf16
 * (nfk_coupling_bwd), B3T [512, K3p], B2T [512, 512] bf16 (nfk_coupling_prep_batch, transposed operands), masks as
 * written by nfk_cnet_fwd_fused / nfk_gemm_nt_bf16 (word-major, [16][ldmask >= M]). Replaces two nfk_gemm_nt_bf16
 * calls with NFK_EPI_MASK_BF16 (autograd of models/flows.py:25-34). Shapes: nfk_cnet_fused_supported(hid, K3p). */
int nfk_cnet_bwd_fused(const void* dhcol, int K3p, const void* B3T, const void* B2T, const void* mask_h2,
                       const void* mask_h1, long long ldmask, void* dpre2, void* dpre1, float* dbias2, float* dbias1,
                       int M, int hid, void* stream);
/* Same kernel for MADE's masked linears: the second weight matrix is block lower triangular (degree-sorted hidden
 * units), so for output channels [0, 256) only its first kb2_end_half0 k-blocks of 64 input channels are non-zero;
 * the remaining B2 tiles of that half are neither loaded nor multiplied (1 <= kb2_end_half0 <= 8; 8 = dense). */
int nfk_cnet_fwd_fused_ranged(const void* col, int K1p, const void* B1, const void* B2, const float* bias1,
                              const float* bias2, void* h1, void* h2, void* mask1, void* mask2, long long ldmask,
                              int M, int hid, int kb2_end_half0, void* stream);

/* ---- the tail of the KD training step (csrc/loss_optim.cu) -------------------------------------------------------
 * NFModel.loss (pl_module.py:257-320) in ONE launch: per sample
 *     kd[b]   = (1/L) sum_l mean_i (s_l[b,i] - t_l[b,i])^2                          (pl_module.py:266-282)
 *     nll[b]  = -(logdet[b] + sum_i log N(z_last[b,i]; mean_i, exp(logs_i))) * nll_scale
 *               (models/layers.py:10-23, models/kd_flows.py:134-150; prior rows NULL = zeros), or nll_in[b] when
 *               z_last is NULL (objective already computed by the model's forward)
 *     res[b]  = (w_nll nll + w_kd kd + w_perc perc[b]) * sample_w[b]                (pl_module.py:306-313)
 * and means[4] = batch means of (nll, kd, perc, res) (pl_module.py:315-320), added up in a fixed order by the last
 * CTA to finish (deterministic). nll_out / kd_out ([B], optional) receive the per-sample terms. scratch:
 * nfk_kd_nll_loss_scratch_floats(B) floats. The backward takes the gradient of the four means (device, [4]) plus
 * optional per-sample gradients of nll / kd and writes ds_l for every level with a non-NULL ds pointer, dz_last,
 * dlogdet (or dnll_in), dperc. Up to NFK_LOSS_MAX_LEVELS levels; the struct is read on the host. */
#define NFK_LOSS_MAX_LEVELS 8
typedef struct {
  const float* s[NFK_LOSS_MAX_LEVELS]; /* student taps [B, n_l] */
  const float* t[NFK_LOSS_MAX_LEVELS]; /* teacher taps [B, n_l] */
  float* ds[NFK_LOSS_MAX_LEVELS];      /* backward only: gradient of s_l (NULL = not needed) */
  int n[NFK_LOSS_MAX_LEVELS];
  int L;
} nfk_loss_levels;
int nfk_kd_nll_loss_scratch_floats(int B);
int nfk_kd_nll_loss_fwd(const nfk_loss_levels* levels, const float* z_last, int nz, const float* prior_mean,
                        const float* prior_logs, const float* logdet, float nll_scale, const float* nll_in,
                        const float* perc, const float* sample_w, float w_nll, float w_kd, float w_perc, int B,
                        float* nll_out, float* kd_out, float* means, float* scratch, void* stream);
int nfk_kd_nll_loss_bwd(const nfk_loss_levels* levels, const float* z_last, int nz, const float* prior_mean,
                        const float* prior_logs, float nll_scale, const float* sample_w, float w_nll, float w_kd,
                        float w_perc, int B, const float* g_means, const float* g_nll, const float* g_kd,
                        float* dz_last, float* dlogdet, float* dnll_in, float* dperc, void* stream);

/* Gradient clipping + optimiser on FLAT fp32 buffers (train.py:46 gradient_clip_val, pl_module.py:348-363 Adam /
 * Adamax): nfk_grad_sqnorm writes nfk_optim_partials() per-CTA partial sums of |g|^2 and adds one to *step (device
 * int, optional); nfk_adam_step re-adds the partials in a fixed order, scales the gradient by
 * min(1, max_norm / (norm + 1e-6)) (max_norm <= 0: no clipping) and applies torch.optim.Adam's (adamax != 0:
 * Adamax's) update with bias correction from *step. norm_out (optional) receives the unclipped norm. */
int nfk_optim_partials(void);
int nfk_grad_sqnorm(const float* g, long long n, float* partials, int* step, void* stream);
int nfk_adam_step(float* p, const float* g, float* m, float* v, long long n, const float* partials, const int* step,
                  float max_norm, float lr, float beta1, float beta2, float eps, float weight_decay, int adamax,
                  float* norm_out, void* stream);

/* ---- fp32-class coupling network on the bf16 tiles: "bf16x3" precision mode (csrc/split3.cu) ---------------------
 * The reference's convolutions are fp32 (models/layers.py:209,249). Each fp32 operand is split a = hi + lo into two
 * bf16 numbers and a*b ~= hi*hi + hi*lo + lo*hi (2^-16 relative) is computed by the SAME tensor-core GEMMs in one pass
 * over K-concatenated operands: activations as [hi | hi | lo] (pattern 0), weights as [hi | lo | hi] (pattern 1).
 * `pattern` selects the operand layout: 0 = A [h|h|m], 1 = B [h|m|h] (three terms, 2^-16); 2 = A [h|h|h|m|m|l],
 * 3 = B [h|m|l|h|m|h] (six terms, 2^-24: used for the forward pre-activations, whose signs are the ReLU masks).
 *   nfk_split3_rows      src fp32 [rows, lds] (first Ksrc columns; zero padded to K) -> out bf16 [rows, terms*K]
 *   nfk_im2col3x3_split3 3x3 'same' im2col (k = tap*Cc + c, zero padded to Kp) of an NCHW channel slice (layout 0) or a
 *                        pixel-major [M, Cc] matrix (layout 1); flip != 0 mirrors the taps (transposed conv);
 *                        pattern 0 or 2 -> [M, terms*Kp]
 *   nfk_act_split3       mode 0: relu(pre); mode 1: pre where gate > 0 (gate: bf16, row stride ldg); pattern 0 or 2
 *                        -> [M, terms*N], and colsum[n] += column sums of the fp32 result (bias gradients)
 *   nfk_coupling_bwd_f32 backward of the affine coupling (models/flows.py:160-168) with an fp32 pixel-major dh [M, C]
 *   nfk_coupling_inv_bwd_f32  backward of the INVERSE coupling (models/flows.py:185-193), the fp32-dh form of
 *                        nfk_coupling_inv_bwd: g_zc = dL/dzc, zc = the post-coupling tensor, hsave its (shift, logit)
 *                        pairs, g_ld [B] -> dz (z1 half = g_zc1, z2 half = g_zc2 / s), dh [M, C] (shift, logit
 *                        interleaved), dbias3 += column sums of dh (zeroed by the caller). C in {12, 24, 48, 96} */
int nfk_split3_rows(const float* src, long long lds, long long rows, int K, int Ksrc, int pattern, void* out,
                    void* stream);
int nfk_im2col3x3_split3(const float* src, int layout, int Ctot, int c0, int Cc, int B, int H, int W, int flip,
                         int Kp, int pattern, void* out, void* stream);
int nfk_act_split3(const float* pre, long long M, int N, int mode, const void* gate, long long ldg, int pattern,
                   void* out, float* colsum, void* stream);
int nfk_coupling_bwd_f32(const float* g_out, const float* g_ld, const float* z_out, const float* hsave, float* dy,
                         float* dh, float* dbias3, int B, int C, int H, int W, void* stream);
int nfk_coupling_inv_bwd_f32(const float* g_zc, const float* g_ld, const float* zc, const float* hsave, float* dz,
                             float* dh, float* dbias3, int B, int C, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NFK_H_ */
