/*
 * barvae.h -- C ABI of libbarvae.so: the B200 (sm_100a) kernels behind the bar-VAE train / decode hot path.
 *
 * The reference (KMU-AELAB-MusicProject/MusicGeneration_VAE-torch) has no native layer: every op on the path is a
 * stock torch.nn layer (SURVEY.md section 8b).  The seam this library sits under is therefore the set of ATen ops
 * the reference's nn.Modules dispatch; each entry point below names the reference lines whose work it replaces.
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch's allocator); the library never frees or
 *     retains one beyond the call; all scratch is passed in explicitly.
 *   - every call is asynchronous on the given stream (a cudaStream_t passed as void*).
 *   - return value: 0 = ok, otherwise a BVAE_ERR_* code; bvae_last_error() gives the message (thread local).
 *   - activations: NHWC, bf16, addressed as ptr[((n*H + h)*W + w)*pitch + c]; `pitch` (elements per pixel)
 *     may exceed C so that a branch can write straight into its slice of a concatenated tensor
 *     (torch.cat at graph/encoder.py:30, graph/decoder.py:100,145,208 is never materialised).
 *   - parameters and their gradients: fp32, in the reference's own state_dict layouts.
 */
#ifndef BARVAE_H_
#define BARVAE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BVAE_OK 0
#define BVAE_ERR_SHAPE 1
#define BVAE_ERR_ALIGN 2
#define BVAE_ERR_ARCH 3
#define BVAE_ERR_CUDA 4
#define BVAE_ERR_UNSUPPORTED 5

#define BVAE_MAX_TAPS 16
#define BVAE_MAX_PHASES 6

/* implementation selector for the contraction kernels */
#define BVAE_IMPL_AUTO 0  /* tcgen05 when the shape allows, else SIMT */
#define BVAE_IMPL_SIMT 1  /* CUDA-core reference kernel (debug / odd shapes such as C_in = 1) */
#define BVAE_IMPL_TC 2    /* tcgen05 + TMEM + TMA; error if the shape is not eligible */

int bvae_version(void);
const char* bvae_last_error(void);
/* number of kernels launched by this library since load / since the last reset (bench.py's gpu_launches) */
uint64_t bvae_launch_count(void);
void bvae_launch_count_reset(void);
/* kernels of this library launched by REPLAYING a captured CUDA graph do not pass through the entry points: the caller
 * that replays adds the number of launches it counted while capturing */
void bvae_launch_count_add(uint64_t n);
/* 1 if the current device is sm_100 (B200); kernels refuse to run elsewhere */
int bvae_device_ok(void);
/* name (with template arguments) of the kernel the calling thread's last bvae_conv_gemm / bvae_wgrad_gemm call launched:
 * lets bench.py attribute CUDA-event times to kernel instances ("conv_tc2_kernel<64,256,4,0>") for the per-kernel roofline */
const char* bvae_last_kernel(void);
/* Deterministic mode (default: env BVAE_DETERMINISTIC, else 0).  When on, every reduction of the FORWARD pass (InstanceNorm
 * statistics, CBAM pooling, BCE loss) runs in a fixed order -- shared-memory accumulations warp by warp, no cross-CTA float
 * atomics -- so two runs on the same inputs are bit-identical (slower; a diagnostic that separates summation-order noise from
 * races).  Weight gradients use one split per output tile (one ordered accumulation per element); the norm-block BACKWARD
 * reductions stay atomic (DESIGN.md section 7). */
void bvae_set_deterministic(int on);
int bvae_deterministic(void);
/* Norm-block kernel-variant switches kept for A/B measurements (DESIGN.md section 4.3): BVAE_NB_MLP, BVAE_NB_MODE, BVAE_NB_SPLIT,
 * BVAE_NB_FAST, BVAE_NB_SMALL (+ its thresholds BVAE_NB_SMALL_HW / BVAE_NB_SMALL_N).  Each is read per call as: the value set here,
 * else the environment variable of the same name, else its default; value < 0 removes the override.  Every variant is
 * parity-tested (tests/test_gpu_kernels.py::test_kernel_variants_*). */
void bvae_set_option(const char* name, int value);
int bvae_get_option(const char* name, int dflt);

/* ------------------------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution  (forward of Conv2d / ConvTranspose2d / Linear and their data gradients).
 *
 *   out[n, qy*osy+ooy, qx*osx+oox, co] = epi( sum_{t < ntaps} sum_{c < C}
 *                                              x[n, qy*sy + dy[t], qx*sx + dx[t], c] * w[co, t*C + c] )
 *   for qy < QH, qx < QW; out-of-range input pixels contribute zero (padding).
 *   epi(v) = act(v + bias[co]) (+ addend) (* act'(mask))  ->  bf16 or fp32 store.
 *
 * One call covers one "phase": a strided transposed convolution is 4 calls (sub-pixel decomposition), a
 * k == stride transposed convolution is one call per tap.  Replaces aten::convolution as dispatched by
 * nn.Conv2d (graph/encodingBlock.py:12-15,43-46,74-77,107-108; graph/decoder.py:79,122,172,175),
 * nn.ConvTranspose2d (graph/decoder.py:12-15,43-46,73-77,116-120), nn.Linear (graph/encoder.py:22,
 * graph/phrase_encoder.py:23, graph/decoder.py:166-167) and their convolution_backward data-gradient halves.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct bvae_conv_desc {
  const void* x;     /* bf16 NHWC [N, H, W, C], pitch x_pitch */
  const void* w;     /* bf16 [Cout, w_pitch] rows; this phase uses columns [0, ntaps*C) (K-major, tap-major) */
  void* y;           /* bf16 (or fp32 if out_f32) NHWC [N, OH, OW, Cout], pitch y_pitch */
  const float* bias; /* [Cout] or NULL */
  const void* addend; /* same geometry/dtype as y (pitch add_pitch) or NULL: out += addend */
  const void* mask;  /* bf16, same geometry as y (pitch mask_pitch) or NULL: out *= (mask > 0 ? 1 : mask_slope) */
  void* stats;       /* optional, 24*N*Cout bytes, zero before the first phase: the epilogue accumulates the
                        InstanceNorm statistics of the output -- double sum[N*Cout], double sumsq[N*Cout],
                        uint32 max key[N*Cout], uint32 min key[N*Cout] (order-preserving float keys) -- so that
                        bvae_nb_forward (stats_fused = 1) needs no statistics pass; see bvae_conv_stats_ok */
  int32_t N, H, W, C, x_pitch;
  int32_t Cout, w_pitch;
  int32_t ntaps;
  int32_t dy[BVAE_MAX_TAPS], dx[BVAE_MAX_TAPS];
  int32_t sy, sx;    /* input stride */
  int32_t QH, QW;    /* output grid of this phase */
  int32_t OH, OW, y_pitch;
  int32_t osy, osx, ooy, oox; /* output stride / offset of this phase */
  int32_t add_pitch, mask_pitch;
  int32_t act;       /* 0 none, 1 leaky-relu with `slope` (0 = ReLU) applied after bias */
  int32_t out_f32;
  float slope, mask_slope;
  /* Several phases in ONE call (all sub-pixel phases of a strided transposed convolution / of a strided
   * convolution's data gradient): nphase > 0, taps listed phase-major in dy/dx (ntaps = total), phase i uses
   * ph_ntaps[i] taps and weight columns starting at (taps before it)*C, writes at offset (ph_ooy[i], ph_oox[i]) on the
   * grid ph_QH[i] x ph_QW[i].  QH/QW/ooy/oox above are ignored then.  Tiles of the same input patch run back to back,
   * so the patch is read from HBM once for all phases.  nphase == 0: the single phase described above. */
  int32_t nphase;
  int32_t ph_ntaps[BVAE_MAX_PHASES], ph_ooy[BVAE_MAX_PHASES], ph_oox[BVAE_MAX_PHASES];
  int32_t ph_QH[BVAE_MAX_PHASES], ph_QW[BVAE_MAX_PHASES];
} bvae_conv_desc;

int bvae_conv_gemm(const bvae_conv_desc* d, int impl, void* stream);
/* 1 if bvae_conv_gemm(d, BVAE_IMPL_AUTO) can fuse the statistics (tcgen05 path, fp32 output, every M tile inside one
 * sample) */
int bvae_conv_stats_ok(const bvae_conv_desc* d);

/* ------------------------------------------------------------------------------------------------------------
 * Weight gradient of the same contractions:
 *   dw[(ra*Cs + rs)*T + tap_idx[t]] (+)= sum_{n, ay, ax} a[n, ay, ax, ra] * s[n, ay*sy + dy[t], ax*sx + dx[t], rs]
 * a = "anchor" tensor (dY for Conv2d/Linear, X for ConvTranspose2d), s = "shifted" tensor (the other one).
 * dw is fp32 in the reference parameter layout (Conv2d [Cout][Cin][kh*kw], ConvTranspose2d [Cin][Cout][kh*kw]);
 * the result is ACCUMULATED (atomically) -- zero it first for a plain gradient.
 * Replaces the weight-gradient half of aten::convolution_backward / addmm backward for the layers listed above.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct bvae_wgrad_desc {
  const void* a;  /* bf16 NHWC [N, AH, AW, Ca], pitch a_pitch */
  const void* s;  /* bf16 NHWC [N, SH, SW, Cs], pitch s_pitch */
  float* dw;
  float* scratch; /* optional fp32 [Ca*T*Cs], all zeros on entry and on exit: lets the tcgen05 kernel reduce with
                     16-byte vector atomics into a packed [ra][tap][rs] layout before unpacking into dw */
  int32_t N, AH, AW, Ca, a_pitch;
  int32_t SH, SW, Cs, s_pitch;
  int32_t sy, sx;
  int32_t ntaps, T;
  int32_t dy[BVAE_MAX_TAPS], dx[BVAE_MAX_TAPS], tap_idx[BVAE_MAX_TAPS];
} bvae_wgrad_desc;

int bvae_wgrad_gemm(const bvae_wgrad_desc* d, int impl, void* stream);

/* fp32 parameter (reference layout) -> bf16 GEMM operand:
 *   dst[r*dst_pitch + tp*Cc + c] = bf16(src[r*sr + c*sc + perm[tp]])   r < R, tp < T, c < Cc   */
int bvae_pack_weight(const float* src, void* dst, int R, int T, int Cc, int64_t sr, int64_t sc,
                     const int32_t* perm /* host array [T] */, int dst_pitch, void* stream);

/* The same repack for MANY parameters in one launch (all contraction weights of the model after each optimiser step;
 * replaces ~100 bvae_pack_weight launches).  Jobs are copied to the device when the plan is created; the plan keeps
 * the src/dst pointers, so it is valid while those buffers live.  `perm` must hold T entries. */
typedef struct bvae_pack_job {
  const float* src;
  void* dst;                        /* bf16 */
  int32_t R, T, Cc, dst_pitch;
  int64_t sr, sc;
  int32_t perm[BVAE_MAX_TAPS];
} bvae_pack_job;
typedef struct bvae_pack_plan bvae_pack_plan;
int bvae_pack_plan_create(const bvae_pack_job* jobs /* host */, int njobs, bvae_pack_plan** out);
int bvae_pack_plan_run(const bvae_pack_plan* plan, void* stream);
void bvae_pack_plan_destroy(bvae_pack_plan* plan);

/* column sums: out[c] += sum over rows of x[row*pitch + c]  (bias gradients; x bf16 or fp32) */
int bvae_colsum(const void* x, int x_f32, int64_t rows, int C, int pitch, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * "Norm block": InstanceNorm2d(affine) [+ CBAM] [+ residual] + (Leaky)ReLU on a raw convolution output.
 *
 *   u   = (y - mean_nc) * rstd_nc * gamma_c + beta_c                       (graph/encodingBlock.py:30,61,92,120)
 *   cb  = u * gc[n,c] * gs[n,h,w]                                          (graph/cbam.py:22-29,43-52,64-68)
 *         gc = sigmoid(W2 relu(W1 avgpool(u)) + W2 relu(W1 maxpool(u)))
 *         gs = sigmoid(conv3x3_{2->1}([mean_c(u*gc), max_c(u*gc)]))
 *   out = act( res_mode 0: u | 1: u + cb | 2: res + cb | 3: cb )
 * Replaces aten::instance_norm, adaptive_avg/max_pool2d, the 1x1 MLP convs, mean/max over C, cat, the 3x3
 * attention conv, sigmoid, mul, add and (leaky_)relu at every site listed in SURVEY.md section 8 rows a3-a14.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct bvae_nb_desc {
  int32_t N, H, W, C;
  int32_t y_pitch, out_pitch, res_pitch, dout_pitch, dy_pitch, dres_pitch;
  int32_t has_cbam, Cr, res_mode; /* res_mode: 0 u | 1 u + cbam(u) | 2 res + cbam(u) | 3 cbam(u) */
  int32_t y_f32;        /* raw conv output dtype: 1 = fp32 (default: survives |mean| >> std), 0 = bf16 */
  int32_t stats_fused;  /* 1: `stats` was filled by bvae_conv_gemm's epilogue (see bvae_conv_desc.stats) */
  float slope, eps;
  const void* y;        /* raw conv output [N,H,W,C] (forward only; not needed by backward) */
  void* uhat;           /* bf16 [N,H,W,C] dense: normalised activations, saved for backward; NULL in bvae_nb_forward = inference, not written */
  void* out;            /* bf16 block output */
  void* stats;          /* forward scratch, 24*N*C bytes */
  const void* res;      /* bf16 external residual (res_mode 2) */
  const float* gamma;   /* [C] */
  const float* beta;    /* [C] */
  const float* w1;      /* [Cr][C]  channel_attention.conv1.weight */
  const float* w2;      /* [C][Cr]  channel_attention.conv2.weight */
  const float* wsp;     /* [2][3][3] spatial_attention.conv.weight */
  /* saved per block (caller-allocated) */
  float* nc;            /* [N][C][8]: mean, rstd, a, b, gc, ext_u (max-pooled u), ext_uhat, spare */
  int32_t* nc_idx;      /* [N][C]: pixel index of the max-pooled element */
  float* sa;            /* [N][H*W][2]: mean_c, max_c of u*gc */
  int32_t* cidx;        /* [N][H*W]: argmax channel */
  float* gs;            /* [N][H*W] */
  /* backward */
  const void* dout;     /* bf16 grad wrt out */
  void* dy;             /* bf16 grad wrt y (also used as scratch for du) */
  void* dres;           /* bf16 grad wrt res (res_mode 2) or NULL */
  float* dgamma;        /* [C], accumulated */
  float* dbeta;         /* [C], accumulated */
  float* dw1;           /* accumulated */
  float* dw2;           /* accumulated */
  float* dwsp;          /* accumulated */
  float* bwd_nc;        /* scratch [N][C][4]: dgc, S1, S2, dmx  (zeroed by the call) */
  float* bwd_px;        /* scratch [N][H*W][4]: dq, dsa_mean, dsa_max, spare */
  float* bwd_h;         /* scratch [N][192]: per-sample channel-MLP factors (CBAM only) */
} bvae_nb_desc;

int bvae_nb_forward(const bvae_nb_desc* d, void* stream);
int bvae_nb_backward(const bvae_nb_desc* d, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * fit2 (1x1 conv 64->1) + sigmoid + BCE(mean, log clamp -100) [+ pitch-prior label smoothing] + the
 * non-differentiable missed-note count  (graph/decoder.py:175,220; graph/loss/bar_loss.py:23-33).
 *   x [rows, C] bf16 (rows = N*96*60), w [C] fp32, target [rows] fp32 {0,1}
 *   recon [rows] fp32 = sigmoid(x.w);  loss_out[0] += BCE sum / rows;  loss_out[1] += missed-note count
 * smoothing: 0 = pre-training (plain labels), 1 = 0.82*t + 0.1/60 + 0.08*prior[pitch], pitch = row % 60.
 * Backward: dx[row, c] = g[row] * w[c],  dw[c] += sum_row g[row]*x[row,c],
 *   g = gscale * (p - t') / max(p(1-p), 1e-12) * p(1-p)    (BCELoss backward then sigmoid backward, as autograd)
 * ------------------------------------------------------------------------------------------------------------ */
int bvae_fit_sigmoid_fwd(const void* x, int x_pitch, const float* w, int64_t rows, int C, float* logits,
                         float* recon, void* stream);
int bvae_bce_fwd(const float* recon, const float* target, int64_t rows, int smoothing, float* loss_out,
                 void* stream);
/* autograd's BCELoss backward alone: drecon[i] = gscale * (p - t') / max(p(1-p), 1e-12)   (gscale = dL / rows) */
int bvae_bce_bwd(const float* recon, const float* target, int64_t rows, int smoothing, float gscale, float* drecon,
                 void* stream);
int bvae_fit_sigmoid_bce_bwd(const void* x, int x_pitch, const float* w, const float* recon, const float* target,
                             const float* drecon /* NULL: use BCE grad with gscale */, float gscale, int smoothing,
                             int64_t rows, int C, void* dx, int dx_pitch, float* dw, void* stream);

/* reparameterise + KL  (old/graphs/models/bar_v1/encoder.py:60-63, old/graphs/losses/loss.py:16)
 *   z = mu + eps*exp(0.5*logvar);  kl_out[0] += -0.5*sum(1 + logvar - mu^2 - exp(logvar))
 *   backward: dmu = dz + gkl*mu ; dlogvar = dz*eps*0.5*exp(0.5*logvar) + gkl*0.5*(exp(logvar) - 1) */
int bvae_reparam_kl_fwd(const float* mu, const float* logvar, const float* eps, float* z, float* kl_out,
                        int64_t n, void* stream);
int bvae_reparam_kl_bwd(const float* mu, const float* logvar, const float* eps, const float* dz, float gkl,
                        float* dmu, float* dlogvar, int64_t n, void* stream);

/* torch.optim.Adam (agent/barGen.py:61-62,327,333) on ONE flat fp32 bucket holding every generator parameter
 * (p, g, m, v each contiguous, 16-byte aligned): p -= lr/(1-b1^t) * m / (sqrt(v)/sqrt(1-b2^t) + eps), g is
 * pre-multiplied by grad_scale (1/world_size when the bucket holds an NCCL sum).  16 B read + 12 B written/param. */
int bvae_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps,
                   int step, float grad_scale, void* stream);
/* The same update with the step-dependent scalars read from DEVICE memory, so that a captured CUDA graph of the whole
 * training step can be replayed unchanged: bvae_adam_hyper (host, no device work) fills out6 = {lr/(1-b1^t),
 * 1/sqrt(1-b2^t), b1, b2, eps, grad_scale}; the caller copies those 6 floats to hyper_dev on the stream before the launch
 * (or before the graph replay). */
void bvae_adam_hyper(float lr, float b1, float b2, float eps, int step, float grad_scale, float* out6);
/* ... or in one call: a one-thread kernel writes them (launch parameters are captured at launch time, so the host may run
 * any number of steps ahead of the device) */
int bvae_adam_hyper_upload(float lr, float b1, float b2, float eps, int step, float grad_scale, float* hyper_dev,
                           void* stream);
int bvae_adam_step_dev(float* p, const float* g, float* m, float* v, int64_t n, const float* hyper_dev, void* stream);

/* fp32 -> bf16 cast of a contiguous buffer (piano-roll inputs: [N,1,H,W] with C == 1 is already NHWC) */
int bvae_f32_to_bf16(const float* src, void* dst, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Bit-packed piano-rolls (SURVEY.md section 8f N3).  The reference moves every batch to the device as fp32
 * (data/bar_dataset.py:22-25 -> agent/barGen.py:134-141 -> .cuda() at :302-306) and reads every generated bar back
 * as fp32 (maker_bar.py:38-40).  Cells are binary, so one bit per cell is lossless: MSB first within a byte, cells
 * in C order -- the layout of numpy.packbits(x.reshape(-1)).
 *   bvae_unpack_bits: out_bf16[i] (encoder / phrase-encoder input, nullable) and out_f32[i] for i < nbits_f32 (the
 *     BCE target, nullable) = bit i of `bits`, as 0.0 / 1.0.  nbits_f32 is a multiple of 8 or equals nbits.
 *   bvae_threshold_pack: bit i of `bits` (nullable) = p[i] > threshold, and out_f32[i] (nullable) the same as
 *     0.0 / 1.0 -- torch.gt(pre_bar, 0.3).type(FloatTensor) of maker_bar.py:39 fused with the packing of the result.
 * Outputs 16-byte aligned; `bits` holds ceil(n / 8) bytes, unused low bits of the last byte are written as 0.
 * ------------------------------------------------------------------------------------------------------------ */
int bvae_unpack_bits(const void* bits, int64_t nbits, void* out_bf16, float* out_f32, int64_t nbits_f32,
                     void* stream);
int bvae_threshold_pack(const float* p, int64_t n, float threshold, void* bits, float* out_f32, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Bernoulli draw per piano-roll cell with temperature, from a counter-based stream (the torch.gt(., 0.3) of
 * maker_bar.py:39 replaced by a draw):
 *   p = 1.f / (1.f + expf(-(logit * inv_temperature))),  cell = (u < p) ? 1 : 0,  u = (float)(r >> 8) * 2^-24,
 *   r = word (i % 4) of Philox4x32-10(counter = {i / 4, bar_index, song lo32, song hi32}, key = {seed lo32, seed hi32}),
 *   i = cell index in the bar (0..5759, C order [96][60]), song = song_base + b for bar row b of `logits`.
 * A cell's draw depends only on (seed, song, bar_index, i): not on the batch size or the split of songs across calls.
 * p is fit_sigmoid_fwd's expression, so at inv_temperature 1 it equals the decoder's probability bit for bit.
 * A NaN logit gives 0, +inf gives 1, -inf gives 0.  inv_temperature finite and > 0 and bars >= 0, else
 * BVAE_ERR_SHAPE; logits and out_f32 16-byte aligned, else BVAE_ERR_ALIGN.
 * ------------------------------------------------------------------------------------------------------------ */
int bvae_bernoulli_sample(const float* logits /* [bars][5760] */, int64_t bars, float inv_temperature,
                          uint64_t seed, int64_t song_base, int32_t bar_index,
                          float* out_f32 /* [bars][5760] {0,1} */, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Per-bar score of a given piano-roll under the decoder's Bernoulli distribution at a temperature.  For each bar,
 * with l = logit * inv_temperature, p = 1.f / (1.f + expf(-l)) (the expression of bvae_bernoulli_sample) and t = 1 for
 * a nonzero target cell, else 0:
 *   nll_out[b]        = sum over the 5760 cells of (t ? softplus(-l) : softplus(l)),  softplus(x) = max(x,0) +
 *                       log1pf(expf(-|x|))  -- in nats; the ATen equivalent is, per bar,
 *                       binary_cross_entropy_with_logits(l, t, reduction='sum')
 *   counts_out[b][0..2] = { #(p > threshold and t), #(p > threshold), #t }   (true positives, predicted on, target on)
 * +-inf logits give the limits (t=1, l=+inf: 0; t=0, l=+inf: +inf); a NaN logit gives a NaN nll and is never counted
 * as predicted on.  No atomics, fixed summation order: a bar's result depends only on its logits and target, so a call
 * split into chunks returns the same bits as one call.  bars >= 0, inv_temperature finite and > 0, threshold finite,
 * else BVAE_ERR_SHAPE; logits and target 16-byte aligned, nll_out and counts_out 4-byte aligned, else BVAE_ERR_ALIGN.
 * ------------------------------------------------------------------------------------------------------------ */
int bvae_bar_score(const float* logits /* [bars][5760] */, const float* target /* [bars][5760] {0,1} */, int64_t bars,
                   float inv_temperature, float threshold, float* nll_out /* [bars] */,
                   int32_t* counts_out /* [bars][3] */, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * First and second moments of n latents of width d (row i at z + i*ld), accumulated in place in fp64 -- the statistics
 * of the Gaussian prior fitted to the encoder's output (prior.py):
 *   sum[j]     += sum_i z[i][j]
 *   gram[j][k] += sum_i z[i][j] * z[i][k]      for k >= j; entries with k < j are neither read nor written
 * Every product is formed in fp64 (exact for two fp32 values), and every output element adds its rows one at a time in
 * increasing row order, starting from the value already in memory.  No atomics, no split of the rows across CTAs, no
 * DMMA: a sequence of calls over consecutive chunks of rows gives the same bits as one call over all of them.
 * n >= 0, d >= 1, ld >= d, else BVAE_ERR_SHAPE; z 4-byte and sum / gram 8-byte aligned, else BVAE_ERR_ALIGN.  n == 0
 * writes nothing.
 * ------------------------------------------------------------------------------------------------------------ */
int bvae_latent_moments(const float* z /* [n][ld] */, int64_t n, int32_t d, int64_t ld, double* sum /* [d] */,
                        double* gram /* [d][d] row-major */, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * nn.BatchNorm2d(C, eps, momentum, affine) (+ optional (Leaky)ReLU) on an NHWC tensor with few channels: the norm of the
 * GAN-phase piano-roll discriminator (graph/bar_discriminator.py:19-23,69,113-114,153: BatchNorm2d(8..64, eps=1e-5,
 * momentum=0.01), OnOffFeature's default-momentum BatchNorm2d(8)) and of the Refiner (graph/refiner.py:13,20,37,43).
 * Replaces ATen's batch_norm / cudnn_batch_norm (+ relu) and their backward.
 *   training != 0: statistics over all P = N*H*W pixels of THIS rank (the reference does not synchronise them across ranks,
 *     SURVEY.md section 8e); running_mean / running_var (nullable) are updated with `momentum` and the unbiased variance.
 *   training == 0: running statistics.
 *   y = act(gamma * (x - mean) * rstd + beta);  backward: dx (bf16), dgamma += , dbeta += (both nullable).
 * C is a power of two <= 64.  `save` holds 4*C floats (mean, rstd written by forward; two sums by backward), `scratch`
 * bvae_bn_scratch_floats(C) floats.  Every reduction is two-stage with a fixed order: no float atomics, bit-reproducible.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct bvae_bn_desc {
  int64_t P;                     /* pixels: N * H * W */
  int32_t C, x_pitch, y_pitch, dy_pitch, dx_pitch;
  int32_t x_f32, y_f32, dy_f32;  /* element types: 1 = fp32, 0 = bf16 (dx is always bf16) */
  int32_t act;                   /* 1: (Leaky)ReLU with `slope` after the affine transform */
  int32_t training;
  float slope, eps, momentum;
  const void* x;                 /* raw input (kept by the caller for backward) */
  void* y;                       /* output; with act != 0 it must be bf16 (backward reads the mask from it) */
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  float* save;
  float* scratch;
  const void* dy;
  void* dx;
  float* dgamma;
  float* dbeta;
} bvae_bn_desc;
int bvae_bn_scratch_floats(int C);
int bvae_bn_forward(const bvae_bn_desc* d, void* stream);
int bvae_bn_backward(const bvae_bn_desc* d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BARVAE_H_ */
