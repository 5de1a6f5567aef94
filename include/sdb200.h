/* sdb200 — C ABI of the B200 (sm_100a) kernel library behind the Stable-Diffusion denoising hot path.
 *
 * The reference (dnnhhuy/stable-diffusion-pytorch) is pure Python/PyTorch and has NO FFI of its own;
 * every entry point below replaces a span of eager PyTorch calls in the reference, cited as
 * file:line relative to the reference root.  The Python host (stable-diffusion-pytorch_b200/) binds
 * these with ctypes; INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; all pointers are DEVICE pointers unless stated.
 *   - every function returns int: 0 = ok, <0 = error (SDK_ERR_*); text via sdk_last_error().
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*), never synchronise,
 *     never allocate: graph-capturable.  Scratch memory is caller-provided.
 *   - activations are NHWC ("rows x channels", rows = B*H*W); dtype codes: 0 = fp32, 1 = bf16.
 *   - handles are not thread-safe; use one stream per caller thread.
 */
#ifndef SDB200_H
#define SDB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDK_OK 0
#define SDK_ERR_ARG (-1)
#define SDK_ERR_CUDA (-2)
#define SDK_ERR_UNSUPPORTED (-3)
#define SDK_F32 0
#define SDK_BF16 1

/* ---- library ------------------------------------------------------------------------------ */
const char* sdk_last_error(void);
int sdk_version(void);
/* stream-ordered memset to zero (graph-capturable) */
int sdk_zero(void* ptr, int64_t bytes, void* stream);
/* out[0]=SM count, out[1..2]=compute capability, out[3]=max opt-in shared memory per block (of the current device) */
int sdk_device_info(int* out, int n);
/* programmatic dependent launch for all kernels (1 = on; default off): kernel N+1's prologue overlaps kernel N's tail */
int sdk_set_pdl(int enabled);
/* 1: all kernels request the max-shared-memory L1 carve-out (0 = driver heuristic, default; measured no difference) */
int sdk_set_uniform_carveout(int enabled);

/* ---- sampler: fused CFG blend + scheduler update (models/diffusion.py:233-236) ------------------
 * coef_table: [T][8] fp32 per-timestep scalars built by the host sampler; the timestep is read from
 * t_dev[0] (device int64) when t_dev != NULL, else t_host.  eps_c == NULL -> no CFG blend.
 * DDIM  replaces models/scheduler/ddim.py:58-87 ; prediction_type 0 = epsilon, 1 = v_prediction.
 * DDPM  replaces models/scheduler/ddpm.py:62-82 (noise = the randn draw of :80, caller-supplied). */
int sdk_ddim_step(const float* x, const float* eps_u, const float* eps_c, float cfg_scale,
                  const float* noise, float* out, int64_t n, const float* coef_table, int T,
                  const int64_t* t_dev, int64_t t_host, int prediction_type, void* stream);
int sdk_ddpm_step(const float* x, const float* eps_u, const float* eps_c, float cfg_scale,
                  const float* noise, float* out, int64_t n, const float* coef_table, int T,
                  const int64_t* t_dev, int64_t t_host, void* stream);
/* Inpainting loop body after the UNet (models/diffusion.py:387-398) in one pass: model output ordered [cond ; uncond] and blended as
 * s*(c-u)+c (eps_u == NULL: no CFG), orig = VAE-encoded image re-noised to the step's timestep with that prediction
 * (forward_process, ddim.py:46-55; orig_batch 1 broadcasts), kept wherever mask[pixel] == 0, then the DDIM update.
 * x, out: [batch][channels][hw] fp32 (may alias); mask: [hw] bytes, non-zero = region to repaint. */
int sdk_ddim_inpaint_step(const float* x, const float* eps_c, const float* eps_u, float cfg_scale,
                          const float* orig, int64_t orig_batch, const uint8_t* mask, float* out,
                          int64_t batch, int64_t channels, int64_t hw, const float* coef_table, int T,
                          const int64_t* t_dev, int64_t t_host, int prediction_type, void* stream);
/* the same loop body with the DDPM update (the reference's inpaint also takes sampler='ddpm', models/diffusion.py:314-316;
 * ddpm.py:62-82); noise = the randn draw of ddpm.py:80, [batch][channels][hw] */
int sdk_ddpm_inpaint_step(const float* x, const float* eps_c, const float* eps_u, float cfg_scale,
                          const float* orig, int64_t orig_batch, const uint8_t* mask, const float* noise, float* out,
                          int64_t batch, int64_t channels, int64_t hw, const float* coef_table, int T,
                          const int64_t* t_dev, int64_t t_host, void* stream);
/* DPM-Solver++(2M) (diffusers' DPMSolverMultistepScheduler, dpmsolver++ / midpoint): the same CFG blend and x0 prediction as
 * sdk_ddim_step, then x' = A*x + B*x0 + C*(x0 - history), the C term only where the table row flags it (column 7) and
 * hist_valid != 0 (history is not read otherwise).  history: [n] fp32, the previous step's x0 prediction, replaced by this
 * step's.  x and out may alias.  The table is the DPMSolverSampler's: it depends on the whole timestep grid. */
int sdk_dpmpp_step(const float* x, const float* eps_u, const float* eps_c, float cfg_scale, float* history, int hist_valid,
                   float* out, int64_t n, const float* coef_table, int T, const int64_t* t_dev, int64_t t_host,
                   int prediction_type, void* stream);
/* the inpainting loop body of sdk_ddim_inpaint_step with the DPM-Solver++(2M) update of sdk_dpmpp_step;
 * history: [batch][channels][hw] */
int sdk_dpmpp_inpaint_step(const float* x, const float* eps_c, const float* eps_u, float cfg_scale,
                           const float* orig, int64_t orig_batch, const uint8_t* mask, float* out,
                           int64_t batch, int64_t channels, int64_t hw, const float* coef_table, int T,
                           const int64_t* t_dev, int64_t t_host, int prediction_type, float* history, int hist_valid,
                           void* stream);
/* models/scheduler/ddim.py:46-55 — per-sample timesteps t_dev[batch] */
int sdk_forward_process(const float* x0, const float* noise, float* out, int64_t batch, int64_t per_sample,
                        const float* coef_table, int T, const int64_t* t_dev, void* stream);
/* models/diffusion.py:111-113 — one-step x0 = (x - sigma*eps)/alpha */
int sdk_x0_from_eps(const float* x, const float* eps, float sigma, float alpha, float* out, int64_t n, void* stream);

/* device-side walk of the (host-built) timestep grid: t_out[0] = table[counter[0]++]  (models/diffusion.py:223) */
int sdk_next_timestep(const int64_t* table, int n, int* counter, int64_t* t_out, void* stream);
/* out[0:row_elems] = table[counter[0] + delta][:] (NaN when out of range): per-step row of a table precomputed for the whole
 * timestep grid -- the loop uses it for the time-embedding projections, which depend only on the timestep (unet.py:182-183,209-220) */
int sdk_gather_row(const float* table, int64_t row_elems, int n_rows, const int* counter, int delta, float* out, void* stream);

/* ---- normalisation / layout (models/unet/unet.py:66,102-108,157,160,250,343,399) ------------- */
int64_t sdk_groupnorm_workspace_bytes(int B, int HW);
/* GroupNorm(32) statistics over the channel-concat [src0 | src1] (src1 may be NULL with C1 = 0);
 * stats = [B][32][2] (mean, rstd).  workspace: sdk_groupnorm_workspace_bytes, zeroed once. */
int sdk_groupnorm_stats(const float* src0, int C0, const float* src1, int C1, int B, int HW, float eps,
                        float* stats, void* workspace, void* stream);
/* y = (x-mean)*rstd*gamma+beta, optional SiLU, written as out_dtype; raw_out (optional) receives the
 * un-normalised concat in the same dtype (operand of the ResBlock's 1x1 shortcut conv). */
int sdk_groupnorm_apply(const float* src0, int C0, const float* src1, int C1, int B, int HW,
                        const float* stats, const float* gamma, const float* beta, int silu,
                        void* out, void* raw_out, int out_dtype, void* stream);
/* GroupNorm apply fed by per-channel (sum, sum of squares) tables cs0 [B][C0][2], cs1 [B][C1][2] (double) of the sources --
 * accumulated by the producing GEMM's epilogue (sdk_tc_gemm_set_stats) or written by sdk_channel_stats -- instead of a statistics
 * pass over the tensor (what the bf16 step program uses; the group fold of nn.GroupNorm, unet.py:156,160,65,398, happens in
 * the kernel's prologue). */
int sdk_groupnorm_apply_cs(const float* src0, int C0, const double* cs0, const float* src1, int C1, const double* cs1,
                           int B, int HW, float eps, const float* gamma, const float* beta, int silu,
                           void* out, void* raw_out, int out_dtype, void* stream);
/* per-channel (sum, sum of squares) of an fp32 [B][HW][C] tensor, ACCUMULATED into out [B][C][2] (double; zero it first) */
int sdk_channel_stats(const float* src, int B, int HW, int C, double* out, void* stream);
/* statistics + apply in ONE cooperative launch; same workspace as sdk_groupnorm_stats */
int sdk_groupnorm_fused(const float* src0, int C0, const float* src1, int C1, int B, int HW, float eps,
                        const float* gamma, const float* beta, int silu, void* out, void* raw_out, int out_dtype,
                        void* workspace, void* stream);
/* statistics + apply in ONE launch, one thread-block cluster per sample, DSMEM reduction (optional mode SDB200_GN_MODE=cluster;
 * the bf16 step program takes its statistics from the producing GEMM's epilogue instead: sdk_groupnorm_apply_cs) */
int sdk_groupnorm_cluster(const float* src0, int C0, const float* src1, int C1, int B, int HW, float eps,
                          const float* gamma, const float* beta, int silu, void* out, void* raw_out, int out_dtype,
                          void* stream);
int sdk_layernorm(const float* x, const float* gamma, const float* beta, float eps, void* out,
                  int out_dtype, int64_t rows, int C, void* stream);
/* out[r][:] = softmax(scale * in[r][:]) over rows of a materialised fp32 score matrix (cols %% 4 == 0, <= 16384): the single-head
 * head_dim = 512 attention of the VAE decoder (models/vae/vae.py:55-80), whose Q K^T and P V products run as sdk_tc_gemm launches */
int sdk_softmax_rows(const float* in, void* out, int out_dtype, int64_t rows, int cols, float scale, void* stream);
/* ---- text encoder front end (models/clip/openclip.py:53-71, clip.py:37-57) and MLP activation ------- */
/* out[r][:] = tok_emb[ids[r]][:] + pos_emb[r %% S][:]   (rows = B*S token ids, int64) */
int sdk_embed_tokens(const int64_t* ids, const float* tok_emb, const float* pos_emb, float* out,
                     int64_t rows, int S, int C, int vocab, void* stream);
/* elementwise activation of an fp32 tensor, written as out_dtype: kind 1 = exact-erf GELU (openclip.py:78), 2 = QuickGELU
 * x*sigmoid(1.702x) (activation_fn.py:4-9) */
int sdk_activation(const float* in, void* out, int out_dtype, int64_t n, int kind, void* stream);
/* fp32 NHWC -> out_dtype NHWC, nearest upsample by `up` (1 or 2)  (unet.py:250) */
int sdk_cast_upsample(const float* src, void* dst, int out_dtype, int B, int H, int W, int C, int up, void* stream);
/* dst[b][p][c] = src[b % B_src][c][p]: NCHW latent -> NHWC, with latent.repeat(2,...) (diffusion.py:228) folded in */
int sdk_nchw_to_nhwc(const float* src, float* dst, int B_src, int B_dst, int C, int HW, void* stream);

/* ---- time embedding (unet.py:209-220 and the per-ResBlock Linear(SiLU(t_emb)) :182-183) ---- */
/* out[i][0:half] = cos(t_i f_j), out[i][half:] = sin(t_i f_j), f_j = exp(-ln(1e4) j/half) */
int sdk_time_sinusoid(const int64_t* t_dev, int n, int dim, float* out, void* stream);
/* y[i][r] = act_out( dot(W[r][:], act_in(x[i][:])) + bias[r] ); act codes: 0 none, 1 SiLU.  W dtype fp32|bf16. */
int sdk_gemv(const void* W, int w_dtype, const float* bias, const float* x, float* y,
             int n, int R, int K, int act_in, int act_out, void* stream);

/* ---- implicit-GEMM convolution / linear --------------------------------------------------------
 * out[m][n] = epilogue( sum_{tap,c} A(m,tap,c) * W[n][tap*Cin + c] ),  m = (b*Hout + oy)*Wout + ox.
 * A is the channel-concat of up to two NHWC sources (skip concat, unet.py:343), optionally read
 * through a nearest 2x upsample (unet.py:250), with ksize 1|3, stride 1|2, zero pad ksize/2.
 * A Linear is ksize=1 on a [1][1][rows] "image".  Weights are K-major [N][ksize*ksize*Cin].
 * Epilogue: + bias[n] + tbias[b*tb_stride + n] + residual[m][n]; geglu: columns are (value, gate)
 * pairs and out[m][j] = v * gelu_erf(g)  (models/activation_fn.py:17-20); out as NHWC or NCHW. */
typedef struct SdkConvParams {
    const void* src0; const void* src1;   /* NHWC activations, in_dtype */
    const void* weight;                   /* [N][K] K-major, w_dtype == in_dtype */
    const float* bias;                    /* [N] or NULL */
    const float* tbias;                   /* per-sample additive term or NULL */
    const float* residual;                /* [M][N_out] fp32 or NULL */
    void* out;
    int64_t tb_stride;                    /* 0: one row broadcast over the batch */
    int C0, C1;
    int B, Hin, Win, Hout, Wout;
    int ksize, stride, upsample;
    int N;                                /* GEMM N (2*N_out when geglu) */
    int in_dtype, out_dtype;
    int out_nchw, geglu;
} SdkConvParams;
/* exact fp32 path (FFMA); also serves shapes the tensor-core path does not take (Cin = 4). in_dtype must be fp32. */
int sdk_conv_gemm_f32(const SdkConvParams* p, void* stream);
/* conv_in (unet.py:256): 3x3 / pad 1 / Cin = 4 on the fp32 NHWC latent x [B][H][W][4], w_t [3][3][4][N] (transposed), out fp32 [B][H][W][N];
 * chan_stats (optional, zeroed by the caller) accumulates the per-channel (sum, sum of squares) table of the output. */
int sdk_conv_in(const float* x, const float* w_t, const float* bias, float* out, double* chan_stats,
                int B, int H, int W, int N, void* stream);

/* ---- attention (models/unet/attention.py:29-50): out = softmax(q k^T * scale) v per head ------
 * q/k/v/out element strides: row stride (between tokens) and batch stride; head h occupies columns
 * [h*D, (h+1)*D).  kv_batch_stride may be 0 (context broadcast, SURVEY §3.4). */
int sdk_attention_f32(const float* q, int64_t q_row, int64_t q_batch, const float* k, int64_t k_row, int64_t k_batch,
                      const float* v, int64_t v_row, int64_t v_batch, float* out, int64_t o_row, int64_t o_batch,
                      int B, int heads, int Sq, int Sk, int D, float scale, void* stream);

/* same with an optional causal (look-ahead) mask: the text encoders' attention in the exact-fp32 mode */
int sdk_attention_f32_ex(const float* q, int64_t q_row, int64_t q_batch, const float* k, int64_t k_row, int64_t k_batch,
                         const float* v, int64_t v_row, int64_t v_batch, float* out, int64_t o_row, int64_t o_batch,
                         int B, int heads, int Sq, int Sk, int D, float scale, int causal, void* stream);

/* bf16 tensor-core attention (mma.sync m16n8k16, fp32 softmax statistics); same contract as sdk_attention_f32 with bf16 tensors */
int sdk_attention_bf16(const void* q, int64_t q_row, int64_t q_batch, const void* k, int64_t k_row, int64_t k_batch,
                       const void* v, int64_t v_row, int64_t v_batch, void* out, int64_t o_row, int64_t o_batch,
                       int B, int heads, int Sq, int Sk, int D, float scale, void* stream);

/* tcgen05 flash attention for head_dim 40 | 64 (S in TMEM, thread-per-row softmax, P V on the tensor core, operands by TMA
 * from per-head 4-D tensor maps).  Plan object = the TMA descriptors; same stride contract as sdk_attention_bf16. */
int sdk_attention_tc_create(const void* q, int64_t q_row, int64_t q_batch, const void* k, int64_t k_row, int64_t k_batch,
                            const void* v, int64_t v_row, int64_t v_batch, void* out, int64_t o_row, int64_t o_batch,
                            int B, int heads, int Sq, int Sk, int D, float scale, void** handle);
/* causal = 1: query i sees keys <= i (text encoders, models/clip/attention.py:38-45 with lookahead_mask=True) */
int sdk_attention_tc_set_causal(void* handle, int causal);
int sdk_attention_tc_launch(void* handle, void* stream);
int sdk_attention_tc_destroy(void* handle);

/* ---- tcgen05 / TMEM / TMA implicit GEMM (bf16 operands, fp32 accumulate) -----------------------------
 * Same math as sdk_conv_gemm_f32 for stride-1 "same" convolutions (ksize 1|3) and linears, with up to two
 * (activation, weight) segments accumulated into one output (segment 1 = a fused 1x1 shortcut conv,
 * unet.py:192).  Activations: NHWC bf16 [B][H][W][C], C % 64 == 0; weights bf16 [N][ksize*ksize*C] or k-block-major (w_kmajor).
 * A plan object holds the TMA descriptors; launches are async and graph-capturable.
 * Replaces nn.Conv2d/nn.Linear at unet.py:67,71,158,161,168,246,401; attention.py:19-25; activation_fn.py:14. */
typedef struct SdkTcGemmDesc {
    const void* a[2];
    const void* w[2];
    int C[2];
    int ksize[2];
    int nseg;
    int B, H, W;
    int N;
    const float* bias; const float* tbias; int64_t tb_stride; const float* residual;
    void* out;
    int out_dtype, geglu, out_nchw;
    int block_n;        /* 0 = auto (32|64|128|160|256) */
    int splits;         /* 0 = auto split-K */
    int w_kmajor;       /* 0: weights [N][K] row-major; 1: k-block-major [K/64][N][64] (contiguous B stages) */
    int two_cta;        /* 0 = auto, 1 = never, 2 = always (when the number of m-tiles is even): tcgen05 cta_group::2 CTA pairs */
    /* --- fusions around LayerNorm (unet.py:102-108,137-149); all optional (NULL / 0), fp32 NHWC outputs only for the first two --- */
    void* out2;               /* bf16 copy [M][N] of the output, written by the same epilogue (raw A operand of the next GEMM) */
    float* row_stats;         /* [M][N/32][2]: (sum, sum of squares) of every output row over each 32-column chunk = the LayerNorm
                                 statistics of the consumer, written by the thread that owns the row (no extra pass over the tensor) */
    const float* ln_stats;    /* LayerNorm FOLDED into this GEMM: `a` holds the raw rows x (bf16), `w` the gamma-scaled weights W' = W*gamma,
                                 `bias` = bias + W beta; ln_stats = the producer's row_stats [M][ln_parts][2] (ln_parts*32 = row width C),
                                 ln_colsum[n] = sum_k W'[n][k].  out = rstd[m]*(x W'^T - mean[m]*ln_colsum) + bias  ==  LN(x) W^T + bias */
    const float* ln_colsum;
    int ln_parts;
    float ln_eps;
    /* --- conv gathers folded into the TMA coordinates (no im2col / upsampled tensor in memory); one 3x3 k-block-major segment --- */
    int a_stride;             /* 2: stride-2 3x3 conv, pad 1 (unet.py:236-240): `a` is the INPUT image [B][a_h][a_w][C], H x W the output size */
    int a_h, a_w;
    int up2;                  /* 1: nearest-2x upsample + 3x3 conv (unet.py:248-251): `a` is the LOW-RES input [B][H][W][C], `out` is
                                 [B][2H][2W][N]; `w` holds FOUR parity sets of 2x2 taps, [py][px][2][2][C/64][N][64] (3x3 taps that
                                 read the same input pixel pre-summed by the host) */
    int w_const;              /* 1: `w` is never written by a kernel of the same stream (packed weights): with programmatic dependent launch
                                 the first weight tiles are fetched BEFORE the wait on the preceding kernel.  0 when `w` is an activation. */
    int weight_stationary;    /* persistent kernel, short K: each CTA keeps the weight tile of ONE n-tile resident in shared memory and walks
                                 m-tiles (a k-block then costs 16 KiB of L2->smem traffic instead of 16 KiB + block_n*128 B).
                                 0 = library default (SDB200_TC_WS, off), 1 = never, 2 = whenever it fits */
} SdkTcGemmDesc;
int sdk_tc_gemm_create(const SdkTcGemmDesc* desc, void** handle);
int64_t sdk_tc_gemm_workspace_bytes(void* handle);
int sdk_tc_gemm_set_workspace(void* handle, void* workspace);   /* zeroed ONCE by the caller (it starts with the split-K tile counters, which the kernels re-arm); shared across plans run on one stream */
int sdk_tc_gemm_info(void* handle, int* out, int n);            /* block_n, splits, grid.x, grid.y, TW, TH, TB, k-blocks [, cta group size, in-kernel split-K reduction, persistent if n >= 11] */
int sdk_tc_gemm_launch(void* handle, void* stream);
int sdk_tc_gemm_destroy(void* handle);
/* Also ACCUMULATE the per-channel (sum, sum of squares) table chan_stats [B][N][2] (double; input of sdk_groupnorm_apply_cs) of
 * the fp32 NHWC output: the caller zeroes the table before every launch (sdk_zero; the step program zeroes all its tables with one
 * call).  SDK_ERR_UNSUPPORTED when this plan cannot (bf16/GEGLU/NCHW output, tiles that straddle samples): use sdk_channel_stats. */
int sdk_tc_gemm_set_stats(void* handle, double* chan_stats);
/* developer aid: record 7 %globaltimer stamps of CTA (0,0,0) into device memory stamps[8] (NULL = off) */
int sdk_tc_gemm_set_debug(void* handle, void* stamps);
/* stride-2 3x3 conv (unet.py:236): gather fp32 NHWC -> bf16 [B*Ho*Wo][9*C] rows, then a 1-tap sdk_tc_gemm */
int sdk_im2col_s2(const float* src, void* dst, int B, int H, int W, int C, void* stream);

/* ---- Linear (+ bias + residual) fused with the LayerNorm of its output rows (unet.py:86,137-149; attention.py:25,50) --------
 * out[m][:] = a[m][:] W^T + bias + residual[m][:]   (fp32, the transformer block's residual stream)
 * ln_out[m][:] = LayerNorm(out[m][:]) * gamma + beta (bf16, the A operand of the next projection)
 * in ONE launch: the N/160 (or N/128) n-tiles of a 128-row block form a thread-block cluster (<= 8 CTAs) that exchanges the
 * per-row statistics (exact two-pass mean / variance) through distributed shared memory; the finished fp32 values stay in TMEM
 * between the passes.  a: bf16 [M][K], K % 64 == 0; w: bf16 k-block-major [K/64][N][64] (as SdkTcGemmDesc.w_kmajor).
 * SDK_ERR_UNSUPPORTED when N is not 160*k or 128*k with k <= 8: use sdk_tc_gemm + sdk_layernorm. */
typedef struct SdkLinearLnDesc {
    const void* a;
    const void* w;
    const float* bias;        /* [N] or NULL */
    const float* residual;    /* fp32 [M][N] or NULL */
    float* out;               /* fp32 [M][N] */
    void* ln_out;             /* bf16 [M][N] */
    const float* gamma; const float* beta;   /* [N] */
    float eps;
    int64_t M;
    int K, N;
} SdkLinearLnDesc;
int sdk_linear_ln_create(const SdkLinearLnDesc* desc, void** handle);
int sdk_linear_ln_info(void* handle, int* out, int n);          /* block_n, cluster size, grid, dynamic shared memory bytes */
int sdk_linear_ln_launch(void* handle, void* stream);
int sdk_linear_ln_destroy(void* handle);

/* ---- LoRA merge into packed weights (the low-rank update W + up*down of a LoRA / LoCon adapter, merged at inference) -------------
 *   dst[row_off + row_step*n][k] = cast( base[n][k] + sum_j up[n][j] * down[j][k] )      n < N, k < K
 * base: fp32 [N][ld_base], the master weight in the packed k order (conv taps NHWC: [kh][kw][Cin]); up: fp32 [N][r] with the adapter
 * scales folded in; down: fp32 [r][K]; several adapters on one target are concatenated along r.  r = 0 is a plain repack (up and
 * down may be NULL).  fp32 FFMA, j in increasing order.  dst_dtype SDK_F32 | SDK_BF16 (round to nearest even).
 * dst_layout SDK_LORA_ROW_MAJOR: dst is [dst_rows][K]; SDK_LORA_KBLOCK_MAJOR: dst is [K/64][dst_rows][64] (K % 64 == 0), the
 * tensor-core weight layout (SdkTcGemmDesc.w_kmajor).  Not launched with programmatic dependent launch: kernels that follow it may
 * read the weights it writes before their own griddepcontrol.wait (SdkTcGemmDesc.w_const).  SDK_ERR_ARG before any launch for
 * NULL base / dst, non-positive sizes, ld_base < K, r < 0, missing factors, an unknown dtype or layout, or rows outside dst_rows. */
#define SDK_LORA_ROW_MAJOR 0
#define SDK_LORA_KBLOCK_MAJOR 1
int sdk_lora_merge(const float* base, int64_t ld_base, const float* up, const float* down, int r, void* dst,
                   int dst_dtype, int dst_layout, int dst_rows, int row_off, int row_step, int N, int K, void* stream);

/* ---- plan-level entry: a program's LAUNCH LIST behind the C ABI, replayable, serialisable (engine file) -------------------------
 * The planning host records every launch of a program (one UNet forward = models/unet/unet.py:431-443, the context program, one
 * whole sampler step = the loop body of models/diffusion.py:223-236, a VAE decode, ...) with sdk_plan_add_launch; the plan ADOPTS the
 * tensor-core handles together with the descriptors they were created from (tuned tilings included), replays a program with ONE
 * call, and sdk_plan_save / sdk_plan_load move the whole thing -- launch lists, descriptors, packed weights, tables -- to a host
 * that has neither Python nor PyTorch (tools/c_host/denoise.c).  Up to 16 programs per plan; the package uses
 * 0 = UNet forward, 1 = context program, 2 = time-embedding chain, 3 = forward without that chain, 4 = one sampler step. */
typedef struct SdkAttentionTcDesc {      /* the arguments of sdk_attention_tc_create, as a struct (what a plan stores for the handle) */
    const void* q; const void* k; const void* v; void* out;
    int64_t q_row, q_batch, k_row, k_batch, v_row, v_batch, o_row, o_batch;
    int B, heads, Sq, Sk, D;
    float scale;
} SdkAttentionTcDesc;
int sdk_plan_create(void** plan);
int sdk_plan_destroy(void* plan);       /* also destroys the adopted handles and, for a loaded plan, frees its device memory */
/* Declare a device buffer the program touches: kind 0 = constant (weights / tables: contents are saved), 1 = scratch (zero-filled on
 * load), 2 = scratch with a NAME the loading host can look up (inputs / outputs / loop state). */
int sdk_plan_add_region(void* plan, const void* base, int64_t bytes, int kind, const char* name);
/* handle_kind 1 = sdk_tc_gemm (desc = SdkTcGemmDesc, aux = {chan_stats pointer or 0, workspace pointer or 0}), 2 = sdk_attention_tc
 * (desc = SdkAttentionTcDesc, aux = {causal}), 3 = sdk_linear_ln (desc = SdkLinearLnDesc).  The plan owns the handle from here on. */
int sdk_plan_adopt(void* plan, int handle_kind, void* handle, const void* desc, int desc_bytes, const uint64_t* aux, int n_aux);
/* Append one launch to `program`: fn_name = a launch-type entry point of this header ("sdk_layernorm", "sdk_tc_gemm_launch", ...),
 * args = its arguments WITHOUT the trailing stream, each widened to 64 bits (pointers and integers as they are, floats as their
 * IEEE-754 bit pattern, parameter structs by host address -- they are copied). */
int sdk_plan_add_launch(void* plan, int program, const char* fn_name, const uint64_t* args, int nargs);
int sdk_plan_num_launches(void* plan, int program);   /* -1 on a bad argument */
int sdk_plan_launch(void* plan, int program, void* stream);
/* capture `program` into a CUDA graph owned by the plan (after one eager launch); sdk_plan_launch then replays the graph */
int sdk_plan_capture(void* plan, int program, void* stream);
int sdk_plan_save(void* plan, const char* path);      /* synchronous (reads the constant regions back); fails if a pointer is in no region */
int sdk_plan_load(const char* path, void** plan);     /* allocates ONE device slab for all regions on the current device */
int sdk_plan_region(void* plan, const char* name, void** ptr, int64_t* bytes);
/* conveniences for hosts without the CUDA runtime headers: async copies into / out of a named region, stream handling */
int sdk_plan_upload(void* plan, const char* name, const void* host, int64_t bytes, void* stream);
int sdk_plan_download(void* plan, const char* name, void* host, int64_t bytes, void* stream);
int sdk_stream_create(void** stream);
int sdk_stream_sync(void* stream);
int sdk_stream_destroy(void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SDB200_H */
