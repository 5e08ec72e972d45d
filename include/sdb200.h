/*
 * sdb200.h — C-ABI of libsdb200.so: the B200 (sm_100a) kernels behind the latent-diffusion
 * sampling hot path of ProgramerSalar/stable-diffusion-from-scratch.
 *
 * The reference has no FFI: the boundary is its Python nn.Module API (UNetModel.forward,
 * DDIMSampler.sample, AutoencoderKL.decode).  The host-side mirror of that API lives in
 * stable-diffusion-from-scratch_b200/*.py and binds these entry points with ctypes.  Each entry
 * point below names the reference op (file:line under the reference tree) whose arithmetic it
 * replaces.
 *
 * Conventions (all entry points):
 *   - plain pointers + sizes only; every pointer is a DEVICE pointer unless marked host
 *   - activations are channels-last: images [N, H, W, C] ("NHWC"), tokens [rows, C]
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued, never synchronised
 *   - returns 0 on success, negative sdb code otherwise (sdb_last_error_string() explains);
 *     no entry point allocates device memory: workspaces are passed in by the caller
 *   - dtype codes: SDB_F32 = 0, SDB_BF16 = 1
 */
#ifndef SDB200_H
#define SDB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDB_OK            0
#define SDB_ERR_INVALID  -1   /* bad argument / unsupported shape */
#define SDB_ERR_CUDA     -2   /* CUDA runtime/driver error at enqueue time */
#define SDB_ERR_NOTMA    -3   /* cuTensorMapEncode* entry point unavailable */

#define SDB_F32   0
#define SDB_BF16  1

/* ---- library ------------------------------------------------------------------------------ */
int         sdb_version(void);                 /* 10000*major + 100*minor + patch */
const char* sdb_last_error_string(void);       /* thread-local, valid until the next failing call */
int         sdb_device_sm_count(void);         /* SMs of the current device (148 on B200) */
/* number of kernel launches enqueued by this library in this process (bench `gpu_launches`) */
unsigned long long sdb_launch_count(void);
/* Every kernel of the library is launched with programmatic stream serialization (it may start while its predecessor in the
 * stream drains and blocks in griddepcontrol.wait until that predecessor is complete).  The next `n` launches of the calling
 * host thread are made WITHOUT the attribute: they start only after ALL prior work of their stream — cross-stream event waits
 * included — has completed.  Callers use it for the first launch after a fork to / join from a side stream.  Returns the
 * previous pending count. */
int sdb_pdl_skip_next(int n);

/* ---- layout ------------------------------------------------------------------------------- */
/* NCHW fp32 <-> NHWC fp32/bf16.  Replaces nothing arithmetic: the reference computes in NCHW
 * (openai_model/model.py:572-595); the kernels compute in NHWC, this is the boundary transpose. */
/* dst_C (0 = C): channel count of dst; channels C..dst_C-1 are written as zeros (the 4-channel latent is padded to 32
 * bf16 channels so that conv_in, openai_model/model.py:365, runs on the tensor cores). */
int sdb_nchw_to_nhwc(const float* src, void* dst, int dst_dtype, int N, int C, int dst_C, int HW, void* stream);
/* Same layout change with a bf16 destination of dst_C >= 2*C channels that keeps fp32 information: channels 0..C-1 = bf16(x),
 * channels C..2C-1 = bf16(x - float(bf16(x))) (the rounding residual), the rest zero.  A bf16 contraction whose weights are
 * repeated for both halves then sees x to ~2^-17: the UNet's first conv (openai_model/model.py:531, 4 latent channels) runs on
 * the tensor cores without rounding x_t itself to bf16. */
int sdb_nchw_to_nhwc_split(const float* src, void* dst /* bf16 */, int N, int C, int dst_C, int HW, void* stream);
int sdb_nhwc_to_nchw(const float* src, float* dst, int N, int C, int HW, void* stream);
/* The same layout change from TWO channel-concatenated sources, in one pass: the channel order of dst is src0's C0 channels,
 * then src1's C1 channels (C = C0 + C1), then zeros up to dst_C (0 = C, or 2*C with split).  Replaces
 * torch.cat([x] + c_concat, dim=1) of DiffusionWrapper.forward (ldm/diffusion/ddpm.py:1992-2034, conditioning_key "concat" /
 * "hybrid": the inpainting UNet's latent | mask | masked-image latent) together with the boundary transpose feeding conv_in.
 * src0 [N,C0,HW], src1 [N,C1,HW] fp32 (src1 = NULL exactly when C1 = 0); dst [N,HW,dst_C] of dst_dtype.  split != 0 (bf16 dst,
 * dst_C >= 2*C): channels C..2C-1 hold the rounding residual of channels 0..C-1, as sdb_nchw_to_nhwc_split.  sdb_nchw_to_nhwc
 * and sdb_nchw_to_nhwc_split are its C1 = 0 case. */
int sdb_nchw_concat_to_nhwc(const float* src0, int C0, const float* src1, int C1, void* dst, int dst_dtype, int dst_C, int split,
                            int N, int HW, void* stream);

/* ---- GroupNorm(32) [+ SiLU] over NHWC, optional two-source channel concat -------------------
 * Replaces GroupNorm32.forward + nn.SiLU (openai_model/utils.py:15-22, model.py:178-181,202-205,
 * 528-531), Normalize eps=1e-6 (openai_model/attention.py:10-11,317; ldm/modules/
 * diffusionmodules/model.py:40-41) and `nonlinearity` x*sigmoid(x) (model.py:35-37), and the
 * torch.cat([h, hs.pop()], 1) feeding it (openai_model/model.py:586).
 *   x0 [N,HW,C0] fp32, x1 [N,HW,C1] fp32 or NULL (C1 = 0); C = C0 + C1, C % (4*groups)... see .cu
 *   out [N,HW,C] (out_dtype), ws: float/double scratch of sdb_groupnorm_ws_bytes() bytes.
 *   raw_out: NULL, or [N,HW,C] bf16 receiving the un-normalised concat input as well (the operand
 *   of the ResBlock's 1x1 skip_connection, openai_model/model.py:207-218,252) from the same read.
 *   counters: >= N ints, ZERO on entry and left zero on exit (ticket of the CTA that folds the
 *   per-chunk partial sums of a sample into its mean / rstd); one buffer per stream.
 *   act: 0 = none, 1 = SiLU.  exact != 0 uses expf (fp32 parity mode) instead of __expf.
 *   gb_stride: 0 = one gamma / beta row [C] shared by the batch; otherwise gamma / beta are [N, gb_stride]
 *   per-sample rows — how `out_norm(h) * (1 + scale) + shift` of the use_scale_shift_norm ResBlock
 *   (openai_model/model.py:244-248) is served: sdb_scale_shift_affine folds scale / shift into them. */
long long sdb_groupnorm_ws_bytes(int N, int HW, int C, int groups);
int sdb_groupnorm_nhwc(const float* x0, int C0, const float* x1, int C1, int N, int HW, int groups,
                       float eps, const float* gamma, const float* beta, long long gb_stride, int act, int exact,
                       void* out, int out_dtype, void* raw_out, void* ws, int* counters, void* stream);
/* gamma_out[n, c] = gamma[c] * (1 + ss[n, c]),  beta_out[n, c] = beta[c] * (1 + ss[n, c]) + ss[n, C + c];
 * ss [N, >= 2C] fp32 with row stride ld_ss = the (scale | shift) halves torch.chunk takes from emb_out
 * (openai_model/model.py:246).  gamma_out / beta_out [N, C]. */
int sdb_scale_shift_affine(const float* gamma, const float* beta, const float* ss, long long ld_ss, int N, int C,
                           float* gamma_out, float* beta_out, void* stream);

/* Same GroupNorm, statistics taken from the column sums the producing tcgen05 convs wrote (sdb_tc_args.colstats:
 * cs = fp32 [2][slots][C*]), so the tensor is read once.  layout (host, 4 values per source) = {slots, consecutive 32-row
 * slots per sample, regions, slots between regions}: regions > 1 is the output of a sub-pixel upsampling conv, whose four
 * phase convolutions each filled one region.  ws: >= N*groups*8 bytes.  Other arguments as sdb_groupnorm_nhwc. */
int sdb_groupnorm_from_colstats(const float* x0, int C0, const float* cs0, const long long* layout0 /* host */,
                                const float* x1, int C1, const float* cs1, const long long* layout1 /* host */,
                                int N, int HW, int groups, float eps,
                                const float* gamma, const float* beta, long long gb_stride, int act, int exact,
                                void* out, int out_dtype, void* raw_out, void* ws, void* stream);

/* ---- LayerNorm over the last dim ---------------------------------------------------------------
 * Replaces nn.LayerNorm(dim) x3 per BasicTransformerBlock (openai_model/attention.py:216-218,
 * 251-253), eps 1e-5.  x [rows, C] fp32 -> out [rows, C] (out_dtype). C % 4 == 0, C <= 2048. */
int sdb_layernorm(const float* x, int rows, int C, float eps, const float* gamma, const float* beta,
                  void* out, int out_dtype, void* stream);

/* ---- elementwise ---------------------------------------------------------------------------
 * sdb_cast_concat: out[n, oh, ow, :] = concat(x0, x1)[n, oh/up, ow/up, :] as out_dtype.
 * Replaces torch.cat (openai_model/model.py:586), F.interpolate(scale_factor=2, "nearest")
 * (openai_model/model.py:127; ldm/modules/diffusionmodules/model.py:56) and the dtype cast
 * feeding a conv. up is 1 or 2. H, W are the INPUT spatial dims. */
int sdb_cast_concat(const float* x0, int C0, const float* x1, int C1, int N, int H, int W, int up,
                    void* out, int out_dtype, void* stream);
/* bilinear x2 upsampling with align_corners=True (DDPM/models/layers.py:68-72); x [N,H,W,C] fp32. */
/* 2x2 average pooling, stride 2 (Downsample(use_conv=False).op = avg_pool2d, openai_model/model.py:88-93; used by
 * ResBlock(down=True), :184-189): x [N,H,W,C] fp32 -> out [N,H/2,W/2,C] (out_dtype).  H, W even, C % 4 == 0. */
int sdb_avgpool2x2(const float* x, int N, int H, int W, int C, void* out, int out_dtype, void* stream);
int sdb_upsample_bilinear2x(const float* x, int N, int H, int W, int C, void* out, int out_dtype, void* stream);
/* out = act(x) (+ optional cast); act 0 none, 1 SiLU (emb_layers' nn.SiLU, model.py:195-196),
 * 2 GELU-erf (DDPM/models/unet.py:29), 3 quick-GELU x * sigmoid(1.702 x) (the CLIP text tower's MLP, clip_encoder/modules.py:246).
 * n elements. */
int sdb_activation(const float* x, void* out, int out_dtype, long long n, int act, void* stream);
/* GEGLU: out[r, j] = h[r, j] * gelu_erf(h[r, inner + j]) (openai_model/attention.py:140-141).
 * h [rows, 2*inner] fp32 -> out [rows, inner] (out_dtype). */
int sdb_geglu(const float* h, int rows, int inner, void* out, int out_dtype, void* stream);
/* row softmax with pre-scale: out[r,:] = softmax(scale * s[r,:]) ; s fp32 [rows, L], row stride lds.
 * Replaces softmax in AttnBlock (ldm/modules/diffusionmodules/model.py:191-192) and the fp32-mode
 * attention (flash_attn_func semantics, openai_model/attention.py:106-112). */
int sdb_softmax_rows(const float* s, long long rows, int L, long long lds, float scale, void* out,
                     int out_dtype, long long ldo, void* stream);
/* the same with a causal mask (fp32-mode attention of the CLIP text tower, clip_encoder/modules.py:246-250): row r belongs to
 * query r % Sq and sees keys 0 .. r % Sq; masked probabilities are written as exact zeros. */
int sdb_softmax_rows_causal(const float* s, long long rows, int L, int Sq, long long lds, float scale, void* out,
                            int out_dtype, long long ldo, void* stream);
/* out = a + b (fp32), n elements: residual adds that follow a norm (DDPM/models/layers.py:338). */
int sdb_add(const float* a, const float* b, float* out, long long n, void* stream);
/* out[n,p,c] = x[n,p,c] + rowvec[n*ldv + c]: `time_emb[:, :, None, None] + h` (DDPM/models/layers.py:331-333). */
int sdb_add_rowvec(const float* x, const float* rowvec, long long ldv, int N, long long HW, int C, void* out,
                   int out_dtype, void* stream);

/* ---- timestep embedding ------------------------------------------------------------------------
 * Replaces timestep_embedding (openai_model/utils.py:225-245): emb[b] = [cos(t_b*f), sin(t_b*f)].
 * freqs: device fp32 [half] (built on the host exactly as the reference does). t: device fp32 [B].
 * round_fp16 != 0 rounds every value through IEEE half, restating `t_emb.half()`
 * (openai_model/model.py:566), which is part of the reference's result even in fp32. */
int sdb_timestep_embedding(const float* t, const float* freqs, int B, int half, int round_fp16, float* emb,
                           void* stream);
/* pe_matrix[t] lookup for the DDPM UNet (DDPM/models/layers.py:32-34): table fp32 [T, dim]. */
int sdb_gather_rows(const float* table, const long long* idx, int B, int dim, float* out, void* stream);

/* ---- skinny GEMM (M <= 32 rows): y[M,N] = act_in(x)[M,K] @ W[N,K]^T + b ------------------------
 * Replaces time_embed / emb_layers Linear on [B,1280] (openai_model/model.py:353-357,195-201,241).
 * W fp32 [N,K] row-major. act_in: 0 none, 1 SiLU applied to x on load. act_out: 0 none, 1 SiLU,
 * 2 GELU-erf (DDPM/models/unet.py:26-31). */
int sdb_skinny_linear(const float* x, int M, int K, const float* W, const float* bias, int N,
                      int act_in, int act_out, float* y, void* stream);
/* Same with the weight matrix stored in bf16 ([N,K] row-major, K % 8 == 0; x, bias, y and the accumulation stay fp32): the
 * bf16 compute mode's form of the 20160 x 1280 ResBlock time-embedding matrix, whose streaming is this kernel's whole cost. */
int sdb_skinny_linear_bf16w(const float* x, int M, int K, const void* W /* bf16 */, const float* bias, int N,
                            int act_in, int act_out, float* y, void* stream);

/* ---- DDIM update ---------------------------------------------------------------------------
 * Replaces p_sample_ddim's arithmetic (ldm/diffusion/ddim.py:175-205 == DDIM/ddim.py):
 *   e = e_uncond + cfg_scale*(e_cond - e_uncond)      (if e_uncond != NULL)
 *   pred_x0 = (x - sqrt_one_minus_at*e) / sqrt_at
 *   x_prev  = sqrt_aprev*pred_x0 + dir_coef*e + sigma_t*noise*temperature
 * all fp32, every operation individually rounded (no FMA contraction) like the eager reference.
 * The caller passes the derived per-step scalars sqrt_at = a_t.sqrt(), sqrt_aprev = a_prev.sqrt(),
 * dir_coef = (1 - a_prev - sigma_t**2).sqrt() (ddim.py:197-205) so that it can evaluate them with the
 * reference's own expressions.  noise may be NULL when sigma_t == 0.  n = number of elements. */
int sdb_ddim_step(const float* x, const float* e_cond, const float* e_uncond, float cfg_scale,
                  const float* noise, float sqrt_at, float sqrt_aprev, float dir_coef, float sigma_t,
                  float sqrt_one_minus_at, float temperature, float* x_prev, float* pred_x0, long long n,
                  void* stream);
/* Second half of the same update for the quantize_denoised branch (ldm/diffusion/ddim.py:198-205): pred_x0 is GIVEN
 * (the caller replaced it by first_stage_model.quantize(pred_x0)), x_prev = sqrt_aprev*pred_x0 + dir_coef*e + sigma_t*noise*temperature. */
int sdb_ddim_xprev(const float* pred_x0, const float* e_cond, const float* e_uncond, float cfg_scale, const float* noise,
                   float sqrt_aprev, float dir_coef, float sigma_t, float temperature, float* x_prev, long long n, void* stream);
/* ---- ancestral (DDPM) update ---------------------------------------------------------------
 * Replaces LatentDiffusion.p_sample's arithmetic (ldm/diffusion/ddpm.py:1528-1793: predict_start_from_noise,
 * x_recon.clamp_, q_posterior, `model_mean + nonzero_mask * (0.5 * model_log_variance).exp() * noise`):
 *   x0     = x0_in != NULL ? x0_in : sqrt_recip[t]*x - sqrt_recipm1[t]*eps
 *   x0     = clip ? clamp(x0, -1, 1) : x0                  (NaN passes through, like torch.clamp)
 *   mean   = coef1[t]*x0 + coef2[t]*x
 *   x_prev = noise != NULL ? mean + ((t != 0) * std[t]) * (noise*temperature) : mean
 * all fp32, every operation individually rounded (no FMA contraction) in the reference's order.
 * x / eps / x0_in / noise / x_prev / x0_out [B, per] fp32; t: device int64 [B]; table: device fp32 [5, T] with rows
 * sqrt_recip_alphas_cumprod, sqrt_recipm1_alphas_cumprod, posterior_mean_coef1, posterior_mean_coef2 and
 * posterior_std = exp(0.5 * posterior_log_variance_clipped), gathered per sample inside the kernel.  eps may be NULL
 * when x0_in is given; x_prev and x0_out are each optional, not both (x0_out only: predict_start_from_noise; no noise:
 * the posterior mean).  A t[b] outside [0, T) writes NaN into sample b and is never used as an index. */
int sdb_ddpm_step(const float* x, const float* eps, const float* x0_in, const float* noise, const long long* t,
                  const float* table, int T, int clip, float temperature, float* x_prev, float* x0_out, int B, long long per,
                  void* stream);
/* Inpainting blend of ddim_sampling (ldm/diffusion/ddim.py:144-149) fused with LatentDiffusion.q_sample
 * (ldm/diffusion/ddpm.py:407-412): img_orig = a[b]*x0 + c[b]*noise; out = img_orig*mask + (1 - mask)*img.
 * x0 / noise / img / out [B,C,HW] fp32, mask [B,Cm,HW] with Cm == 1 (broadcast over channels) or Cm == C; a / c: B per-sample
 * coefficients (sqrt_alphas_cumprod[t], sqrt_one_minus_alphas_cumprod[t]); individually rounded fp32 operations. */
int sdb_inpaint_blend(const float* x0, const float* noise, const float* a, const float* c, const float* mask, const float* img,
                      int B, int C, int Cm, long long HW, float* out, void* stream);

/* ---- VAE posterior and img2img entry ('next' row f3) ------------------------------------------
 * sdb_diag_gaussian replaces DiagonalGaussianDistribution.__init__ / .sample
 * (ldm/modules/distributions/distributions.py:24-37): moments [N,2C,HW] fp32 (NCHW, the quant_conv output)
 * -> mean, logvar = clamp(., -30, 20), std = exp(0.5 logvar), var = exp(logvar), and, when noise != NULL,
 * sample = mean + std * noise; every output [N,C,HW] fp32.
 * sdb_q_sample replaces DDIMSampler.stochastic_encode's arithmetic (ldm/diffusion/ddim.py:218-222):
 * out[b, :] = a[b] * x0[b, :] + c[b] * noise[b, :], a / c device vectors of B per-sample coefficients,
 * per = elements per sample; individually rounded fp32 operations like the eager reference. */
int sdb_diag_gaussian(const float* moments, const float* noise, int N, int C, long long HW, float* mean, float* logvar,
                      float* stdv, float* var, float* sample, void* stream);
int sdb_q_sample(const float* x0, const float* noise, const float* a, const float* c, int B, long long per, float* out,
                 void* stream);

/* ---- fp32 SIMT contraction (the fp32 parity mode; also the C_in=4 / tiny layers) --------------
 * One kernel family: out[m, n] = alpha * sum_k A(m,k) * B(n,k) + bias[n] + rowvec[img(m), n]
 *                                + residual[m, n]
 * conv mode (kh*kw > 0 and H > 0): A(m,k) gathers x NHWC fp32 [NB,IH,IW,Cin] with stride/pad
 *   (+ nearest-2x fold: `up`), B = weights packed [kh*kw][Cout][Cin] ("RSKC").
 *   Replaces nn.Conv2d 3x3/1x1 (openai_model/model.py:88-90,117,181,207,218,365,531;
 *   openai_model/attention.py:319-334; ldm/modules/diffusionmodules/model.py:49,94,104,...).
 * gemm mode: A [M,K] lda, B [N,K] ldb (b_kn = 0) or [K,N] ldb (b_kn = 1); two-level batch.
 *   Replaces nn.Linear (openai_model/attention.py:40-47,133,159-167) and torch.bmm
 *   (ldm/modules/diffusionmodules/model.py:188,197). */
typedef struct sdb_simt_args {
    const float* A; const float* B; float* out;
    const float* bias;       /* [N] or NULL */
    const float* rowvec;     /* [NB, ldv] per-image vector (time-emb add) or NULL; conv mode only */
    const float* residual;   /* [M, ldr] or NULL */
    long long lda, ldb, ldc, ldr, ldv;
    int M, N, K;
    float alpha;
    int b_kn;
    /* batch: z = b1*nb2 + b2 */
    int nb1, nb2;
    long long sa1, sa2, sb1, sb2, sc1, sc2;
    /* conv geometry; kh = 0 means plain gemm */
    int kh, kw, stride, pad, up;
    int NB, IH, IW, Cin, OH, OW;
    int out_dtype;           /* SDB_F32 or SDB_BF16 */
} sdb_simt_args;
int sdb_simt_contract(const sdb_simt_args* args /* host */, void* stream);

/* ---- tcgen05 contraction (bf16 operands, fp32 TMEM accumulation) -----------------------------
 * TMA -> 128B-swizzled smem ring -> tcgen05.mma (cta_group::1, M=128, N=BN, K=16) -> TMEM ->
 * tcgen05.ld epilogue.  Same algebra as sdb_simt_contract with bf16 A/B:
 *   gemm mode: A bf16 [M,K] (lda), B bf16 [N,K] (ldb)
 *   conv mode: A bf16 NHWC [NB,IH,IW,Cin] (pixel stride ldx), B bf16 packed [taps][CoutPad][Cin]
 * epilogue: + bias[n] + rowvec[img, n] + residual[m, n]; optional GEGLU pairing
 * (openai_model/attention.py:140-141) when geglu != 0 (B rows packed a|gate per BN tile);
 * optional column-group remap (n -> (n / cg)*cgs + n % cg) used to write q/k/v heads padded.
 * split_k > 1: every K-split writes its fp32 partial tile to the workspace and a second kernel sums
 * the splits in a fixed order and applies bias / rowvec / residual (deterministic, no atomics). */
typedef struct sdb_tc_args {
    const void* A; const void* B; void* out;
    const float* bias; const float* rowvec; const float* residual;
    long long lda, ldb, ldc, ldr, ldv;   /* elements */
    int M, N, K;
    int out_dtype;
    int geglu;
    int col_group, col_group_stride;     /* 0 = no remap */
    int split_k;
    int block_n;                          /* 0 = auto; else 16/32/64/128/160/256 */
    /* conv geometry; taps = 0 means gemm */
    int taps;                             /* 1, 4 (2x2) or 9 (3x3) */
    int kw;                               /* kernel width (taps = kh*kw) */
    int stride, pad_h, pad_w;
    int NB, IH, IW, Cin, OH, OW;          /* OH/OW: conv output dims (before out_* remap) */
    int cout_pad;                         /* rows of B per tap */
    /* output pixel remap (sub-pixel upsample phases): oh' = oh*out_sh + out_oh etc. */
    int out_sh, out_sw, out_oh, out_ow, OHF, OWF;
    /* split-K workspace (device, 16-byte aligned) for the per-split partial tiles; may be NULL when
     * split_k == 1.  split_k == 0 lets the library choose (it only splits when `ws` is given). */
    void* ws; long long ws_bytes;
    /* gemm mode: rows of A owned by ONE independent sample (tokens per image), 0 = unknown.  Only used so
     * that the automatic split-K choice does not depend on the batch size (batch-invariant bit patterns). */
    int rows_per_item;
    /* kernel variant: 0 = library default (see sdb_tc_set_pair_kernel), 1 = one-CTA 128 x BN kernel,
     * 2 = CTA-pair persistent 256 x BN kernel (block_n >= 128).  Same results up to summation order. */
    int variant;
    /* optional, conv mode: fp32 [2][colstats_slots][N] receiving, for every 32-row slot of the output (4 per 128-row
     * m-tile, slot = 4*tile + row/32) and every column, the sum and the sum of squares of the values this call stores
     * — the statistics pass of the GroupNorm that consumes the output (openai_model/utils.py:15-22) comes for free.
     * Size it with sdb_tc_colstats_layout(); NULL = off. */
    float* colstats; long long colstats_slots;
    /* != 0: B is a constant of the stream (a weight matrix no earlier launch writes).  The kernels then fetch their first B
     * tiles BEFORE the programmatic-dependent-launch wait, i.e. while the preceding kernel is still draining: the weights come
     * from DRAM (1.7 GB streamed per UNet call), so their latency leaves the critical path.  0 = B may have been produced by the
     * preceding launch (e.g. torch.bmm operands): everything waits. */
    int b_const;
} sdb_tc_args;
/* slots the column statistics of these args occupy and how many consecutive slots belong to one sample (both 0 when
 * the plan cannot produce them: split-K, several samples per tile, bf16 / remapped output). */
int sdb_tc_colstats_layout(const sdb_tc_args* args /* host */, long long* slots, long long* slots_per_item);
/* bytes of workspace sdb_tc_contract may use for these args (0 = none; -1 = invalid args).  With
 * split_k == 0 this is what the library's automatic split choice needs. */
long long sdb_tc_workspace_bytes(const sdb_tc_args* args /* host */);
int sdb_tc_contract(const sdb_tc_args* args /* host */, void* stream);
/* Tuning switch (measurement only, same results either way): 1 = CTA-pair persistent kernel
 * (cta_group::2, 256 x BN tiles) for block_n >= 128 [default], 0 = one-CTA 128 x BN kernel everywhere.
 * Returns the previous setting. */
int sdb_tc_set_pair_kernel(int enable);
/* Tuning switch (measurement only, bit-identical results either way): 1 = the CTA-pair kernel's epilogue stages 32 x 32 boxes
 * in swizzled shared memory and moves them with TMA (cp.async.bulk.tensor stores, residual tiles by TMA loads) whenever the
 * output layout allows [default], 0 = register-store epilogue everywhere.  Returns the previous setting. */
int sdb_tc_set_tma_epilogue(int enable);
/* Tuning switch (measurement only, bit-identical results either way): 1 = the one-CTA kernel with 160-column tiles issues the
 * tiles of its last, partial wave (tiles mod SM count) as two sub-tiles of 96 and 64 columns, so the tail of the launch is handed
 * out in half-size pieces [default; SDB200_TC_TAILSPLIT=0 at load time], 0 = whole tiles only.  Returns the previous setting. */
int sdb_tc_set_tail_split(int enable);

/* ---- fused attention forward (bf16, tcgen05) ---------------------------------------------------
 * Replaces flash_attn_func(q,k,v, softmax_scale, causal=False) (openai_model/attention.py:106-112).
 * q [B,Sq,H,*], k/v [B,Sk,H,*] bf16 with explicit element strides.  The kernel works on heads of dpad (multiple of 64,
 * <= 192) channels: dense == 0: the heads are stored zero-padded from d to dpad channels; dense != 0: the heads are stored
 * with their d channels only (e.g. the plain [rows, H*d] output of a projection GEMM) and the TMA tensor maps are d wide,
 * so the pad channels of every shared-memory tile are the zeros TMA fills in for out-of-bounds elements.
 * out [B,Sq,H,d] bf16 with explicit strides. */
typedef struct sdb_attn_args {
    const void* q; const void* k; const void* v; void* out;
    long long q_bs, q_ss, q_hs;   /* batch / seq / head strides (elements) */
    long long k_bs, k_ss, k_hs;
    long long v_bs, v_ss, v_hs;
    long long o_bs, o_ss, o_hs;
    int B, H, Sq, Sk, d, dpad;
    float scale;
    int dense;
    /* != 0: causal mask — query i attends to keys 0..i only, as HF CLIPTextModel builds it for the text tower behind
     * FrozenCLIPEmbedder (clip_encoder/modules.py:212-256); needs Sq == Sk. */
    int causal;
} sdb_attn_args;
int sdb_attention_fwd(const sdb_attn_args* args /* host */, void* stream);
/* Tuning switch (measurement only): 1 = problems with ONE key tile (Sk <= 128, head pad <= 128, no causal mask — the
 * cross-attention over the 77 text tokens, openai_model/attention.py:99-112) run on tc_attention_kv1_kernel, whose CTAs keep
 * K / V resident and walk query items [default; SDB200_XATTN=0 turns it off at load time]; 0 = the key-tile-walking kernel
 * everywhere.  Returns the previous setting. */
int sdb_attention_set_short_key_kernel(int enable);

/* ---- fused attention forward for one WIDE head (d = 256 or 512): the VAE AttnBlock -------------------------------
 * Replaces  w_ = bmm(q, k) * c**-0.5;  w_ = softmax(w_);  h_ = bmm(v, w_)  of AttnBlock.forward
 * (ldm/modules/diffusionmodules/model.py:180-204; one head over all C channels, 4096 tokens in the SD decoder's mid block)
 * without materialising the [Sq, Sk] score matrix: a CTA owns a 128-row query tile and ONE 256-channel half of the output
 * (the 512 TMEM columns cannot hold S and a 512-wide O), recomputes S = Q K^T over the full d on tcgen05 and accumulates
 * O[:, half] += P V[:, half].  q / k / v bf16 [B, S, d] with explicit batch / sequence strides in elements (d contiguous,
 * e.g. the three column blocks of one [B*S, 3d] projection output); out [B, Sq, d] bf16. */
int sdb_attention_wide_fwd(const void* q, const void* k, const void* v, void* out, long long q_bs, long long q_ss,
                           long long k_bs, long long k_ss, long long v_bs, long long v_ss, long long o_bs, long long o_ss,
                           int B, int Sq, int Sk, int d, float scale, void* stream);

/* ---- vector quantisation: the VQ first stage's codebook lookup ------------------------------------------------------
 * sdb_vq_quantize replaces taming's VectorQuantizer2.forward in eval with legacy=True (ldm/tamming/quantize.py:213-311,
 * the `quantize` of VQModel / VQModelInterface, ldm/models/autoencoder.py):
 *   zf   = z as [M = N*HW, D] rows in (n, h, w) order
 *   d    = (sum(zf**2, 1) + sum(W**2, 1)) - 2 * zf @ W.T          fp32, never materialised
 *   idx  = argmin(d, 1)                                           first index of the minimum; NaN counts as the minimum
 *   z_q  = z + (W[idx] - z)                                       straight-through, fp32, each operation rounded
 *   loss = mean((W[idx] - z)**2) + beta * mean((W[idx] - z)**2)   one fp32 scalar, fp64 partials in a fixed order
 * z fp32 in z_layout (SDB_NCHW: [N, D, HW]; SDB_NHWC: [N, HW, D]); z_q fp32 in zq_layout; idx int64 [M]; codebook W fp32
 * [n_e, D], 1 <= D <= 16, any n_e >= 1.  z_q, idx and loss are each optional (NULL), not all three.  ws: device scratch of
 * sdb_vq_ws_bytes(M, n_e) bytes; counters: >= 1 int, zero on entry and left zero (ticket of the CTA that folds the loss
 * partials; only used when loss != NULL), the same buffer kind sdb_groupnorm_nhwc takes.  When M rows alone cannot fill the
 * GPU the codebook is split into slices scanned by separate CTAs whose minima are merged by (NaN first, d, index): the
 * split depends on M and n_e only, and the result does not depend on it. */
#define SDB_NCHW  0
#define SDB_NHWC  1
long long sdb_vq_ws_bytes(long long M, int n_e);                    /* -1 on bad arguments */
int sdb_vq_quantize(const float* z, int z_layout, int N, int HW, int D, const float* codebook, int n_e, float beta,
                    float* z_q, int zq_layout, long long* idx, float* loss, void* ws, int* counters, void* stream);
/* VectorQuantizer2.get_codebook_entry (ldm/tamming/quantize.py:313-329): out = W[idx] for M = N*HW indices in (n, h, w)
 * order, written as out_layout ([N, D, HW] or [N, HW, D]) fp32.  An index outside [0, n_e) writes a NaN row and is never
 * dereferenced. */
int sdb_vq_codebook_gather(const long long* idx, long long M, const float* codebook, int n_e, int D, float* out, int out_layout,
                           int HW, void* stream);

/* ---- patch-distributed fold / unfold: LatentDiffusion's split_input_params branch -----------------------------------
 * (ldm/diffusion/ddpm.py:1344-1437 apply_model, 1097-1139 decode_first_stage.)  The crop grid of an image of H x W with
 * crops kh x kw at stride (sh, sw) is Ly = (H - kh) / sh + 1 by Lx = (W - kw) / sw + 1, crop l = ly * Lx + lx with its
 * origin at (ly * sh, lx * sw).  Crops are stored crop-major, [L*B, C, kh, kw] with row l*B + b, so that the L crops of a
 * batch of B images are one batch of L*B samples.  Both use 64-bit element indices, never allocate and never sync.
 *
 * sdb_patch_unfold: out = unfold(x).view(B, C, kh, kw, L)[..., l] for every l (torch.nn.Unfold, dilation 1, no padding),
 * x fp32 NCHW [B, C, H, W]; a pure copy. */
int sdb_patch_unfold(const float* x, int B, int C, int H, int W, int kh, int kw, int sh, int sw, float* out, void* stream);
/* sdb_patch_fold: out = fold(o * weighting) / fold(weighting) on an fp32 NCHW [B, C, OH, OW] output, o fp32 [L*B, C, KH, KW]
 * crop-major, with the per-crop weight w_l(p) = wpix[p] (wcrop == NULL) or fl(wpix[p] * wcrop[l]) (the tie breaker), wpix
 * fp32 [KH*KW], wcrop fp32 [L]:
 *   out[b, c, y, x] = (sum_l fl(o_l * w_l)) / (sum_l w_l)     over the crops l covering (y, x)
 * Both sums start at 0.0f and run in fp32 in increasing l, the order of torch's CUDA col2im, so the result is the bits of
 * the reference's torch.nn.Fold expression.  A pixel no crop covers is 0 / 0 = NaN, as in the reference.  L must equal
 * Ly * Lx and the grid must lie inside (OH, OW). */
int sdb_patch_fold(const float* o, int B, int C, int KH, int KW, int Ly, int Lx, int SH, int SW, int OH, int OW,
                   const float* wpix, const float* wcrop, int L, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SDB200_H */
