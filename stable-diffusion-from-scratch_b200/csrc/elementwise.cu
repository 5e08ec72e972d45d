// sdb200 — layout, elementwise and small-matrix kernels (all HBM/launch-bound).
#include "common.cuh"
#include <cuda_fp16.h>

namespace sdb {

// ---- NCHW <-> NHWC (32x32 smem tile transpose, padded against bank conflicts) -------------------
// Two sources: channels 0..C0-1 come from src0 [N, C0, HW], channels C0..C0+C1-1 from src1 [N, C1, HW] (C1 = 0: src0 only), so the
// channel concat in front of a conditioned UNet's conv_in (ldm/diffusion/ddpm.py:1992-2034, torch.cat([x] + c_concat, dim=1)) is
// done by the same pass that changes the layout.  C = C0 + C1.
// SPLIT (bf16 output only): channels C..2C-1 carry the rounding residual x - float(bf16(x)) of channels 0..C-1, so a bf16
// contraction whose weights are repeated for both halves sees x to ~2^-17 instead of 2^-9 (the UNet's conv_in on the tensor
// cores without rounding the latent x_t itself).
template <bool OUT_BF16, bool SPLIT>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src0, int C0, const float* __restrict__ src1, int C1,
                                    void* __restrict__ dst, int Cd, int HW) {
    pdl_trigger();
    pdl_wait();
    __shared__ float tile[32][33];
    const int C = C0 + C1;
    const int n = blockIdx.z;
    const int hw0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const float* s0 = src0 + (long long)n * C0 * HW;
    const float* s1 = src1 + (long long)n * C1 * HW;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int c = c0 + i, hw = hw0 + threadIdx.x;
        if (SPLIT && c >= C && c < 2 * C) c -= C;
        float v = 0.f;                                                                  // the remaining channels up to Cd are zero padding
        if (hw < HW) {
            if (c < C0) v = s0[(long long)c * HW + hw];
            else if (c < C) v = s1[(long long)(c - C0) * HW + hw];
        }
        tile[i][threadIdx.x] = v;
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int hw = hw0 + i, c = c0 + threadIdx.x;
        if (hw < HW && c < Cd) {
            long long o = ((long long)n * HW + hw) * Cd + c;
            float v = tile[threadIdx.x][i];
            if (SPLIT && c >= C && c < 2 * C) v = v - __bfloat162float(__float2bfloat16_rn(v));
            if (OUT_BF16) reinterpret_cast<__nv_bfloat16*>(dst)[o] = __float2bfloat16_rn(v);
            else reinterpret_cast<float*>(dst)[o] = v;
        }
    }
}

__global__ void nhwc_to_nchw_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int HW) {
    pdl_trigger();
    pdl_wait();
    __shared__ float tile[32][33];
    const int n = blockIdx.z;
    const int hw0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const float* s = src + (long long)n * C * HW;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int hw = hw0 + i, c = c0 + threadIdx.x;
        tile[i][threadIdx.x] = (c < C && hw < HW) ? s[(long long)hw * C + c] : 0.f;
    }
    __syncthreads();
    float* d = dst + (long long)n * C * HW;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        int c = c0 + i, hw = hw0 + threadIdx.x;
        if (c < C && hw < HW) d[(long long)c * HW + hw] = tile[threadIdx.x][i];
    }
}

// ---- cast (+ channel concat, + nearest 2x upsample) ---------------------------------------------
// One thread per float4 of the OUTPUT. out [N, H*up, W*up, C0+C1].
template <bool OUT_BF16>
__global__ void cast_concat_kernel(const float* __restrict__ x0, int C0, const float* __restrict__ x1, int C1,
                                   int H, int W, int up, long long total_vec, void* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int C = C0 + C1, V = C >> 2;
    const int OW = W * up;
    const long long OHW = (long long)H * up * OW;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
         i += (long long)gridDim.x * blockDim.x) {
        int v = (int)(i % V);
        long long pix = i / V;
        long long n = pix / OHW;
        int rem = (int)(pix % OHW);
        int oh = rem / OW, ow = rem % OW;
        long long ipix = (n * H + oh / up) * W + ow / up;
        int c = v * 4;
        float4 a = (c < C0) ? __ldg(reinterpret_cast<const float4*>(x0 + ipix * C0 + c))
                            : __ldg(reinterpret_cast<const float4*>(x1 + ipix * C1 + (c - C0)));
        long long o = pix * C + c;
        if (OUT_BF16) st_stream_u2(reinterpret_cast<__nv_bfloat16*>(out) + o, pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w));
        else st_stream_f4(reinterpret_cast<float*>(out) + o, a);
    }
}

template <bool OUT_BF16>
__global__ void activation_kernel(const float* __restrict__ x, void* __restrict__ out, long long n, int act) {
    pdl_trigger();
    pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = x[i];
        if (act == 1) v = silu_exact(v);
        else if (act == 2) v = gelu_erf(v);
        else if (act == 3) v = v / (1.0f + expf(-1.702f * v));      // quick_gelu = x * sigmoid(1.702 x) (CLIP text tower MLP)
        if (OUT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
        else reinterpret_cast<float*>(out)[i] = v;
    }
}

template <bool OUT_BF16>
__global__ void geglu_kernel(const float* __restrict__ h, int rows, int inner, void* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const long long total = (long long)rows * inner;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        long long r = i / inner;
        int j = (int)(i % inner);
        float a = h[r * 2 * inner + j], g = h[r * 2 * inner + inner + j];
        float v = a * gelu_erf(g);
        if (OUT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
        else reinterpret_cast<float*>(out)[i] = v;
    }
}

// out[n, p, c] = x[n, p, c] + rowvec[n, c]  (time-embedding broadcast add, DDPM/models/layers.py:331-333)
template <bool OUT_BF16>
__global__ void add_rowvec_kernel(const float* __restrict__ x, const float* __restrict__ rv, long long ldv,
                                  long long HW, int C, long long total_vec, void* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int V = C >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec; i += (long long)gridDim.x * blockDim.x) {
        int v = (int)(i % V);
        long long n = (i / V) / HW;
        float4 a = __ldg(reinterpret_cast<const float4*>(x) + i);
        const float* r = rv + n * ldv + v * 4;
        a.x += r[0]; a.y += r[1]; a.z += r[2]; a.w += r[3];
        if (OUT_BF16) st_stream_u2(reinterpret_cast<__nv_bfloat16*>(out) + i * 4, pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w));
        else st_stream_f4(reinterpret_cast<float*>(out) + i * 4, a);
    }
}

__global__ void add_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long n) {
    pdl_trigger();
    pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = a[i] + b[i];
}

// ---- row softmax: one CTA per row, fp32 statistics ----------------------------------------------
// causal_sq > 0: row r is query r % causal_sq and sees keys 0 .. (r % causal_sq) only (masked probabilities are written as 0)
template <bool OUT_BF16>
__global__ void softmax_rows_kernel(const float* __restrict__ s, int L_all, long long lds, float scale,
                                    void* __restrict__ out, long long ldo, int causal_sq) {
    pdl_trigger();
    pdl_wait();
    __shared__ float red[32];
    const long long row = blockIdx.x;
    const float* p = s + row * lds;
    int L = L_all;
    if (causal_sq > 0) {
        const int qi = (int)(row % causal_sq);
        L = qi + 1 < L_all ? qi + 1 : L_all;
        for (int i = L + threadIdx.x; i < L_all; i += blockDim.x) {
            if (OUT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[row * ldo + i] = __float2bfloat16_rn(0.f);
            else reinterpret_cast<float*>(out)[row * ldo + i] = 0.f;
        }
    }
    float m = -INFINITY;
    for (int i = threadIdx.x; i < L; i += blockDim.x) m = fmaxf(m, p[i] * scale);
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : -INFINITY;
        t = warp_max(t);
        if (threadIdx.x == 0) red[0] = t;
    }
    __syncthreads();
    m = red[0];
    __syncthreads();
    float sum = 0.f;
    for (int i = threadIdx.x; i < L; i += blockDim.x) sum += expf(p[i] * scale - m);
    sum = warp_sum(sum);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = (threadIdx.x < (blockDim.x >> 5)) ? red[threadIdx.x] : 0.f;
        t = warp_sum(t);
        if (threadIdx.x == 0) red[0] = t;
    }
    __syncthreads();
    const float inv = 1.0f / red[0];
    for (int i = threadIdx.x; i < L; i += blockDim.x) {
        float v = expf(p[i] * scale - m) * inv;
        if (OUT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[row * ldo + i] = __float2bfloat16_rn(v);
        else reinterpret_cast<float*>(out)[row * ldo + i] = v;
    }
}

// ---- timestep embedding (reference openai_model/utils.py:225-245): [cos | sin] ------------------
__global__ void timestep_embedding_kernel(const float* __restrict__ t, const float* __restrict__ freqs,
                                          int B, int half, int round_fp16, float* __restrict__ emb) {
    pdl_trigger();
    pdl_wait();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * half) return;
    int b = i / half, j = i % half;
    float a = t[b] * freqs[j];
    float c = cosf(a), s = sinf(a);
    if (round_fp16) { c = __half2float(__float2half_rn(c)); s = __half2float(__float2half_rn(s)); }
    emb[(long long)b * 2 * half + j] = c;
    emb[(long long)b * 2 * half + half + j] = s;
}

__global__ void gather_rows_kernel(const float* __restrict__ table, const long long* __restrict__ idx,
                                   int B, int dim, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * dim) return;
    int b = i / dim, j = i % dim;
    out[i] = table[idx[b] * dim + j];
}

// ---- skinny linear: M <= 32 rows; one warp per output column, weights streamed once -------------
// NC output columns per warp: the activated input rows are read from shared memory once per NC weight rows (with one column per
// warp the kernel is bound by those reads — 16 LDS.128 per 16-byte weight load at M = 8 — at ~0.7 TB/s of weight streaming).
template <int MT, bool WBF16, int NC>
__global__ void skinny_linear_kernel(const float* __restrict__ x, int M, int K, const void* __restrict__ Wv,
                                     const float* __restrict__ bias, int N, int act_in, int act_out,
                                     float* __restrict__ y) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ float xs[];   // [M][K] activated input
    for (int i = threadIdx.x; i < M * K; i += blockDim.x) {
        float v = x[i];
        if (act_in == 1) v = silu_exact(v);
        xs[i] = v;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int warps = blockDim.x >> 5;
    constexpr int EPL = WBF16 ? 8 : 4;        // weights per 16-byte load
    // the weight rows are streamed once: KU 16-byte loads per lane and column are in flight before the first FMA (one load in
    // flight per lane made this kernel latency-bound at ~1 TB/s on the ResBlock time-embedding matrix)
    constexpr int KU = (WBF16 ? 5 : 10) / (NC > 1 ? (WBF16 ? 1 : 2) : 1);
    for (int n0 = (blockIdx.x * warps + (threadIdx.x >> 5)) * NC; n0 < N; n0 += gridDim.x * warps * NC) {
        float acc[NC][MT];
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
            for (int m = 0; m < MT; ++m) acc[c][m] = 0.f;
        for (int k0 = lane * EPL; k0 < K; k0 += 32 * EPL * KU) {
            float4 wv[NC][KU];
#pragma unroll
            for (int c = 0; c < NC; ++c)
#pragma unroll
                for (int u = 0; u < KU; ++u) {
                    wv[c][u] = make_float4(0.f, 0.f, 0.f, 0.f);
                    const int k = k0 + 32 * EPL * u;
                    if (k < K && n0 + c < N) {
                        if (WBF16) wv[c][u] = ld_stream_f4(reinterpret_cast<const float*>(reinterpret_cast<const __nv_bfloat16*>(Wv) + (long long)(n0 + c) * K + k));
                        else wv[c][u] = ld_stream_f4(reinterpret_cast<const float*>(Wv) + (long long)(n0 + c) * K + k);
                    }
                }
#pragma unroll
            for (int u = 0; u < KU; ++u) {
                const int k = k0 + 32 * EPL * u;
                if (k < K) {
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
                        if (m < M) {
                            const float4 xa = *reinterpret_cast<const float4*>(xs + m * K + k);
                            if (WBF16) {
                                const float4 xb = *reinterpret_cast<const float4*>(xs + m * K + k + 4);
#pragma unroll
                                for (int c = 0; c < NC; ++c) {
                                    // 8 bf16 weights: a bf16 is the high half of the fp32 with the same value
                                    const uint32_t q0 = __float_as_uint(wv[c][u].x), q1 = __float_as_uint(wv[c][u].y);
                                    const uint32_t q2 = __float_as_uint(wv[c][u].z), q3 = __float_as_uint(wv[c][u].w);
                                    acc[c][m] += (__uint_as_float(q0 << 16) * xa.x + __uint_as_float(q0 & 0xffff0000u) * xa.y +
                                                  __uint_as_float(q1 << 16) * xa.z + __uint_as_float(q1 & 0xffff0000u) * xa.w) +
                                                 (__uint_as_float(q2 << 16) * xb.x + __uint_as_float(q2 & 0xffff0000u) * xb.y +
                                                  __uint_as_float(q3 << 16) * xb.z + __uint_as_float(q3 & 0xffff0000u) * xb.w);
                                }
                            } else {
#pragma unroll
                                for (int c = 0; c < NC; ++c)
                                    acc[c][m] += wv[c][u].x * xa.x + wv[c][u].y * xa.y + wv[c][u].z * xa.z + wv[c][u].w * xa.w;
                            }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int c = 0; c < NC; ++c) {
#pragma unroll
            for (int m = 0; m < MT; ++m) {
                if (m < M) {
                    float v = warp_sum(acc[c][m]);
                    if (lane == 0 && n0 + c < N) {
                        if (bias) v += bias[n0 + c];
                        if (act_out == 1) v = silu_exact(v);
                        else if (act_out == 2) v = gelu_erf(v);
                        y[(long long)m * N + n0 + c] = v;
                    }
                }
            }
        }
    }
}

// ---- fused sampler updates: one pointwise driver, one op per update ------------------------------------------------------
// sampler_update_kernel<VEC, Op> runs Op over n fp32 elements.  VEC = 4: 128-bit loads / stores (every pointer 16-byte aligned
// and n % 4 == 0; DdpmStep also needs per % 4 == 0, so that a vector never straddles two samples), VEC = 1: any alignment.
// An op names its NIN elementwise inputs in `ins` and its NOUT outputs in `outs`.  The first NREQ inputs are never NULL.  The
// kernel reads exactly the inputs that are non-NULL (a NULL one reads as 0; the host sets to NULL every input the call does not
// read) and stores exactly the outputs that are non-NULL.  op.apply(in, out, i0) maps the VEC elements of every input that start
// at element i0 to those of every output.
// At SD-1.x sizes a launch is latency-bound (about 2.5 us on a B200; figures in DESIGN.md §0, sampler-update driver).  Two
// choices here bring PLMS close to the 2.58 us per launch of its former kernel: 2.60 us with both, 2.77 with a NULL test on the
// NREQ inputs, 2.64 without __grid_constant__.  __grid_constant__ costs the DDIM and DDPM updates 0.02-0.06 us; they stay
// faster than their former kernels.
template <int VEC, class Op>
__global__ void __launch_bounds__(256) sampler_update_kernel(const __grid_constant__ Op op, long long n) {
    pdl_trigger();
    pdl_wait();
    const long long nv = n / VEC;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
        float in[Op::NIN][VEC], out[Op::NOUT][VEC];
#pragma unroll
        for (int k = 0; k < Op::NIN; ++k) {
            const bool read = k < Op::NREQ || op.ins[k];
            if constexpr (VEC == 4) {
                const float4 a = read ? __ldg(reinterpret_cast<const float4*>(op.ins[k]) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                in[k][0] = a.x; in[k][1] = a.y; in[k][2] = a.z; in[k][3] = a.w;
            } else {
                in[k][0] = read ? __ldg(op.ins[k] + i) : 0.f;
            }
        }
        op.apply(in, out, i * VEC);
#pragma unroll
        for (int k = 0; k < Op::NOUT; ++k) {
            if (!op.outs[k]) continue;
            if constexpr (VEC == 4) reinterpret_cast<float4*>(op.outs[k])[i] = make_float4(out[k][0], out[k][1], out[k][2], out[k][3]);
            else op.outs[k][i] = out[k][0];
        }
    }
}

// ---- DDIM update (reference ldm/diffusion/ddim.py:175-205) --------------------------------------
// Every operation is a separately rounded fp32 op (__f*_rn blocks FMA contraction) so that, given
// the same eps, x_prev / pred_x0 are bit-identical to the eager reference arithmetic.
// Classifier-free guidance combine e_u + cfg * (e_c - e_u) (ddim.py:176-179).
__device__ __forceinline__ float cfg_combine_1(float e, float u, float cfg) {
    return __fadd_rn(u, __fmul_rn(cfg, __fsub_rn(e, u)));
}

// One element of the update; `p0_given`: pred_x0 is given (quantize_denoised branch, ddim.py:198-199) and only x_prev is formed.
__device__ __forceinline__ void ddim_update_1(float xv, float e, bool has_u, float u, float cfg, bool has_nz, float nzv,
                                              float sqrt_at, float sqrt_aprev, float dir_coef, float sigma_t,
                                              float sqrt_one_minus_at, float temperature, bool p0_given, float& p0, float& xp) {
    if (has_u) e = cfg_combine_1(e, u, cfg);
    if (!p0_given) p0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(sqrt_one_minus_at, e)), sqrt_at);
    const float dir = __fmul_rn(dir_coef, e);
    float nz = 0.f;
    if (has_nz) nz = __fmul_rn(__fmul_rn(sigma_t, nzv), temperature);
    xp = __fadd_rn(__fadd_rn(__fmul_rn(sqrt_aprev, p0), dir), nz);
}

// HBM-bound: 16 B / element at eta = 0 (x, e in; x_prev, pred_x0 out), + 4 with noise, + 4 with classifier-free guidance.
// p0_in given: the quantize_denoised branch (ddim.py:198-205); x is not read and pred_x0 is not written.
struct DdimStep {
    static constexpr int NIN = 5, NOUT = 2, NREQ = 1;
    const float* ins[NIN];   // e_cond, x, e_uncond, noise, p0_in
    float* outs[NOUT];       // x_prev, pred_x0
    float cfg, sqrt_at, sqrt_aprev, dir_coef, sigma_t, sqrt_one_minus_at, temperature;
    template <int VEC>
    __device__ __forceinline__ void apply(const float (&in)[NIN][VEC], float (&out)[NOUT][VEC], long long) const {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            out[1][j] = in[4][j];
            ddim_update_1(in[1][j], in[0][j], ins[2] != nullptr, in[2][j], cfg, ins[3] != nullptr, in[3][j], sqrt_at, sqrt_aprev,
                          dir_coef, sigma_t, sqrt_one_minus_at, temperature, ins[4] != nullptr, out[1][j], out[0][j]);
        }
    }
};

// ---- PLMS update (ldm/models/diffusion/plms.py, p_sample_plms) ------------------------------------------------------------
//   e  = e_u given ? e_u + cfg * (e - e_u) : e                       (written to e_out: what the eps history keeps)
//   e' = order 0: (o1 + e) / 2                                        (second half of the first step; o1 = the first eval)
//        order 1: e
//        order 2: (3 e - o1) / 2
//        order 3: (23 e - 16 o1 + 5 o2) / 12
//        order 4: (55 e - 59 o1 + 37 o2 - 9 o3) / 24                  (o1 = old_eps[-1], o2 = old_eps[-2], o3 = old_eps[-3])
//   then the DDIM update (ddim_update_1) with e'.
// Separately rounded fp32 operations, left to right as the eager reference evaluates them; / 2, / 12, / 24 are divisions.
__device__ __forceinline__ float plms_combine_1(int order, float e, float o1, float o2, float o3) {
    switch (order) {
    case 0: return __fdiv_rn(__fadd_rn(o1, e), 2.f);
    case 2: return __fdiv_rn(__fsub_rn(__fmul_rn(3.f, e), o1), 2.f);
    case 3: return __fdiv_rn(__fadd_rn(__fsub_rn(__fmul_rn(23.f, e), __fmul_rn(16.f, o1)), __fmul_rn(5.f, o2)), 12.f);
    case 4: return __fdiv_rn(__fsub_rn(__fadd_rn(__fsub_rn(__fmul_rn(55.f, e), __fmul_rn(59.f, o1)), __fmul_rn(37.f, o2)),
                                       __fmul_rn(9.f, o3)), 24.f);
    default: return e;
    }
}

struct PlmsOut { float e, ep, p0, xp; };

__device__ __forceinline__ PlmsOut plms_update_1(int order, float xv, float e, bool has_u, float u, float cfg, float o1, float o2,
                                                 float o3, bool has_nz, float nzv, float sqrt_at, float sqrt_aprev, float dir_coef,
                                                 float sigma_t, float sqrt_one_minus_at, float temperature) {
    PlmsOut r;
    r.e = has_u ? cfg_combine_1(e, u, cfg) : e;
    r.ep = plms_combine_1(order, r.e, o1, o2, o3);
    ddim_update_1(xv, r.ep, false, 0.f, 1.f, has_nz, nzv, sqrt_at, sqrt_aprev, dir_coef, sigma_t, sqrt_one_minus_at, temperature,
                  false, r.p0, r.xp);
    return r;
}

struct PlmsStep {
    static constexpr int NIN = 7, NOUT = 4, NREQ = 2;
    const float* ins[NIN];   // x, e, e_uncond, o1, o2, o3, noise
    float* outs[NOUT];       // e_out, ep_out, pred_x0, x_prev
    float cfg;
    int order;
    float sqrt_at, sqrt_aprev, dir_coef, sigma_t, sqrt_one_minus_at, temperature;
    template <int VEC>
    __device__ __forceinline__ void apply(const float (&in)[NIN][VEC], float (&out)[NOUT][VEC], long long) const {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const PlmsOut r = plms_update_1(order, in[0][j], in[1][j], ins[2] != nullptr, in[2][j], cfg, in[3][j], in[4][j], in[5][j],
                                            ins[6] != nullptr, in[6][j], sqrt_at, sqrt_aprev, dir_coef, sigma_t, sqrt_one_minus_at,
                                            temperature);
            out[0][j] = r.e; out[1][j] = r.ep; out[2][j] = r.p0; out[3][j] = r.xp;
        }
    }
};

// ---- multistep DPM-Solver++ update (CompVis ldm/models/diffusion/dpm_solver/dpm_solver.py, predict_x0, 'dpm_solver') ------
//   e   = e_u given ? e_u + cfg * (e - e_u) : e                              (model_wrapper, classifier-free)
//   m0  = (x - sigma_s * e) / alpha_s                                        (data_prediction_fn at the evaluated time)
//   order 1: x_t = c_x x - c_0 m0                                            (dpm_solver_first_update)
//   order 2: D1_0 = inv_r0 (m0 - m1); x_t = c_x x - c_0 m0 - c_1 D1_0        (multistep_dpm_solver_second_update)
//   order 3: D1_0 = inv_r0 (m0 - m1); D1_1 = inv_r1 (m1 - m2); D1 = D1_0 + c_r (D1_0 - D1_1); D2 = c_d2 (D1_0 - D1_1);
//            x_t = c_x x - c_0 m0 + c_1 D1 - c_2 D2                          (multistep_dpm_solver_third_update)
// Separately rounded fp32 operations, left to right as the eager reference evaluates them.
struct DpmCoef { float sigma_s, alpha_s, c_x, c_0, c_1, c_2, inv_r0, inv_r1, c_r, c_d2; };
struct DpmOut { float m0, xn; };

__device__ __forceinline__ DpmOut dpm_update_1(int order, float xv, float e, bool has_u, float u, float cfg, float m1, float m2,
                                               const DpmCoef& k) {
    if (has_u) e = cfg_combine_1(e, u, cfg);
    DpmOut r;
    r.m0 = __fdiv_rn(__fsub_rn(xv, __fmul_rn(k.sigma_s, e)), k.alpha_s);
    r.xn = __fsub_rn(__fmul_rn(k.c_x, xv), __fmul_rn(k.c_0, r.m0));
    if (order >= 2) {
        const float d10 = __fmul_rn(k.inv_r0, __fsub_rn(r.m0, m1));
        if (order == 2) {
            r.xn = __fsub_rn(r.xn, __fmul_rn(k.c_1, d10));
        } else {
            const float d11 = __fmul_rn(k.inv_r1, __fsub_rn(m1, m2));
            const float dd = __fsub_rn(d10, d11);
            const float d1 = __fadd_rn(d10, __fmul_rn(k.c_r, dd));
            const float d2 = __fmul_rn(k.c_d2, dd);
            r.xn = __fsub_rn(__fadd_rn(r.xn, __fmul_rn(k.c_1, d1)), __fmul_rn(k.c_2, d2));
        }
    }
    return r;
}

struct DpmSolverStep {
    static constexpr int NIN = 5, NOUT = 2, NREQ = 2;
    const float* ins[NIN];   // x, e, e_uncond, m1, m2
    float* outs[NOUT];       // x_next, m0_out
    float cfg;
    int order;
    DpmCoef k;
    template <int VEC>
    __device__ __forceinline__ void apply(const float (&in)[NIN][VEC], float (&out)[NOUT][VEC], long long) const {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const DpmOut r = dpm_update_1(order, in[0][j], in[1][j], ins[2] != nullptr, in[2][j], cfg, in[3][j], in[4][j], k);
            out[0][j] = r.xn; out[1][j] = r.m0;
        }
    }
};

// ---- ancestral (DDPM) update of LatentDiffusion.p_sample (ldm/diffusion/ddpm.py:1528-1793) -----------------------
//   x0   = x0_in given ? x0_in : sqrt_recip[t]*x - sqrt_recipm1[t]*eps     (predict_start_from_noise)
//   x0   = clip ? clamp(x0, -1, 1) : x0                                     (x_recon.clamp_, NaN passes through)
//   mean = coef1[t]*x0 + coef2[t]*x                                          (q_posterior)
//   out  = noise ? mean + ((t != 0) * std[t]) * (noise * temperature) : mean
// Separately rounded fp32 operations in the reference's order.  The per-sample coefficients are gathered from the
// [5, T] device table by t[b]; a t outside [0, T) makes that sample NaN and is never used as an index.
__device__ __forceinline__ void ddpm_update_1(float xv, float e, float x0v, bool x0_given, bool clip, bool has_nz, float nzv,
                                              float sr, float srm1, float c1, float c2, float s, float temperature,
                                              float& x0, float& xp) {
    x0 = x0_given ? x0v : __fsub_rn(__fmul_rn(sr, xv), __fmul_rn(srm1, e));
    if (clip) x0 = x0 < -1.f ? -1.f : (x0 > 1.f ? 1.f : x0);
    const float mean = __fadd_rn(__fmul_rn(c1, x0), __fmul_rn(c2, xv));
    xp = has_nz ? __fadd_rn(mean, __fmul_rn(s, __fmul_rn(nzv, temperature))) : mean;
}

// The five coefficients are gathered once per vector: every element of a vector belongs to the same sample.
struct DdpmStep {
    static constexpr int NIN = 4, NOUT = 2, NREQ = 1;
    const float* ins[NIN];   // x, eps, x0_in, noise
    float* outs[NOUT];       // x_prev, x0_out
    const long long* t;
    const float* table;
    int T, clip;
    float temperature;
    long long per;
    template <int VEC>
    __device__ __forceinline__ void apply(const float (&in)[NIN][VEC], float (&out)[NOUT][VEC], long long i0) const {
        const long long tb = __ldg(t + i0 / per);
        if (tb < 0 || tb >= T) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) out[0][j] = out[1][j] = __int_as_float(0x7fc00000);
            return;
        }
        const float sr = __ldg(table + tb), srm1 = __ldg(table + T + tb);
        const float c1 = __ldg(table + 2 * (long long)T + tb), c2 = __ldg(table + 3 * (long long)T + tb);
        const float s = __fmul_rn(tb != 0 ? 1.f : 0.f, __ldg(table + 4 * (long long)T + tb));   // nonzero_mask * std
#pragma unroll
        for (int j = 0; j < VEC; ++j)
            ddpm_update_1(in[0][j], in[1][j], in[2][j], ins[2] != nullptr, clip != 0, ins[3] != nullptr, in[3][j], sr, srm1, c1, c2,
                          s, temperature, out[1][j], out[0][j]);
    }
};

// ---- inpainting blend of ddim_sampling (ldm/diffusion/ddim.py:144-149) with q_sample (ldm/diffusion/ddpm.py:407-412) fused:
//   img_orig = a[b] * x0 + c[b] * noise;   out = img_orig * mask + (1 - mask) * img
// mask [B, Cm, HW] with Cm in {1, C} (broadcast over channels); separately rounded fp32 operations like the eager reference.
__global__ void inpaint_blend_kernel(const float* __restrict__ x0, const float* __restrict__ noise, const float* __restrict__ a,
                                     const float* __restrict__ c, const float* __restrict__ mask, const float* __restrict__ img,
                                     int C, int Cm, long long HW, long long n, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const long long per = (long long)C * HW;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / per, r = i - b * per;
        const long long mi = Cm == 1 ? b * HW + r % HW : i;
        const float m = mask[mi];
        const float orig = __fadd_rn(__fmul_rn(a[b], x0[i]), __fmul_rn(c[b], noise[i]));
        out[i] = __fadd_rn(__fmul_rn(orig, m), __fmul_rn(__fsub_rn(1.0f, m), img[i]));
    }
}

// ---- posterior of the VAE encoder: DiagonalGaussianDistribution (ldm/modules/distributions/distributions.py:24-37) ----
// moments [N, 2C, HW] fp32 (NCHW) -> mean, logvar (clamped to [-30, 20]), std = exp(0.5 logvar), var = exp(logvar),
// sample = mean + std * noise (when noise != NULL), each [N, C, HW].
__global__ void diag_gaussian_kernel(const float* __restrict__ moments, const float* __restrict__ noise, int C, long long HW,
                                     long long n, float* __restrict__ mean, float* __restrict__ logvar,
                                     float* __restrict__ stdv, float* __restrict__ var, float* __restrict__ sample) {
    pdl_trigger();
    pdl_wait();
    const long long per = (long long)C * HW;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long img = i / per, r = i - img * per;
        const float m = moments[img * 2 * per + r];
        float lv = moments[img * 2 * per + per + r];
        lv = fminf(fmaxf(lv, -30.0f), 20.0f);
        const float sd = expf(__fmul_rn(0.5f, lv));
        mean[i] = m;
        logvar[i] = lv;
        stdv[i] = sd;
        var[i] = expf(lv);
        if (sample) sample[i] = __fadd_rn(m, __fmul_rn(sd, noise[i]));
    }
}

// ---- q_sample with per-sample coefficients: out = a[b] * x0 + c[b] * noise (DDIMSampler.stochastic_encode,
// ldm/diffusion/ddim.py:208-222; separately rounded fp32 operations like the eager reference) ----
__global__ void q_sample_kernel(const float* __restrict__ x0, const float* __restrict__ noise, const float* __restrict__ a,
                                const float* __restrict__ c, long long per, long long n, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / per;
        out[i] = __fadd_rn(__fmul_rn(a[b], x0[i]), __fmul_rn(c[b], noise[i]));
    }
}

// ---- scale-shift GroupNorm affine rows and 2x2 average pooling (UNet variants, SURVEY.md §8 f4) ----------------
__global__ void scale_shift_affine_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                          const float* __restrict__ ss, long long ld_ss, int C, long long n,
                                          float* __restrict__ go, float* __restrict__ bo) {
    pdl_trigger();
    pdl_wait();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / C;
        const int c = (int)(i - b * C);
        const float one_plus = 1.0f + ss[b * ld_ss + c];
        go[i] = gamma[c] * one_plus;
        bo[i] = fmaf(beta[c], one_plus, ss[b * ld_ss + C + c]);
    }
}

template <bool OUT_BF16>
__global__ void avgpool2x2_kernel(const float* __restrict__ x, int H, int W, int C, long long total_vec, void* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int OH = H >> 1, OW = W >> 1, V = C >> 2;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec; i += (long long)gridDim.x * blockDim.x) {
        const int v = (int)(i % V);
        long long pix = i / V;
        const int ow = (int)(pix % OW);
        long long t = pix / OW;
        const int oh = (int)(t % OH);
        const long long img = t / OH;
        const float* p = x + ((img * H + 2 * oh) * W + 2 * ow) * (long long)C + 4 * v;
        const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + C);
        const float4 c = *reinterpret_cast<const float4*>(p + (long long)W * C), d = *reinterpret_cast<const float4*>(p + (long long)W * C + C);
        // summation order of ATen's avg_pool2d: row-major over the window, then one division
        float4 r;
        r.x = (((a.x + b.x) + c.x) + d.x) * 0.25f;
        r.y = (((a.y + b.y) + c.y) + d.y) * 0.25f;
        r.z = (((a.z + b.z) + c.z) + d.z) * 0.25f;
        r.w = (((a.w + b.w) + c.w) + d.w) * 0.25f;
        if (OUT_BF16) reinterpret_cast<uint2*>(out)[i] = make_uint2(pack_bf16x2(r.x, r.y), pack_bf16x2(r.z, r.w));
        else reinterpret_cast<float4*>(out)[i] = r;
    }
}

// ---- bilinear x2 upsample, align_corners=True (DDPM/models/layers.py:68-72), NHWC ----------------
template <bool OUT_BF16>
__global__ void upsample_bilinear2x_kernel(const float* __restrict__ x, int H, int W, int C, long long total_vec,
                                           void* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int OH = 2 * H, OW = 2 * W, V = C >> 2;
    // PyTorch's area_pixel_compute_scale for align_corners=True: (in - 1) / (out - 1), 0 when out == 1
    const float sh = OH > 1 ? (float)(H - 1) / (float)(OH - 1) : 0.f;
    const float sw = OW > 1 ? (float)(W - 1) / (float)(OW - 1) : 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total_vec;
         i += (long long)gridDim.x * blockDim.x) {
        int v = (int)(i % V);
        long long pix = i / V;
        int ow = (int)(pix % OW);
        long long t = pix / OW;
        int oh = (int)(t % OH);
        long long n = t / OH;
        float fh = sh * oh, fw = sw * ow;
        int h0 = (int)fh, w0 = (int)fw;
        int h1 = h0 + (h0 < H - 1 ? 1 : 0), w1 = w0 + (w0 < W - 1 ? 1 : 0);
        float lh = fh - h0, lw = fw - w0;
        const float* b = x + (n * H) * (long long)W * C + v * 4;
        float4 a00 = __ldg(reinterpret_cast<const float4*>(b + ((long long)h0 * W + w0) * C));
        float4 a01 = __ldg(reinterpret_cast<const float4*>(b + ((long long)h0 * W + w1) * C));
        float4 a10 = __ldg(reinterpret_cast<const float4*>(b + ((long long)h1 * W + w0) * C));
        float4 a11 = __ldg(reinterpret_cast<const float4*>(b + ((long long)h1 * W + w1) * C));
        float w00 = (1.f - lh) * (1.f - lw), w01 = (1.f - lh) * lw, w10 = lh * (1.f - lw), w11 = lh * lw;
        float4 r;
        r.x = w00 * a00.x + w01 * a01.x + w10 * a10.x + w11 * a11.x;
        r.y = w00 * a00.y + w01 * a01.y + w10 * a10.y + w11 * a11.y;
        r.z = w00 * a00.z + w01 * a01.z + w10 * a10.z + w11 * a11.z;
        r.w = w00 * a00.w + w01 * a01.w + w10 * a10.w + w11 * a11.w;
        long long o = pix * C + v * 4;
        if (OUT_BF16) st_stream_u2(reinterpret_cast<__nv_bfloat16*>(out) + o, pack_bf16x2(r.x, r.y), pack_bf16x2(r.z, r.w));
        else st_stream_f4(reinterpret_cast<float*>(out) + o, r);
    }
}

static inline int grid_for(long long n, int threads) {
    long long b = (n + threads - 1) / threads;
    long long cap = 148LL * 16;
    return (int)(b < cap ? (b < 1 ? 1 : b) : cap);
}

}  // namespace sdb

using namespace sdb;

template <bool WBF16>
static int launch_skinny(const float* x, int M, int K, const void* W, const float* bias, int N, int act_in, int act_out, float* y, void* stream) {
    SDB_REQUIRE(x && W && y && M > 0 && M <= 32 && K > 0 && K % (WBF16 ? 8 : 4) == 0 && N > 0, "skinny_linear: bad args M=%d K=%d N=%d", M, K, N);
    SDB_REQUIRE(((uintptr_t)W & 15) == 0, "skinny_linear: W must be 16-byte aligned");
    size_t smem = (size_t)M * K * sizeof(float);
    SDB_REQUIRE(smem <= 200 * 1024, "skinny_linear: M*K too large");
    int threads = 256;
    // four columns per warp when there are enough columns to keep every SM busy that way (the ResBlock embedding matrix)
    const int nc = (M <= 8 && N >= 4 * 8 * 148 * 2) ? 4 : 1;
    int blocks = ceil_div(N, (threads / 32) * nc);
    if (blocks > 148 * 4) blocks = 148 * 4;
    cudaStream_t st = (cudaStream_t)stream;
#define SK(MT, NC)                                                                                          \
    do {                                                                                                    \
        if (smem > 48 * 1024) cudaFuncSetAttribute(skinny_linear_kernel<MT, WBF16, NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        launch_pdl(skinny_linear_kernel<MT, WBF16, NC>, dim3(blocks), dim3(threads), smem, st, x, M, K, W, bias, N, act_in, act_out, y);   \
    } while (0)
    if (nc == 4) { if (M <= 4) SK(4, 4); else SK(8, 4); }
    else if (M <= 4) SK(4, 1); else if (M <= 8) SK(8, 1); else if (M <= 16) SK(16, 1); else SK(32, 1);
#undef SK
    return check_launch("skinny_linear_kernel");
}

// [a, a + n) and [b, b + n) (fp32 elements) share an element; NULL never overlaps.
static bool ranges_overlap(const float* a, const float* b, long long n) {
    if (!a || !b) return false;
    const uintptr_t pa = reinterpret_cast<uintptr_t>(a), pb = reinterpret_cast<uintptr_t>(b), len = (uintptr_t)n * sizeof(float);
    return pa < pb + len && pb < pa + len;
}

// Launches sampler_update_kernel over n elements.  It first rejects any output that overlaps an input or another output: the
// kernel reads its inputs through the read-only data cache (__ldg), which needs them unwritten while it runs.  VEC 4 needs every
// pointer 16-byte aligned and `unit` a multiple of 4.  Every error message starts with "<entry>: ".
template <class Op>
static int launch_sampler_update(const char* entry, const Op& op, long long n, long long unit, void* stream) {
    for (int j = 0; j < Op::NOUT; ++j) {
        for (const float* in : op.ins) SDB_REQUIRE(!ranges_overlap(op.outs[j], in, n), "%s: output %d overlaps an input", entry, j);
        for (int k = 0; k < j; ++k) SDB_REQUIRE(!ranges_overlap(op.outs[j], op.outs[k], n), "%s: outputs %d and %d overlap", entry, k, j);
    }
    uintptr_t al = 0;
    for (const float* p : op.ins) al |= reinterpret_cast<uintptr_t>(p);
    for (const float* p : op.outs) al |= reinterpret_cast<uintptr_t>(p);
    if ((al & 15) == 0 && unit % 4 == 0)
        launch_pdl(sampler_update_kernel<4, Op>, dim3(grid_for(n / 4, 256)), dim3(256), 0, (cudaStream_t)stream, op, n);
    else
        launch_pdl(sampler_update_kernel<1, Op>, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, op, n);
    return check_launch(entry);
}

extern "C" {

int sdb_nchw_concat_to_nhwc(const float* src0, int C0, const float* src1, int C1, void* dst, int dst_dtype, int dst_C, int split,
                            int N, int HW, void* stream) {
    SDB_REQUIRE(src0 && dst && N > 0 && C0 > 0 && C1 >= 0 && HW > 0, "nchw_concat_to_nhwc: bad args");
    SDB_REQUIRE((C1 == 0) == (src1 == nullptr), "nchw_concat_to_nhwc: src1 must be given exactly when C1 > 0 (C1=%d)", C1);
    SDB_REQUIRE(dst_dtype == SDB_F32 || dst_dtype == SDB_BF16, "nchw_concat_to_nhwc: bad dst_dtype %d", dst_dtype);
    const int C = C0 + C1;
    const int Cd = dst_C > 0 ? dst_C : C;
    if (split) {
        SDB_REQUIRE(dst_dtype == SDB_BF16, "nchw_concat_to_nhwc: split needs a bf16 destination");
        SDB_REQUIRE(Cd >= 2 * C, "nchw_concat_to_nhwc: dst_C=%d < 2*C=%d", Cd, 2 * C);
    } else {
        SDB_REQUIRE(Cd >= C, "nchw_concat_to_nhwc: dst_C=%d < C=%d", Cd, C);
    }
    dim3 grid(ceil_div(HW, 32), ceil_div(Cd, 32), N), block(32, 8);
    cudaStream_t st = (cudaStream_t)stream;
    if (split) launch_pdl(nchw_to_nhwc_kernel<true, true>, grid, block, 0, st, src0, C0, src1, C1, dst, Cd, HW);
    else if (dst_dtype == SDB_BF16) launch_pdl(nchw_to_nhwc_kernel<true, false>, grid, block, 0, st, src0, C0, src1, C1, dst, Cd, HW);
    else launch_pdl(nchw_to_nhwc_kernel<false, false>, grid, block, 0, st, src0, C0, src1, C1, dst, Cd, HW);
    return check_launch(split ? "nchw_to_nhwc_kernel(split)" : "nchw_to_nhwc_kernel");
}

int sdb_nchw_to_nhwc(const float* src, void* dst, int dst_dtype, int N, int C, int dst_C, int HW, void* stream) {
    SDB_REQUIRE(src && dst && N > 0 && C > 0 && HW > 0, "nchw_to_nhwc: bad args");
    const int Cd = dst_C > 0 ? dst_C : C;
    SDB_REQUIRE(Cd >= C, "nchw_to_nhwc: dst_C=%d < C=%d", Cd, C);
    return sdb_nchw_concat_to_nhwc(src, C, nullptr, 0, dst, dst_dtype == SDB_BF16 ? SDB_BF16 : SDB_F32, Cd, 0, N, HW, stream);
}

int sdb_nchw_to_nhwc_split(const float* src, void* dst, int N, int C, int dst_C, int HW, void* stream) {
    SDB_REQUIRE(src && dst && N > 0 && C > 0 && HW > 0, "nchw_to_nhwc_split: bad args");
    SDB_REQUIRE(dst_C >= 2 * C, "nchw_to_nhwc_split: dst_C=%d < 2*C=%d", dst_C, 2 * C);
    return sdb_nchw_concat_to_nhwc(src, C, nullptr, 0, dst, SDB_BF16, dst_C, 1, N, HW, stream);
}

int sdb_nhwc_to_nchw(const float* src, float* dst, int N, int C, int HW, void* stream) {
    SDB_REQUIRE(src && dst && N > 0 && C > 0 && HW > 0, "nhwc_to_nchw: bad args");
    dim3 grid(ceil_div(HW, 32), ceil_div(C, 32), N), block(32, 8);
    launch_pdl(nhwc_to_nchw_kernel, dim3(grid), dim3(block), 0, (cudaStream_t)stream, src, dst, C, HW);
    return check_launch("nhwc_to_nchw_kernel");
}

int sdb_cast_concat(const float* x0, int C0, const float* x1, int C1, int N, int H, int W, int up,
                    void* out, int out_dtype, void* stream) {
    SDB_REQUIRE(x0 && out && N > 0 && H > 0 && W > 0, "cast_concat: bad args");
    SDB_REQUIRE(C0 > 0 && C0 % 4 == 0 && C1 % 4 == 0 && (C1 == 0) == (x1 == nullptr), "cast_concat: bad channels %d %d", C0, C1);
    SDB_REQUIRE(up == 1 || up == 2, "cast_concat: up must be 1 or 2");
    long long total = (long long)N * H * up * W * up * ((C0 + C1) / 4);
    int threads = 256, blocks = grid_for(total, threads);
    if (out_dtype == SDB_BF16) launch_pdl(cast_concat_kernel<true>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x0, C0, x1, C1, H, W, up, total, out);
    else launch_pdl(cast_concat_kernel<false>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x0, C0, x1, C1, H, W, up, total, out);
    return check_launch("cast_concat_kernel");
}

int sdb_upsample_bilinear2x(const float* x, int N, int H, int W, int C, void* out, int out_dtype, void* stream) {
    SDB_REQUIRE(x && out && N > 0 && H > 0 && W > 0 && C > 0 && C % 4 == 0, "upsample_bilinear2x: bad args");
    long long total = (long long)N * 2 * H * 2 * W * (C / 4);
    int threads = 256, blocks = grid_for(total, threads);
    if (out_dtype == SDB_BF16) launch_pdl(upsample_bilinear2x_kernel<true>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, H, W, C, total, out);
    else launch_pdl(upsample_bilinear2x_kernel<false>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, H, W, C, total, out);
    return check_launch("upsample_bilinear2x_kernel");
}

int sdb_activation(const float* x, void* out, int out_dtype, long long n, int act, void* stream) {
    SDB_REQUIRE(x && out && n > 0, "activation: bad args");
    int threads = 256, blocks = grid_for(n, threads);
    if (out_dtype == SDB_BF16) launch_pdl(activation_kernel<true>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, out, n, act);
    else launch_pdl(activation_kernel<false>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, out, n, act);
    return check_launch("activation_kernel");
}

int sdb_geglu(const float* h, int rows, int inner, void* out, int out_dtype, void* stream) {
    SDB_REQUIRE(h && out && rows > 0 && inner > 0, "geglu: bad args");
    int threads = 256, blocks = grid_for((long long)rows * inner, threads);
    if (out_dtype == SDB_BF16) launch_pdl(geglu_kernel<true>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, h, rows, inner, out);
    else launch_pdl(geglu_kernel<false>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, h, rows, inner, out);
    return check_launch("geglu_kernel");
}

static int launch_softmax_rows(const float* s, long long rows, int L, long long lds, float scale, void* out,
                               int out_dtype, long long ldo, int causal_sq, void* stream) {
    SDB_REQUIRE(s && out && rows > 0 && L > 0 && causal_sq >= 0, "softmax_rows: bad args");
    SDB_REQUIRE(rows < (1LL << 31), "softmax_rows: too many rows");
    int threads = L >= 1024 ? 256 : (L >= 256 ? 128 : 32);
    if (out_dtype == SDB_BF16) launch_pdl(softmax_rows_kernel<true>, dim3((unsigned)rows), dim3(threads), 0, (cudaStream_t)stream, s, L, lds, scale, out, ldo, causal_sq);
    else launch_pdl(softmax_rows_kernel<false>, dim3((unsigned)rows), dim3(threads), 0, (cudaStream_t)stream, s, L, lds, scale, out, ldo, causal_sq);
    return check_launch("softmax_rows_kernel");
}

int sdb_softmax_rows(const float* s, long long rows, int L, long long lds, float scale, void* out,
                     int out_dtype, long long ldo, void* stream) {
    return launch_softmax_rows(s, rows, L, lds, scale, out, out_dtype, ldo, 0, stream);
}

int sdb_softmax_rows_causal(const float* s, long long rows, int L, int Sq, long long lds, float scale, void* out,
                            int out_dtype, long long ldo, void* stream) {
    SDB_REQUIRE(Sq > 0, "softmax_rows_causal: Sq must be positive");
    return launch_softmax_rows(s, rows, L, lds, scale, out, out_dtype, ldo, Sq, stream);
}

int sdb_add_rowvec(const float* x, const float* rowvec, long long ldv, int N, long long HW, int C, void* out,
                   int out_dtype, void* stream) {
    SDB_REQUIRE(x && rowvec && out && N > 0 && HW > 0 && C > 0 && C % 4 == 0, "add_rowvec: bad args");
    long long total = (long long)N * HW * (C / 4);
    int threads = 256, blocks = grid_for(total, threads);
    if (out_dtype == SDB_BF16) launch_pdl(add_rowvec_kernel<true>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, rowvec, ldv, HW, C, total, out);
    else launch_pdl(add_rowvec_kernel<false>, dim3(blocks), dim3(threads), 0, (cudaStream_t)stream, x, rowvec, ldv, HW, C, total, out);
    return check_launch("add_rowvec_kernel");
}

int sdb_add(const float* a, const float* b, float* out, long long n, void* stream) {
    SDB_REQUIRE(a && b && out && n > 0, "add: bad args");
    launch_pdl(add_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, a, b, out, n);
    return check_launch("add_kernel");
}

int sdb_timestep_embedding(const float* t, const float* freqs, int B, int half, int round_fp16, float* emb,
                           void* stream) {
    SDB_REQUIRE(t && freqs && emb && B > 0 && half > 0, "timestep_embedding: bad args");
    int n = B * half;
    launch_pdl(timestep_embedding_kernel, dim3(ceil_div(n, 256)), dim3(256), 0, (cudaStream_t)stream, t, freqs, B, half, round_fp16, emb);
    return check_launch("timestep_embedding_kernel");
}

int sdb_gather_rows(const float* table, const long long* idx, int B, int dim, float* out, void* stream) {
    SDB_REQUIRE(table && idx && out && B > 0 && dim > 0, "gather_rows: bad args");
    launch_pdl(gather_rows_kernel, dim3(ceil_div(B * dim, 256)), dim3(256), 0, (cudaStream_t)stream, table, idx, B, dim, out);
    return check_launch("gather_rows_kernel");
}

int sdb_skinny_linear(const float* x, int M, int K, const float* W, const float* bias, int N,
                      int act_in, int act_out, float* y, void* stream) {
    return launch_skinny<false>(x, M, K, W, bias, N, act_in, act_out, y, stream);
}

int sdb_skinny_linear_bf16w(const float* x, int M, int K, const void* W, const float* bias, int N,
                            int act_in, int act_out, float* y, void* stream) {
    return launch_skinny<true>(x, M, K, W, bias, N, act_in, act_out, y, stream);
}

int sdb_ddim_step(const float* x, const float* e_cond, const float* e_uncond, float cfg_scale,
                  const float* noise, float sqrt_at, float sqrt_aprev, float dir_coef, float sigma_t,
                  float sqrt_one_minus_at, float temperature, float* x_prev, float* pred_x0, long long n,
                  void* stream) {
    SDB_REQUIRE(x && e_cond && x_prev && pred_x0 && n > 0, "ddim_step: bad args");
    SDB_REQUIRE(noise || sigma_t == 0.0f, "ddim_step: sigma_t != 0 needs a noise tensor");
    const DdimStep op{{e_cond, x, e_uncond, noise, nullptr}, {x_prev, pred_x0}, cfg_scale, sqrt_at, sqrt_aprev, dir_coef, sigma_t,
                      sqrt_one_minus_at, temperature};
    return launch_sampler_update("ddim_step", op, n, n, stream);
}

int sdb_ddim_xprev(const float* pred_x0, const float* e_cond, const float* e_uncond, float cfg_scale, const float* noise,
                   float sqrt_aprev, float dir_coef, float sigma_t, float temperature, float* x_prev, long long n, void* stream) {
    SDB_REQUIRE(pred_x0 && e_cond && x_prev && n > 0, "ddim_xprev: bad args");
    SDB_REQUIRE(noise || sigma_t == 0.0f, "ddim_xprev: sigma_t != 0 needs a noise tensor");
    const DdimStep op{{e_cond, nullptr, e_uncond, noise, pred_x0}, {x_prev, nullptr}, cfg_scale, 1.0f, sqrt_aprev, dir_coef, sigma_t, 0.0f,
                      temperature};
    return launch_sampler_update("ddim_xprev", op, n, n, stream);
}

int sdb_plms_step(const float* x, const float* e, const float* e_uncond, float cfg_scale, const float* e_old1, const float* e_old2,
                  const float* e_old3, int order, const float* noise, float sqrt_at, float sqrt_aprev, float dir_coef, float sigma_t,
                  float sqrt_one_minus_at, float temperature, float* e_out, float* e_prime_out, float* pred_x0, float* x_prev,
                  long long n, void* stream) {
    SDB_REQUIRE(x && e && n > 0, "plms_step: null input or empty problem (n=%lld)", n);
    SDB_REQUIRE(order >= 0 && order <= 4, "plms_step: order %d outside 0..4", order);
    SDB_REQUIRE(e_out || e_prime_out || pred_x0 || x_prev, "plms_step: no output requested");
    SDB_REQUIRE(order < 2 || e_old1, "plms_step: order %d needs e_old1", order);
    SDB_REQUIRE(order != 0 || e_old1, "plms_step: order 0 needs the first evaluation in e_old1");
    SDB_REQUIRE(order < 3 || e_old2, "plms_step: order %d needs e_old2", order);
    SDB_REQUIRE(order < 4 || e_old3, "plms_step: order 4 needs e_old3");
    SDB_REQUIRE(noise || sigma_t == 0.0f, "plms_step: sigma_t != 0 needs a noise tensor");
    const float* o1 = (order == 0 || order >= 2) ? e_old1 : nullptr;
    const float* o2 = order >= 3 ? e_old2 : nullptr;
    const float* o3 = order >= 4 ? e_old3 : nullptr;
    const PlmsStep op{{x, e, e_uncond, o1, o2, o3, noise}, {e_out, e_prime_out, pred_x0, x_prev}, cfg_scale, order, sqrt_at,
                      sqrt_aprev, dir_coef, sigma_t, sqrt_one_minus_at, temperature};
    return launch_sampler_update("plms_step", op, n, n, stream);
}

int sdb_dpm_solver_step(const float* x, const float* e, const float* e_uncond, float cfg_scale, float sigma_s, float alpha_s,
                        const float* m1, const float* m2, int order, float c_x, float c_0, float c_1, float c_2, float inv_r0,
                        float inv_r1, float c_r, float c_d2, float* x_next, float* m0_out, long long n, void* stream) {
    SDB_REQUIRE(x && e && n > 0, "dpm_solver_step: null input or empty problem (n=%lld)", n);
    SDB_REQUIRE(order >= 1 && order <= 3, "dpm_solver_step: order %d outside 1..3", order);
    SDB_REQUIRE(order < 2 || m1, "dpm_solver_step: order %d needs m1", order);
    SDB_REQUIRE(order < 3 || m2, "dpm_solver_step: order 3 needs m2");
    SDB_REQUIRE(x_next || m0_out, "dpm_solver_step: no output requested");
    const float* h1 = order >= 2 ? m1 : nullptr;
    const float* h2 = order >= 3 ? m2 : nullptr;
    const DpmSolverStep op{{x, e, e_uncond, h1, h2}, {x_next, m0_out}, cfg_scale, order,
                           {sigma_s, alpha_s, c_x, c_0, c_1, c_2, inv_r0, inv_r1, c_r, c_d2}};
    return launch_sampler_update("dpm_solver_step", op, n, n, stream);
}

int sdb_ddpm_step(const float* x, const float* eps, const float* x0_in, const float* noise, const long long* t,
                  const float* table, int T, int clip, float temperature, float* x_prev, float* x0_out, int B, long long per,
                  void* stream) {
    SDB_REQUIRE(x && t && table, "ddpm_step: null pointer");
    SDB_REQUIRE(eps || x0_in, "ddpm_step: needs eps or a given x0");
    SDB_REQUIRE(x_prev || x0_out, "ddpm_step: no output requested");
    SDB_REQUIRE(T > 0 && B > 0 && per > 0, "ddpm_step: bad shape B=%d per=%lld T=%d", B, per, T);
    const DdpmStep op{{x, x0_in ? nullptr : eps, x0_in, noise}, {x_prev, x0_out}, t, table, T, clip, temperature, per};
    return launch_sampler_update("ddpm_step", op, (long long)B * per, per, stream);
}

int sdb_inpaint_blend(const float* x0, const float* noise, const float* a, const float* c, const float* mask, const float* img,
                      int B, int C, int Cm, long long HW, float* out, void* stream) {
    SDB_REQUIRE(x0 && noise && a && c && mask && img && out, "inpaint_blend: null pointer");
    SDB_REQUIRE(B > 0 && C > 0 && HW > 0 && (Cm == 1 || Cm == C), "inpaint_blend: bad shape B=%d C=%d Cm=%d", B, C, Cm);
    const long long n = (long long)B * C * HW;
    launch_pdl(inpaint_blend_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, x0, noise, a, c, mask, img, C, Cm, HW, n, out);
    return check_launch("inpaint_blend_kernel");
}

int sdb_diag_gaussian(const float* moments, const float* noise, int N, int C, long long HW, float* mean, float* logvar,
                      float* stdv, float* var, float* sample, void* stream) {
    SDB_REQUIRE(moments && mean && logvar && stdv && var, "diag_gaussian: null pointer");
    SDB_REQUIRE(N > 0 && C > 0 && HW > 0, "diag_gaussian: empty problem");
    SDB_REQUIRE((sample == nullptr) == (noise == nullptr), "diag_gaussian: sample and noise go together");
    const long long n = (long long)N * C * HW;
    launch_pdl(diag_gaussian_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream,
        moments, noise, C, HW, n, mean, logvar, stdv, var, sample);
    return check_launch("diag_gaussian_kernel");
}

int sdb_q_sample(const float* x0, const float* noise, const float* a, const float* c, int B, long long per, float* out,
                 void* stream) {
    SDB_REQUIRE(x0 && noise && a && c && out, "q_sample: null pointer");
    SDB_REQUIRE(B > 0 && per > 0, "q_sample: empty problem");
    const long long n = (long long)B * per;
    launch_pdl(q_sample_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream, x0, noise, a, c, per, n, out);
    return check_launch("q_sample_kernel");
}

int sdb_scale_shift_affine(const float* gamma, const float* beta, const float* ss, long long ld_ss, int N, int C,
                           float* gamma_out, float* beta_out, void* stream) {
    SDB_REQUIRE(gamma && beta && ss && gamma_out && beta_out, "scale_shift_affine: null pointer");
    SDB_REQUIRE(N > 0 && C > 0 && ld_ss >= 2LL * C, "scale_shift_affine: bad shape N=%d C=%d ld=%lld", N, C, ld_ss);
    const long long n = (long long)N * C;
    launch_pdl(scale_shift_affine_kernel, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)stream,
        gamma, beta, ss, ld_ss, C, n, gamma_out, beta_out);
    return check_launch("scale_shift_affine_kernel");
}

int sdb_avgpool2x2(const float* x, int N, int H, int W, int C, void* out, int out_dtype, void* stream) {
    SDB_REQUIRE(x && out, "avgpool2x2: null pointer");
    SDB_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && H % 2 == 0 && W % 2 == 0 && C % 4 == 0, "avgpool2x2: bad shape %dx%dx%dx%d", N, H, W, C);
    SDB_REQUIRE(out_dtype == SDB_F32 || out_dtype == SDB_BF16, "avgpool2x2: bad out_dtype");
    const long long tv = (long long)N * (H / 2) * (W / 2) * (C / 4);
    if (out_dtype == SDB_BF16) launch_pdl(avgpool2x2_kernel<true>, dim3(grid_for(tv, 256)), dim3(256), 0, (cudaStream_t)stream, x, H, W, C, tv, out);
    else launch_pdl(avgpool2x2_kernel<false>, dim3(grid_for(tv, 256)), dim3(256), 0, (cudaStream_t)stream, x, H, W, C, tv, out);
    return check_launch("avgpool2x2_kernel");
}

}  // extern "C"
