// sdb200 — the conditioning stages of the latent-diffusion family beside CLIP (ldm/modules/encoders/modules.py,
// ldm/modules/x_transformer.py): the bounded embedding lookup of TransformerWrapper / ClassEmbedder and the resize of
// SpatialRescaler.
//
//   embed_rows_kernel   out[i] = table[ids[i]] (+ pos[i % seq_len]): token_emb(x) + pos_emb(x) in one pass, and
//                       nn.Embedding alone; an id outside [0, vocab) gives a NaN row and is never dereferenced
//   interp_kernel       one F.interpolate stage on NCHW fp32 (align_corners=False, recompute_scale_factor=None) with the
//                       coordinate rules and evaluation order of torch's CUDA kernels (upsample_nearest2d,
//                       upsample_bilinear2d, upsample_bicubic2d, adaptive_avg_pool2d), optionally followed by a 1x1
//                       channel map computed from the interpolated pixel in registers
#include "common.cuh"

namespace sdb {

constexpr int EMB_THREADS = 128;
constexpr int INTERP_THREADS = 256;
constexpr int INTERP_COUT = 4;                     // output channels a thread of the channel-map kernel accumulates

__global__ void __launch_bounds__(EMB_THREADS)
embed_rows_kernel(const float* __restrict__ table, const long long* __restrict__ ids, long long n, int dim, int vocab,
                  const float* __restrict__ pos, int seq_len, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    for (long long r = blockIdx.x; r < n; r += gridDim.x) {
        const long long j = __ldg(ids + r);
        const bool ok = j >= 0 && j < vocab;
        const float* p = pos ? pos + (r % seq_len) * dim : nullptr;
        float* dst = out + r * dim;
        for (int c = threadIdx.x; c < dim; c += EMB_THREADS) {
            float v = ok ? __ldg(table + j * dim + c) : __int_as_float(0x7fc00000);
            if (p) v = __fadd_rn(v, __ldg(p + c));
            dst[c] = v;
        }
    }
}

// Where an output pixel reads its input and with which weights; which fields are used depends on the mode.
//   nearest   y[0], x[0]
//   bilinear  rows y[0], y[1] with weights wy[0], wy[1]; likewise along x
//   bicubic   rows y[0..3] (clamped) with weights wy[0..3]; likewise along x
//   area      window rows [y[0], y[1]), columns [x[0], x[1])
struct InterpPix {
    int y[4], x[4];
    float wy[4], wx[4];
};

// torch's area_pixel_compute_source_index with align_corners=False, written as torch writes it so that the compiler
// forms the same fused multiply-add
__device__ __forceinline__ float interp_src(float scale, int dst, bool cubic) {
    const float s = scale * (dst + 0.5f) - 0.5f;
    return (!cubic && s < 0.0f) ? 0.0f : s;
}

// get_cubic_upsample_coefficients, A = -0.75
__device__ __forceinline__ void cubic_coeffs(float t, float* c) {
    const float A = -0.75f;
    const float x1 = t + 1.0f, x2 = 1.0f - t, x3 = x2 + 1.0f;
    c[0] = ((A * x1 - 5 * A) * x1 + 8 * A) * x1 - 4 * A;
    c[1] = ((A + 2) * t - (A + 3)) * t * t + 1;
    c[2] = ((A + 2) * x2 - (A + 3)) * x2 * x2 + 1;
    c[3] = ((A * x3 - 5 * A) * x3 + 8 * A) * x3 - 4 * A;
}

// adaptive_avg_pool2d's window bounds (start_index / end_index)
__device__ __forceinline__ int area_start(int o, int out, int in) { return (int)floorf(__fdiv_rn((float)(o * in), (float)out)); }
__device__ __forceinline__ int area_end(int o, int out, int in) { return (int)ceilf(__fdiv_rn((float)((o + 1) * in), (float)out)); }

template <int MODE>
__device__ __forceinline__ void interp_axis(int o, int in, int out, float scale, int* idx, float* w) {
    if (MODE == SDB_INTERP_NEAREST) {
        idx[0] = min((int)floorf(o * scale), in - 1);
    } else if (MODE == SDB_INTERP_BILINEAR) {
        const float r = interp_src(scale, o, false);
        const int i0 = (int)r;
        const float l1 = r - i0;
        idx[0] = i0;
        idx[1] = i0 + (i0 < in - 1 ? 1 : 0);
        w[0] = 1.0f - l1;
        w[1] = l1;
    } else if (MODE == SDB_INTERP_BICUBIC) {
        const float r = interp_src(scale, o, true);
        const int i0 = (int)floorf(r);
        cubic_coeffs(r - i0, w);
#pragma unroll
        for (int k = 0; k < 4; ++k) idx[k] = max(min(i0 - 1 + k, in - 1), 0);
    } else {
        idx[0] = area_start(o, out, in);
        idx[1] = area_end(o, out, in);
    }
}

template <int MODE>
__device__ __forceinline__ float interp_eval(const float* __restrict__ p, int W, const InterpPix& q) {
    if (MODE == SDB_INTERP_NEAREST) {
        return __ldg(p + (long long)q.y[0] * W + q.x[0]);
    } else if (MODE == SDB_INTERP_BILINEAR) {
        const float* r0 = p + (long long)q.y[0] * W;
        const float* r1 = p + (long long)q.y[1] * W;
        // upsample_bilinear2d_out_frame's h0l * (w0l * a + w1l * b) + h1l * (w0l * c + w1l * d)
        return q.wy[0] * (q.wx[0] * __ldg(r0 + q.x[0]) + q.wx[1] * __ldg(r0 + q.x[1])) +
               q.wy[1] * (q.wx[0] * __ldg(r1 + q.x[0]) + q.wx[1] * __ldg(r1 + q.x[1]));
    } else if (MODE == SDB_INTERP_BICUBIC) {
        float row[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float* r = p + (long long)q.y[k] * W;
            row[k] = __ldg(r + q.x[0]) * q.wx[0] + __ldg(r + q.x[1]) * q.wx[1] + __ldg(r + q.x[2]) * q.wx[2] +
                     __ldg(r + q.x[3]) * q.wx[3];
        }
        return row[0] * q.wy[0] + row[1] * q.wy[1] + row[2] * q.wy[2] + row[3] * q.wy[3];
    } else {
        float sum = 0.0f;
        for (int y = q.y[0]; y < q.y[1]; ++y) {
            const float* r = p + (long long)y * W;
            for (int x = q.x[0]; x < q.x[1]; ++x) sum = __fadd_rn(sum, __ldg(r + x));
        }
        return __fdiv_rn(__fdiv_rn(sum, (float)(q.y[1] - q.y[0])), (float)(q.x[1] - q.x[0]));
    }
}

// grid.x walks the OH*OW output pixels (32-bit: checked on the host), grid.y the output planes: [N*C] without the channel
// map, [N * ceil(Cout / INTERP_COUT)] with it.  A thread sets up its pixel's taps once and reuses them for every plane.
template <int MODE, bool MAP>
__global__ void __launch_bounds__(INTERP_THREADS)
interp_kernel(const float* __restrict__ x, int C, int H, int W, int OH, int OW, float rh, float rw, long long planes,
              const float* __restrict__ wmap, const float* __restrict__ bias, int Cout, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const long long in_plane = (long long)H * W, out_plane = (long long)OH * OW;
    const int np = OH * OW;
    const int cgroups = MAP ? (Cout + INTERP_COUT - 1) / INTERP_COUT : 1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < np; i += gridDim.x * blockDim.x) {
        const int oy = i / OW, ox = i - oy * OW;
        InterpPix q;
        interp_axis<MODE>(oy, H, OH, rh, q.y, q.wy);
        interp_axis<MODE>(ox, W, OW, rw, q.x, q.wx);
        for (long long r = blockIdx.y; r < planes; r += gridDim.y) {
            if (!MAP) {
                out[r * out_plane + i] = interp_eval<MODE>(x + r * in_plane, W, q);
                continue;
            }
            const long long n = r / cgroups;
            const int co0 = (int)(r - n * cgroups) * INTERP_COUT;
            const int nco = min(INTERP_COUT, Cout - co0);
            float acc[INTERP_COUT];
#pragma unroll
            for (int k = 0; k < INTERP_COUT; ++k) acc[k] = 0.0f;
            // rows past Cout repeat the last row: computed, never stored
            const float* wr[INTERP_COUT];
#pragma unroll
            for (int k = 0; k < INTERP_COUT; ++k) wr[k] = wmap + (long long)(co0 + min(k, nco - 1)) * C;
            const float* xn = x + n * C * in_plane;
            for (int ci = 0; ci < C; ++ci) {
                const float v = interp_eval<MODE>(xn + ci * in_plane, W, q);
#pragma unroll
                for (int k = 0; k < INTERP_COUT; ++k) acc[k] = fmaf(__ldg(wr[k] + ci), v, acc[k]);
            }
#pragma unroll
            for (int k = 0; k < INTERP_COUT; ++k)
                if (k < nco)
                    out[(n * Cout + co0 + k) * out_plane + i] = bias ? __fadd_rn(acc[k], __ldg(bias + co0 + k)) : acc[k];
        }
    }
}

template <int MODE>
static void launch_interp(dim3 grid, cudaStream_t st, const float* x, int C, int H, int W, int OH, int OW, float rh, float rw,
                          long long planes, const float* wmap, const float* bias, int Cout, float* out) {
    if (wmap)
        launch_pdl(interp_kernel<MODE, true>, grid, dim3(INTERP_THREADS), 0, st, x, C, H, W, OH, OW, rh, rw, planes, wmap, bias,
                   Cout, out);
    else
        launch_pdl(interp_kernel<MODE, false>, grid, dim3(INTERP_THREADS), 0, st, x, C, H, W, OH, OW, rh, rw, planes, wmap,
                   bias, Cout, out);
}

// compute_scales_value<float>: 1 / scale_factor when one was given, else in / out
static float interp_scale(double s, int in, int out) { return s > 0.0 ? (float)(1.0 / s) : (float)in / out; }

}  // namespace sdb

using namespace sdb;

extern "C" {

int sdb_embed_rows(const float* table, const long long* ids, long long n_ids, int dim, int vocab, const float* pos_table,
                   int seq_len, float* out, void* stream) {
    SDB_REQUIRE(table && ids && out, "embed_rows: null pointer");
    SDB_REQUIRE(n_ids > 0 && dim > 0 && vocab > 0, "embed_rows: bad size n_ids=%lld dim=%d vocab=%d", n_ids, dim, vocab);
    SDB_REQUIRE(!pos_table || seq_len > 0, "embed_rows: a position table needs seq_len > 0 (got %d)", seq_len);
    const long long g = n_ids < (1LL << 20) ? n_ids : (1LL << 20);
    launch_pdl(embed_rows_kernel, dim3((unsigned)g), dim3(EMB_THREADS), 0, (cudaStream_t)stream, table, ids, n_ids, dim, vocab,
               pos_table, seq_len, out);
    return check_launch("embed_rows_kernel");
}

int sdb_interpolate_nchw(const float* x, int N, int C, int H, int W, int OH, int OW, int mode, double scale_h, double scale_w,
                         const float* weight, const float* bias, int Cout, float* out, void* stream) {
    SDB_REQUIRE(x && out, "interpolate: null pointer");
    SDB_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0 && OH > 0 && OW > 0,
                "interpolate: bad size N=%d C=%d in=(%d, %d) out=(%d, %d)", N, C, H, W, OH, OW);
    SDB_REQUIRE(mode >= SDB_INTERP_NEAREST && mode <= SDB_INTERP_AREA, "interpolate: unknown mode %d", mode);
    SDB_REQUIRE(scale_h >= 0.0 && scale_w >= 0.0, "interpolate: negative scale factor (%g, %g)", scale_h, scale_w);
    SDB_REQUIRE(weight || (Cout == 0 && !bias), "interpolate: Cout=%d or a bias without a channel-map weight", Cout);
    SDB_REQUIRE(!weight || Cout > 0, "interpolate: a channel-map weight needs Cout > 0 (got %d)", Cout);
    SDB_REQUIRE((long long)OH * OW < (1LL << 31), "interpolate: output (%d, %d) too large", OH, OW);
    SDB_REQUIRE(mode != SDB_INTERP_AREA || ((long long)OH * H < (1LL << 31) && (long long)OW * W < (1LL << 31)),
                "interpolate: area window bounds of (%d, %d) -> (%d, %d) overflow", H, W, OH, OW);
    const float rh = interp_scale(scale_h, H, OH), rw = interp_scale(scale_w, W, OW);
    const long long planes = weight ? (long long)N * ceil_div(Cout, INTERP_COUT) : (long long)N * C;
    const dim3 grid((unsigned)ceil_div_ll((long long)OH * OW, INTERP_THREADS), (unsigned)(planes < 65535 ? planes : 65535));
    const cudaStream_t st = (cudaStream_t)stream;
    switch (mode) {
        case SDB_INTERP_NEAREST: launch_interp<SDB_INTERP_NEAREST>(grid, st, x, C, H, W, OH, OW, rh, rw, planes, weight, bias, Cout, out); break;
        case SDB_INTERP_BILINEAR: launch_interp<SDB_INTERP_BILINEAR>(grid, st, x, C, H, W, OH, OW, rh, rw, planes, weight, bias, Cout, out); break;
        case SDB_INTERP_BICUBIC: launch_interp<SDB_INTERP_BICUBIC>(grid, st, x, C, H, W, OH, OW, rh, rw, planes, weight, bias, Cout, out); break;
        default: launch_interp<SDB_INTERP_AREA>(grid, st, x, C, H, W, OH, OW, rh, rw, planes, weight, bias, Cout, out); break;
    }
    return check_launch("interp_kernel");
}

}  // extern "C"
