// sdb200 — the patch-distributed ("split_input_params") branch of LatentDiffusion (ldm/diffusion/ddpm.py:1344-1437,
// 1097-1139): overlapping crops cut out of an image, run through a model as one batch, and stitched back with a
// border-weighted fold.
//
//   patch_unfold_kernel  torch.nn.Unfold(ks, stride) followed by view(B, C, kh, kw, L), written crop-major as
//                        [L*B, C, kh, kw] (row l*B + b) so that the L crops of a call form one batch; a pure copy
//   patch_fold_kernel    fold(o * weighting) / fold(weighting): one thread per output element gathers over the crops
//                        that cover it, in increasing l (row-major crop order, the order of torch's CUDA col2im), with both
//                        sums starting at 0.0f in fp32 and every product rounded on its own; no atomics, no workspace
#include "common.cuh"

namespace sdb {

constexpr int PATCH_THREADS = 256;

// (pixel blocks of a plane, planes) -> launch grid; gridDim.y is at most 65535, the kernels loop over the rest
static dim3 patch_grid(long long plane_px, long long planes) {
    return dim3((unsigned)ceil_div_ll(plane_px, PATCH_THREADS), (unsigned)(planes < 65535 ? planes : 65535));
}

// grid.y walks the [L*B*C] (crop, image, channel) planes, grid.x the kh*kw pixels of a plane (32-bit: checked on the host)
__global__ void __launch_bounds__(PATCH_THREADS)
patch_unfold_kernel(const float* __restrict__ x, int B, int C, int H, int W, int kh, int kw, int sh, int sw, int Lx,
                    long long planes, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const int np = kh * kw;
    for (long long r = blockIdx.y; r < planes; r += gridDim.y) {
        // out plane r = (l * B + b) * C + c
        const int c = (int)(r % C);
        const long long lb = r / C;
        const int b = (int)(lb % B);
        const int l = (int)(lb / B);
        const int ly = l / Lx, lx = l - ly * Lx;
        const float* src = x + (((long long)b * C + c) * H + (long long)ly * sh) * W + (long long)lx * sw;
        float* dst = out + r * np;
        for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < np; p += gridDim.x * blockDim.x) {
            const int u = p / kw, v = p - u * kw;
            dst[p] = __ldg(src + (long long)u * W + v);
        }
    }
}

// grid.y walks the [B*C] output planes, grid.x the OH*OW pixels of a plane (32-bit: checked on the host)
__global__ void __launch_bounds__(PATCH_THREADS)
patch_fold_kernel(const float* __restrict__ o, int B, int C, int KH, int KW, int Ly, int Lx, int SH, int SW, int OH, int OW,
                  const float* __restrict__ wpix, const float* __restrict__ wcrop, float* __restrict__ out) {
    pdl_trigger();
    pdl_wait();
    const long long crop = (long long)KH * KW, planes = (long long)B * C;
    const int np = OH * OW;
    for (long long bc = blockIdx.y; bc < planes; bc += gridDim.y) {
        const int c = (int)(bc % C);
        const long long b = bc / C;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < np; i += gridDim.x * blockDim.x) {
            const int yo = i / OW, xo = i - yo * OW;
            // crops ly with ly*SH <= yo < ly*SH + KH (col2im's h_col_start / h_col_end), likewise along x
            const int ly0 = yo < KH ? 0 : (yo - KH) / SH + 1, ly1 = min(yo / SH + 1, Ly);
            const int lx0 = xo < KW ? 0 : (xo - KW) / SW + 1, lx1 = min(xo / SW + 1, Lx);
            float acc = 0.0f, nrm = 0.0f;
            for (int ly = ly0; ly < ly1; ++ly) {
                for (int lx = lx0; lx < lx1; ++lx) {
                    const int l = ly * Lx + lx;
                    const long long p = (long long)(yo - ly * SH) * KW + (xo - lx * SW);
                    const float w = wcrop ? __fmul_rn(__ldg(wpix + p), __ldg(wcrop + l)) : __ldg(wpix + p);
                    const float v = __ldg(o + (((long long)l * B + b) * C + c) * crop + p);
                    acc = __fadd_rn(acc, __fmul_rn(v, w));
                    nrm = __fadd_rn(nrm, w);
                }
            }
            out[bc * np + i] = __fdiv_rn(acc, nrm);      // 0 / 0 = NaN where no crop covers the pixel, as in the reference
        }
    }
}

}  // namespace sdb

using namespace sdb;

extern "C" {

int sdb_patch_unfold(const float* x, int B, int C, int H, int W, int kh, int kw, int sh, int sw, float* out, void* stream) {
    SDB_REQUIRE(x && out, "patch_unfold: null pointer");
    SDB_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && kh > 0 && kw > 0 && sh > 0 && sw > 0,
                "patch_unfold: bad size B=%d C=%d H=%d W=%d ks=(%d, %d) stride=(%d, %d)", B, C, H, W, kh, kw, sh, sw);
    SDB_REQUIRE(kh <= H && kw <= W, "patch_unfold: crop (%d, %d) larger than the image (%d, %d)", kh, kw, H, W);
    SDB_REQUIRE((long long)kh * kw < (1LL << 31), "patch_unfold: crop (%d, %d) too large", kh, kw);
    const int Ly = (H - kh) / sh + 1, Lx = (W - kw) / sw + 1;
    SDB_REQUIRE((long long)Ly * Lx * B < (1LL << 31), "patch_unfold: %d x %d crops of %d images is too many", Ly, Lx, B);
    const long long planes = (long long)Ly * Lx * B * C;
    launch_pdl(patch_unfold_kernel, patch_grid((long long)kh * kw, planes), dim3(PATCH_THREADS), 0, (cudaStream_t)stream, x, B, C,
               H, W, kh, kw, sh, sw, Lx, planes, out);
    return check_launch("patch_unfold_kernel");
}

int sdb_patch_fold(const float* o, int B, int C, int KH, int KW, int Ly, int Lx, int SH, int SW, int OH, int OW,
                   const float* wpix, const float* wcrop, int L, float* out, void* stream) {
    SDB_REQUIRE(o && wpix && out, "patch_fold: null pointer");
    SDB_REQUIRE(B > 0 && C > 0 && KH > 0 && KW > 0 && Ly > 0 && Lx > 0 && SH > 0 && SW > 0 && OH > 0 && OW > 0,
                "patch_fold: bad size B=%d C=%d ks=(%d, %d) grid=(%d, %d) stride=(%d, %d) out=(%d, %d)", B, C, KH, KW, Ly, Lx,
                SH, SW, OH, OW);
    SDB_REQUIRE((long long)L == (long long)Ly * Lx, "patch_fold: L=%d is not Ly*Lx = %d*%d", L, Ly, Lx);
    SDB_REQUIRE((long long)(Ly - 1) * SH + KH <= OH && (long long)(Lx - 1) * SW + KW <= OW,
                "patch_fold: a %dx%d grid of (%d, %d) crops at stride (%d, %d) reaches outside (%d, %d)", Ly, Lx, KH, KW, SH, SW,
                OH, OW);
    SDB_REQUIRE((long long)OH * OW < (1LL << 31), "patch_fold: output (%d, %d) too large", OH, OW);
    launch_pdl(patch_fold_kernel, patch_grid((long long)OH * OW, (long long)B * C), dim3(PATCH_THREADS), 0, (cudaStream_t)stream,
               o, B, C, KH, KW, Ly, Lx, SH, SW, OH, OW, wpix, wcrop, out);
    return check_launch("patch_fold_kernel");
}

}  // extern "C"
