// sdb200 — nearest-codebook vector quantisation (taming's VectorQuantizer2.forward in eval, legacy=True, and
// get_codebook_entry; ldm/tamming/quantize.py:213-329), the quantizer of the VQ-regularised first stage.
//
// The reference forms the full [M, n_e] fp32 distance matrix d = (||z||^2 + ||w||^2) - 2 z.w and reads it back with
// argmin.  Here a thread keeps the running minimum of its rows in registers while the codebook streams through shared
// memory, so the matrix is never written.  fp32 SIMT in both compute modes: tensor-core operands would change which
// code wins, and with D <= 16 they would be mostly padding.
//
//   vq_search_kernel    one CTA = VQ_ROWS rows x one codebook slice; per (slice, row) the minimum (d, index)
//   vq_finalize_kernel  per row: merge the slice minima (lexicographic, NaN first), gather the code, write the
//                       index, z_q = z + (e - z) and the fp64 partial of the commitment loss; the last CTA (ticket)
//                       folds the partials in a fixed order
//   vq_gather_kernel    get_codebook_entry: W[idx] in NCHW or NHWC, NaN rows for out-of-range indices
#include "common.cuh"

namespace sdb {

constexpr int VQ_THREADS = 128;
constexpr int VQ_RPT = 2;                          // rows per thread
constexpr int VQ_ROWS = VQ_THREADS * VQ_RPT;       // rows per CTA
constexpr int VQ_CHUNK = 256;                      // codes staged in shared memory per pass
constexpr int VQ_MIN_SLICE = 256;                  // smallest codebook slice a CTA scans
constexpr int VQ_TARGET_CTAS = 148 * 8;            // 8 resident 4-warp CTAs on each of the B200's 148 SMs
constexpr int VQ_FIN_THREADS = 256;
constexpr int VQ_FIN_MAX_CTAS = 1024;

// Codebook slices for M rows and n_e codes: enough (row block, slice) CTAs to fill the GPU when M alone does not,
// never a slice shorter than VQ_MIN_SLICE codes.  A function of (M, n_e) only, so results are reproducible.
static int vq_splits(long long M, int n_e) {
    const long long blocks_m = ceil_div_ll(M, VQ_ROWS);
    long long s = ceil_div_ll(VQ_TARGET_CTAS, blocks_m);
    const long long smax = n_e / VQ_MIN_SLICE > 1 ? n_e / VQ_MIN_SLICE : 1;
    if (s > smax) s = smax;
    if (s < 1) s = 1;
    const int slice = (int)ceil_div_ll(n_e, s);
    return (int)ceil_div_ll(n_e, slice);           // no empty slice
}

static int vq_fin_ctas(long long M) {
    const long long g = ceil_div_ll(M, VQ_FIN_THREADS);
    return (int)(g < VQ_FIN_MAX_CTAS ? g : VQ_FIN_MAX_CTAS);
}

static long long vq_cand_bytes(long long M, int S) { return ceil_div_ll(8 * (long long)S * M, 256) * 256; }

// z row m = (n, p) of an [N, D, HW] (NCHW) or [N, HW, D] (NHWC) tensor, element k
__device__ __forceinline__ long long vq_off(long long m, int k, int D, int HW, bool nhwc) {
    if (nhwc) return m * D + k;
    const long long n = m / HW, p = m - n * HW;
    return (n * D + k) * HW + p;
}

// (d, j) ranks before (bd, bj): NaN first (torch.argmin), then smaller d, then the smaller index
__device__ __forceinline__ bool vq_better(float d, int j, float bd, int bj) {
    const bool dn = d != d, bn = bd != bd;
    if (dn != bn) return dn;
    if (dn) return j < bj;
    return d < bd || (d == bd && j < bj);
}

template <int D>
__global__ void __launch_bounds__(VQ_THREADS)
vq_search_kernel(const float* __restrict__ z, int z_nhwc, long long M, int HW, const float* __restrict__ W, int n_e,
                 int slice_len, float2* __restrict__ cand) {
    constexpr int DP = (D + 1 + 3) / 4 * 4;        // smem code row: w[0..D-1], ||w||^2, zero padding to 16 bytes
    __shared__ __align__(16) float sw[VQ_CHUNK * DP];
    pdl_trigger();
    pdl_wait();
    const int s = blockIdx.y;
    const int j0 = s * slice_len;
    const int j1 = min(n_e, j0 + slice_len);
    float zr[VQ_RPT][D], zz[VQ_RPT], best[VQ_RPT];
    int bi[VQ_RPT];
#pragma unroll
    for (int r = 0; r < VQ_RPT; ++r) {
        const long long m = (long long)blockIdx.x * VQ_ROWS + r * VQ_THREADS + threadIdx.x;
        float acc = 0.f;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            zr[r][k] = m < M ? __ldg(z + vq_off(m, k, D, HW, z_nhwc != 0)) : 0.f;
            acc = k == 0 ? __fmul_rn(zr[r][k], zr[r][k]) : __fadd_rn(acc, __fmul_rn(zr[r][k], zr[r][k]));
        }
        zz[r] = acc;
        best[r] = __int_as_float(0x7f800000);      // +inf with index j0: a row whose every d is +inf gets the first code
        bi[r] = j0;
    }
    for (int c0 = j0; c0 < j1; c0 += VQ_CHUNK) {
        const int cn = min(VQ_CHUNK, j1 - c0);
        __syncthreads();
        for (int t = threadIdx.x; t < cn; t += VQ_THREADS) {
            const float* w = W + (long long)(c0 + t) * D;
            float* o = sw + t * DP;
            float ee = 0.f;
#pragma unroll
            for (int k = 0; k < D; ++k) {
                const float v = __ldg(w + k);
                o[k] = v;
                ee = k == 0 ? __fmul_rn(v, v) : __fadd_rn(ee, __fmul_rn(v, v));
            }
            o[D] = ee;
#pragma unroll
            for (int k = D + 1; k < DP; ++k) o[k] = 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int j = 0; j < cn; ++j) {
            float w[DP];
#pragma unroll
            for (int q = 0; q < DP / 4; ++q) {
                const float4 v = reinterpret_cast<const float4*>(sw + j * DP)[q];
                w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
            }
#pragma unroll
            for (int r = 0; r < VQ_RPT; ++r) {
                float dot = __fmul_rn(zr[r][0], w[0]);
#pragma unroll
                for (int k = 1; k < D; ++k) dot = fmaf(zr[r][k], w[k], dot);
                // (zz + ee) - 2 dot in the reference's association; 2 dot is exact, so one fma rounds the same
                const float d = fmaf(-2.f, dot, __fadd_rn(zz[r], w[D]));
                // codes are visited in ascending order: a tie keeps the earlier one, a NaN replaces any number
                if (d < best[r] || (d != d && best[r] == best[r])) { best[r] = d; bi[r] = c0 + j; }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < VQ_RPT; ++r) {
        const long long m = (long long)blockIdx.x * VQ_ROWS + r * VQ_THREADS + threadIdx.x;
        if (m < M) cand[(long long)s * M + m] = make_float2(best[r], __int_as_float(bi[r]));
    }
}

__global__ void __launch_bounds__(VQ_FIN_THREADS)
vq_finalize_kernel(const float* __restrict__ z, int z_nhwc, long long M, int HW, int D, const float* __restrict__ W,
                   const float2* __restrict__ cand, int S, float* __restrict__ zq, int zq_nhwc, long long* __restrict__ idx,
                   float* __restrict__ loss, float beta, double* __restrict__ partial, int* __restrict__ counter) {
    __shared__ double red[VQ_FIN_THREADS];
    __shared__ int s_last;
    pdl_trigger();
    pdl_wait();
    double sq = 0.0;
    for (long long m = (long long)blockIdx.x * VQ_FIN_THREADS + threadIdx.x; m < M; m += (long long)gridDim.x * VQ_FIN_THREADS) {
        float2 c = cand[m];
        float bd = c.x;
        int bj = __float_as_int(c.y);
        for (int s = 1; s < S; ++s) {
            c = cand[(long long)s * M + m];
            if (vq_better(c.x, __float_as_int(c.y), bd, bj)) { bd = c.x; bj = __float_as_int(c.y); }
        }
        if (idx) idx[m] = bj;
        const float* e = W + (long long)bj * D;
        for (int k = 0; k < D; ++k) {
            const float zv = __ldg(z + vq_off(m, k, D, HW, z_nhwc != 0));
            const float diff = __fsub_rn(__ldg(e + k), zv);
            if (zq) zq[vq_off(m, k, D, HW, zq_nhwc != 0)] = __fadd_rn(zv, diff);   // straight-through z + (e - z)
            sq += (double)__fmul_rn(diff, diff);
        }
    }
    if (!loss) return;
    red[threadIdx.x] = sq;
    __syncthreads();
    for (int o = VQ_FIN_THREADS / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = red[0];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(counter, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    double t = 0.0;
    for (int b = threadIdx.x; b < (int)gridDim.x; b += VQ_FIN_THREADS) t += __ldcg(partial + b);
    red[threadIdx.x] = t;
    __syncthreads();
    for (int o = VQ_FIN_THREADS / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        // legacy: mean((e - z)^2) + beta * mean((e - z)^2), the two means being the same fp32 number
        const float mse = (float)(red[0] / ((double)M * D));
        *loss = __fadd_rn(mse, __fmul_rn(beta, mse));
        *counter = 0;
    }
}

__global__ void __launch_bounds__(256)
vq_gather_kernel(const long long* __restrict__ idx, long long M, const float* __restrict__ W, int n_e, int D,
                 float* __restrict__ out, int out_nhwc, int HW) {
    pdl_trigger();
    pdl_wait();
    for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < M; m += (long long)gridDim.x * blockDim.x) {
        const long long j = __ldg(idx + m);
        const bool ok = j >= 0 && j < n_e;
        for (int k = 0; k < D; ++k)
            out[vq_off(m, k, D, HW, out_nhwc != 0)] = ok ? __ldg(W + j * D + k) : __int_as_float(0x7fc00000);
    }
}

template <int D>
static void launch_search(dim3 grid, cudaStream_t st, const float* z, int z_nhwc, long long M, int HW, const float* W, int n_e,
                          int slice, float2* cand) {
    launch_pdl(vq_search_kernel<D>, grid, dim3(VQ_THREADS), 0, st, z, z_nhwc, M, HW, W, n_e, slice, cand);
}

}  // namespace sdb

using namespace sdb;

extern "C" {

long long sdb_vq_ws_bytes(long long M, int n_e) {
    SDB_REQUIRE(M > 0 && n_e > 0, "vq_ws_bytes: bad shape M=%lld n_e=%d", M, n_e);
    return vq_cand_bytes(M, vq_splits(M, n_e)) + 8LL * VQ_FIN_MAX_CTAS;
}

int sdb_vq_quantize(const float* z, int z_layout, int N, int HW, int D, const float* codebook, int n_e, float beta,
                    float* z_q, int zq_layout, long long* idx, float* loss, void* ws, int* counters, void* stream) {
    SDB_REQUIRE(z && codebook && ws, "vq_quantize: null pointer");
    SDB_REQUIRE(z_q || idx || loss, "vq_quantize: no output requested");
    SDB_REQUIRE(!loss || counters, "vq_quantize: the loss needs a ticket counter");
    SDB_REQUIRE(N > 0 && HW > 0 && n_e > 0, "vq_quantize: bad shape N=%d HW=%d n_e=%d", N, HW, n_e);
    SDB_REQUIRE(D >= 1 && D <= 16, "vq_quantize: codebook dimension D=%d outside [1, 16]", D);
    SDB_REQUIRE((z_layout == SDB_NCHW || z_layout == SDB_NHWC) && (zq_layout == SDB_NCHW || zq_layout == SDB_NHWC),
                "vq_quantize: bad layout %d / %d", z_layout, zq_layout);
    const long long M = (long long)N * HW;
    SDB_REQUIRE(M < (1LL << 40), "vq_quantize: M=%lld too large", M);
    const int S = vq_splits(M, n_e);
    const int slice = (int)ceil_div_ll(n_e, S);
    float2* cand = reinterpret_cast<float2*>(ws);
    double* partial = reinterpret_cast<double*>(reinterpret_cast<char*>(ws) + vq_cand_bytes(M, S));
    const dim3 grid((unsigned)ceil_div_ll(M, VQ_ROWS), (unsigned)S);
    const cudaStream_t st = (cudaStream_t)stream;
    const int zn = z_layout == SDB_NHWC;
    switch (D) {
#define VQ_CASE(d) case d: launch_search<d>(grid, st, z, zn, M, HW, codebook, n_e, slice, cand); break;
        VQ_CASE(1) VQ_CASE(2) VQ_CASE(3) VQ_CASE(4) VQ_CASE(5) VQ_CASE(6) VQ_CASE(7) VQ_CASE(8)
        VQ_CASE(9) VQ_CASE(10) VQ_CASE(11) VQ_CASE(12) VQ_CASE(13) VQ_CASE(14) VQ_CASE(15) VQ_CASE(16)
#undef VQ_CASE
    }
    int rc = check_launch("vq_search_kernel");
    if (rc) return rc;
    launch_pdl(vq_finalize_kernel, dim3(vq_fin_ctas(M)), dim3(VQ_FIN_THREADS), 0, st, z, zn, M, HW, D, codebook,
               (const float2*)cand, S, z_q, (int)(zq_layout == SDB_NHWC), idx, loss, beta, partial, counters);
    return check_launch("vq_finalize_kernel");
}

int sdb_vq_codebook_gather(const long long* idx, long long M, const float* codebook, int n_e, int D, float* out, int out_layout,
                           int HW, void* stream) {
    SDB_REQUIRE(idx && codebook && out, "vq_codebook_gather: null pointer");
    SDB_REQUIRE(M > 0 && n_e > 0 && HW > 0 && M % HW == 0, "vq_codebook_gather: bad shape M=%lld n_e=%d HW=%d", M, n_e, HW);
    SDB_REQUIRE(D >= 1 && D <= 16, "vq_codebook_gather: codebook dimension D=%d outside [1, 16]", D);
    SDB_REQUIRE(out_layout == SDB_NCHW || out_layout == SDB_NHWC, "vq_codebook_gather: bad layout %d", out_layout);
    const long long g = ceil_div_ll(M, 256);
    launch_pdl(vq_gather_kernel, dim3((unsigned)(g < 4096 ? g : 4096)), dim3(256), 0, (cudaStream_t)stream, idx, M, codebook, n_e, D,
               out, (int)(out_layout == SDB_NHWC), HW);
    return check_launch("vq_gather_kernel");
}

}  // extern "C"
