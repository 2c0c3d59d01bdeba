// Error plumbing, input pyramid packing and weight packing.
#include "common.cuh"
#include "../../include/mpnn.h"
#include <cstdarg>
#include <cstdio>

static thread_local char g_err[512] = "";

void mpnn_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int mpnn_check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        mpnn_set_error("%s: %s", what, cudaGetErrorString(e));
        return MPNN_ERR_CUDA;
    }
    return MPNN_OK;
}

extern "C" const char* mpnn_last_error(void) { return g_err; }
extern "C" int mpnn_version(void) { return 100; }

// --------------------------------------------------------------------------- //
// ToPyramid: strided subsample of NHWC fp32 into padded planes.
// One thread per (plane kg, valid pixel); 8 channels each.
// --------------------------------------------------------------------------- //
// CNT: the first min(*count, g.B) images only (g.B: the capacity the grid was sized for)
template <typename T, bool CNT = false>
__global__ void pack_input_kernel(const float* __restrict__ x0, int H0, int W0, int C0, int step,
                                  T* __restrict__ planes, int Cpad, Geom g, const int* __restrict__ count) {
    const int KG = Cpad / 8;
    if (CNT) g.B = min(max(*count, 0), g.B);
    const long long total = (long long)KG * g.B * g.H * g.W;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        int w = i % g.W;
        long long r = i / g.W;
        int h = r % g.H; r /= g.H;
        int n = r % g.B;
        int kg = r / g.B;
        const float* src = x0 + (((size_t)n * H0 + (size_t)h * step) * W0 + (size_t)w * step) * C0;
        float v[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            int ch = kg * 8 + c;
            v[c] = ch < C0 ? __ldg(src + ch) : 0.f;
        }
        Row8<T>::store(plane_row(planes, kg, g.P, row_of(g, n, h, w)), v);
    }
}

static int pack_input_impl(const float* x0, int B, int H0, int W0, int C0, int step,
                           void* planes, int Cpad, int G, int P, int dtype, const int* count, void* stream) {
    MPNN_REQUIRE(step >= 1 && H0 % step == 0 && W0 % step == 0, "pack_input: bad step %d", step);
    MPNN_REQUIRE(Cpad % 8 == 0 && Cpad >= C0, "pack_input: Cpad=%d C0=%d", Cpad, C0);
    Geom g = make_geom(B, H0 / step, W0 / step, G, P);
    MPNN_REQUIRE(G + g.rows <= P, "pack_input: P too small");
    long long total = (long long)(Cpad / 8) * B * g.H * g.W;
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    if (grid < 1) grid = 1;
    if (count) {
        MPNN_DISPATCH_DTYPE(dtype, (pack_input_kernel<T, true><<<grid, 256, 0, (cudaStream_t)stream>>>(
            x0, H0, W0, C0, step, (T*)planes, Cpad, g, count)));
    } else {
        MPNN_DISPATCH_DTYPE(dtype, (pack_input_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(
            x0, H0, W0, C0, step, (T*)planes, Cpad, g, nullptr)));
    }
    return mpnn_check_launch("pack_input");
}

extern "C" int mpnn_pack_input(const float* x0, int B, int H0, int W0, int C0, int step,
                               void* planes, int Cpad, int G, int P, int dtype, void* stream) {
    return pack_input_impl(x0, B, H0, W0, C0, step, planes, Cpad, G, P, dtype, nullptr, stream);
}

extern "C" int mpnn_pack_input_counted(const float* x0, int B, int H0, int W0, int C0, int step,
                                       void* planes, int Cpad, int G, int P, int dtype, const int* count,
                                       void* stream) {
    return pack_input_impl(x0, B, H0, W0, C0, step, planes, Cpad, G, P, dtype, count, stream);
}

// --------------------------------------------------------------------------- //
// MultiscaleLLN (lib/layer_types.py:126-147) on one pyramid scale of an RGB image: local luminance
//   lum(h, w) = sum_{|u|,|v| <= s} g(u, v) * (0.2126 R + 0.7152 G + 0.0722 B)(h + u, w + v)    (zero outside the image)
// with g(u, v) = exp(-(u^2 + v^2) / (2 sigma^2)) / (2 pi sigma^2), s = ceil(2 sigma); density = the same sum over
// an image of ones (so borders are normalised by the weight that falls inside); out = x / (lum / density + eps).
// x0 is the full-resolution NHWC image, the scale is its `step`-strided subsample (ToPyramid, :118-125);
// out is NHWC fp32 at the scale's size.  One thread per output pixel.
// --------------------------------------------------------------------------- //
__global__ void __launch_bounds__(256)
lln_kernel(const float* __restrict__ x0, int B, int H0, int W0, int step, float sigma, float eps, int s,
           float* __restrict__ out) {
    const int H = H0 / step, W = W0 / step;
    const int total = B * H * W;
    const float inv2s2 = 1.f / (2.f * sigma * sigma), norm = 1.f / (2.f * 3.14159265358979323846f * sigma * sigma);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int w = i % W, h = (i / W) % H, n = i / (W * H);
        float lum = 0.f, den = 0.f;
        for (int u = -s; u <= s; ++u) {
            const int hh = h + u;
            if (hh < 0 || hh >= H) continue;
            for (int v = -s; v <= s; ++v) {
                const int ww = w + v;
                if (ww < 0 || ww >= W) continue;
                const float gk = expf(-(float)(u * u + v * v) * inv2s2) * norm;
                const float* p = x0 + (((size_t)n * H0 + (size_t)hh * step) * W0 + (size_t)ww * step) * 3;
                lum = fmaf(gk, 0.2126f * __ldg(p) + 0.7152f * __ldg(p + 1) + 0.0722f * __ldg(p + 2), lum);
                den = fmaf(gk, 0.2126f + 0.7152f + 0.0722f, den);
            }
        }
        const float k = 1.f / (lum / den + eps);
        const float* p = x0 + (((size_t)n * H0 + (size_t)h * step) * W0 + (size_t)w * step) * 3;
        float* o = out + (size_t)i * 3;
        o[0] = __ldg(p) * k; o[1] = __ldg(p + 1) * k; o[2] = __ldg(p + 2) * k;
    }
}

extern "C" int mpnn_lln(const float* x0, int B, int H0, int W0, int C0, int step, float sigma, float eps,
                        float* out, void* stream) {
    MPNN_REQUIRE(x0 && out && C0 == 3, "lln: the luminance weights are defined for 3 channels (C0=%d)", C0);
    MPNN_REQUIRE(step >= 1 && H0 % step == 0 && W0 % step == 0 && sigma > 0.f, "lln: step=%d sigma=%g", step, (double)sigma);
    const int s = (int)ceilf(2.f * sigma);
    const long long total = (long long)B * (H0 / step) * (W0 / step);
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    lln_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x0, B, H0, W0, step, sigma, eps, s, out);
    return mpnn_check_launch("lln");
}

// --------------------------------------------------------------------------- //
// Weight packing:  w[t][i][o] (HWIO / (n_in,n_chan)) -> Wp[tap][Ktot/8][Ntot][8]
// --------------------------------------------------------------------------- //
template <typename T> __device__ __forceinline__ T cvt_from_float(float v);
template <> __device__ __forceinline__ float cvt_from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 cvt_from_float<__nv_bfloat16>(float v) {
    return __float2bfloat16_rn(v);
}

// mode & 4: the residual of one bf16 rounding, w - bf16(w) (second part of a split weight);
// mode & 8: the residual of two, w - bf16(w) - bf16(w - bf16(w)) (third part, "bf16x6" mode)
__device__ __forceinline__ float bf16_residual(float v, int mode) {
    if (mode & 12) v -= __bfloat162float(__float2bfloat16_rn(v));
    if (mode & 8) v -= __bfloat162float(__float2bfloat16_rn(v));
    return v;
}

template <typename T>
__global__ void pack_weights_kernel(const float* __restrict__ w, int ntaps, int I, int O, int mode,
                                    int k_off, int Ktot, int n_off, int Ntot, T* __restrict__ packed) {
    const int total = ntaps * I * O;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        int o = e % O;
        int i = (e / O) % I;
        int t = e / (O * I);
        int k, n, tap;
        if ((mode & 3) == 0) { k = k_off + i; n = n_off + o; tap = t; }
        else                 { k = k_off + o; n = n_off + i; tap = ntaps - 1 - t; }
        size_t dst = (((size_t)tap * (Ktot / 8) + (k >> 3)) * Ntot + n) * 8 + (k & 7);
        packed[dst] = cvt_from_float<T>(bf16_residual(w[e], mode));
    }
}

// all weight tensors of a step in ONE launch: blockIdx.y selects the descriptor
template <typename T>
__global__ void pack_weights_batched_kernel(const mpnn_pack_desc* __restrict__ descs) {
    const mpnn_pack_desc d = descs[blockIdx.y];
    const int total = d.ntaps * d.I * d.O;
    if (d.mode == 2) {          // fp32 vector copy (bias vectors of fused heads)
        float* pf = static_cast<float*>(d.packed);
        for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < d.O; e += gridDim.x * blockDim.x)
            pf[d.n_off + e] = __ldg(d.w + e);
        return;
    }
    T* packed = static_cast<T*>(d.packed);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        int o = e % d.O;
        int i = (e / d.O) % d.I;
        int t = e / (d.O * d.I);
        int k, n, tap;
        if ((d.mode & 3) == 0) { k = d.k_off + i; n = d.n_off + o; tap = t; }
        else                   { k = d.k_off + o; n = d.n_off + i; tap = d.ntaps - 1 - t; }
        size_t dst = (((size_t)tap * (d.Ktot / 8) + (k >> 3)) * d.Ntot + n) * 8 + (k & 7);
        packed[dst] = cvt_from_float<T>(bf16_residual(__ldg(d.w + e), d.mode));
    }
}

extern "C" int mpnn_pack_weights_batched(const mpnn_pack_desc* descs, int n, int blocks_per_desc,
                                         int dtype, void* stream) {
    MPNN_REQUIRE(n >= 1 && n <= 65535 && blocks_per_desc >= 1, "pack_weights_batched: n=%d", n);
    dim3 grid(blocks_per_desc, n);
    MPNN_DISPATCH_DTYPE(dtype, (pack_weights_batched_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(descs)));
    return mpnn_check_launch("pack_weights_batched");
}

extern "C" int mpnn_pack_weights(const float* w, int ntaps, int I, int O, int mode,
                                 int k_off, int Ktot, int n_off, int Ntot,
                                 void* packed, int dtype, void* stream) {
    MPNN_REQUIRE(Ktot % 8 == 0, "pack_weights: Ktot %% 8");
    if ((mode & 3) == 0) MPNN_REQUIRE(k_off + I <= Ktot && n_off + O <= Ntot, "pack_weights: range");
    else           MPNN_REQUIRE(k_off + O <= Ktot && n_off + I <= Ntot, "pack_weights: range (dgrad)");
    int total = ntaps * I * O;
    int grid = (total + 255) / 256;
    if (grid > 148 * 8) grid = 148 * 8;
    MPNN_DISPATCH_DTYPE(dtype, (pack_weights_kernel<T><<<grid, 256, 0, (cudaStream_t)stream>>>(
        w, ntaps, I, O, mode, k_off, Ktot, n_off, Ntot, (T*)packed)));
    return mpnn_check_launch("pack_weights");
}

// --------------------------------------------------------------------------- //
// fp32 planes -> two bf16 planes sets (hi | lo) with x = hi + lo up to 2^-17 |x|: the operand format of the
// "bf16x3" precision mode, where a fp32 product a*b is evaluated on the tensor cores as
// a_hi*b_hi + a_lo*b_hi + a_hi*b_lo (relative error ~2^-16) with fp32 accumulation.
// src [C/8][P][8] fp32, dst [2*C/8][P][8] bf16: planes [0, C/8) = hi, [C/8, 2*C/8) = lo.
// --------------------------------------------------------------------------- //
__global__ void __launch_bounds__(256)
split_planes_kernel(const float* __restrict__ src, long long rows, __nv_bfloat16* __restrict__ dst) {
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x) {
        float v[8], hi[8], lo[8];
        Row8<float>::load(src + r * 8, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            hi[j] = __bfloat162float(__float2bfloat16_rn(v[j]));
            lo[j] = v[j] - hi[j];
        }
        Row8<__nv_bfloat16>::store(dst + r * 8, hi);
        Row8<__nv_bfloat16>::store(dst + (rows + r) * 8, lo);
    }
}

// three-way split (hi | mid | lo), x = hi + mid + lo up to 2^-25 |x|: operand format of the "bf16x6" mode, where a
// product is a_hi*b_hi + a_mid*b_hi + a_lo*b_hi + a_hi*b_mid + a_mid*b_mid + a_hi*b_lo (every term above 2^-24).
// Row r of the C/8 * P source rows; `rows` = C/8 * P is the distance between the three parts of dst.  Shared by the
// whole-tensor and the counted launch, so both write the same bits.
__device__ __forceinline__ void split3_row(const float* __restrict__ src, long long rows, long long r,
                                           __nv_bfloat16* __restrict__ dst) {
    float v[8], hi[8], mid[8], lo[8];
    Row8<float>::load(src + r * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        hi[j] = __bfloat162float(__float2bfloat16_rn(v[j]));
        const float r1 = v[j] - hi[j];
        mid[j] = __bfloat162float(__float2bfloat16_rn(r1));
        lo[j] = r1 - mid[j];
    }
    Row8<__nv_bfloat16>::store(dst + r * 8, hi);
    Row8<__nv_bfloat16>::store(dst + (rows + r) * 8, mid);
    Row8<__nv_bfloat16>::store(dst + (2 * rows + r) * 8, lo);
}

__global__ void __launch_bounds__(256)
split_planes3_kernel(const float* __restrict__ src, long long rows, __nv_bfloat16* __restrict__ dst) {
    for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < rows; r += (long long)gridDim.x * blockDim.x)
        split3_row(src, rows, r, dst);
}

// counted: rows [0, G + m*S) of every plane (blockIdx.y), m = min(*count, g.B); m = 0 writes nothing
__global__ void __launch_bounds__(256)
split_planes3_counted_kernel(const float* __restrict__ src, Geom g, __nv_bfloat16* __restrict__ dst,
                             const int* __restrict__ count) {
    const int m = count ? min(max(*count, 0), g.B) : g.B;
    if (m == 0) return;
    const long long live = (long long)g.G + (long long)m * g.S;
    const long long rows = (long long)gridDim.y * g.P;
    const long long base = (long long)blockIdx.y * g.P;
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < live; p += (long long)gridDim.x * blockDim.x)
        split3_row(src, rows, base + p, dst);
}

extern "C" int mpnn_split_planes3(const float* src, int C, int P, void* dst, void* stream) {
    MPNN_REQUIRE(src && dst && C % 8 == 0 && C > 0 && P > 0, "split_planes3: C=%d P=%d", C, P);
    const long long rows = (long long)(C / 8) * P;
    long long g = (rows + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    split_planes3_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(src, rows, (__nv_bfloat16*)dst);
    return mpnn_check_launch("split_planes3");
}

extern "C" int mpnn_split_planes3_counted(const float* src, int C, int B, int H, int W, int G, int P, void* dst,
                                          const int* count, void* stream) {
    MPNN_REQUIRE(src && dst && C % 8 == 0 && C > 0 && B >= 0 && H > 0 && W > 0,
                 "split_planes3_counted: C=%d B=%d H=%d W=%d", C, B, H, W);
    MPNN_REQUIRE(C / 8 <= 65535, "split_planes3_counted: C=%d", C);
    Geom g = make_geom(B, H, W, G, P);
    MPNN_REQUIRE(G + g.rows <= P, "split_planes3_counted: P=%d < G + B*(H+1)*(W+1)", P);
    if (B == 0) return MPNN_OK;
    const int planes = C / 8;
    long long gx = ((long long)G + g.rows + 255) / 256;              // sized for the capacity
    const long long cap = (148 * 16 + planes - 1) / planes;
    if (gx > cap) gx = cap;
    split_planes3_counted_kernel<<<dim3((unsigned)gx, planes), 256, 0, (cudaStream_t)stream>>>(
        src, g, (__nv_bfloat16*)dst, count);
    return mpnn_check_launch("split_planes3_counted");
}

extern "C" int mpnn_split_planes(const float* src, int C, int P, void* dst, void* stream) {
    MPNN_REQUIRE(src && dst && C % 8 == 0 && C > 0 && P > 0, "split_planes: C=%d P=%d", C, P);
    const long long rows = (long long)(C / 8) * P;
    long long g = (rows + 255) / 256;
    if (g > 148 * 16) g = 148 * 16;
    split_planes_kernel<<<(int)g, 256, 0, (cudaStream_t)stream>>>(src, rows, (__nv_bfloat16*)dst);
    return mpnn_check_launch("split_planes");
}
