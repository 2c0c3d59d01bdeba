// MaxPool and GlobalMaxPool of lib/layer_types.py:86-100 on padded-planes tensors, forward and backward.
//
// MaxPool: the reference hands (strides, k_shape) to tf.nn.max_pool(value, ksize, strides), i.e. the window is
// `stride` wide and the step is `supp` (SURVEY F8); the 2 / 2 case -- the only one where both readings agree and
// the one a conv block uses -- is what these kernels serve: 2x2 window, step 2, even sizes (SAME = VALID).
// GlobalMaxPool: tf.reduce_max over the image dimensions.
// Gradients go to the first maximal element in window / row-major order (ties only arise between equal
// activations, e.g. zeros behind the ReLU, where the ReLU gradient is zero anyway).
#include "common.cuh"
#include "../../include/mpnn.h"

// one thread per (pooled pixel, 8-channel plane): out = max of the 2x2 block; optionally also in the flattened
// (h, w, c) feature layout [F/8][Balloc][8] the head GEMMs read
template <typename T>
__global__ void __launch_bounds__(256)
maxpool2_fwd_kernel(const T* __restrict__ x, int C, Geom g, T* __restrict__ out, Geom gp,
                    T* __restrict__ feat, int Balloc) {
    const int kg = blockIdx.y, KG = C / 8;
    const int HH = g.H / 2, WW = g.W / 2, total = g.B * HH * WW;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int w = i % WW, r = i / WW, h = r % HH, n = r / HH;
        const int p00 = row_of(g, n, 2 * h, 2 * w);
        float v[4][8], m[8];
        Row8<T>::load(plane_row(x, kg, g.P, p00), v[0]);
        Row8<T>::load(plane_row(x, kg, g.P, p00 + 1), v[1]);
        Row8<T>::load(plane_row(x, kg, g.P, p00 + g.Wp), v[2]);
        Row8<T>::load(plane_row(x, kg, g.P, p00 + g.Wp + 1), v[3]);
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] = fmaxf(fmaxf(v[0][j], v[1][j]), fmaxf(v[2][j], v[3][j]));
        if (out) Row8<T>::store(plane_row(out, kg, gp.P, row_of(gp, n, h, w)), m);
        if (feat) Row8<T>::store(plane_row(feat, (h * WW + w) * KG + kg, Balloc, n), m);
    }
}

extern "C" int mpnn_maxpool2_fwd(const void* x, int C, int B, int H, int W, int G, int P,
                                 void* out, int Pp, void* feat, int Balloc, int dtype, void* stream) {
    MPNN_REQUIRE(x && (out || feat) && C % 8 == 0 && H % 2 == 0 && W % 2 == 0, "maxpool2_fwd: C=%d H=%d W=%d", C, H, W);
    Geom g = make_geom(B, H, W, G, P), gp = make_geom(B, H / 2, W / 2, G, Pp);
    const long long total = (long long)B * (H / 2) * (W / 2);
    int gx = (int)((total + 255) / 256);
    if (gx > 148 * 8) gx = 148 * 8;
    MPNN_DISPATCH_DTYPE(dtype, (maxpool2_fwd_kernel<T><<<dim3(gx, C / 8), 256, 0, (cudaStream_t)stream>>>(
        (const T*)x, C, g, (T*)out, gp, (T*)feat, Balloc)));
    return mpnn_check_launch("maxpool2_fwd");
}

// dx of the 2x2 block = (dout + dfeat) at the first maximum, zero elsewhere (every row of dx is written)
template <typename T>
__global__ void __launch_bounds__(256)
maxpool2_bwd_kernel(const T* __restrict__ x, const T* __restrict__ dout, const T* __restrict__ dfeat, int Balloc,
                    int C, Geom g, Geom gp, T* __restrict__ dx) {
    const int kg = blockIdx.y, KG = C / 8;
    const int HH = g.H / 2, WW = g.W / 2, total = g.B * HH * WW;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int w = i % WW, r = i / WW, h = r % HH, n = r / HH;
        const int p00 = row_of(g, n, 2 * h, 2 * w);
        const int pk[4] = {p00, p00 + 1, p00 + g.Wp, p00 + g.Wp + 1};
        float v[4][8], d[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) Row8<T>::load(plane_row(x, kg, g.P, pk[k]), v[k]);
#pragma unroll
        for (int j = 0; j < 8; ++j) d[j] = 0.f;
        if (dout) Row8<T>::load(plane_row(dout, kg, gp.P, row_of(gp, n, h, w)), d);
        if (dfeat) {
            float d2[8];
            Row8<T>::load(plane_row(dfeat, (h * WW + w) * KG + kg, Balloc, n), d2);
#pragma unroll
            for (int j = 0; j < 8; ++j) d[j] += d2[j];
        }
        int best[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            best[j] = 0;
            float bv = v[0][j];
#pragma unroll
            for (int k = 1; k < 4; ++k)
                if (v[k][j] > bv) { bv = v[k][j]; best[j] = k; }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = best[j] == k ? d[j] : 0.f;
            Row8<T>::store(plane_row(dx, kg, g.P, pk[k]), o);
        }
    }
}

extern "C" int mpnn_maxpool2_bwd(const void* x, const void* dout, const void* dfeat, int Balloc,
                                 int C, int B, int H, int W, int G, int P, int Pp, void* dx, int dtype, void* stream) {
    MPNN_REQUIRE(x && dx && (dout || dfeat) && C % 8 == 0 && H % 2 == 0 && W % 2 == 0, "maxpool2_bwd: args");
    Geom g = make_geom(B, H, W, G, P), gp = make_geom(B, H / 2, W / 2, G, Pp);
    const long long total = (long long)B * (H / 2) * (W / 2);
    int gx = (int)((total + 255) / 256);
    if (gx > 148 * 8) gx = 148 * 8;
    MPNN_DISPATCH_DTYPE(dtype, (maxpool2_bwd_kernel<T><<<dim3(gx, C / 8), 256, 0, (cudaStream_t)stream>>>(
        (const T*)x, (const T*)dout, (const T*)dfeat, Balloc, C, g, gp, (T*)dx)));
    return mpnn_check_launch("maxpool2_bwd");
}

// GlobalMaxPool: one warp per (image, 8-channel plane); lanes stride over the pixels in row-major order and keep
// (value, pixel) of their first maximum per channel; the warp reduction prefers the smaller pixel on ties.
// feat [C/8][Balloc][8] (the layout of a flattened 1x1 image), arg [C/8][Balloc][8] int32 = h * W + w.
// CNT: count and arg may be NULL; a count limits the launch to the first min(*count, g.B) images (g.B: the capacity
// the grid was sized for).
template <typename T, bool CNT = false>
__global__ void __launch_bounds__(256)
global_maxpool_fwd_kernel(const T* __restrict__ x, int C, Geom g, T* __restrict__ feat, int* __restrict__ arg,
                          int Balloc, const int* __restrict__ count) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int KG = C / 8;
    if (CNT && count) g.B = min(max(*count, 0), g.B);
    if (warp >= g.B * KG) return;
    const int n = warp / KG, kg = warp % KG;
    float bv[8];
    int bi[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { bv[j] = -INFINITY; bi[j] = 0x7fffffff; }
    for (int px = lane; px < g.H * g.W; px += 32) {
        float v[8];
        Row8<T>::load(plane_row(x, kg, g.P, row_of(g, n, px / g.W, px % g.W)), v);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (v[j] > bv[j]) { bv[j] = v[j]; bi[j] = px; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv[j], o);
            const int oi = __shfl_xor_sync(0xffffffffu, bi[j], o);
            if (ov > bv[j] || (ov == bv[j] && oi < bi[j])) { bv[j] = ov; bi[j] = oi; }
        }
    }
    if (lane == 0) {
        Row8<T>::store(plane_row(feat, kg, Balloc, n), bv);
        if (!CNT || arg) {
            int* a = arg + ((size_t)kg * Balloc + n) * 8;
#pragma unroll
            for (int j = 0; j < 8; ++j) a[j] = bi[j];
        }
    }
}

extern "C" int mpnn_global_maxpool_fwd(const void* x, int C, int B, int H, int W, int G, int P,
                                       void* feat, int* arg, int Balloc, int dtype, void* stream) {
    MPNN_REQUIRE(x && feat && arg && C % 8 == 0 && Balloc >= B, "global_maxpool_fwd: args");
    Geom g = make_geom(B, H, W, G, P);
    const long long warps = (long long)B * (C / 8);
    MPNN_DISPATCH_DTYPE(dtype, (global_maxpool_fwd_kernel<T><<<(int)((warps * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const T*)x, C, g, (T*)feat, arg, Balloc, nullptr)));
    return mpnn_check_launch("global_maxpool_fwd");
}

// the forward on the live images of a counted launch (grid sized for the capacity B, live images min(*count, B));
// arg may be NULL (the 'ev' pass needs no argmax).  count NULL: the uncounted launch at B.
extern "C" int mpnn_global_maxpool_fwd_counted(const void* x, int C, int B, int H, int W, int G, int P,
                                               void* feat, int* arg, int Balloc, int dtype, const int* count,
                                               void* stream) {
    MPNN_REQUIRE(x && feat && C % 8 == 0 && B >= 0 && Balloc >= B,
                 "global_maxpool_fwd_counted: C=%d B=%d Balloc=%d", C, B, Balloc);
    if (arg && !count) return mpnn_global_maxpool_fwd(x, C, B, H, W, G, P, feat, arg, Balloc, dtype, stream);
    if (B == 0) return MPNN_OK;
    Geom g = make_geom(B, H, W, G, P);
    const long long warps = (long long)B * (C / 8);
    MPNN_DISPATCH_DTYPE(dtype, (global_maxpool_fwd_kernel<T, true><<<(int)((warps * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const T*)x, C, g, (T*)feat, arg, Balloc, count)));
    return mpnn_check_launch("global_maxpool_fwd_counted");
}

// dx[n][h][w][c] = dfeat[n][c] where (h, w) is the recorded maximum of channel c, zero elsewhere
template <typename T>
__global__ void __launch_bounds__(256)
global_maxpool_bwd_kernel(const T* __restrict__ dfeat, const int* __restrict__ arg, int Balloc, int C, Geom g,
                          T* __restrict__ dx) {
    const int kg = blockIdx.y;
    const int total = g.B * g.H * g.W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int px = i % (g.H * g.W), n = i / (g.H * g.W);
        float d[8], o[8];
        Row8<T>::load(plane_row(dfeat, kg, Balloc, n), d);
        const int* a = arg + ((size_t)kg * Balloc + n) * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = a[j] == px ? d[j] : 0.f;
        Row8<T>::store(plane_row(dx, kg, g.P, row_of(g, n, px / g.W, px % g.W)), o);
    }
}

extern "C" int mpnn_global_maxpool_bwd(const void* dfeat, const int* arg, int Balloc, int C, int B, int H, int W,
                                       int G, int P, void* dx, int dtype, void* stream) {
    MPNN_REQUIRE(dfeat && arg && dx && C % 8 == 0, "global_maxpool_bwd: args");
    Geom g = make_geom(B, H, W, G, P);
    const long long total = (long long)B * H * W;
    int gx = (int)((total + 255) / 256);
    if (gx > 148 * 8) gx = 148 * 8;
    MPNN_DISPATCH_DTYPE(dtype, (global_maxpool_bwd_kernel<T><<<dim3(gx, C / 8), 256, 0, (cudaStream_t)stream>>>(
        (const T*)dfeat, arg, Balloc, C, g, (T*)dx)));
    return mpnn_check_launch("global_maxpool_bwd");
}
