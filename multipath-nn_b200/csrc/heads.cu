// Fully-connected heads on feature planes, softmax + cross-entropy, and the
// router tail (BN-ReLU-FC-BN-ReLU-FC).  fp32 arithmetic throughout: routing
// decisions must stay bit-stable (SURVEY section 7, "bit-exact routing").
// Reference: lib/layer_types.py:39-53 (LinTrans), :81-84 (Softmax),
// :262-272 (CrossEntropyError), :219-239 (BatchNorm); arch_and_hypers.py:45-49.
#include "common.cuh"
#include "../../include/mpnn.h"

#define FC_NMAX 16
#define FC_NWIDE 64          // widest FC head: the first layer of a 64-wide router, in FC_NMAX-column slices

// ---------------------------------------------------------------- fc forward
// CNT: only the rows b < min(*count, B) are stored (B: the capacity the grid was sized for).  blockIdx.y selects the
// FC_NMAX-column slice j0 = 16 * blockIdx.y of the n outputs (one slice for n <= 16).
template <typename T, bool CNT = false>
__global__ void __launch_bounds__(256)
fc_fwd_kernel(const T* __restrict__ X, int F, int Balloc, int B, const float* __restrict__ W,
              const float* __restrict__ bias, const float* __restrict__ extra, int n,
              float* __restrict__ Z, const int* __restrict__ count) {
    const int lane = threadIdx.x, ky = threadIdx.y;   // 32 x 8
    const int b = blockIdx.x * 32 + lane;
    const int bl = b < B ? b : B - 1;
    const int Bn = CNT ? min(max(*count, 0), B) : B;
    if (CNT && (int)blockIdx.x * 32 >= Bn) return;
    const int j0 = blockIdx.y * FC_NMAX, nj = min(FC_NMAX, n - j0);
    float acc[FC_NMAX];
#pragma unroll
    for (int j = 0; j < FC_NMAX; ++j) acc[j] = 0.f;
    for (int fg = ky; fg < F / 8; fg += 8) {
        float x[8];
        Row8<T>::load(plane_row(X, fg, Balloc, bl), x);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const float* wr = W + (size_t)(fg * 8 + c) * n + j0;
#pragma unroll
            for (int j = 0; j < FC_NMAX; ++j)
                if (j < nj) acc[j] = fmaf(x[c], __ldg(wr + j), acc[j]);
        }
    }
    __shared__ float red[8][32][FC_NMAX + 1];
#pragma unroll
    for (int j = 0; j < FC_NMAX; ++j) red[ky][lane][j] = acc[j];
    __syncthreads();
    // thread (lane, ky) finalises outputs j = ky, ky+8
    for (int j = ky; j < nj; j += 8) {
        float t = 0.f;
#pragma unroll
        for (int s = 0; s < 8; ++s) t += red[s][lane][j];
        if (extra) t = fmaf(extra[bl], __ldg(W + (size_t)F * n + j0 + j), t);
        t += bias ? bias[j0 + j] : 0.f;
        if (b < Bn) Z[(size_t)b * n + j0 + j] = t;
    }
}

extern "C" int mpnn_fc_fwd_counted(const void* X, int F, int Balloc, int B, const float* W, const float* bias,
                                   const float* extra, int n, float* Z, int dtype, const int* count, void* stream) {
    MPNN_REQUIRE(F % 8 == 0 && n >= 1 && n <= FC_NWIDE, "fc_fwd: F=%d n=%d (n<=%d)", F, n, FC_NWIDE);
    MPNN_REQUIRE(B >= 1 && Balloc >= B, "fc_fwd: B=%d Balloc=%d", B, Balloc);
    dim3 block(32, 8), grid(ceil_div(B, 32), ceil_div(n, FC_NMAX));
    if (count) {
        MPNN_DISPATCH_DTYPE(dtype, (fc_fwd_kernel<T, true><<<grid, block, 0, (cudaStream_t)stream>>>(
            (const T*)X, F, Balloc, B, W, bias, extra, n, Z, count)));
    } else {
        MPNN_DISPATCH_DTYPE(dtype, (fc_fwd_kernel<T, false><<<grid, block, 0, (cudaStream_t)stream>>>(
            (const T*)X, F, Balloc, B, W, bias, extra, n, Z, nullptr)));
    }
    return mpnn_check_launch("fc_fwd");
}

extern "C" int mpnn_fc_fwd(const void* X, int F, int Balloc, int B, const float* W, const float* bias,
                           const float* extra, int n, float* Z, int dtype, void* stream) {
    return mpnn_fc_fwd_counted(X, F, Balloc, B, W, bias, extra, n, Z, dtype, nullptr, stream);
}

// ---------------------------------------------------------- fc backward data
// N1MAX: register row of the second operand (FC_NMAX, or FC_NWIDE for the first layer of a wide router)
template <typename T, int N1MAX = FC_NMAX>
__global__ void __launch_bounds__(256)
fc_bwd_data_kernel(const float* __restrict__ dZ0, const float* __restrict__ W0, int n0,
                   const float* __restrict__ dZ1, const float* __restrict__ W1, int n1,
                   int F, int Balloc, int B, T* __restrict__ dX) {
    const int lane = threadIdx.x, ky = threadIdx.y;
    const int b = blockIdx.x * 32 + lane;
    if (b >= B) return;
    float d0[FC_NMAX], d1[N1MAX];
#pragma unroll
    for (int j = 0; j < FC_NMAX; ++j) d0[j] = j < n0 ? dZ0[(size_t)b * n0 + j] : 0.f;
#pragma unroll
    for (int j = 0; j < N1MAX; ++j) d1[j] = (dZ1 && j < n1) ? dZ1[(size_t)b * n1 + j] : 0.f;
    for (int fg = blockIdx.y * 8 + ky; fg < F / 8; fg += 8 * gridDim.y) {
        float v[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int f = fg * 8 + c;
            float t = 0.f;
#pragma unroll
            for (int j = 0; j < FC_NMAX; ++j)
                if (j < n0) t = fmaf(d0[j], __ldg(W0 + (size_t)f * n0 + j), t);
            if (dZ1) {
#pragma unroll
                for (int j = 0; j < N1MAX; ++j)
                    if (j < n1) t = fmaf(d1[j], __ldg(W1 + (size_t)f * n1 + j), t);
            }
            v[c] = t;
        }
        Row8<T>::store(plane_row(dX, fg, Balloc, b), v);
    }
}

extern "C" int mpnn_fc_bwd_data(const float* dZ0, const float* W0, int n0,
                                const float* dZ1, const float* W1, int n1,
                                int F, int Balloc, int B, void* dX, int dtype, void* stream) {
    MPNN_REQUIRE(F % 8 == 0 && n0 >= 1 && n0 <= FC_NWIDE && n1 <= FC_NWIDE && (n0 <= FC_NMAX || n1 == 0),
                 "fc_bwd_data: n0=%d n1=%d (n0 <= %d beside a second operand, each <= %d)", n0, n1, FC_NMAX, FC_NWIDE);
    if (n0 > FC_NMAX) {          // a wide operand alone takes the wide slot (same summation order)
        dZ1 = dZ0; W1 = W0; n1 = n0;
        dZ0 = nullptr; W0 = nullptr; n0 = 0;
    }
    int gy = ceil_div(F / 8, 8 * 4);
    if (gy < 1) gy = 1;
    dim3 block(32, 8), grid(ceil_div(B, 32), gy);
    if (n1 <= FC_NMAX) {
        MPNN_DISPATCH_DTYPE(dtype, (fc_bwd_data_kernel<T><<<grid, block, 0, (cudaStream_t)stream>>>(
            dZ0, W0, n0, dZ1, W1, n1, F, Balloc, B, (T*)dX)));
    } else {
        MPNN_DISPATCH_DTYPE(dtype, (fc_bwd_data_kernel<T, FC_NWIDE><<<grid, block, 0, (cudaStream_t)stream>>>(
            dZ0, W0, n0, dZ1, W1, n1, F, Balloc, B, (T*)dX)));
    }
    return mpnn_check_launch("fc_bwd_data");
}

// -------------------------------------------------------- fc backward weight
// block (8 c, n j): outputs dW[fg*8+c][j]; blockIdx.y splits the batch.
template <typename T>
__global__ void fc_bwd_weight_kernel(const T* __restrict__ X, int F, int Balloc, int B,
                                     const float* __restrict__ extra, const float* __restrict__ dZ, int n,
                                     float* __restrict__ dW, float* __restrict__ db, int bchunk) {
    const int fg = blockIdx.x;
    const int j = threadIdx.x, c = threadIdx.y;
    const int b0 = blockIdx.y * bchunk, b1 = min(b0 + bchunk, B);
    float acc = 0.f;
    if (fg < F / 8) {
        const T* xc = X + (size_t)fg * Balloc * 8 + c;
        for (int b = b0; b < b1; ++b) {
            float xv;
            if (sizeof(T) == 4) xv = reinterpret_cast<const float*>(xc)[(size_t)b * 8];
            else xv = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(xc)[(size_t)b * 8]);
            acc = fmaf(xv, dZ[(size_t)b * n + j], acc);
        }
        atomicAdd(dW + (size_t)(fg * 8 + c) * n + j, acc);
    } else {
        // tail block: c==0 -> bias, c==1 -> extra feature row
        if (c == 0 && db) {
            for (int b = b0; b < b1; ++b) acc += dZ[(size_t)b * n + j];
            atomicAdd(db + j, acc);
        } else if (c == 1 && extra) {
            for (int b = b0; b < b1; ++b) acc = fmaf(extra[b], dZ[(size_t)b * n + j], acc);
            atomicAdd(dW + (size_t)F * n + j, acc);
        }
    }
}

extern "C" int mpnn_fc_bwd_weight(const void* X, int F, int Balloc, int B, const float* extra,
                                  const float* dZ, int n, float* dW, float* db, int dtype, void* stream) {
    MPNN_REQUIRE(F % 8 == 0 && n >= 1 && n <= FC_NWIDE, "fc_bwd_weight: F=%d n=%d (n<=%d)", F, n, FC_NWIDE);
    int bchunk = 512;
    dim3 block(n, 8), grid(F / 8 + 1, ceil_div(B, bchunk));
    MPNN_DISPATCH_DTYPE(dtype, (fc_bwd_weight_kernel<T><<<grid, block, 0, (cudaStream_t)stream>>>(
        (const T*)X, F, Balloc, B, extra, dZ, n, dW, db, bchunk)));
    return mpnn_check_launch("fc_bwd_weight");
}

// ------------------------------------------------------ softmax + CE forward
// LPR lanes per example (16 for n <= 16, else 32), one class per lane, reductions by shuffles inside the lane
// group.  (One thread per example with the class loop unrolled to 32 was ~2600 dependent instructions in a
// single warp: 7.6 us for B = 128, n = 10 under ncu, all of it issue latency.)
#define CE_NMAX 32
template <int LPR>
__device__ __forceinline__ float grp_sum(float v) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <int LPR>
__device__ __forceinline__ float grp_max(float v) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// index of the first maximum of v over the lanes j < n of the group (tf.argmax)
template <int LPR>
__device__ __forceinline__ int grp_argmax(float v, int j) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oj = __shfl_xor_sync(0xffffffffu, j, o);
        if (ov > v || (ov == v && oj < j)) { v = ov; j = oj; }
    }
    return j;
}

template <int LPR>
__global__ void __launch_bounds__(128)
softmax_ce_fwd_kernel(const float* __restrict__ Z, int ldz, const float* __restrict__ y, int B,
                      int n, float eps, float* __restrict__ prob, float* __restrict__ c_err,
                      float* __restrict__ d_cor) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = t / LPR, j = t % LPR;
    const bool on = b < B && j < n;
    const float z = on ? Z[(size_t)b * ldz + j] : -INFINITY;
    const float yy = on ? y[(size_t)b * n + j] : -INFINITY;
    const float mx = grp_max<LPR>(z);
    const float e = on ? expf(z - mx) : 0.f;
    const float p = e * (1.f / grp_sum<LPR>(e));
    if (on) prob[(size_t)b * n + j] = p;
    const float ce = grp_sum<LPR>(on ? -yy * logf(eps / n + (1.f - eps) * p) : 0.f);
    const int am_p = grp_argmax<LPR>(on ? p : -INFINITY, j);
    const int am_y = grp_argmax<LPR>(yy, j);
    if (b < B && j == 0) {
        c_err[b] = ce;
        d_cor[b] = am_p == am_y ? 1.f : 0.f;
    }
}

extern "C" int mpnn_softmax_ce_fwd(const float* Z, int ldz, const float* y, int B, int n, float eps,
                                   float* prob, float* c_err, float* d_cor, void* stream) {
    MPNN_REQUIRE(n >= 1 && n <= CE_NMAX && ldz >= n, "softmax_ce_fwd: n=%d ldz=%d", n, ldz);
    if (n <= 16)
        softmax_ce_fwd_kernel<16><<<ceil_div(B * 16, 128), 128, 0, (cudaStream_t)stream>>>(Z, ldz, y, B, n, eps, prob, c_err, d_cor);
    else
        softmax_ce_fwd_kernel<32><<<ceil_div(B * 32, 128), 128, 0, (cudaStream_t)stream>>>(Z, ldz, y, B, n, eps, prob, c_err, d_cor);
    return mpnn_check_launch("softmax_ce_fwd");
}

// ------------------------------------------------------ routed inference: results at one classifier
// The softmax and first argmax of softmax_ce_fwd_kernel (same lane groups, same expressions, so prob is the same
// bits as the dense path's for the same logits) on rows pos[j] of the parent's compact batch, written at the
// examples' original ids orig[j] into rows of ldp >= n floats (columns n .. ldp-1 zero).  The live count is read on
// the device; the grid covers the host bound.
template <int LPR>
__global__ void __launch_bounds__(128)
leaf_emit_kernel(const float* __restrict__ Z, int ldz, int n, const int* __restrict__ pos,
                 const int* __restrict__ orig, const int* __restrict__ count, int n_max, int leaf, double path_ops,
                 float* __restrict__ prob, int ldp, int* __restrict__ cls, int* __restrict__ exit_id,
                 double* __restrict__ ops) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = t / LPR, j = t % LPR;
    const int nb = count ? min(*count, n_max) : n_max;
    const bool live = b < nb;
    const bool on = live && j < n;
    const int row = !live ? 0 : pos ? pos[b] : b;
    const int o = !live ? 0 : orig ? orig[b] : b;
    const float z = on ? Z[(size_t)row * ldz + j] : -INFINITY;
    const float mx = grp_max<LPR>(z);
    const float e = on ? expf(z - mx) : 0.f;
    const float p = e * (1.f / grp_sum<LPR>(e));
    if (on) prob[(size_t)o * ldp + j] = p;
    if (live)
        for (int c = n + j; c < ldp; c += LPR) prob[(size_t)o * ldp + c] = 0.f;
    const int am = grp_argmax<LPR>(on ? p : -INFINITY, j);
    if (live && j == 0) {
        cls[o] = am;
        exit_id[o] = leaf;
        ops[o] = path_ops;
    }
}

extern "C" int mpnn_leaf_emit_strided(const float* Z, int ldz, int n_out, const int* pos, const int* orig,
                                      const int* count, int n, int leaf, double path_ops, float* prob, int ldp,
                                      int* cls, int* exit_id, double* ops, void* stream) {
    MPNN_REQUIRE(n >= 0 && n_out >= 1 && n_out <= CE_NMAX && ldz >= n_out && ldp >= n_out,
                 "leaf_emit: n=%d n_out=%d ldz=%d ldp=%d", n, n_out, ldz, ldp);
    if (n == 0) return MPNN_OK;
    MPNN_REQUIRE(Z && prob && cls && exit_id && ops, "leaf_emit: NULL operand");
    if (n_out <= 16)
        leaf_emit_kernel<16><<<ceil_div(n, 128 / 16), 128, 0, (cudaStream_t)stream>>>(
            Z, ldz, n_out, pos, orig, count, n, leaf, path_ops, prob, ldp, cls, exit_id, ops);
    else
        leaf_emit_kernel<32><<<ceil_div(n, 128 / 32), 128, 0, (cudaStream_t)stream>>>(
            Z, ldz, n_out, pos, orig, count, n, leaf, path_ops, prob, ldp, cls, exit_id, ops);
    return mpnn_check_launch("leaf_emit");
}

extern "C" int mpnn_leaf_emit(const float* Z, int ldz, int n_cls, const int* pos, const int* orig, const int* count,
                              int n, int leaf, double path_ops, float* prob, int* cls, int* exit_id, double* ops,
                              void* stream) {
    return mpnn_leaf_emit_strided(Z, ldz, n_cls, pos, orig, count, n, leaf, path_ops, prob, n_cls, cls, exit_id, ops,
                                  stream);
}

// ------------------------------------------------------ compacted statistics at one classifier
// Statistics of the examples routed to one classifier (train-nets:117-130 with p_ev one-hot), with the correctness
// target and the class bins apart:
//   cor = [first argmax of the softmax of Z[pos[j]] == first argmax of t[orig[j]]] over the leaf's n_out columns --
//         the comparison of softmax_ce_fwd_kernel (same lane groups and expressions), so it is the dense d_cor bit;
//   out[0] += #cor, out[1] += #(1 - cor), out[2 + c] += sum cor * y[orig][c], out[2 + n_cls + c] += sum (1 - cor) * y[c]
// over the n_cls one-hot labels y.  t = y for Softmax + CrossEntropyError leaves, y @ w_cls for superclass leaves.
// Warp-uniform loop over the examples (the lane groups shuffle); the live count is read on the device.
template <int LPR>
__global__ void __launch_bounds__(128)
leaf_stats_kernel(const float* __restrict__ Z, int ldz, int n, const float* __restrict__ t,
                  const float* __restrict__ y, int n_cls, const int* __restrict__ pos, const int* __restrict__ orig,
                  const int* __restrict__ count, int n_fixed, double* __restrict__ out) {
    const int nb = count ? *count : n_fixed;
    extern __shared__ float sacc[];                       // [2 + 2 * n_cls]
    const int na = 2 + 2 * n_cls;
    for (int i = threadIdx.x; i < na; i += blockDim.x) sacc[i] = 0.f;
    __syncthreads();
    const int j = threadIdx.x % LPR;
    for (int b = (blockIdx.x * blockDim.x + threadIdx.x) / LPR; b - (int)(threadIdx.x & 31) / LPR < nb;
         b += gridDim.x * blockDim.x / LPR) {
        const bool live = b < nb;
        const bool on = live && j < n;
        const int row = !live ? 0 : pos ? pos[b] : b;
        const int o = !live ? 0 : orig ? orig[b] : b;
        const float z = on ? Z[(size_t)row * ldz + j] : -INFINITY;
        const float tt = on ? t[(size_t)o * n + j] : -INFINITY;
        const float mx = grp_max<LPR>(z);
        const float e = on ? expf(z - mx) : 0.f;
        const float p = e * (1.f / grp_sum<LPR>(e));
        const int am_p = grp_argmax<LPR>(on ? p : -INFINITY, j);
        const int am_t = grp_argmax<LPR>(tt, j);
        if (live) {
            const bool cor = am_p == am_t;
            if (j == 0) atomicAdd(sacc + (cor ? 0 : 1), 1.f);
            const float* yy = y + (size_t)o * n_cls;
            for (int c = j; c < n_cls; c += LPR)
                if (yy[c] != 0.f) atomicAdd(sacc + 2 + (cor ? 0 : n_cls) + c, yy[c]);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < na; i += blockDim.x)
        if (sacc[i] != 0.f) atomicAdd(out + i, (double)sacc[i]);
}

extern "C" int mpnn_leaf_stats_targets(const float* Z, int ldz, int n_out, const float* t, const float* y, int n_cls,
                                       const int* pos, const int* orig, const int* count, int n, double* out,
                                       void* stream) {
    MPNN_REQUIRE(Z && t && y && out && n_out >= 1 && n_out <= CE_NMAX && ldz >= n_out && n_cls >= 1 && n_cls <= 1024
                 && n >= 0, "leaf_stats: n_out=%d ldz=%d n_cls=%d n=%d", n_out, ldz, n_cls, n);
    const int lpr = n_out <= 16 ? 16 : 32;
    int grid = ceil_div(n > 0 ? n : 1, 128 / lpr);
    if (grid > 148) grid = 148;
    const size_t smem = (2 + 2 * n_cls) * sizeof(float);
    if (lpr == 16)
        leaf_stats_kernel<16><<<grid, 128, smem, (cudaStream_t)stream>>>(Z, ldz, n_out, t, y, n_cls, pos, orig, count, n, out);
    else
        leaf_stats_kernel<32><<<grid, 128, smem, (cudaStream_t)stream>>>(Z, ldz, n_out, t, y, n_cls, pos, orig, count, n, out);
    return mpnn_check_launch("leaf_stats");
}

// dZ in fp32 [B][n] and/or as two bf16 planes [2][Balloc][8] (columns >= n zero) for the
// tcgen05 head GEMMs; dbias += column sums of dZ.  squared: the error layer is SquaredError on x = prob.
template <int LPR>
__global__ void __launch_bounds__(128)
softmax_ce_bwd_kernel(const float* __restrict__ prob, const float* __restrict__ y, int B, int n,
                      float eps, const float* __restrict__ coef, float coef_scale,
                      float* __restrict__ dZ, __nv_bfloat16* __restrict__ dZp, int Balloc,
                      float* __restrict__ dbias, int squared) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = t / LPR, j = t % LPR;
    const bool on = b < B && j < n;
    float v = 0.f;
    {
        const float s = on ? prob[(size_t)b * n + j] : 0.f;
        const float yy = on ? y[(size_t)b * n + j] : 0.f;
        const float g = !on ? 0.f : (squared ? 2.f * (s - yy) : -yy * (1.f - eps) / (eps / n + (1.f - eps) * s));
        const float dot = grp_sum<LPR>(s * g);
        const float k = (b < B ? (coef ? coef[b] : 1.f) : 0.f) * coef_scale;
        v = !on ? 0.f : (squared ? k * g : k * s * (g - dot));
    }
    if (on && dZ) dZ[(size_t)b * n + j] = v;
    if (dZp && b < B && j < 16) plane_row(dZp, j >> 3, Balloc, b)[j & 7] = __float2bfloat16_rn(v);
    if (dbias) {
        // column sums over the examples of this CTA: across the lane groups of a warp, then across the warps
        float c = v;
#pragma unroll
        for (int o = 16; o >= LPR; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
        __shared__ float red[4][LPR];
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (lane < LPR) red[warp][lane] = c;
        __syncthreads();
        if (threadIdx.x < n && threadIdx.x < 16)
            atomicAdd(dbias + threadIdx.x, red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x]);
    }
}

static void softmax_ce_bwd_launch(const float* prob, const float* y, int B, int n, float eps, const float* coef,
                                  float coef_scale, float* dZ, void* dZp, int Balloc, float* dbias, int squared,
                                  void* stream) {
    if (n <= 16)
        softmax_ce_bwd_kernel<16><<<ceil_div(B * 16, 128), 128, 0, (cudaStream_t)stream>>>(
            prob, y, B, n, eps, coef, coef_scale, dZ, (__nv_bfloat16*)dZp, Balloc, dbias, squared);
    else
        softmax_ce_bwd_kernel<32><<<ceil_div(B * 32, 128), 128, 0, (cudaStream_t)stream>>>(
            prob, y, B, n, eps, coef, coef_scale, dZ, (__nv_bfloat16*)dZp, Balloc, dbias, squared);
}

extern "C" int mpnn_softmax_ce_bwd(const float* prob, const float* y, int B, int n, float eps,
                                   const float* coef, float coef_scale, float* dZ,
                                   void* dZp, int Balloc, float* dbias, void* stream) {
    MPNN_REQUIRE(n >= 1 && n <= CE_NMAX, "softmax_ce_bwd: n=%d", n);
    MPNN_REQUIRE((!dZp && !dbias) || n <= 16, "softmax_ce_bwd: planes / bias output need n <= 16 (n=%d)", n);
    softmax_ce_bwd_launch(prob, y, B, n, eps, coef, coef_scale, dZ, dZp, Balloc, dbias, 0, stream);
    return mpnn_check_launch("softmax_ce_bwd");
}

// ------------------------------------------------------ SquaredError (lib/layer_types.py:255-260)
// on the LinTrans output x: c_err = sum_j (x_j - y_j)^2, d_cor = [argmax x == argmax y] (first maximum).
// `out` keeps a dense copy of x for the backward (the head GEMM's own buffer has a wider row stride).
__global__ void squared_err_fwd_kernel(const float* __restrict__ Z, int ldz, const float* __restrict__ y, int B, int n,
                                       float* __restrict__ out, float* __restrict__ c_err, float* __restrict__ d_cor) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float ce = 0.f, best_x = -INFINITY, best_y = -INFINITY;
    int am_x = 0, am_y = 0;
    for (int j = 0; j < n; ++j) {
        const float x = Z[(size_t)b * ldz + j], yy = y[(size_t)b * n + j];
        out[(size_t)b * n + j] = x;
        const float d = x - yy;
        ce = fmaf(d, d, ce);
        if (x > best_x) { best_x = x; am_x = j; }
        if (yy > best_y) { best_y = yy; am_y = j; }
    }
    c_err[b] = ce;
    d_cor[b] = am_x == am_y ? 1.f : 0.f;
}

extern "C" int mpnn_squared_err_fwd(const float* Z, int ldz, const float* y, int B, int n,
                                    float* out, float* c_err, float* d_cor, void* stream) {
    MPNN_REQUIRE(n >= 1 && n <= CE_NMAX && ldz >= n, "squared_err_fwd: n=%d ldz=%d", n, ldz);
    squared_err_fwd_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(Z, ldz, y, B, n, out, c_err, d_cor);
    return mpnn_check_launch("squared_err_fwd");
}

extern "C" int mpnn_squared_err_bwd(const float* out, const float* y, int B, int n,
                                    const float* coef, float coef_scale, float* dZ,
                                    void* dZp, int Balloc, float* dbias, void* stream) {
    MPNN_REQUIRE(n >= 1 && n <= CE_NMAX, "squared_err_bwd: n=%d", n);
    MPNN_REQUIRE((!dZp && !dbias) || n <= 16, "squared_err_bwd: planes / bias output need n <= 16 (n=%d)", n);
    softmax_ce_bwd_launch(out, y, B, n, 0.f, coef, coef_scale, dZ, dZp, Balloc, dbias, 1, stream);
    return mpnn_check_launch("squared_err_bwd");
}

// ------------------------------------- SuperclassCrossEntropyError targets (lib/layer_types.py:274-285)
// y_sup = y @ w_cls, [B][n_cls] x [n_cls][n_sup]; softmax_ce_fwd / bwd then run on y_sup.
__global__ void superclass_targets_kernel(const float* __restrict__ y, const float* __restrict__ w, int B, int n_cls,
                                          int n_sup, float* __restrict__ y_sup) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= B * n_sup) return;
    const int b = e / n_sup, k = e % n_sup;
    float t = 0.f;
    for (int j = 0; j < n_cls; ++j) t = fmaf(y[(size_t)b * n_cls + j], w[(size_t)j * n_sup + k], t);
    y_sup[e] = t;
}

extern "C" int mpnn_superclass_targets(const float* y, const float* w_cls, int B, int n_cls, int n_sup,
                                       float* y_sup, void* stream) {
    MPNN_REQUIRE(y && w_cls && y_sup && B >= 1 && n_cls >= 1 && n_sup >= 1, "superclass_targets: args");
    superclass_targets_kernel<<<ceil_div(B * n_sup, 256), 256, 0, (cudaStream_t)stream>>>(y, w_cls, B, n_cls, n_sup, y_sup);
    return mpnn_check_launch("superclass_targets");
}

// ----------------------------------------------------------------- router tail
#define RT_C 16
#define RT_THREADS 512
#define RT_NSMAX 8

// per-channel sum over B rows of f(row) for a [B][16] array; result in out[16] (smem)
__device__ void rt_channel_stats(const float* __restrict__ Zin, int B, float* mean, float* rstd,
                                 float eps, float* sred /*RT_THREADS*/) {
    const int tid = threadIdx.x, c = tid % RT_C;
    float s = 0.f;
    for (int e = tid; e < B * RT_C; e += RT_THREADS) s += Zin[e];
    sred[tid] = s;
    __syncthreads();
    if (tid < RT_C) {
        double t = 0.0;
        for (int k = tid; k < RT_THREADS; k += RT_C) t += sred[k];
        mean[tid] = (float)(t / B);
    }
    __syncthreads();
    float m = mean[c];
    s = 0.f;
    for (int e = tid; e < B * RT_C; e += RT_THREADS) { float d = Zin[e] - m; s += d * d; }
    sred[tid] = s;
    __syncthreads();
    if (tid < RT_C) {
        double t = 0.0;
        for (int k = tid; k < RT_THREADS; k += RT_C) t += sred[k];
        rstd[tid] = (float)(t / B);          // variance for now
    }
    __syncthreads();
}

__device__ __forceinline__ void
router_tail_fwd_body(const float* Z1, int B,
                       const float* __restrict__ g1, const float* __restrict__ b1, float* m1, float* v1,
                       const float* __restrict__ W2, const float* __restrict__ bias2,
                       const float* __restrict__ g2, const float* __restrict__ b2, float* m2, float* v2,
                       const float* __restrict__ W3, const float* __restrict__ bias3, int ns,
                       float d, float eps, int train, float* Z2, float* __restrict__ R,
                       float* __restrict__ save) {
    __shared__ float sred[RT_THREADS];
    __shared__ float mean[RT_C], var[RT_C], a[RT_C], c[RT_C];
    __shared__ float sW2[RT_C * RT_C], sW3[RT_C * RT_NSMAX], sb2[RT_C], sb3[RT_NSMAX];
    const int tid = threadIdx.x;
    if (tid < RT_C * RT_C) sW2[tid] = W2[tid];
    if (tid < RT_C * ns) sW3[tid] = W3[tid];
    if (tid < RT_C) sb2[tid] = bias2[tid];
    if (tid < ns) sb3[tid] = bias3[tid];
    for (int layer = 0; layer < 2; ++layer) {
        const float* Zin = layer == 0 ? Z1 : Z2;
        const float* gg = layer == 0 ? g1 : g2;
        const float* bb = layer == 0 ? b1 : b2;
        float* ma = layer == 0 ? m1 : m2;
        float* va = layer == 0 ? v1 : v2;
        __syncthreads();
        if (train) {
            rt_channel_stats(Zin, B, mean, var, eps, sred);
            if (tid < RT_C) {
                ma[tid] = d * ma[tid] + (1.f - d) * mean[tid];
                va[tid] = d * va[tid] + (1.f - d) * var[tid];
            }
        } else if (tid < RT_C) {
            mean[tid] = ma[tid]; var[tid] = va[tid];
        }
        __syncthreads();
        if (tid < RT_C) {
            float rs = 1.f / sqrtf(var[tid] + eps);
            a[tid] = gg[tid] * rs;
            c[tid] = bb[tid] - mean[tid] * a[tid];
            save[layer * 2 * RT_C + tid] = mean[tid];
            save[layer * 2 * RT_C + RT_C + tid] = rs;
        }
        __syncthreads();
        for (int b = tid; b < B; b += RT_THREADS) {
            float h[RT_C];
#pragma unroll
            for (int i = 0; i < RT_C; ++i) h[i] = fmaxf(fmaf(a[i], Zin[(size_t)b * RT_C + i], c[i]), 0.f);
            if (layer == 0) {
#pragma unroll
                for (int j = 0; j < RT_C; ++j) {
                    float t = sb2[j];
#pragma unroll
                    for (int i = 0; i < RT_C; ++i) t = fmaf(h[i], sW2[i * RT_C + j], t);
                    Z2[(size_t)b * RT_C + j] = t;
                }
            } else {
                for (int k = 0; k < ns; ++k) {
                    float t = sb3[k];
#pragma unroll
                    for (int i = 0; i < RT_C; ++i) t = fmaf(h[i], sW3[i * ns + k], t);
                    R[(size_t)b * ns + k] = t;
                }
            }
        }
        __threadfence_block();
    }
}

__global__ void __launch_bounds__(RT_THREADS)
router_tail_fwd_kernel(const float* Z1, int B, const float* g1, const float* b1, float* m1, float* v1,
                       const float* W2, const float* bias2, const float* g2, const float* b2, float* m2,
                       float* v2, const float* W3, const float* bias3, int ns, float d, float eps, int train,
                       float* Z2, float* R, float* save) {
    router_tail_fwd_body(Z1, B, g1, b1, m1, v1, W2, bias2, g2, b2, m2, v2, W3, bias3, ns, d, eps, train, Z2, R, save);
}

// (the batched variants -- every router in one launch -- live in router_cluster.cu)

extern "C" int mpnn_router_tail_fwd(const float* Z1, int B, int C,
                                    const float* g1, const float* b1, float* m1, float* v1,
                                    const float* W2, const float* bias2,
                                    const float* g2, const float* b2, float* m2, float* v2,
                                    const float* W3, const float* bias3, int ns,
                                    float d, float eps, int train,
                                    float* Z2, float* R, float* save, void* stream) {
    MPNN_REQUIRE(C == RT_C, "router_tail_fwd: C=%d (only %d; wider routers run in mpnn_router_tail_fwd_batched)", C, RT_C);
    MPNN_REQUIRE(ns >= 2 && ns <= RT_NSMAX, "router_tail_fwd: ns=%d", ns);
    router_tail_fwd_kernel<<<1, RT_THREADS, 0, (cudaStream_t)stream>>>(
        Z1, B, g1, b1, m1, v1, W2, bias2, g2, b2, m2, v2, W3, bias3, ns, d, eps, train, Z2, R, save);
    return mpnn_check_launch("router_tail_fwd");
}

// block-wide sum of a per-thread vector into smem acc[n] (acc must be zeroed before)
template <int N>
__device__ __forceinline__ void rt_block_add(const float (&v)[N], float* acc) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        float t = warp_sum(v[i]);
        if (lane == 0) atomicAdd(acc + i, t);
    }
}

__device__ __forceinline__ void
router_tail_bwd_body(const float* __restrict__ Z1, const float* __restrict__ Z2,
                       const float* __restrict__ dR, int B, int ns,
                       const float* __restrict__ g1, const float* __restrict__ b1,
                       const float* __restrict__ W2,
                       const float* __restrict__ g2, const float* __restrict__ b2,
                       const float* __restrict__ W3, const float* __restrict__ save,
                       float* dg1, float* dbt1, float* dW2, float* dbias2,
                       float* dg2, float* dbt2, float* dW3, float* dbias3,
                       float* __restrict__ dZ1, float* __restrict__ scratch,
                       __nv_bfloat16* __restrict__ dZ1p, int Balloc, float* dbias1) {
    __shared__ float sW2[RT_C * RT_C], sW3[RT_C * RT_NSMAX];
    __shared__ float a1[RT_C], c1[RT_C], a2[RT_C], c2[RT_C], mn1[RT_C], rs1[RT_C], mn2[RT_C], rs2[RT_C];
    __shared__ float sacc[2 * RT_C];
    __shared__ float part[2][RT_C * RT_C];
    const int tid = threadIdx.x;
    float* sH = scratch;                       // [B][C] activations (h2 then h1)
    float* sD = scratch + (size_t)B * RT_C;    // [B][C] dz2n then dz2
    if (tid < RT_C * RT_C) sW2[tid] = W2[tid];
    if (tid < RT_C * ns) sW3[tid] = W3[tid];
    if (tid < RT_C) {
        mn1[tid] = save[tid]; rs1[tid] = save[RT_C + tid];
        mn2[tid] = save[2 * RT_C + tid]; rs2[tid] = save[3 * RT_C + tid];
        a1[tid] = g1[tid] * rs1[tid]; c1[tid] = b1[tid] - mn1[tid] * a1[tid];
        a2[tid] = g2[tid] * rs2[tid]; c2[tid] = b2[tid] - mn2[tid] * a2[tid];
    }
    if (tid < 2 * RT_C) sacc[tid] = 0.f;
    __syncthreads();
    const float invB = 1.f / (float)B;

    // Phase A: through FC3 and ReLU2; BN2 reduction terms
    {
        float s01[2 * RT_C];
#pragma unroll
        for (int i = 0; i < 2 * RT_C; ++i) s01[i] = 0.f;
        for (int b = tid; b < B; b += RT_THREADS) {
            float dr[RT_NSMAX];
            for (int k = 0; k < ns; ++k) dr[k] = dR[(size_t)b * ns + k];
#pragma unroll
            for (int i = 0; i < RT_C; ++i) {
                float z = Z2[(size_t)b * RT_C + i];
                float h = fmaxf(fmaf(a2[i], z, c2[i]), 0.f);
                float dh = 0.f;
                for (int k = 0; k < ns; ++k) dh = fmaf(dr[k], sW3[i * ns + k], dh);
                float dz = h > 0.f ? dh : 0.f;
                float xh = (z - mn2[i]) * rs2[i];
                sH[(size_t)b * RT_C + i] = h;
                sD[(size_t)b * RT_C + i] = dz;
                s01[i] += dz; s01[RT_C + i] += dz * xh;
            }
        }
        rt_block_add<2 * RT_C>(s01, sacc);
    }
    __syncthreads();
    // Phase A2: dW3, dbias3   (threads (half, i, k))
    {
        const int half = tid / 256, t = tid % 256;
        const int i = t / RT_NSMAX, k = t % RT_NSMAX;
        float acc = 0.f, accb = 0.f;
        if (i < RT_C && k < ns) {
            for (int b = half; b < B; b += 2) {
                float drv = dR[(size_t)b * ns + k];
                acc = fmaf(sH[(size_t)b * RT_C + i], drv, acc);
                if (i == 0) accb += drv;
            }
        }
        part[half][t] = acc;
        __syncthreads();
        if (half == 0 && i < RT_C && k < ns) dW3[i * ns + k] += part[0][t] + part[1][t];
        __syncthreads();
        part[half][t] = accb;
        __syncthreads();
        if (half == 0 && i == 0 && k < ns) dbias3[k] += part[0][t] + part[1][t];
        __syncthreads();
    }
    float m0_2[RT_C], m1_2[RT_C];
#pragma unroll
    for (int i = 0; i < RT_C; ++i) { m0_2[i] = sacc[i] * invB; m1_2[i] = sacc[RT_C + i] * invB; }
    __syncthreads();
    if (tid < RT_C) { dbt2[tid] += sacc[tid]; dg2[tid] += sacc[RT_C + tid]; }
    __syncthreads();
    if (tid < 2 * RT_C) sacc[tid] = 0.f;
    __syncthreads();
    // Phase B: BN2 backward, FC2 backward data, ReLU1; BN1 reduction terms
    {
        float s01[2 * RT_C];
#pragma unroll
        for (int i = 0; i < 2 * RT_C; ++i) s01[i] = 0.f;
        for (int b = tid; b < B; b += RT_THREADS) {
            float dz2[RT_C];
#pragma unroll
            for (int j = 0; j < RT_C; ++j) {
                float z = Z2[(size_t)b * RT_C + j];
                float xh = (z - mn2[j]) * rs2[j];
                dz2[j] = a2[j] * (sD[(size_t)b * RT_C + j] - m0_2[j] - xh * m1_2[j]);
                sD[(size_t)b * RT_C + j] = dz2[j];
            }
#pragma unroll
            for (int i = 0; i < RT_C; ++i) {
                float z = Z1[(size_t)b * RT_C + i];
                float h = fmaxf(fmaf(a1[i], z, c1[i]), 0.f);
                float dh = 0.f;
#pragma unroll
                for (int j = 0; j < RT_C; ++j) dh = fmaf(dz2[j], sW2[i * RT_C + j], dh);
                float dz = h > 0.f ? dh : 0.f;
                float xh = (z - mn1[i]) * rs1[i];
                sH[(size_t)b * RT_C + i] = h;
                dZ1[(size_t)b * RT_C + i] = dz;
                s01[i] += dz; s01[RT_C + i] += dz * xh;
            }
        }
        rt_block_add<2 * RT_C>(s01, sacc);
    }
    __syncthreads();
    // Phase B2: dW2, dbias2
    {
        const int half = tid / 256, t = tid % 256;
        const int i = t / RT_C, j = t % RT_C;
        float acc = 0.f, accb = 0.f;
        for (int b = half; b < B; b += 2) {
            float dv = sD[(size_t)b * RT_C + j];
            acc = fmaf(sH[(size_t)b * RT_C + i], dv, acc);
            if (i == 0) accb += dv;
        }
        part[half][t] = acc;
        __syncthreads();
        if (half == 0) dW2[t] += part[0][t] + part[1][t];
        __syncthreads();
        part[half][t] = accb;
        __syncthreads();
        if (half == 0 && i == 0) dbias2[j] += part[0][t] + part[1][t];
        __syncthreads();
    }
    if (tid < RT_C) { dbt1[tid] += sacc[tid]; dg1[tid] += sacc[RT_C + tid]; }
    // Phase C: BN1 backward in place (+ bf16 planes copy for the tcgen05 head GEMMs)
    float bsum[RT_C];
#pragma unroll
    for (int i = 0; i < RT_C; ++i) bsum[i] = 0.f;
    for (int b = tid; b < B; b += RT_THREADS) {
        float o[RT_C];
#pragma unroll
        for (int i = 0; i < RT_C; ++i) {
            float z = Z1[(size_t)b * RT_C + i];
            float xh = (z - mn1[i]) * rs1[i];
            float dz = dZ1[(size_t)b * RT_C + i];
            dz = a1[i] * (dz - sacc[i] * invB - xh * sacc[RT_C + i] * invB);
            dZ1[(size_t)b * RT_C + i] = dz;
            o[i] = dz;
            bsum[i] += dz;
        }
        if (dZ1p) {
            Row8<__nv_bfloat16>::store(plane_row(dZ1p, 0, Balloc, b), o);
            Row8<__nv_bfloat16>::store(plane_row(dZ1p, 1, Balloc, b), o + 8);
        }
    }
    if (dbias1) {          // bias of the first router FC (zero up to rounding under train-mode BN)
        __syncthreads();
        if (tid < RT_C) sacc[tid] = 0.f;
        __syncthreads();
        rt_block_add<RT_C>(bsum, sacc);
        __syncthreads();
        if (tid < RT_C) dbias1[tid] += sacc[tid];
    }
}

__global__ void __launch_bounds__(RT_THREADS)
router_tail_bwd_kernel(const float* Z1, const float* Z2, const float* dR, int B, int ns,
                       const float* g1, const float* b1, const float* W2, const float* g2, const float* b2,
                       const float* W3, const float* save, float* dg1, float* dbt1, float* dW2, float* dbias2,
                       float* dg2, float* dbt2, float* dW3, float* dbias3, float* dZ1, float* scratch) {
    router_tail_bwd_body(Z1, Z2, dR, B, ns, g1, b1, W2, g2, b2, W3, save, dg1, dbt1, dW2, dbias2, dg2, dbt2,
                         dW3, dbias3, dZ1, scratch, nullptr, 0, nullptr);
}

// (the batched variant -- every router in one launch -- lives in router_cluster.cu)

extern "C" int mpnn_router_tail_bwd(const float* Z1, const float* Z2, const float* dR, int B, int C, int ns,
                                    const float* g1, const float* b1, const float* W2,
                                    const float* g2, const float* b2, const float* W3,
                                    const float* save,
                                    float* dg1, float* dbt1, float* dW2, float* dbias2,
                                    float* dg2, float* dbt2, float* dW3, float* dbias3,
                                    float* dZ1, float* scratch, void* stream) {
    MPNN_REQUIRE(C == RT_C, "router_tail_bwd: C=%d (only %d; wider routers run in mpnn_router_tail_bwd_batched)", C, RT_C);
    MPNN_REQUIRE(ns >= 2 && ns <= RT_NSMAX, "router_tail_bwd: ns=%d", ns);
    router_tail_bwd_kernel<<<1, RT_THREADS, 0, (cudaStream_t)stream>>>(
        Z1, Z2, dR, B, ns, g1, b1, W2, g2, b2, W3, save, dg1, dbt1, dW2, dbias2, dg2, dbt2, dW3, dbias3,
        dZ1, scratch);
    return mpnn_check_launch("router_tail_bwd");
}
