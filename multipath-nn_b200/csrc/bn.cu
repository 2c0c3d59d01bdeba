// BatchNorm (+ReLU, +2x2 max-pool, +feature flatten) forward and backward on
// padded-planes tensors.  All kernels touch VALID pixels only, so the zero
// pads of act / pooled / dLin survive from the one-time memset.
// Reference: lib/layer_types.py:109-110 (pool), :196-199 (ReLU), :219-249 (BN).
#include "common.cuh"
#include "../../include/mpnn.h"
#include "bn_fuse.cuh"

// ------------------------------------------------------------------ finalize
__global__ void bn_finalize_kernel(const float* __restrict__ partials, int n_parts, int C, double count,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float* __restrict__ m_avg, float* __restrict__ v_avg,
                                   float d, float eps, int train,
                                   float* __restrict__ ss, float* __restrict__ mr) {
    // one warp per channel: lanes stride over the partial rows (fixed order -> deterministic)
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= C) return;
    float mean, var;
    if (train) {
        double s = 0.0, s2 = 0.0;
        for (int i = lane; i < n_parts; i += 32) {
            s += (double)partials[((size_t)i * 2) * C + c];
            s2 += (double)partials[((size_t)i * 2 + 1) * C + c];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if (lane != 0) return;
        double m = s / count;
        double v = s2 / count - m * m;
        if (v < 0.0) v = 0.0;
        mean = (float)m; var = (float)v;
        if (m_avg) {
            m_avg[c] = d * m_avg[c] + (1.f - d) * mean;
            v_avg[c] = d * v_avg[c] + (1.f - d) * var;
        }
    } else {
        if (lane != 0) return;
        mean = m_avg[c]; var = v_avg[c];
    }
    float rstd = 1.0f / sqrtf(var + eps);
    float a = gamma[c] * rstd;
    ss[c] = a;
    ss[C + c] = beta[c] - mean * a;
    mr[c] = mean;
    mr[C + c] = rstd;
}

extern "C" int mpnn_bn_finalize(const float* partials, int n_parts, int C, double count,
                                const float* gamma, const float* beta, float* m_avg, float* v_avg,
                                float d, float eps, int train, float* ss, float* mr, void* stream) {
    MPNN_REQUIRE(C > 0 && (train == 0 || (partials && n_parts > 0)), "bn_finalize: args");
    bn_finalize_kernel<<<ceil_div(C, 4), 128, 0, (cudaStream_t)stream>>>(
        partials, n_parts, C, count, gamma, beta, m_avg, v_avg, d, eps, train, ss, mr);
    return mpnn_check_launch("bn_finalize");
}

// ------------------------------------------------------------------ forward
// One thread per (plane kg, image n, row pair h2, full-resolution column w) when pooling,
// per pixel otherwise: consecutive lanes touch consecutive 16/32-byte rows, so every
// load and store instruction is fully coalesced; the 2x2 maximum is taken in-thread
// over the row pair and across the lane pair (w, w^1) with one shuffle per channel.
// grid.y = plane, so the per-channel constants are loaded once per thread.
// CNT: only the first min(*count, g.B) images are read and written (g.B: the capacity the grid was sized for).
template <typename T, bool POOL, bool CNT = false>
__global__ void __launch_bounds__(256)
bn_relu_pool_fwd_kernel(const T* __restrict__ lin, int C, Geom g,
                        const float* __restrict__ ss, T* __restrict__ act,
                        T* __restrict__ pooled, Geom gp,
                        T* __restrict__ feat, int Balloc, const mpnn_bn_fuse bn, const int* __restrict__ count) {
    pdl_launch_dependents();
    pdl_wait();
    const int KG = C / 8, kg = blockIdx.y;
    const int HH = POOL ? g.H / 2 : g.H;
    const int nb = CNT ? min(max(*count, 0), g.B) : g.B;
    const unsigned total = (unsigned)nb * HH * g.W;           // host guarantees < 2^31
    if (CNT && total == 0) return;
    float a[8], c[8];
    const bool affine = (ss || bn.acc) && (act || feat);
    if (bn.acc) {
        // deferred train-mode statistics: the producer left the totals in bn.acc; every thread derives the constants
        // of its 8 channels, the first CTA of the plane publishes them and updates the running moments
        const bool pub = blockIdx.x == 0 && threadIdx.x == 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int ch = kg * 8 + j;
            float mean, var, rstd;
            mpnn_bn_consts_from_acc(bn, C, ch, a[j], c[j], mean, var, rstd);
            if (pub) {
                bn.ss[ch] = a[j]; bn.ss[C + ch] = c[j];
                bn.mr[ch] = mean; bn.mr[C + ch] = rstd;
                if (bn.m_avg) {
                    bn.m_avg[ch] = bn.d * bn.m_avg[ch] + (1.f - bn.d) * mean;
                    bn.v_avg[ch] = bn.d * bn.v_avg[ch] + (1.f - bn.d) * var;
                }
            }
        }
    } else if (affine) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { a[j] = __ldg(ss + kg * 8 + j); c[j] = __ldg(ss + C + kg * 8 + j); }
    }
    const unsigned lane = threadIdx.x & 31;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i - lane < total; i += gridDim.x * blockDim.x) {
        const bool ok = i < total;
        const unsigned ii = ok ? i : 0;
        const int w = ii % (unsigned)g.W;
        const unsigned r = ii / (unsigned)g.W;
        const int h = r % (unsigned)HH;
        const int n = r / (unsigned)HH;
        if (POOL) {
            const int p0 = row_of(g, n, 2 * h, w), p1 = p0 + g.Wp;
            float v0[8], v1[8], mx[8];
            if (ok) {
                Row8<T>::load(plane_row(lin, kg, g.P, p0), v0);
                Row8<T>::load(plane_row(lin, kg, g.P, p1), v1);
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) { v0[j] = 0.f; v1[j] = 0.f; }
            }
            if (ok && act && affine) {
                float o[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = fmaxf(fmaf(a[j], v0[j], c[j]), 0.f);
                Row8<T>::store(plane_row(act, kg, g.P, p0), o);
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = fmaxf(fmaf(a[j], v1[j], c[j]), 0.f);
                Row8<T>::store(plane_row(act, kg, g.P, p1), o);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                mx[j] = fmaxf(v0[j], v1[j]);
                mx[j] = fmaxf(mx[j], __shfl_xor_sync(0xffffffffu, mx[j], 1));
            }
            if (ok && !(w & 1)) Row8<T>::store(plane_row(pooled, kg, gp.P, row_of(gp, n, h, w >> 1)), mx);
        } else if (ok) {
            const int p = row_of(g, n, h, w);
            float v[8], o[8];
            Row8<T>::load(plane_row(lin, kg, g.P, p), v);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaxf(fmaf(a[j], v[j], c[j]), 0.f);
            if (act) Row8<T>::store(plane_row(act, kg, g.P, p), o);
            if (feat) Row8<T>::store(plane_row(feat, (h * g.W + w) * KG + kg, Balloc, n), o);
        }
    }
}

static int bn_relu_pool_fwd_impl(const void* lin, int C, int B, int H, int W, int G, int P,
                                 const float* ss, const mpnn_bn_fuse* bnp, void* act, void* pooled, int Pp,
                                 void* feat, int Balloc, int dtype, void* stream, const int* count = nullptr) {
    MPNN_REQUIRE(C % 8 == 0, "bn_relu_pool_fwd: C=%d", C);
    MPNN_REQUIRE(!count || !bnp, "bn_relu_pool_fwd_counted: no train-mode statistics");
    MPNN_REQUIRE(!(pooled && feat), "bn_relu_pool_fwd: pooled and feat are exclusive");
    MPNN_REQUIRE(pooled || ss || bnp, "bn_relu_pool_fwd: nothing to do");
    MPNN_REQUIRE(!pooled || (H % 2 == 0 && W % 2 == 0), "bn_relu_pool_fwd: odd size");
    MPNN_REQUIRE(!bnp || (bnp->acc && bnp->gamma && bnp->beta && bnp->ss && bnp->mr && bnp->count > 0),
                 "bn_relu_pool_fwd_acc: incomplete mpnn_bn_fuse");
    Geom g = make_geom(B, H, W, G, P);
    Geom gp = make_geom(B, H / 2, W / 2, G, Pp);
    long long total = (long long)B * (pooled ? (H / 2) * W : H * W);
    MPNN_REQUIRE(total < (1ll << 31), "bn_relu_pool_fwd: too many pixels");
    int gx = (int)((total + 255) / 256);
    int cap = 148 * 16 / (C / 8);
    if (cap < 148) cap = 148;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    dim3 grid(gx, C / 8);
    cudaStream_t st = (cudaStream_t)stream;
    mpnn_bn_fuse bn = {};
    if (bnp) bn = *bnp;
#define GO(POOL, CNT) MPNN_DISPATCH_DTYPE(dtype, (mpnn_launch_pdl(bn_relu_pool_fwd_kernel<T, POOL, CNT>, grid, dim3(256), \
        0, st, (const T*)lin, C, g, ss, (T*)act, (T*)pooled, gp, (T*)feat, Balloc, bn, count)))
    if (pooled) {
        if (count) GO(true, true); else GO(true, false);
    } else {
        if (count) GO(false, true); else GO(false, false);
    }
#undef GO
    return mpnn_check_launch("bn_relu_pool_fwd");
}

extern "C" int mpnn_bn_relu_pool_fwd(const void* lin, int C, int B, int H, int W, int G, int P,
                                     const float* ss, void* act, void* pooled, int Pp,
                                     void* feat, int Balloc, int dtype, void* stream) {
    return bn_relu_pool_fwd_impl(lin, C, B, H, W, G, P, ss, nullptr, act, pooled, Pp, feat, Balloc, dtype, stream);
}

extern "C" int mpnn_bn_relu_pool_fwd_counted(const void* lin, int C, int B, int H, int W, int G, int P,
                                             const float* ss, void* act, void* pooled, int Pp,
                                             void* feat, int Balloc, int dtype, const int* count, void* stream) {
    return bn_relu_pool_fwd_impl(lin, C, B, H, W, G, P, ss, nullptr, act, pooled, Pp, feat, Balloc, dtype, stream,
                                 count);
}

extern "C" int mpnn_bn_relu_pool_fwd_acc(const void* lin, int C, int B, int H, int W, int G, int P,
                                         const mpnn_bn_fuse* bn, void* act, void* pooled, int Pp,
                                         void* feat, int Balloc, int dtype, void* stream) {
    MPNN_REQUIRE(bn, "bn_relu_pool_fwd_acc: bn is NULL");
    return bn_relu_pool_fwd_impl(lin, C, B, H, W, G, P, nullptr, bn, act, pooled, Pp, feat, Balloc, dtype, stream);
}

// ---------------------------------------------------------------------------
// Small tensors (B*H*W <= MPNN_BN_SMALL_MAX_PIXELS, no pooled output: the coarsest scale of a stage at the
// reference's batch): train-mode statistics AND BN / ReLU (/ feature flatten) in ONE launch.  With the statistics
// riding on the conv launch, a small conv ends in a chain of global round trips (fp64 atomics -> fence -> ticket ->
// last CTA reads the totals back and writes the constants: 6.0 us instead of 2.6 for the same conv without them,
// profiles/r02_mb_chain.txt).  Here the conv stores `lin` and nothing else; one 8-CTA cluster per 8-channel plane
// loads its pixels once (<= 4 per thread, kept in registers), sums x and x^2 warp -> CTA -> cluster (distributed
// shared memory, fixed rank order, fp64 across CTAs) behind ONE cluster barrier, and every CTA derives the
// constants and writes its part of act / feat; rank 0 publishes ss / mr and updates the running moments
// (lib/layer_types.py:219-249).
// ---------------------------------------------------------------------------
#include <cooperative_groups.h>
namespace cgf = cooperative_groups;
constexpr int kFwdCL = 8, kFwdT = 256;
static_assert(kFwdCL * kFwdT * 4 == MPNN_BN_SMALL_MAX_PIXELS, "bn_fwd_small capacity");

template <typename T, int RPT>
__global__ void __cluster_dims__(kFwdCL, 1, 1) __launch_bounds__(kFwdT)
bn_fwd_small_kernel(const T* __restrict__ lin, int C, Geom g, const float* __restrict__ gamma,
                    const float* __restrict__ beta, float* __restrict__ m_avg, float* __restrict__ v_avg,
                    float d, float eps, double count, float* __restrict__ ss, float* __restrict__ mr,
                    T* __restrict__ act, T* __restrict__ feat, int Balloc) {
    cgf::cluster_group cluster = cgf::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int kg = blockIdx.y, KG = C / 8, tid = threadIdx.x;
    const int total = g.B * g.H * g.W;
    const int per = (total + kFwdCL - 1) / kFwdCL;
    __shared__ float red[kFwdT / 32][16];
    __shared__ float part[16];
    __shared__ float sa[8], sc[8];
    float lv[RPT][8];
    int prow[RPT], pfeat[RPT], pn[RPT];
    float s1[8], s2[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { s1[j] = 0.f; s2[j] = 0.f; }
#pragma unroll
    for (int u = 0; u < RPT; ++u) {
        const int k = u * kFwdT + tid, i = rank * per + k;
        prow[u] = -1;
        if (k < per && i < total) {
            const int w = i % g.W, r = i / g.W, h = r % g.H, n = r / g.H;
            prow[u] = row_of(g, n, h, w);
            pfeat[u] = (h * g.W + w) * KG + kg;
            pn[u] = n;
            Row8<T>::load(plane_row(lin, kg, g.P, prow[u]), lv[u]);
#pragma unroll
            for (int j = 0; j < 8; ++j) { s1[j] += lv[u][j]; s2[j] = fmaf(lv[u][j], lv[u][j], s2[j]); }
        }
    }
    const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float t1 = warp_sum(s1[j]), t2 = warp_sum(s2[j]);
        if (lane == 0) { red[warp][j] = t1; red[warp][8 + j] = t2; }
    }
    __syncthreads();
    if (tid < 16) {
        float t = 0.f;
#pragma unroll
        for (int wv = 0; wv < kFwdT / 32; ++wv) t += red[wv][tid];
        part[tid] = t;
    }
    cluster.sync();
    if (tid < 8) {
        double t1 = 0.0, t2 = 0.0;
        for (int k = 0; k < kFwdCL; ++k) {
            const float* pp = cluster.map_shared_rank(&part[0], k);
            t1 += (double)pp[tid]; t2 += (double)pp[8 + tid];
        }
        const int ch = kg * 8 + tid;
        const double m = t1 / count;
        double v = t2 / count - m * m;
        if (v < 0.0) v = 0.0;
        const float mean = (float)m, var = (float)v;
        const float rstd = 1.0f / sqrtf(var + eps);
        const float a = gamma[ch] * rstd, sh = beta[ch] - mean * a;
        sa[tid] = a; sc[tid] = sh;
        if (rank == 0) {
            ss[ch] = a; ss[C + ch] = sh;
            mr[ch] = mean; mr[C + ch] = rstd;
            if (m_avg) {
                m_avg[ch] = d * m_avg[ch] + (1.f - d) * mean;
                v_avg[ch] = d * v_avg[ch] + (1.f - d) * var;
            }
        }
    }
    __syncthreads();
    float a[8], c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { a[j] = sa[j]; c[j] = sc[j]; }
#pragma unroll
    for (int u = 0; u < RPT; ++u) {
        if (prow[u] >= 0) {
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaxf(fmaf(a[j], lv[u][j], c[j]), 0.f);
            if (act) Row8<T>::store(plane_row(act, kg, g.P, prow[u]), o);
            if (feat) Row8<T>::store(plane_row(feat, pfeat[u], Balloc, pn[u]), o);
        }
    }
    cluster.sync();          // keep this CTA's shared memory alive until every peer has read it
}

extern "C" int mpnn_bn_fwd_small(const void* lin, int C, int B, int H, int W, int G, int P,
                                 const float* gamma, const float* beta, float* m_avg, float* v_avg,
                                 float d, float eps, float* ss, float* mr,
                                 void* act, void* feat, int Balloc, int dtype, void* stream) {
    MPNN_REQUIRE(C % 8 == 0 && lin && gamma && beta && ss && mr && (act || feat), "bn_fwd_small: args");
    MPNN_REQUIRE((m_avg == nullptr) == (v_avg == nullptr), "bn_fwd_small: m_avg / v_avg");
    const long long total = (long long)B * H * W;
    MPNN_REQUIRE(total <= MPNN_BN_SMALL_MAX_PIXELS,
                 "bn_fwd_small: %lld pixels (at most %d: use mpnn_conv_bn_stats + mpnn_bn_relu_pool_fwd)", total,
                 MPNN_BN_SMALL_MAX_PIXELS);
    Geom g = make_geom(B, H, W, G, P);
    const int per = ((int)total + kFwdCL - 1) / kFwdCL;
    const int rpt = (per + kFwdT - 1) / kFwdT;
    dim3 grid(kFwdCL, C / 8);
    cudaStream_t st = (cudaStream_t)stream;
#define MPNN_BN_FWD_SMALL_LAUNCH(R)                                                                        \
    MPNN_DISPATCH_DTYPE(dtype, (bn_fwd_small_kernel<T, R><<<grid, kFwdT, 0, st>>>(                          \
        (const T*)lin, C, g, gamma, beta, m_avg, v_avg, d, eps, (double)total, ss, mr, (T*)act, (T*)feat, Balloc)))
    if (rpt <= 1) { MPNN_BN_FWD_SMALL_LAUNCH(1); }
    else if (rpt <= 2) { MPNN_BN_FWD_SMALL_LAUNCH(2); }
    else { MPNN_BN_FWD_SMALL_LAUNCH(4); }
#undef MPNN_BN_FWD_SMALL_LAUNCH
    return mpnn_check_launch("bn_fwd_small");
}
