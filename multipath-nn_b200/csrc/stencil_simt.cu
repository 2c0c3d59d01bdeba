// fp32-accumulate SIMT implementation of the stencil GEMM (conv fwd / dgrad /
// 1-tap FC-as-GEMM) and its weight gradient.  This is the exact-arithmetic
// ("fp32 mode") path the parity tests anchor on; the tcgen05 path lives in
// stencil_umma.cu and is selected with impl=1.
#include "common.cuh"
#include "../../include/mpnn.h"
#include "bn_fuse.cuh"

int mpnn_stencil_gemm_umma(const void* A0, int K0, const void* A1, int K1, const void* Wp, int ntaps,
                           const float* bias, void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                           Geom g, float* stats, int stats_cap, int* n_parts, int out_dtype,
                           const mpnn_bn_fuse* bn, const mpnn_bn_bwd_epi* bwd, const int* count, cudaStream_t st);
int mpnn_stencil_wgrad_umma(const void* A0, int K0, int K0real, float* dW0, const void* A1, int K1,
                            int K1real, float* dW1, const void* Gd, int N, int Nreal, float* dbias,
                            int ntaps, Geom g, cudaStream_t st);

__device__ __forceinline__ int tap_offset(int ntaps, int tap, int Wp) {
    return ntaps == 9 ? (tap / 3 - 1) * Wp + (tap % 3 - 1) : 0;
}

// CNT: the live batch is min(*count, g.B) (g.B: the capacity the grid was sized for); only its rows are stored.
template <typename T, typename TO, int NB, bool CNT = false>
__global__ void __launch_bounds__(128)
stencil_gemm_simt(const T* __restrict__ A0, int K0, const T* __restrict__ A1, int K1,
                  const T* __restrict__ Wp, int ntaps, const float* __restrict__ bias,
                  TO* __restrict__ out0, int N0, int acc0, TO* __restrict__ out1, int N1, int acc1,
                  Geom g, int n_tiles, float* __restrict__ stats, const mpnn_bn_fuse bn, const int* __restrict__ count) {
    const int N = N0 + N1;
    int row_end = g.rows + 128 - 1;              // the tiles' pad rows beyond the batch are stored too (unspecified)
    if (CNT) {
        row_end = min(max(*count, 0), g.B) * g.S;
        n_tiles = (row_end + 127) >> 7;
    }
    const int n0 = blockIdx.y * NB;
    const int KG0 = K0 / 8, KG = (K0 + K1) / 8;
    float ssum[NB], ssq[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) { ssum[j] = 0.f; ssq[j] = 0.f; }

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int q = tile * 128 + threadIdx.x;
        const int p = g.G + q;
        float acc[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) acc[j] = bias ? __ldg(bias + n0 + j) : 0.f;
        for (int tap = 0; tap < ntaps; ++tap) {
            const int pr = p + tap_offset(ntaps, tap, g.Wp);
            for (int kg = 0; kg < KG; ++kg) {
                float a[8];
                if (kg < KG0) Row8<T>::load(plane_row(A0, kg, g.P, pr), a);
                else          Row8<T>::load(plane_row(A1, kg - KG0, g.P, pr), a);
                const T* wrow = Wp + (((size_t)tap * KG + kg) * N + n0) * 8;
#pragma unroll
                for (int j = 0; j < NB; ++j) {
                    float w[8];
                    Row8<T>::load(wrow + j * 8, w);
#pragma unroll
                    for (int c = 0; c < 8; ++c) acc[j] = fmaf(a[c], w[c], acc[j]);
                }
            }
        }
        int n_, h_, w_;
        const bool valid = row_valid(g, q, n_, h_, w_);
        if (q < row_end && p < g.P) {
#pragma unroll
            for (int j8 = 0; j8 < NB / 8; ++j8) {
                int col = n0 + j8 * 8;
                TO* dst; int accf;
                if (col < N0) { dst = plane_row(out0, col / 8, g.P, p); accf = acc0; }
                else          { dst = plane_row(out1, (col - N0) / 8, g.P, p); accf = acc1; }
                float v[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) v[c] = acc[j8 * 8 + c];
                if (accf) {
                    float o[8];
                    Row8<TO>::load(dst, o);
#pragma unroll
                    for (int c = 0; c < 8; ++c) v[c] += o[c];
                }
                Row8<TO>::store(dst, v);
            }
        }
        if ((stats || bn.acc) && valid) {
#pragma unroll
            for (int j = 0; j < NB; ++j) { ssum[j] += acc[j]; ssq[j] += acc[j] * acc[j]; }
        }
    }
    if (stats || bn.acc) {
        __shared__ float red[4][2 * NB];
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            float s = warp_sum(ssum[j]), s2 = warp_sum(ssq[j]);
            if (lane == 0) { red[warp][j] = s; red[warp][NB + j] = s2; }
        }
        __syncthreads();
        if (stats && threadIdx.x < 2 * NB) {
            float t = red[0][threadIdx.x] + red[1][threadIdx.x] + red[2][threadIdx.x] + red[3][threadIdx.x];
            int which = threadIdx.x / NB, j = threadIdx.x % NB;
            stats[((size_t)blockIdx.x * 2 + which) * N + n0 + j] = t;
        }
        if (bn.acc && bn.defer) {
            mpnn_acc_only(bn.acc, N, n0, NB, [&](int i) { return red[0][i] + red[1][i] + red[2][i] + red[3][i]; });
        } else if (bn.acc) {
            const bool last = mpnn_acc_and_ticket(bn.acc, N, n0, NB, gridDim.x * gridDim.y,
                                                  [&](int i) { return red[0][i] + red[1][i] + red[2][i] + red[3][i]; });
            if (last) mpnn_bn_fwd_finalize_last(bn, N);
        }
    }
}

template <typename T, typename TO, bool CNT>
static int launch_gemm_simt(const void* A0, int K0, const void* A1, int K1, const void* Wp, int ntaps,
                            const float* bias, void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                            Geom g, float* stats, int stats_cap, int* n_parts, const mpnn_bn_fuse* bnp,
                            const int* count, cudaStream_t st) {
    const int N = N0 + N1;
    mpnn_bn_fuse bn = {};
    if (bnp) bn = *bnp;
    const int n_tiles = ceil_div(g.rows, 128);
    int gx = n_tiles;
    if (stats) { if (gx > stats_cap) gx = stats_cap; }
    else if (bnp) { if (gx > 148 * 4) gx = 148 * 4; }
    else if (gx > 148 * 32) gx = 148 * 32;
    if (n_parts) *n_parts = stats ? gx : 0;
    if (N % 32 == 0 && N0 % 32 == 0) {
        dim3 grid(gx, N / 32);
        stencil_gemm_simt<T, TO, 32, CNT><<<grid, 128, 0, st>>>((const T*)A0, K0, (const T*)A1, K1, (const T*)Wp,
            ntaps, bias, (TO*)out0, N0, acc0, (TO*)out1, N1, acc1, g, n_tiles, stats, bn, count);
    } else if (N % 16 == 0 && N0 % 16 == 0) {
        dim3 grid(gx, N / 16);
        stencil_gemm_simt<T, TO, 16, CNT><<<grid, 128, 0, st>>>((const T*)A0, K0, (const T*)A1, K1, (const T*)Wp,
            ntaps, bias, (TO*)out0, N0, acc0, (TO*)out1, N1, acc1, g, n_tiles, stats, bn, count);
    } else {
        dim3 grid(gx, N / 8);
        stencil_gemm_simt<T, TO, 8, CNT><<<grid, 128, 0, st>>>((const T*)A0, K0, (const T*)A1, K1, (const T*)Wp,
            ntaps, bias, (TO*)out0, N0, acc0, (TO*)out1, N1, acc1, g, n_tiles, stats, bn, count);
    }
    return mpnn_check_launch("stencil_gemm_simt");
}

static int stencil_gemm_impl(const void* A0, int K0, const void* A1, int K1,
                             const void* Wp, int ntaps, const float* bias,
                             void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                             int B, int H, int W, int G, int P,
                             float* stats, int stats_cap, int* n_parts, const mpnn_bn_fuse* bn,
                             int dtype, int out_dtype, int impl, void* stream,
                             const mpnn_bn_bwd_epi* bwd = nullptr, const int* count = nullptr) {
    MPNN_REQUIRE(ntaps == 9 || ntaps == 1, "stencil_gemm: ntaps=%d", ntaps);
    MPNN_REQUIRE(!bwd || impl == 1, "conv_dgrad_bn_reduce: only the tcgen05 path fuses the BN-backward sums");
    MPNN_REQUIRE(K0 % 8 == 0 && K1 % 8 == 0 && K0 > 0, "stencil_gemm: K0=%d K1=%d", K0, K1);
    MPNN_REQUIRE(N0 % 8 == 0 && N1 % 8 == 0 && N0 + N1 > 0, "stencil_gemm: N0=%d N1=%d", N0, N1);
    MPNN_REQUIRE(K1 == 0 || A1, "stencil_gemm: A1 null");
    Geom g = make_geom(B, H, W, G, P);
    const int halo = ntaps == 9 ? g.Wp + 1 : 0;
    MPNN_REQUIRE(G >= halo, "stencil_gemm: front guard %d < %d", G, halo);
    MPNN_REQUIRE(P >= G + ceil_div(g.rows, 128) * 128 + halo, "stencil_gemm: back guard too small (P=%d)", P);
    MPNN_REQUIRE(!stats || stats_cap > 0, "stencil_gemm: stats_cap");
    MPNN_REQUIRE(!count || (!stats && !bn && !bwd), "stencil_gemm_counted: a counted launch computes no statistics");
    MPNN_REQUIRE(!bn || (bn->acc && bn->gamma && bn->beta && bn->ss && bn->mr && bn->count > 0),
                 "conv_bn_stats: incomplete mpnn_bn_fuse");
    cudaStream_t st = (cudaStream_t)stream;
    if (impl == 1) {
        MPNN_REQUIRE(dtype == MPNN_BF16, "stencil_gemm: tcgen05 path needs bf16 operands");
        return mpnn_stencil_gemm_umma(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1,
                                      g, stats, stats_cap, n_parts, out_dtype, bn, bwd, count, st);
    }
#define GO(T, TO) return count ? launch_gemm_simt<T, TO, true>(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1,  \
                                                               N1, acc1, g, stats, stats_cap, n_parts, bn, count, st) \
                           : launch_gemm_simt<T, TO, false>(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1,  \
                                                            N1, acc1, g, stats, stats_cap, n_parts, bn, nullptr, st)
    if (dtype == MPNN_F32 && out_dtype == MPNN_F32) GO(float, float);
    if (dtype == MPNN_BF16 && out_dtype == MPNN_BF16) GO(__nv_bfloat16, __nv_bfloat16);
    if (dtype == MPNN_BF16 && out_dtype == MPNN_F32) GO(__nv_bfloat16, float);
#undef GO
    mpnn_set_error("stencil_gemm: dtype combo %d/%d", dtype, out_dtype);
    return MPNN_ERR_ARG;
}

extern "C" int mpnn_stencil_gemm(const void* A0, int K0, const void* A1, int K1,
                                 const void* Wp, int ntaps, const float* bias,
                                 void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                                 int B, int H, int W, int G, int P,
                                 float* stats, int stats_cap, int* n_parts,
                                 int dtype, int out_dtype, int impl, void* stream) {
    return stencil_gemm_impl(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1, B, H, W, G, P,
                             stats, stats_cap, n_parts, nullptr, dtype, out_dtype, impl, stream);
}

extern "C" int mpnn_stencil_gemm_counted(const void* A0, int K0, const void* A1, int K1,
                                         const void* Wp, int ntaps, const float* bias,
                                         void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                                         int B, int H, int W, int G, int P,
                                         float* stats, int stats_cap, int* n_parts,
                                         int dtype, int out_dtype, int impl, const int* count, void* stream) {
    return stencil_gemm_impl(A0, K0, A1, K1, Wp, ntaps, bias, out0, N0, acc0, out1, N1, acc1, B, H, W, G, P,
                             stats, stats_cap, n_parts, nullptr, dtype, out_dtype, impl, stream, nullptr, count);
}

extern "C" int mpnn_conv_bn_stats(const void* A0, int K0, const void* A1, int K1,
                                  const void* Wp, const float* bias, void* out, int N,
                                  int B, int H, int W, int G, int P, const mpnn_bn_fuse* bn,
                                  int dtype, int impl, void* stream) {
    MPNN_REQUIRE(bn, "conv_bn_stats: bn is NULL");
    return stencil_gemm_impl(A0, K0, A1, K1, Wp, 9, bias, out, N, 0, nullptr, 0, 0, B, H, W, G, P,
                             nullptr, 0, nullptr, bn, dtype, dtype, impl, stream);
}

// the general form: accumulate into `out` (acc != 0), output dtype chosen separately from the operand dtype; the
// fused BN statistics are those of the values finally stored.  Used by the bf16x3 mode, where a conv is two
// launches (horizontal operand, then the pooled predecessor accumulated on top) with fp32 planes out.
extern "C" int mpnn_conv_acc_bn_stats(const void* A0, int K0, const void* A1, int K1,
                                      const void* Wp, const float* bias, void* out, int N, int acc,
                                      int B, int H, int W, int G, int P, const mpnn_bn_fuse* bn,
                                      int dtype, int out_dtype, int impl, void* stream) {
    return stencil_gemm_impl(A0, K0, A1, K1, Wp, 9, bias, out, N, acc, nullptr, 0, 0, B, H, W, G, P,
                             nullptr, 0, nullptr, bn, dtype, out_dtype, impl, stream);
}

extern "C" int mpnn_conv_dgrad_bn_reduce(const void* Gd, int K, const void* Wp, void* out0, int N0,
                                         void* out1, int N1, int B, int H, int W, int G, int P,
                                         const mpnn_bn_bwd_epi* epi, int dtype, int impl, void* stream) {
    MPNN_REQUIRE(epi, "conv_dgrad_bn_reduce: epi is NULL");
    return stencil_gemm_impl(Gd, K, nullptr, 0, Wp, 9, nullptr, out0, N0, 0, out1, N1, 0, B, H, W, G, P,
                             nullptr, 0, nullptr, nullptr, dtype, dtype, impl, stream, epi);
}

// --------------------------------------------------------------------------- //
// Weight gradient.  grid = (row chunks, ntaps, K/8); block = 128 threads over n.
// dW[tap][k][n] += sum_p A[p+off][k] * Gd[p][n]
// --------------------------------------------------------------------------- //
template <typename T>
__global__ void __launch_bounds__(128)
stencil_wgrad_simt(const T* __restrict__ A0, int K0, int K0real, float* __restrict__ dW0,
                   const T* __restrict__ A1, int K1, int K1real, float* __restrict__ dW1,
                   const T* __restrict__ Gd, int N, int Nreal, float* __restrict__ dbias,
                   int ntaps, Geom g, int chunk) {
    const int tap = blockIdx.y, kg = blockIdx.z;
    const int KG0 = K0 / 8;
    const T* A = kg < KG0 ? A0 + (size_t)kg * g.P * 8 : A1 + (size_t)(kg - KG0) * g.P * 8;
    const int off = tap_offset(ntaps, tap, g.Wp);
    const int q0 = blockIdx.x * chunk;
    const int q1 = min(q0 + chunk, g.rows);
    const bool do_bias = dbias && tap == 0 && kg == 0;
    for (int n = threadIdx.x; n < N; n += 128) {
        const T* gcol = Gd + (size_t)(n >> 3) * g.P * 8 + (n & 7);
        // fp64 accumulators: this is the reference-arithmetic path, and a sequential fp32 sum over ~1000 pixels
        // of terms that largely cancel costs 1e-3 of the result
        double acc[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[c] = 0.0;
        double bsum = 0.0;
        for (int q = q0; q < q1; ++q) {
            const int p = g.G + q;
            float gv;
            if (sizeof(T) == 4) gv = __ldg(reinterpret_cast<const float*>(gcol) + (size_t)p * 8);
            else gv = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(gcol)[(size_t)p * 8]);
            float a[8];
            Row8<T>::load(A + (size_t)(p + off) * 8, a);
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[c] += (double)a[c] * (double)gv;
            bsum += (double)gv;
        }
        if (n < Nreal) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                int k = kg * 8 + c;
                if (kg < KG0) {
                    if (k < K0real) atomicAdd(dW0 + ((size_t)tap * K0real + k) * Nreal + n, (float)acc[c]);
                } else {
                    int k1 = k - K0;
                    if (k1 < K1real) atomicAdd(dW1 + ((size_t)tap * K1real + k1) * Nreal + n, (float)acc[c]);
                }
            }
            if (do_bias) atomicAdd(dbias + n, (float)bsum);
        }
    }
}

extern "C" int mpnn_stencil_wgrad(const void* A0, int K0, int K0real, float* dW0,
                                  const void* A1, int K1, int K1real, float* dW1,
                                  const void* Gd, int N, int Nreal, float* dbias, int ntaps,
                                  int B, int H, int W, int G, int P,
                                  int dtype, int impl, void* stream) {
    MPNN_REQUIRE(ntaps == 9 || ntaps == 1, "stencil_wgrad: ntaps=%d", ntaps);
    MPNN_REQUIRE(K0 % 8 == 0 && K1 % 8 == 0 && N % 8 == 0, "stencil_wgrad: K0=%d K1=%d N=%d", K0, K1, N);
    MPNN_REQUIRE(K0real <= K0 && K1real <= K1 && Nreal <= N, "stencil_wgrad: real > padded");
    Geom g = make_geom(B, H, W, G, P);
    MPNN_REQUIRE(G >= g.Wp + 1 && P >= G + g.rows + 128 + g.Wp + 1, "stencil_wgrad: guards");
    cudaStream_t st = (cudaStream_t)stream;
    if (impl == 1) {
        MPNN_REQUIRE(dtype == MPNN_BF16, "stencil_wgrad: tcgen05 path needs bf16 operands");
        return mpnn_stencil_wgrad_umma(A0, K0, K0real, dW0, A1, K1, K1real, dW1, Gd, N, Nreal, dbias,
                                       ntaps, g, st);
    }
    int chunk = g.rows > (1 << 17) ? 8192 : 2048;      // few fp32 atomics per output: their order is the remaining noise
    dim3 grid(ceil_div(g.rows, chunk), ntaps, (K0 + K1) / 8);
    MPNN_DISPATCH_DTYPE(dtype, (stencil_wgrad_simt<T><<<grid, 128, 0, st>>>(
        (const T*)A0, K0, K0real, dW0, (const T*)A1, K1, K1real, dW1, (const T*)Gd, N, Nreal, dbias,
        ntaps, g, chunk)));
    return mpnn_check_launch("stencil_wgrad_simt");
}
