// Forward and backward of every router tail of the net in ONE launch each, one 8-CTA thread-block
// cluster per router (reference: lib/net_types.py router() = FC16-BN-ReLU-FC16-
// BN-ReLU-FC(n_sinks); TF autodiff through train-mode batch norm).
//
// Train-mode BN makes the backward a chain of two batch-wide reductions
//   (BN2 sums) -> (BN1 sums) -> dZ1,
// which a single CTA can only walk serially over the whole batch.  Here the
// batch is split over the 8 CTAs of a cluster; each CTA reduces its slice, the
// slices are combined through distributed shared memory (fixed rank order, so
// the BN statistics are deterministic) and cluster.sync() separates the phases.
// The two small weight gradients (16x16, 16xns) are accumulated per CTA from
// shared-memory tiles and added to the flat gradient buffer with fp32 atomics.
#include <cooperative_groups.h>
#include <cstdlib>
#include "common.cuh"
#include "../../include/mpnn.h"

namespace cg = cooperative_groups;

namespace {

constexpr int C = 16;            // router width
constexpr int NSMAX = 8;         // max sinks
constexpr int T = 256;           // threads per CTA = rows per tile
constexpr int CL = 8;            // CTAs per cluster
constexpr int LD = C + 1;        // padded tile row

__device__ __forceinline__ void block_add(const float* v, int n, float* acc) {
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < n; ++i) {
        float t = warp_sum(v[i]);
        if (lane == 0) atomicAdd(acc + i, t);
    }
}

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_bwd_cluster_kernel(const mpnn_router_bwd_desc* __restrict__ descs, int B) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_bwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;

    __shared__ float sW2[C * C], sW3[C * NSMAX];
    __shared__ float a1[C], c1[C], a2[C], c2[C], mn1[C], rs1[C], mn2[C], rs2[C];
    __shared__ float tH[T * LD], tD[T * LD], tR[T * (NSMAX + 1)];
    __shared__ float part[T];
    __shared__ float sum2[2 * C], sum1[2 * C];      // this CTA's BN2 / BN1 partial sums (read by the cluster)
    __shared__ float tot2[2 * C], tot1[2 * C];      // cluster totals
    __shared__ float sb1[C];

    sW2[tid] = r.W2[tid];
    if (tid < C * ns) sW3[tid] = r.W3[tid];
    if (tid < C) {
        mn1[tid] = r.save[tid]; rs1[tid] = r.save[C + tid];
        mn2[tid] = r.save[2 * C + tid]; rs2[tid] = r.save[3 * C + tid];
        a1[tid] = r.g1[tid] * rs1[tid]; c1[tid] = r.b1[tid] - mn1[tid] * a1[tid];
        a2[tid] = r.g2[tid] * rs2[tid]; c2[tid] = r.b2[tid] - mn2[tid] * a2[tid];
        sb1[tid] = 0.f;
    }
    if (tid < 2 * C) { sum2[tid] = 0.f; sum1[tid] = 0.f; }
    __syncthreads();

    const int Bc = (B + CL - 1) / CL;
    const int b_lo = rank * Bc, b_hi = min(B, b_lo + Bc);
    const float invB = 1.f / (float)B;

    // forward recompute of one row up to dL/d(BN2 output): h2, masked dz, xhat2
    auto row_top = [&](int b, float* h2, float* dz, float* xh, float* dr) {
        for (int k = 0; k < NSMAX; ++k) dr[k] = k < ns ? r.dR[(size_t)b * ns + k] : 0.f;
#pragma unroll
        for (int i = 0; i < C; ++i) {
            const float z = r.Z2[(size_t)b * C + i];
            const float h = fmaxf(fmaf(a2[i], z, c2[i]), 0.f);
            float dh = 0.f;
            for (int k = 0; k < ns; ++k) dh = fmaf(dr[k], sW3[i * ns + k], dh);
            h2[i] = h;
            dz[i] = h > 0.f ? dh : 0.f;
            xh[i] = (z - mn2[i]) * rs2[i];
        }
    };

    // ---- phase A: FC3 / ReLU2 backward, BN2 sums, dW3, dbias3 --------------------
    {
        float s01[2 * C];
#pragma unroll
        for (int i = 0; i < 2 * C; ++i) s01[i] = 0.f;
        const int q = tid >> 7, t = tid & 127, gi = t >> 3, gk = t & 7;     // (row phase, i, k)
        float acc = 0.f, accb = 0.f;
        for (int base = b_lo; base < b_hi; base += T) {
            const int b = base + tid;
            float h2[C], dz[C], xh[C], dr[NSMAX];
            if (b < b_hi) {
                row_top(b, h2, dz, xh, dr);
#pragma unroll
                for (int i = 0; i < C; ++i) { s01[i] += dz[i]; s01[C + i] += dz[i] * xh[i]; }
            } else {
#pragma unroll
                for (int i = 0; i < C; ++i) h2[i] = 0.f;
#pragma unroll
                for (int k = 0; k < NSMAX; ++k) dr[k] = 0.f;
            }
#pragma unroll
            for (int i = 0; i < C; ++i) tH[tid * LD + i] = h2[i];
#pragma unroll
            for (int k = 0; k < NSMAX; ++k) tR[tid * (NSMAX + 1) + k] = dr[k];
            __syncthreads();
            const int nrow = min(T, b_hi - base);          // rows of this tile that hold examples
            for (int row = q; row < nrow; row += 2) {
                const float drv = tR[row * (NSMAX + 1) + gk];
                acc = fmaf(tH[row * LD + gi], drv, acc);
                accb += drv;
            }
            __syncthreads();
        }
        part[tid] = acc;
        __syncthreads();
        if (tid < 128 && gk < ns) atomicAdd(r.dW3 + gi * ns + gk, part[tid] + part[tid + 128]);
        __syncthreads();
        part[tid] = accb;
        __syncthreads();
        if (tid < 128 && gi == 0 && gk < ns) atomicAdd(r.dbias3 + gk, part[tid] + part[tid + 128]);
        block_add(s01, 2 * C, sum2);
    }
    cluster.sync();
    if (tid < 2 * C) {
        float t = 0.f;
        for (int k = 0; k < CL; ++k) t += cluster.map_shared_rank(sum2, k)[tid];
        tot2[tid] = t;
        if (rank == 0) {
            if (tid < C) r.dbt2[tid] += t; else r.dg2[tid - C] += t;
        }
    }
    __syncthreads();

    // ---- phase B: BN2 / FC2 / ReLU1 backward, BN1 sums, dW2, dbias2 ----------------
    {
        float s01[2 * C];
#pragma unroll
        for (int i = 0; i < 2 * C; ++i) s01[i] = 0.f;
        const int gi = tid >> 4, gj = tid & 15;
        float acc = 0.f, accb = 0.f;
        for (int base = b_lo; base < b_hi; base += T) {
            const int b = base + tid;
            float h[C], dz2[C];
            if (b < b_hi) {
                float dz[C], xh[C], dr[NSMAX];
                row_top(b, h, dz, xh, dr);
#pragma unroll
                for (int j = 0; j < C; ++j)
                    dz2[j] = a2[j] * (dz[j] - tot2[j] * invB - xh[j] * tot2[C + j] * invB);
#pragma unroll
                for (int i = 0; i < C; ++i) {
                    const float z = r.Z1[(size_t)b * C + i];
                    const float h1 = fmaxf(fmaf(a1[i], z, c1[i]), 0.f);
                    float dh = 0.f;
#pragma unroll
                    for (int j = 0; j < C; ++j) dh = fmaf(dz2[j], sW2[i * C + j], dh);
                    const float d1 = h1 > 0.f ? dh : 0.f;
                    const float x1 = (z - mn1[i]) * rs1[i];
                    h[i] = h1;
                    r.dZ1[(size_t)b * C + i] = d1;
                    s01[i] += d1; s01[C + i] += d1 * x1;
                }
            } else {
#pragma unroll
                for (int i = 0; i < C; ++i) { h[i] = 0.f; dz2[i] = 0.f; }
            }
#pragma unroll
            for (int i = 0; i < C; ++i) { tH[tid * LD + i] = h[i]; tD[tid * LD + i] = dz2[i]; }
            __syncthreads();
            const int nrow = min(T, b_hi - base);
            for (int row = 0; row < nrow; ++row) {
                const float dv = tD[row * LD + gj];
                acc = fmaf(tH[row * LD + gi], dv, acc);
                accb += dv;
            }
            __syncthreads();
        }
        atomicAdd(r.dW2 + tid, acc);
        if (gi == 0) atomicAdd(r.dbias2 + gj, accb);
        block_add(s01, 2 * C, sum1);
    }
    cluster.sync();
    if (tid < 2 * C) {
        float t = 0.f;
        for (int k = 0; k < CL; ++k) t += cluster.map_shared_rank(sum1, k)[tid];
        tot1[tid] = t;
        if (rank == 0) {
            if (tid < C) r.dbt1[tid] += t; else r.dg1[tid - C] += t;
        }
    }
    __syncthreads();

    // ---- phase C: BN1 backward in place (+ bf16 planes copy for the tcgen05 head GEMMs) ---
    {
        float bsum[C];
#pragma unroll
        for (int i = 0; i < C; ++i) bsum[i] = 0.f;
        for (int b = b_lo + tid; b < b_hi; b += T) {
            float o[C];
#pragma unroll
            for (int i = 0; i < C; ++i) {
                const float z = r.Z1[(size_t)b * C + i];
                const float x1 = (z - mn1[i]) * rs1[i];
                float d = r.dZ1[(size_t)b * C + i];
                d = a1[i] * (d - tot1[i] * invB - x1 * tot1[C + i] * invB);
                r.dZ1[(size_t)b * C + i] = d;
                o[i] = d;
                bsum[i] += d;
            }
            if (r.dZ1p) {
                __nv_bfloat16* pl = (__nv_bfloat16*)r.dZ1p;
                Row8<__nv_bfloat16>::store(plane_row(pl, 0, r.Balloc, b), o);
                Row8<__nv_bfloat16>::store(plane_row(pl, 1, r.Balloc, b), o + 8);
            }
        }
        if (r.dbias1) {      // bias of the first router FC (zero up to rounding under train-mode BN)
            block_add(bsum, C, sb1);
            __syncthreads();
            if (tid < C) atomicAdd(r.dbias1 + tid, sb1[tid]);
        }
    }
    cluster.sync();          // keep this CTA's shared memory alive until every peer has read it
}

// ---------------------------------------------------------------------------
// Forward of every router tail in one launch (same cluster layout): BN1 -> ReLU -> FC16 -> BN2 ->
// ReLU -> FC(ns).  Train-mode statistics are two-pass (mean, then centred second moment) like
// tf.nn.moments; each pass is a per-CTA partial + a fixed-order fp64 sum over the cluster.
__device__ __forceinline__ void cluster_channel_sum(cg::cluster_group& cluster, const float* v, float* part, double* out) {
    // v[C]: this thread's partial per channel; part[C]: CTA partial (smem, read by the cluster)
    const int tid = threadIdx.x;
    if (tid < C) part[tid] = 0.f;
    __syncthreads();
    block_add(v, C, part);
    cluster.sync();
    if (tid < C) {
        double t = 0.0;
        for (int k = 0; k < CL; ++k) t += (double)cluster.map_shared_rank(part, k)[tid];
        out[tid] = t;
    }
    cluster.sync();          // everyone has read `part` before it is reused
}

// CNT (eval mode only): the rows b < min(*count, B) are computed and stored; the batch is split over the cluster by
// the capacity B, so every row sees the arithmetic of an uncounted launch at batch B
template <bool CNT = false>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_fwd_cluster_kernel(const mpnn_router_fwd_desc* __restrict__ descs, int B, float d, float eps, int train,
                               const int* __restrict__ count) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_fwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;
    __shared__ float sW2[C * C], sW3[C * NSMAX], sb2[C], sb3[NSMAX];
    __shared__ float part[C], a[C], c[C], mean[C];
    __shared__ double tot[C];
    sW2[tid] = r.W2[tid];
    if (tid < C * ns) sW3[tid] = r.W3[tid];
    if (tid < C) sb2[tid] = r.bias2[tid];
    if (tid < ns) sb3[tid] = r.bias3[tid];
    const int Bc = (B + CL - 1) / CL;
    const int b_lo = rank * Bc, b_hi = min(CNT ? min(max(*count, 0), B) : B, b_lo + Bc);
    for (int layer = 0; layer < 2; ++layer) {
        const float* Zin = layer == 0 ? r.Z1 : r.Z2;
        const float* gg = layer == 0 ? r.g1 : r.g2;
        const float* bb = layer == 0 ? r.b1 : r.b2;
        float* ma = layer == 0 ? r.m1 : r.m2;
        float* va = layer == 0 ? r.v1 : r.v2;
        __syncthreads();
        if (train) {
            float v[C];
#pragma unroll
            for (int i = 0; i < C; ++i) v[i] = 0.f;
            for (int b = b_lo + tid; b < b_hi; b += T) {
#pragma unroll
                for (int i = 0; i < C; ++i) v[i] += Zin[(size_t)b * C + i];
            }
            cluster_channel_sum(cluster, v, part, tot);
            if (tid < C) mean[tid] = (float)(tot[tid] / B);
            __syncthreads();
#pragma unroll
            for (int i = 0; i < C; ++i) v[i] = 0.f;
            for (int b = b_lo + tid; b < b_hi; b += T) {
#pragma unroll
                for (int i = 0; i < C; ++i) { const float t = Zin[(size_t)b * C + i] - mean[i]; v[i] = fmaf(t, t, v[i]); }
            }
            cluster_channel_sum(cluster, v, part, tot);
            if (tid < C) {
                const float var = (float)(tot[tid] / B);
                const float rs = 1.f / sqrtf(var + eps);
                a[tid] = gg[tid] * rs;
                c[tid] = bb[tid] - mean[tid] * a[tid];
                if (rank == 0) {
                    ma[tid] = d * ma[tid] + (1.f - d) * mean[tid];
                    va[tid] = d * va[tid] + (1.f - d) * var;
                    r.save[layer * 2 * C + tid] = mean[tid];
                    r.save[layer * 2 * C + C + tid] = rs;
                }
            }
        } else if (tid < C) {
            const float m = ma[tid], rs = 1.f / sqrtf(va[tid] + eps);
            a[tid] = gg[tid] * rs;
            c[tid] = bb[tid] - m * a[tid];
            if (rank == 0) { r.save[layer * 2 * C + tid] = m; r.save[layer * 2 * C + C + tid] = rs; }
        }
        __syncthreads();
        for (int b = b_lo + tid; b < b_hi; b += T) {
            float h[C];
#pragma unroll
            for (int i = 0; i < C; ++i) h[i] = fmaxf(fmaf(a[i], Zin[(size_t)b * C + i], c[i]), 0.f);
            if (layer == 0) {
#pragma unroll
                for (int j = 0; j < C; ++j) {
                    float t = sb2[j];
#pragma unroll
                    for (int i = 0; i < C; ++i) t = fmaf(h[i], sW2[i * C + j], t);
                    r.Z2[(size_t)b * C + j] = t;
                }
            } else {
                for (int k = 0; k < ns; ++k) {
                    float t = sb3[k];
#pragma unroll
                    for (int i = 0; i < C; ++i) t = fmaf(h[i], sW3[i * ns + k], t);
                    r.R[(size_t)b * ns + k] = t;
                }
            }
        }
        __threadfence_block();      // this CTA re-reads its own Z2 rows in the next layer
    }
    cluster.sync();
}


// ---------------------------------------------------------------------------
// Register-resident variants (the ones the entry points use for B <= 8 * 256 * RPT): the tail is a CHAIN --
// at the reference's batch of 128 the kernels above spend their time in dependent round trips (every pass
// re-reads its rows from global memory: three passes per layer forward, three phases backward) and in
// 16..32 serial shuffle-reduce-atomic sequences per reduction.  Here every thread owns RPT rows, loads them
// ONCE, keeps them in registers across all passes / phases, and every batch reduction is a transposing
// column sum (warp_colsum16: 16 shuffles for 16 columns) + one shared-memory hop + one DSMEM hop, in a fixed
// order (deterministic statistics).  Each exchange has its own shared-memory slot, so one cluster.sync()
// per exchange suffices.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void load_row16(const float* p, float (&v)[C]) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 t = *(reinterpret_cast<const float4*>(p) + q);
            v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) v[i] = p[i];
    }
}
__device__ __forceinline__ void store_row16(float* p, const float (&v)[C]) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            *(reinterpret_cast<float4*>(p) + q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) p[i] = v[i];
    }
}
// sum over the 32 lanes of v[0..16): afterwards every lane holds the total of column (lane & 15)
__device__ __forceinline__ float colsum16(float (&v)[C], int lane) {
#pragma unroll
    for (int s = 8; s >= 1; s >>= 1) {
        const bool up = (lane & s) != 0;
#pragma unroll
        for (int i = 0; i < s; ++i) {
            const float send = up ? v[i] : v[i + s];
            const float keep = up ? v[i + s] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
        }
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 16);
}
// CTA total of the per-thread columns v[16] -> out[16] (shared memory, written by threads 0..15; visible after the
// caller's next barrier).  wpart: [T / 32][16] scratch.  Destroys v.
__device__ __forceinline__ void cta_colsum16(float (&v)[C], float* wpart, float* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float t = colsum16(v, lane);
    __syncthreads();                       // earlier readers of wpart are done
    if (lane < C) wpart[warp * C + lane] = t;
    __syncthreads();
    if (threadIdx.x < C) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < T / 32; ++w) s += wpart[w * C + threadIdx.x];
        out[threadIdx.x] = s;
    }
}

template <int RPT, bool CNT = false>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_fwd_fast_kernel(const mpnn_router_fwd_desc* __restrict__ descs, int B, float d, float eps, int train,
                            const int* __restrict__ count) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_fwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;
    __shared__ float sW2[C * C], sW3[C * NSMAX], sb2[C], sb3[NSMAX];
    __shared__ float wpart[(T / 32) * C], part[4][C], a[C], c[C], mean[C];
    sW2[tid] = r.W2[tid];
    if (tid < C * ns) sW3[tid] = r.W3[tid];
    if (tid < C) sb2[tid] = r.bias2[tid];
    if (tid < ns) sb3[tid] = r.bias3[tid];
    const int Bc = (B + CL - 1) / CL;
    const int b_lo = rank * Bc, b_hi = min(CNT ? min(max(*count, 0), B) : B, b_lo + Bc);
    float z[RPT][C];
    bool ok[RPT];
#pragma unroll
    for (int u = 0; u < RPT; ++u) {
        const int b = b_lo + u * T + tid;
        ok[u] = b < b_hi;
        if (ok[u]) load_row16(r.Z1 + (size_t)b * C, z[u]);
        else {
#pragma unroll
            for (int i = 0; i < C; ++i) z[u][i] = 0.f;
        }
    }
    const double invB = 1.0 / (double)B;
#pragma unroll
    for (int layer = 0; layer < 2; ++layer) {
        const float* gg = layer == 0 ? r.g1 : r.g2;
        const float* bb = layer == 0 ? r.b1 : r.b2;
        float* ma = layer == 0 ? r.m1 : r.m2;
        float* va = layer == 0 ? r.v1 : r.v2;
        if (train) {
            // two-pass moments like tf.nn.moments: mean, then the centred second moment
            float v[C];
#pragma unroll
            for (int i = 0; i < C; ++i) {
                v[i] = 0.f;
#pragma unroll
                for (int u = 0; u < RPT; ++u) v[i] += z[u][i];            // rows that do not exist are zero
            }
            cta_colsum16(v, wpart, part[2 * layer]);
            cluster.sync();
            if (tid < C) {
                double t = 0.0;
                for (int k = 0; k < CL; ++k) t += (double)cluster.map_shared_rank(&part[2 * layer][0], k)[tid];
                mean[tid] = (float)(t * invB);
            }
            __syncthreads();
#pragma unroll
            for (int i = 0; i < C; ++i) {
                v[i] = 0.f;
#pragma unroll
                for (int u = 0; u < RPT; ++u) {
                    const float t = z[u][i] - mean[i];
                    v[i] = ok[u] ? fmaf(t, t, v[i]) : v[i];
                }
            }
            cta_colsum16(v, wpart, part[2 * layer + 1]);
            cluster.sync();
            if (tid < C) {
                double t = 0.0;
                for (int k = 0; k < CL; ++k) t += (double)cluster.map_shared_rank(&part[2 * layer + 1][0], k)[tid];
                const float var = (float)(t * invB);
                const float rs = 1.f / sqrtf(var + eps);
                a[tid] = gg[tid] * rs;
                c[tid] = bb[tid] - mean[tid] * a[tid];
                if (rank == 0) {
                    ma[tid] = d * ma[tid] + (1.f - d) * mean[tid];
                    va[tid] = d * va[tid] + (1.f - d) * var;
                    r.save[layer * 2 * C + tid] = mean[tid];
                    r.save[layer * 2 * C + C + tid] = rs;
                }
            }
        } else if (tid < C) {
            const float m = ma[tid], rs = 1.f / sqrtf(va[tid] + eps);
            a[tid] = gg[tid] * rs;
            c[tid] = bb[tid] - m * a[tid];
            if (rank == 0) { r.save[layer * 2 * C + tid] = m; r.save[layer * 2 * C + C + tid] = rs; }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            const int b = b_lo + u * T + tid;
            float h[C];
#pragma unroll
            for (int i = 0; i < C; ++i) h[i] = fmaxf(fmaf(a[i], z[u][i], c[i]), 0.f);
            if (layer == 0) {
                float o[C];
#pragma unroll
                for (int j = 0; j < C; ++j) {
                    float t = sb2[j];
#pragma unroll
                    for (int i = 0; i < C; ++i) t = fmaf(h[i], sW2[i * C + j], t);
                    o[j] = t;
                }
                if (ok[u]) store_row16(r.Z2 + (size_t)b * C, o);
#pragma unroll
                for (int j = 0; j < C; ++j) z[u][j] = ok[u] ? o[j] : 0.f;       // the next layer's input stays in registers
            } else if (ok[u]) {
                for (int k = 0; k < ns; ++k) {
                    float t = sb3[k];
#pragma unroll
                    for (int i = 0; i < C; ++i) t = fmaf(h[i], sW3[i * ns + k], t);
                    r.R[(size_t)b * ns + k] = t;
                }
            }
        }
        __syncthreads();                   // a / c / mean are rewritten by the next layer
    }
    cluster.sync();                        // keep this CTA's shared memory alive until every peer has read it
}

template <int RPT>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_bwd_fast_kernel(const mpnn_router_bwd_desc* __restrict__ descs, int B) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_bwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;

    __shared__ float sW2[C * C], sW3[C * NSMAX];
    __shared__ float a1[C], c1[C], a2[C], c2[C], mn1[C], rs1[C], mn2[C], rs2[C];
    __shared__ float tH[T * LD], tD[T * LD], tR[T * (NSMAX + 1)];
    __shared__ float part[T], wpart[(T / 32) * C];
    __shared__ float sum2[2 * C], sum1[2 * C];      // this CTA's BN2 / BN1 partial sums (read by the cluster)
    __shared__ float tot2[2 * C], tot1[2 * C];      // cluster totals
    __shared__ float sb1[C];

    sW2[tid] = r.W2[tid];
    if (tid < C * NSMAX) sW3[tid] = tid < C * ns ? r.W3[tid] : 0.f;
    if (tid < C) {
        mn1[tid] = r.save[tid]; rs1[tid] = r.save[C + tid];
        mn2[tid] = r.save[2 * C + tid]; rs2[tid] = r.save[3 * C + tid];
        a1[tid] = r.g1[tid] * rs1[tid]; c1[tid] = r.b1[tid] - mn1[tid] * a1[tid];
        a2[tid] = r.g2[tid] * rs2[tid]; c2[tid] = r.b2[tid] - mn2[tid] * a2[tid];
    }
    const int Bc = (B + CL - 1) / CL;
    const int b_lo = rank * Bc, b_hi = min(B, b_lo + Bc);
    const float invB = 1.f / (float)B;
    // the rows of this thread, loaded once
    float z2[RPT][C], z1[RPT][C], dr[RPT][NSMAX], d1[RPT][C];
    bool ok[RPT];
#pragma unroll
    for (int u = 0; u < RPT; ++u) {
        const int b = b_lo + u * T + tid;
        ok[u] = b < b_hi;
        if (ok[u]) {
            load_row16(r.Z2 + (size_t)b * C, z2[u]);
            load_row16(r.Z1 + (size_t)b * C, z1[u]);
#pragma unroll
            for (int k = 0; k < NSMAX; ++k) dr[u][k] = k < ns ? r.dR[(size_t)b * ns + k] : 0.f;
        } else {
#pragma unroll
            for (int i = 0; i < C; ++i) { z2[u][i] = 0.f; z1[u][i] = 0.f; }
#pragma unroll
            for (int k = 0; k < NSMAX; ++k) dr[u][k] = 0.f;
        }
    }
    __syncthreads();
    // one row up to dL/d(BN2 output): h2, masked dz, xhat2 (weights beyond ns are zero-filled: static loop bounds)
    auto row_top = [&](int u, float* h2, float* dz, float* xh) {
#pragma unroll
        for (int i = 0; i < C; ++i) {
            const float z = z2[u][i];
            const float h = fmaxf(fmaf(a2[i], z, c2[i]), 0.f);
            float dh = 0.f;
#pragma unroll
            for (int k = 0; k < NSMAX; ++k) dh = fmaf(dr[u][k], sW3[i * ns + k], dh);
            h2[i] = h;
            dz[i] = h > 0.f ? dh : 0.f;
            xh[i] = (z - mn2[i]) * rs2[i];
        }
    };

    // ---- phase A: FC3 / ReLU2 backward, BN2 sums, dW3, dbias3 --------------------
    {
        float s0[C], s1[C];
#pragma unroll
        for (int i = 0; i < C; ++i) { s0[i] = 0.f; s1[i] = 0.f; }
        const int q = tid >> 7, t = tid & 127, gi = t >> 3, gk = t & 7;     // (row phase, i, k)
        float acc = 0.f, accb = 0.f;
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            float h2[C], dz[C], xh[C];
            row_top(u, h2, dz, xh);
#pragma unroll
            for (int i = 0; i < C; ++i) {
                if (ok[u]) { s0[i] += dz[i]; s1[i] = fmaf(dz[i], xh[i], s1[i]); }
                tH[tid * LD + i] = ok[u] ? h2[i] : 0.f;
            }
#pragma unroll
            for (int k = 0; k < NSMAX; ++k) tR[tid * (NSMAX + 1) + k] = dr[u][k];
            __syncthreads();
            const int nrow = max(0, min(T, b_hi - (b_lo + u * T)));     // rows of this tile that hold examples
            for (int row = q; row < nrow; row += 2) {
                const float drv = tR[row * (NSMAX + 1) + gk];
                acc = fmaf(tH[row * LD + gi], drv, acc);
                accb += drv;
            }
            __syncthreads();
        }
        part[tid] = acc;
        __syncthreads();
        if (tid < 128 && gk < ns) atomicAdd(r.dW3 + gi * ns + gk, part[tid] + part[tid + 128]);
        __syncthreads();
        part[tid] = accb;
        __syncthreads();
        if (tid < 128 && gi == 0 && gk < ns) atomicAdd(r.dbias3 + gk, part[tid] + part[tid + 128]);
        cta_colsum16(s0, wpart, sum2);
        cta_colsum16(s1, wpart, sum2 + C);
    }
    cluster.sync();
    if (tid < 2 * C) {
        float t = 0.f;
        for (int k = 0; k < CL; ++k) t += cluster.map_shared_rank(&sum2[0], k)[tid];
        tot2[tid] = t;
        if (rank == 0) {
            if (tid < C) r.dbt2[tid] += t; else r.dg2[tid - C] += t;
        }
    }
    __syncthreads();

    // ---- phase B: BN2 / FC2 / ReLU1 backward, BN1 sums, dW2, dbias2 ----------------
    {
        float s0[C], s1[C];
#pragma unroll
        for (int i = 0; i < C; ++i) { s0[i] = 0.f; s1[i] = 0.f; }
        const int gi = tid >> 4, gj = tid & 15;
        float acc = 0.f, accb = 0.f;
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            float h[C], dz[C], xh[C], dz2[C];
            row_top(u, h, dz, xh);
#pragma unroll
            for (int j = 0; j < C; ++j)
                dz2[j] = ok[u] ? a2[j] * (dz[j] - tot2[j] * invB - xh[j] * tot2[C + j] * invB) : 0.f;
#pragma unroll
            for (int i = 0; i < C; ++i) {
                const float z = z1[u][i];
                const float h1 = fmaxf(fmaf(a1[i], z, c1[i]), 0.f);
                float dh = 0.f;
#pragma unroll
                for (int j = 0; j < C; ++j) dh = fmaf(dz2[j], sW2[i * C + j], dh);
                const float dd = h1 > 0.f ? dh : 0.f;
                const float x1 = (z - mn1[i]) * rs1[i];
                d1[u][i] = dd;                           // zero for rows that do not exist (dz2 = 0)
                s0[i] += dd; s1[i] = fmaf(dd, x1, s1[i]);
                tH[tid * LD + i] = ok[u] ? h1 : 0.f;
                tD[tid * LD + i] = dz2[i];
            }
            __syncthreads();
            const int nrow = max(0, min(T, b_hi - (b_lo + u * T)));
            for (int row = 0; row < nrow; ++row) {
                const float dv = tD[row * LD + gj];
                acc = fmaf(tH[row * LD + gi], dv, acc);
                accb += dv;
            }
            __syncthreads();
        }
        atomicAdd(r.dW2 + tid, acc);
        if (gi == 0) atomicAdd(r.dbias2 + gj, accb);
        cta_colsum16(s0, wpart, sum1);
        cta_colsum16(s1, wpart, sum1 + C);
    }
    cluster.sync();
    if (tid < 2 * C) {
        float t = 0.f;
        for (int k = 0; k < CL; ++k) t += cluster.map_shared_rank(&sum1[0], k)[tid];
        tot1[tid] = t;
        if (rank == 0) {
            if (tid < C) r.dbt1[tid] += t; else r.dg1[tid - C] += t;
        }
    }
    __syncthreads();

    // ---- phase C: BN1 backward (+ bf16 planes copy for the tcgen05 head GEMMs) ---
    {
        float bsum[C];
#pragma unroll
        for (int i = 0; i < C; ++i) bsum[i] = 0.f;
#pragma unroll
        for (int u = 0; u < RPT; ++u) {
            const int b = b_lo + u * T + tid;
            float o[C];
#pragma unroll
            for (int i = 0; i < C; ++i) {
                const float x1 = (z1[u][i] - mn1[i]) * rs1[i];
                o[i] = a1[i] * (d1[u][i] - tot1[i] * invB - x1 * tot1[C + i] * invB);
                if (ok[u]) bsum[i] += o[i];
            }
            if (ok[u]) {
                store_row16(r.dZ1 + (size_t)b * C, o);
                if (r.dZ1p) {
                    __nv_bfloat16* pl = (__nv_bfloat16*)r.dZ1p;
                    Row8<__nv_bfloat16>::store(plane_row(pl, 0, r.Balloc, b), o);
                    Row8<__nv_bfloat16>::store(plane_row(pl, 1, r.Balloc, b), o + 8);
                }
            }
        }
        if (r.dbias1) {      // bias of the first router FC (zero up to rounding under train-mode BN)
            cta_colsum16(bsum, wpart, sb1);
            __syncthreads();
            if (tid < C) atomicAdd(r.dbias1 + tid, sb1[tid]);
        }
    }
    cluster.sync();          // keep this CTA's shared memory alive until every peer has read it
}

}  // namespace

extern "C" int mpnn_router_tail_bwd_batched(const mpnn_router_bwd_desc* descs, int n, int B, int Cw, void* stream) {
    MPNN_REQUIRE(Cw == C && n >= 1, "router_tail_bwd_batched: C=%d n=%d", Cw, n);
    static const int fast = getenv("MPNN_ROUTER_FAST") ? atoi(getenv("MPNN_ROUTER_FAST")) : 1;
    const int per_cta = ceil_div(B, CL);
    if (fast && per_cta <= T) router_tail_bwd_fast_kernel<1><<<n * CL, T, 0, (cudaStream_t)stream>>>(descs, B);
    else if (fast && per_cta <= 2 * T) router_tail_bwd_fast_kernel<2><<<n * CL, T, 0, (cudaStream_t)stream>>>(descs, B);
    else router_tail_bwd_cluster_kernel<<<n * CL, T, 0, (cudaStream_t)stream>>>(descs, B);
    return mpnn_check_launch("router_tail_bwd_batched");
}

template <bool CNT>
static int router_tail_fwd_launch(const mpnn_router_fwd_desc* descs, int n, int B, float d, float eps, int train,
                                  const int* count, cudaStream_t st) {
    static const int fast = getenv("MPNN_ROUTER_FAST") ? atoi(getenv("MPNN_ROUTER_FAST")) : 1;
    const int per_cta = ceil_div(B, CL);
    if (fast && per_cta <= T) router_tail_fwd_fast_kernel<1, CNT><<<n * CL, T, 0, st>>>(descs, B, d, eps, train, count);
    else if (fast && per_cta <= 2 * T) router_tail_fwd_fast_kernel<2, CNT><<<n * CL, T, 0, st>>>(descs, B, d, eps, train, count);
    else if (fast && per_cta <= 4 * T) router_tail_fwd_fast_kernel<4, CNT><<<n * CL, T, 0, st>>>(descs, B, d, eps, train, count);
    else router_tail_fwd_cluster_kernel<CNT><<<n * CL, T, 0, st>>>(descs, B, d, eps, train, count);
    return mpnn_check_launch("router_tail_fwd_batched");
}

extern "C" int mpnn_router_tail_fwd_batched(const mpnn_router_fwd_desc* descs, int n, int B, int Cw,
                                            float d, float eps, int train, void* stream) {
    MPNN_REQUIRE(Cw == C && n >= 1, "router_tail_fwd_batched: C=%d n=%d", Cw, n);
    return router_tail_fwd_launch<false>(descs, n, B, d, eps, train, nullptr, (cudaStream_t)stream);
}

extern "C" int mpnn_router_tail_fwd_batched_counted(const mpnn_router_fwd_desc* descs, int n, int B, int Cw,
                                                    float d, float eps, int train, const int* count, void* stream) {
    MPNN_REQUIRE(Cw == C && n >= 1, "router_tail_fwd_batched: C=%d n=%d", Cw, n);
    if (!count) return mpnn_router_tail_fwd_batched(descs, n, B, Cw, d, eps, train, stream);
    MPNN_REQUIRE(!train, "router_tail_fwd_batched_counted: eval mode only (train-mode moments need the whole batch)");
    return router_tail_fwd_launch<true>(descs, n, B, d, eps, train, count, (cudaStream_t)stream);
}
