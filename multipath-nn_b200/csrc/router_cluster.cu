// Forward and backward of every router tail of the net in ONE launch each, one 8-CTA thread-block
// cluster per router (reference: arch_and_hypers.py router() = FC(C)-BN-ReLU-FC(C)-BN-ReLU-FC(n_sinks),
// C = router_n_chan; TF autodiff through train-mode batch norm).  The width C is a template parameter:
// 16 (the reference's value), 32 and 64 are compiled.
//
// Train-mode BN makes the backward a chain of two batch-wide reductions
//   (BN2 sums) -> (BN1 sums) -> dZ1,
// which a single CTA can only walk serially over the whole batch.  Here the
// batch is split over the 8 CTAs of a cluster; each CTA reduces its slice, the
// slices are combined through distributed shared memory (fixed rank order, so
// the BN statistics are deterministic) and cluster.sync() separates the phases.
// The two small weight gradients (CxC, Cxns) are accumulated per CTA from
// shared-memory tiles and added to the flat gradient buffer with fp32 atomics.
#include <cooperative_groups.h>
#include <cstdlib>
#include "common.cuh"
#include "../../include/mpnn.h"

namespace cg = cooperative_groups;

namespace {

constexpr int NSMAX = 8;         // max sinks
constexpr int T = 256;           // threads per CTA = rows per tile
constexpr int CL = 8;            // CTAs per cluster

__device__ __forceinline__ void block_add(const float* v, int n, float* acc) {
    const int lane = threadIdx.x & 31;
    for (int i = 0; i < n; ++i) {
        float t = warp_sum(v[i]);
        if (lane == 0) atomicAdd(acc + i, t);
    }
}

// CTA sum of the per-thread columns v[C] added to acc[C]: at C = 16 by shared-memory atomics (the original kernels);
// wider routers add the warp totals in warp order, so their cluster-kernel statistics are reproducible bit for bit.
// wpart: [T / 32][C] scratch (unused at C = 16).  Ends with a barrier.
template <int C>
__device__ __forceinline__ void cta_add(const float* v, float* acc, float* wpart) {
    if constexpr (C == 16) {
        block_add(v, C, acc);
        __syncthreads();
    } else {
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll 1
        for (int i = 0; i < C; ++i) {            // (not unrolled: at C = 32 the unrolled loop spilled)
            const float t = warp_sum(v[i]);
            if (lane == 0) wpart[warp * C + i] = t;
        }
        __syncthreads();
        if (threadIdx.x < C) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < T / 32; ++w) s += wpart[w * C + threadIdx.x];
            acc[threadIdx.x] += s;
        }
        __syncthreads();
    }
}

// Shared memory of the backward kernels.  The row tiles tH / tD are T x (C + 1) floats each: 34 KB at C = 16,
// which stays static; wider routers (67 / 133 KB) take it as opt-in dynamic shared memory.
template <int C>
struct BwdSmem {
    float sW2[C * C], sW3[C * NSMAX];
    float a1[C], c1[C], a2[C], c2[C], mn1[C], rs1[C], mn2[C], rs2[C];
    float tH[T * (C + 1)], tD[T * (C + 1)], tR[T * (NSMAX + 1)];
    float part[T], wpart[(T / 32) * C];
    float sum2[2 * C], sum1[2 * C];      // this CTA's BN2 / BN1 partial sums (read by the cluster)
    float tot2[2 * C], tot1[2 * C];      // cluster totals
    float sb1[C];
};
template <int C>
__device__ __forceinline__ BwdSmem<C>& bwd_smem() {
    if constexpr (C == 16) {
        __shared__ BwdSmem<16> s;
        return s;
    } else {
        extern __shared__ __align__(16) unsigned char dyn_smem[];
        return *reinterpret_cast<BwdSmem<C>*>(dyn_smem);
    }
}
template <int C>
constexpr int bwd_dyn_smem() { return C == 16 ? 0 : (int)sizeof(BwdSmem<C>); }

// Entries of dW3 (C x NSMAX) and dW2 (C x C) over the T threads of the tile accumulation: dW3 at C = 16 has
// 128 entries, so two row phases of 128 threads; wider routers give every thread E3 / E2 entries.
template <int C> struct Acc {
    static constexpr int NP3 = C * NSMAX;
    static constexpr int RP3 = NP3 < T ? T / NP3 : 1;      // row phases of the dW3 accumulation
    static constexpr int E3 = NP3 > T ? NP3 / T : 1;       // dW3 entries per thread
    static constexpr int E2 = C * C / T;                   // dW2 entries per thread
};

// dW3 / dbias3 of this CTA's rows (thread: entries (gi + e * T / NSMAX, gk)); at C = 16 the two row phases are first
// combined through `part`
template <int C>
__device__ __forceinline__ void dw3_commit(const mpnn_router_bwd_desc& r, const float (&acc)[Acc<C>::E3], float accb,
                                           float* part, int gi, int gk, int ns) {
    const int tid = threadIdx.x;
    if constexpr (Acc<C>::RP3 == 2) {
        part[tid] = acc[0];
        __syncthreads();
        if (tid < 128 && gk < ns) atomicAdd(r.dW3 + gi * ns + gk, part[tid] + part[tid + 128]);
        __syncthreads();
        part[tid] = accb;
        __syncthreads();
        if (tid < 128 && gi == 0 && gk < ns) atomicAdd(r.dbias3 + gk, part[tid] + part[tid + 128]);
    } else {
        static_assert(Acc<C>::RP3 == 1, "dW3 row phases");
        if (gk < ns) {
#pragma unroll
            for (int e = 0; e < Acc<C>::E3; ++e) atomicAdd(r.dW3 + (gi + e * (T / NSMAX)) * ns + gk, acc[e]);
            if (gi == 0) atomicAdd(r.dbias3 + gk, accb);
        }
    }
}

// dW2 / dbias2 of this CTA's rows (thread: entries (gi + e * T / C, gj))
template <int C>
__device__ __forceinline__ void dw2_commit(const mpnn_router_bwd_desc& r, const float (&acc)[Acc<C>::E2], float accb,
                                           int gi, int gj) {
#pragma unroll
    for (int e = 0; e < Acc<C>::E2; ++e) atomicAdd(r.dW2 + (gi + e * (T / C)) * C + gj, acc[e]);
    if (gi == 0) atomicAdd(r.dbias2 + gj, accb);
}

template <int C>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_bwd_cluster_kernel(const mpnn_router_bwd_desc* __restrict__ descs, int B) {
    constexpr int LD = C + 1;
    using A = Acc<C>;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_bwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;

    BwdSmem<C>& sm = bwd_smem<C>();
    float *sW2 = sm.sW2, *sW3 = sm.sW3;
    float *a1 = sm.a1, *c1 = sm.c1, *a2 = sm.a2, *c2 = sm.c2, *mn1 = sm.mn1, *rs1 = sm.rs1, *mn2 = sm.mn2, *rs2 = sm.rs2;
    float *tH = sm.tH, *tD = sm.tD, *tR = sm.tR, *part = sm.part;
    float *sum2 = sm.sum2, *sum1 = sm.sum1, *tot2 = sm.tot2, *tot1 = sm.tot1, *sb1 = sm.sb1;

    for (int i = tid; i < C * C; i += T) sW2[i] = r.W2[i];
    for (int i = tid; i < C * ns; i += T) sW3[i] = r.W3[i];
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
        const int q = tid / A::NP3, t = tid % A::NP3, gi = t / NSMAX, gk = t % NSMAX;     // (row phase, i, k)
        float acc[A::E3], accb = 0.f;
#pragma unroll
        for (int e = 0; e < A::E3; ++e) acc[e] = 0.f;
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
            for (int row = q; row < nrow; row += A::RP3) {
                const float drv = tR[row * (NSMAX + 1) + gk];
#pragma unroll
                for (int e = 0; e < A::E3; ++e) acc[e] = fmaf(tH[row * LD + gi + e * (T / NSMAX)], drv, acc[e]);
                accb += drv;
            }
            __syncthreads();
        }
        dw3_commit<C>(r, acc, accb, part, gi, gk, ns);
        cta_add<C>(s01, sum2, sm.wpart);
        cta_add<C>(s01 + C, sum2 + C, sm.wpart);
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
        const int gi = tid / C, gj = tid % C;
        float acc[A::E2], accb = 0.f;
#pragma unroll
        for (int e = 0; e < A::E2; ++e) acc[e] = 0.f;
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
#pragma unroll
                for (int e = 0; e < A::E2; ++e) acc[e] = fmaf(tH[row * LD + gi + e * (T / C)], dv, acc[e]);
                accb += dv;
            }
            __syncthreads();
        }
        dw2_commit<C>(r, acc, accb, gi, gj);
        cta_add<C>(s01, sum1, sm.wpart);
        cta_add<C>(s01 + C, sum1 + C, sm.wpart);
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
#pragma unroll
                for (int p = 0; p < C / 8; ++p) Row8<__nv_bfloat16>::store(plane_row(pl, p, r.Balloc, b), o + 8 * p);
            }
        }
        if (r.dbias1) {      // bias of the first router FC (zero up to rounding under train-mode BN)
            cta_add<C>(bsum, sb1, sm.wpart);
            if (tid < C) atomicAdd(r.dbias1 + tid, sb1[tid]);
        }
    }
    cluster.sync();          // keep this CTA's shared memory alive until every peer has read it
}

// ---------------------------------------------------------------------------
// Forward of every router tail in one launch (same cluster layout): BN1 -> ReLU -> FC(C) -> BN2 ->
// ReLU -> FC(ns).  Train-mode statistics are two-pass (mean, then centred second moment) like
// tf.nn.moments; each pass is a per-CTA partial + a fixed-order fp64 sum over the cluster.
template <int C>
__device__ __forceinline__ void cluster_channel_sum(cg::cluster_group& cluster, const float* v, float* part, double* out,
                                                    float* wpart) {
    // v[C]: this thread's partial per channel; part[C]: CTA partial (smem, read by the cluster)
    const int tid = threadIdx.x;
    if (tid < C) part[tid] = 0.f;
    __syncthreads();
    cta_add<C>(v, part, wpart);
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
template <int C, bool CNT = false>
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
    __shared__ float wpart[(T / 32) * (C == 16 ? 1 : C)];
    for (int i = tid; i < C * C; i += T) sW2[i] = r.W2[i];
    for (int i = tid; i < C * ns; i += T) sW3[i] = r.W3[i];
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
            cluster_channel_sum<C>(cluster, v, part, tot, wpart);
            if (tid < C) mean[tid] = (float)(tot[tid] / B);
            __syncthreads();
#pragma unroll
            for (int i = 0; i < C; ++i) v[i] = 0.f;
            for (int b = b_lo + tid; b < b_hi; b += T) {
#pragma unroll
                for (int i = 0; i < C; ++i) { const float t = Zin[(size_t)b * C + i] - mean[i]; v[i] = fmaf(t, t, v[i]); }
            }
            cluster_channel_sum<C>(cluster, v, part, tot, wpart);
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
// column sum (colsum: C shuffles for C columns) + one shared-memory hop + one DSMEM hop, in a fixed
// order (deterministic statistics).  Each exchange has its own shared-memory slot, so one cluster.sync()
// per exchange suffices.
// ---------------------------------------------------------------------------
template <int C>
__device__ __forceinline__ void load_row(const float* p, float (&v)[C]) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int q = 0; q < C / 4; ++q) {
            const float4 t = *(reinterpret_cast<const float4*>(p) + q);
            v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) v[i] = p[i];
    }
}
template <int C>
__device__ __forceinline__ void store_row(float* p, const float (&v)[C]) {
    if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
#pragma unroll
        for (int q = 0; q < C / 4; ++q)
            *(reinterpret_cast<float4*>(p) + q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) p[i] = v[i];
    }
}
// transposing butterfly over the lanes: at C = 16, stages 8..1 leave lane L with column (L & 15) summed over the
// lanes that agree in bit 4, and the last shuffle adds the other half (out[0]); at C >= 32 every 32-column group g
// takes stages 16..1 and lane L ends with the total of column 32 g + L (out[g]).  C shuffles per call.
template <int C> __host__ __device__ constexpr int colsum_n() { return C == 16 ? 1 : C / 32; }
template <int C>
__device__ __forceinline__ void colsum(float (&v)[C], int lane, float (&out)[colsum_n<C>()]) {
    constexpr int S0 = C == 16 ? 8 : 16;
#pragma unroll
    for (int g = 0; g < colsum_n<C>(); ++g) {
        float* w = v + 32 * g;
#pragma unroll
        for (int s = S0; s >= 1; s >>= 1) {
            const bool up = (lane & s) != 0;
#pragma unroll
            for (int i = 0; i < s; ++i) {
                const float send = up ? w[i] : w[i + s];
                const float keep = up ? w[i + s] : w[i];
                w[i] = keep + __shfl_xor_sync(0xffffffffu, send, s);
            }
        }
        out[g] = C == 16 ? w[0] + __shfl_xor_sync(0xffffffffu, w[0], 16) : w[0];
    }
}
// CTA total of the per-thread columns v[C] -> out[C] (shared memory, written by threads 0..C-1; visible after the
// caller's next barrier).  wpart: [T / 32][C] scratch.  Warps are added in index order.  Destroys v.
template <int C>
__device__ __forceinline__ void cta_colsum(float (&v)[C], float* wpart, float* out) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float t[colsum_n<C>()];
    colsum<C>(v, lane, t);
    __syncthreads();                       // earlier readers of wpart are done
    if constexpr (C == 16) {
        if (lane < C) wpart[warp * C + lane] = t[0];
    } else {
#pragma unroll
        for (int g = 0; g < colsum_n<C>(); ++g) wpart[warp * C + 32 * g + lane] = t[g];
    }
    __syncthreads();
    if (threadIdx.x < C) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < T / 32; ++w) s += wpart[w * C + threadIdx.x];
        out[threadIdx.x] = s;
    }
}

template <int C, int RPT, bool CNT = false>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_fwd_fast_kernel(const mpnn_router_fwd_desc* __restrict__ descs, int B, float d, float eps, int train,
                            const int* __restrict__ count) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_fwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;
    __shared__ float sW2[C * C], sW3[C * NSMAX], sb2[C], sb3[NSMAX];
    __shared__ float wpart[(T / 32) * C], part[4][C], a[C], c[C], mean[C];
    for (int i = tid; i < C * C; i += T) sW2[i] = r.W2[i];
    for (int i = tid; i < C * ns; i += T) sW3[i] = r.W3[i];
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
        if (ok[u]) load_row<C>(r.Z1 + (size_t)b * C, z[u]);
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
            cta_colsum<C>(v, wpart, part[2 * layer]);
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
            cta_colsum<C>(v, wpart, part[2 * layer + 1]);
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
                if (ok[u]) store_row<C>(r.Z2 + (size_t)b * C, o);
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

template <int C, int RPT>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(T)
router_tail_bwd_fast_kernel(const mpnn_router_bwd_desc* __restrict__ descs, int B) {
    constexpr int LD = C + 1;
    using A = Acc<C>;
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const mpnn_router_bwd_desc r = descs[blockIdx.x / CL];
    const int ns = r.ns, tid = threadIdx.x;

    BwdSmem<C>& sm = bwd_smem<C>();
    float *sW2 = sm.sW2, *sW3 = sm.sW3;
    float *a1 = sm.a1, *c1 = sm.c1, *a2 = sm.a2, *c2 = sm.c2, *mn1 = sm.mn1, *rs1 = sm.rs1, *mn2 = sm.mn2, *rs2 = sm.rs2;
    float *tH = sm.tH, *tD = sm.tD, *tR = sm.tR, *part = sm.part, *wpart = sm.wpart;
    float *sum2 = sm.sum2, *sum1 = sm.sum1, *tot2 = sm.tot2, *tot1 = sm.tot1, *sb1 = sm.sb1;

    for (int i = tid; i < C * C; i += T) sW2[i] = r.W2[i];
    for (int i = tid; i < C * NSMAX; i += T) sW3[i] = i < C * ns ? r.W3[i] : 0.f;
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
            load_row<C>(r.Z2 + (size_t)b * C, z2[u]);
            load_row<C>(r.Z1 + (size_t)b * C, z1[u]);
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
        const int q = tid / A::NP3, t = tid % A::NP3, gi = t / NSMAX, gk = t % NSMAX;     // (row phase, i, k)
        float acc[A::E3], accb = 0.f;
#pragma unroll
        for (int e = 0; e < A::E3; ++e) acc[e] = 0.f;
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
            for (int row = q; row < nrow; row += A::RP3) {
                const float drv = tR[row * (NSMAX + 1) + gk];
#pragma unroll
                for (int e = 0; e < A::E3; ++e) acc[e] = fmaf(tH[row * LD + gi + e * (T / NSMAX)], drv, acc[e]);
                accb += drv;
            }
            __syncthreads();
        }
        dw3_commit<C>(r, acc, accb, part, gi, gk, ns);
        cta_colsum<C>(s0, wpart, sum2);
        cta_colsum<C>(s1, wpart, sum2 + C);
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
        const int gi = tid / C, gj = tid % C;
        float acc[A::E2], accb = 0.f;
#pragma unroll
        for (int e = 0; e < A::E2; ++e) acc[e] = 0.f;
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
#pragma unroll
                for (int e = 0; e < A::E2; ++e) acc[e] = fmaf(tH[row * LD + gi + e * (T / C)], dv, acc[e]);
                accb += dv;
            }
            __syncthreads();
        }
        dw2_commit<C>(r, acc, accb, gi, gj);
        cta_colsum<C>(s0, wpart, sum1);
        cta_colsum<C>(s1, wpart, sum1 + C);
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
                store_row<C>(r.dZ1 + (size_t)b * C, o);
                if (r.dZ1p) {
                    __nv_bfloat16* pl = (__nv_bfloat16*)r.dZ1p;
#pragma unroll
                    for (int p = 0; p < C / 8; ++p) Row8<__nv_bfloat16>::store(plane_row(pl, p, r.Balloc, b), o + 8 * p);
                }
            }
        }
        if (r.dbias1) {      // bias of the first router FC (zero up to rounding under train-mode BN)
            cta_colsum<C>(bsum, wpart, sb1);
            __syncthreads();
            if (tid < C) atomicAdd(r.dbias1 + tid, sb1[tid]);
        }
    }
    cluster.sync();          // keep this CTA's shared memory alive until every peer has read it
}

}  // namespace

// Register-resident kernels per width: the largest RPT that compiles without spilling (ptxas -v), up to which the
// entry points use them (B <= 8 * 256 * RPT); 0 = the cluster kernel at every batch.  C = 64 keeps no backward rows
// in registers: z1, z2 and d1 alone would be 192 of the 255 registers a thread can have.
template <int C> constexpr int fwd_rpt_max() { return C == 16 ? 4 : (C == 32 ? 2 : 1); }
template <int C> constexpr int bwd_rpt_max() { return C == 16 ? 2 : (C == 32 ? 1 : 0); }

static bool router_width_ok(int Cw) { return Cw == 16 || Cw == 32 || Cw == 64; }
#define ROUTER_WIDTHS "16, 32 or 64"

// the backward kernels of the wide routers take their tiles as dynamic shared memory beyond the 48 KB default
template <typename K>
static int allow_smem(K kern, int bytes, bool* done) {
    if (bytes == 0) return 0;                // C = 16: static shared memory, no host call
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && done[dev]) return 0;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) { mpnn_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return MPNN_ERR_CUDA; }
    if (dev >= 0 && dev < 64) done[dev] = true;
    return 0;
}

template <int C, int RPT>
static int router_tail_bwd_run(const mpnn_router_bwd_desc* descs, int n, int B, int fast, cudaStream_t st) {
    constexpr int smem = bwd_dyn_smem<C>();
    if constexpr (RPT <= bwd_rpt_max<C>()) {
        if (fast && ceil_div(B, CL) <= RPT * T) {
            static bool done[64] = {};
            if (int rc = allow_smem(router_tail_bwd_fast_kernel<C, RPT>, smem, done)) return rc;
            router_tail_bwd_fast_kernel<C, RPT><<<n * CL, T, smem, st>>>(descs, B);
            return mpnn_check_launch("router_tail_bwd_batched");
        }
        return router_tail_bwd_run<C, RPT * 2>(descs, n, B, fast, st);
    } else {
        static bool done[64] = {};
        if (int rc = allow_smem(router_tail_bwd_cluster_kernel<C>, smem, done)) return rc;
        router_tail_bwd_cluster_kernel<C><<<n * CL, T, smem, st>>>(descs, B);
        return mpnn_check_launch("router_tail_bwd_batched");
    }
}

extern "C" int mpnn_router_tail_bwd_batched(const mpnn_router_bwd_desc* descs, int n, int B, int Cw, void* stream) {
    MPNN_REQUIRE(router_width_ok(Cw) && n >= 1, "router_tail_bwd_batched: C=%d (router widths " ROUTER_WIDTHS ") n=%d",
                 Cw, n);
    static const int fast = getenv("MPNN_ROUTER_FAST") ? atoi(getenv("MPNN_ROUTER_FAST")) : 1;
    const cudaStream_t st = (cudaStream_t)stream;
    if (Cw == 16) return router_tail_bwd_run<16, 1>(descs, n, B, fast, st);
    if (Cw == 32) return router_tail_bwd_run<32, 1>(descs, n, B, fast, st);
    return router_tail_bwd_run<64, 1>(descs, n, B, fast, st);
}

template <int C, int RPT, bool CNT>
static int router_tail_fwd_run(const mpnn_router_fwd_desc* descs, int n, int B, float d, float eps, int train,
                               const int* count, int fast, cudaStream_t st) {
    if constexpr (RPT <= fwd_rpt_max<C>()) {
        if (fast && ceil_div(B, CL) <= RPT * T) {
            router_tail_fwd_fast_kernel<C, RPT, CNT><<<n * CL, T, 0, st>>>(descs, B, d, eps, train, count);
            return mpnn_check_launch("router_tail_fwd_batched");
        }
        return router_tail_fwd_run<C, RPT * 2, CNT>(descs, n, B, d, eps, train, count, fast, st);
    } else {
        router_tail_fwd_cluster_kernel<C, CNT><<<n * CL, T, 0, st>>>(descs, B, d, eps, train, count);
        return mpnn_check_launch("router_tail_fwd_batched");
    }
}

template <bool CNT>
static int router_tail_fwd_launch(const mpnn_router_fwd_desc* descs, int n, int B, int Cw, float d, float eps, int train,
                                  const int* count, cudaStream_t st) {
    static const int fast = getenv("MPNN_ROUTER_FAST") ? atoi(getenv("MPNN_ROUTER_FAST")) : 1;
    if (Cw == 16) return router_tail_fwd_run<16, 1, CNT>(descs, n, B, d, eps, train, count, fast, st);
    if (Cw == 32) return router_tail_fwd_run<32, 1, CNT>(descs, n, B, d, eps, train, count, fast, st);
    return router_tail_fwd_run<64, 1, CNT>(descs, n, B, d, eps, train, count, fast, st);
}

extern "C" int mpnn_router_tail_fwd_batched(const mpnn_router_fwd_desc* descs, int n, int B, int Cw,
                                            float d, float eps, int train, void* stream) {
    MPNN_REQUIRE(router_width_ok(Cw) && n >= 1, "router_tail_fwd_batched: C=%d (router widths " ROUTER_WIDTHS ") n=%d",
                 Cw, n);
    return router_tail_fwd_launch<false>(descs, n, B, Cw, d, eps, train, nullptr, (cudaStream_t)stream);
}

extern "C" int mpnn_router_tail_fwd_batched_counted(const mpnn_router_fwd_desc* descs, int n, int B, int Cw,
                                                    float d, float eps, int train, const int* count, void* stream) {
    MPNN_REQUIRE(router_width_ok(Cw) && n >= 1, "router_tail_fwd_batched: C=%d (router widths " ROUTER_WIDTHS ") n=%d",
                 Cw, n);
    if (!count) return mpnn_router_tail_fwd_batched(descs, n, B, Cw, d, eps, train, stream);
    MPNN_REQUIRE(!train, "router_tail_fwd_batched_counted: eval mode only (train-mode moments need the whole batch)");
    return router_tail_fwd_launch<true>(descs, n, B, Cw, d, eps, train, count, (cudaStream_t)stream);
}
