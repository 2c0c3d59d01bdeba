// tcgen05 / TMEM implementation of the stencil GEMM (conv forward and data
// gradient) for sm_100a, bf16 operands, fp32 accumulation in tensor memory.
//
// Why this shape of kernel: in the padded-planes layout (common.cuh) a 3x3 SAME
// convolution over a tile of 128 consecutive rows needs the rows
// [p0-halo, p0+128+halo) of every 8-channel plane, each a CONTIGUOUS run of
// 16-byte rows in HBM.  One cp.async.bulk per plane lands it in shared memory
// exactly in the UMMA "interleaved / no-swizzle" K-major core-matrix layout
// (8 rows x 16 B contiguous; SBO = 128 B between 8-row groups; LBO = plane
// stride between the two 8-channel halves of a K=16 step).  The nine taps are
// then nine descriptor START ADDRESSES into the same staged tile (row shift
// dh*(W+1)+dw), so the input is read from L2/HBM once, not nine times.
//
// Roles (192 threads): warp 0 bulk-copy producer, warp 1 TMEM owner + MMA
// issuer (one elected lane), warps 2-5 epilogue (tcgen05.ld -> bias -> BN
// partial moments -> coalesced 16 B row stores).  Persistent over tiles, A
// stages ring-buffered with mbarriers, two TMEM accumulators so the epilogue
// of tile i overlaps the MMAs of tile i+1.  Weights for the CTA's N-slice stay
// resident in shared memory for the kernel's lifetime.
#include <cstdlib>
#include "common.cuh"
#include "umma.cuh"
#include "../../include/mpnn.h"
#include "bn_fuse.cuh"

extern "C" int mpnn_has_umma(void) { return 1; }

namespace {

// fused BN-backward reduction on out0 (data-gradient epilogue): with dy' = dAct * [ss0*lin + ss1 > 0]
// the CTA accumulates sum dy' and sum dy'*(lin - mean) per channel of out0; the last CTA converts the totals
// into the xhat form (bn_fuse.cuh).  Replaces the bn_bwd_reduce pass over (lin, dAct).
struct BwdRed {
    const __nv_bfloat16* lin; const float* ss; const float* mr;
    mpnn_bn_bwd_fuse f;
};

struct GemmArgs {
    const __nv_bfloat16* A0; const __nv_bfloat16* A1; const __nv_bfloat16* Wp;
    const float* bias;
    void* out0; void* out1;
    float* stats;
    Geom g;
    int K0, K1, N, N0, NB, ntaps, acc0, acc1, n_tiles, nstage, rowsA, halo;
    int out_mode;      // 0: bf16 planes, 1: fp32 planes, 2: fp32 row-major [row][ld]
    int ld0, ld1;      // leading dimensions of out0 / out1 in row-major mode
    int KC, n_kc;      // planes per pipeline stage and stages per tile (K is streamed for wide FC inputs)
    int stats_mode;    // 0 none, 1 moments of out (forward BN), 2 BN-backward sums on out0 (red)
    mpnn_bn_fuse bn;   // bn.acc != NULL: fused BN statistics (last CTA finalises)
    BwdRed red;
    int dbg;           // tuning aid (MPNN_TUNE_DBG): 1 skip MMAs, 2 skip stores, 4 skip loads; timing probes of the
                       // MMA phase (results wrong by construction): 8 all taps read the unshifted tile, 16 the taps
                       // alternate between the two accumulators, 32 three MMAs of 3x the width instead of nine
    const int* count;  // CNT instantiations: live batch in device memory (g.B is the capacity the grid was sized for)
};

constexpr int kThreads = 192;

__device__ __forceinline__ uint4 pack_bf16x8(const float* v) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    return u;
}
__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float* v) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
}

// NBT = compile-time N-slice width for the hot conv shapes (16, 32): the epilogue is
// fully unrolled and the BN sums stay in per-thread registers across all tiles of
// the CTA (one warp reduction at kernel end instead of one per tile).  NBT = 0 is the
// generic width (any multiple of 16 up to 256) with a per-tile warp reduction.
// KS  = compile-time number of K steps (K = 16*KS) of a 9-tap conv whose K fits one pipeline stage:
// the MMA issue loop is then 9*KS straight-line instructions with immediate descriptor offsets.  In
// round 1 that loop cost ~45 SASS instructions per MMA (runtime trip counts, per-MMA predicate and
// register-file conversions) and, with the issuing warps of all resident CTAs sharing one scheduler,
// bounded the thin layers at ~540 cycles per tile per SM.  KS = 0 is the generic loop.
// EPI = 0: generic epilogue (any output mode, accumulation, either kind of sums); 1: bf16 planes out, no
// accumulation into the outputs, forward BN moments or no sums (stores without the read-modify-write and
// output-mode dispatch); 2: the same with the fused BN-backward sums (separate instantiation: the two kinds
// of sums have different register footprints and the accumulators must not spill).
// CNT: the live batch is min(*count, g.B); only its rows are computed and stored (counted entry point, inference).
template <int NBT, int KS, int EPI, bool CNT = false>
// (32-wide slices at two CTAs per SM: at three the 64 register accumulators of the BN sums spilled -- 96 registers,
//  16-48 bytes of stack -- and H16 32->32 ran at 53 us instead of 49)
__global__ void __launch_bounds__(kThreads, NBT == 16 ? (EPI == 2 ? 3 : 4) : (NBT == 32 ? 2 : 1))
stencil_gemm_umma_kernel(const GemmArgs a) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KG = KS ? 2 * KS : (a.K0 + a.K1) >> 3, KG0 = a.K0 >> 3;
    const int NB = NBT ? NBT : a.NB, n0 = blockIdx.y * NB;
    const uint32_t w_bytes = (uint32_t)a.ntaps * KG * NB * 16;
    const uint32_t PS = (uint32_t)a.rowsA * 16;          // plane stride inside a stage
    const uint32_t stage_bytes = PS * a.KC;
    uint8_t* sW = smem;
    uint8_t* sA = smem + ((w_bytes + 127) & ~127u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(sA + (size_t)a.nstage * stage_bytes);
    // bars: full[nstage], empty[nstage], tfull[2], tempty[2], wbar
    const uint32_t full0 = smem_u32(bars), empty0 = full0 + 8 * a.nstage;
    const uint32_t tfull0 = empty0 + 8 * a.nstage, tempty0 = tfull0 + 16, wbar = tempty0 + 16;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * a.nstage + 6);   // 16-byte aligned
    float* sstat = reinterpret_cast<float*>(tmem_slot + 4);      // [4 warps][2][NB]
    float* sbias = sstat + 4 * 2 * NB;                           // [NB]
    float* sred = sbias + NB;                                    // [3][N0]: scale / shift / mean of the BN behind out0 (mode 2)
    const uint32_t ncols = tmem_cols_pow2(((a.dbg & 32) && NBT ? 6 : 2) * NB);
    constexpr bool FAST = EPI != 0;
    const int stats_mode = EPI == 2 ? 2 : (EPI == 1 ? (a.stats_mode == 1 ? 1 : 0) : a.stats_mode);
    int n_tiles = a.n_tiles, rows = a.g.rows;
    if (CNT) {
        // the count is written by an earlier kernel: wait for it before anything else, and let a CTA without tiles
        // leave before it sets up barriers or allocates tensor memory (a zero count costs one early return)
        pdl_wait();
        rows = min(max(*a.count, 0), a.g.B) * a.g.S;
        n_tiles = (rows + 127) >> 7;
        if ((int)blockIdx.x >= n_tiles) return;
    }

    if (threadIdx.x == 0) {
        for (int s = 0; s < a.nstage; ++s) { mbar_init(full0 + 8 * s, 1); mbar_init(empty0 + 8 * s, 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(tfull0 + 8 * s, 1); mbar_init(tempty0 + 8 * s, 4); }
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (threadIdx.x >= 64) {
        if (stats_mode)
            for (int i = threadIdx.x - 64; i < 4 * 2 * NB; i += 128) sstat[i] = 0.f;
        for (int i = threadIdx.x - 64; i < NB; i += 128) sbias[i] = a.bias ? a.bias[n0 + i] : 0.f;
    }
    pdl_launch_dependents();
    pdl_wait();                  // everything above is independent of the previous kernel in the stream
    if (stats_mode == 2 && threadIdx.x >= 64)
        for (int i = threadIdx.x - 64; i < 3 * a.N0; i += 128) sred[i] = i < 2 * a.N0 ? a.red.ss[i] : a.red.mr[i - 2 * a.N0];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------ producer (whole warp, one elected lane issues)
        {
            const bool leader = elect_one();
            if (leader) mbar_expect_tx(wbar, w_bytes);
            if (NB == a.N) {
                // unsplit N: the packed weights [tap][K/8][N][8] are one contiguous block
                if (leader) bulk_g2s(smem_u32(sW), a.Wp, w_bytes, wbar);
            } else {
                for (int t = 0; t < a.ntaps * KG; ++t)
                    if (leader) bulk_g2s(smem_u32(sW) + (uint32_t)t * NB * 16,
                                         a.Wp + ((size_t)t * a.N + n0) * 8, (uint32_t)NB * 16, wbar);
            }
            // the single-thread issue loops are the per-CTA critical path: no divisions, no
            // 64-bit address rebuilds inside them (ring slot / phase are running counters)
            int s = 0; uint32_t ph = 0;
            const __nv_bfloat16* src0 = a.A0 + (size_t)(a.g.G - a.halo) * 8;
            const __nv_bfloat16* src1 = a.A1 ? a.A1 + (size_t)(a.g.G - a.halo) * 8 : nullptr;
            const size_t plane = (size_t)a.g.P * 8;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const size_t toff = (size_t)tile * (128 * 8);
                for (int ci = 0; ci < a.n_kc; ++ci) {
                    const int kg0 = ci * a.KC, kgn = min(a.KC, KG - kg0);
                    mbar_wait(empty0 + 8 * s, ph ^ 1u);
                    if (a.dbg & 4) { if (leader) mbar_arrive(full0 + 8 * s); }
                    else {
                        if (leader) mbar_expect_tx(full0 + 8 * s, PS * kgn);
                        const uint32_t dst = smem_u32(sA) + (uint32_t)s * stage_bytes;
                        for (int j = 0; j < kgn; ++j) {
                            const int kg = kg0 + j;
                            const __nv_bfloat16* src = kg < KG0 ? src0 + kg * plane + toff
                                                                : src1 + (kg - KG0) * plane + toff;
                            if (leader) bulk_g2s(dst + (uint32_t)j * PS, src, PS, full0 + 8 * s);
                        }
                    }
                    if (++s == a.nstage) { s = 0; ph ^= 1u; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------ MMA issuer (whole warp, one elected lane issues)
        {
            const bool leader = elect_one();
            const uint32_t idesc = make_idesc(NB, 0, 0);
            // descriptors: hi word (SBO = 128 B, version) is constant; the lo word is
            // (address >> 4) | (LBO >> 4) << 16, so a tap shift of `off` rows (16 B each)
            // or a K step is one 32-bit add
            const uint32_t d_hi = (128u >> 4) | (1u << 14);
            const uint32_t a_lo0 = (((smem_u32(sA) + (uint32_t)a.halo * 16) & 0x3FFFFu) >> 4) | ((PS >> 4) << 16);
            const uint32_t b_lo0 = ((smem_u32(sW) & 0x3FFFFu) >> 4) | ((uint32_t)NB << 16);
            const uint32_t a_stage = stage_bytes >> 4, a_kstep = 2 * (PS >> 4), b_kstep = 2 * (uint32_t)NB;
            const uint32_t b_tap = (uint32_t)KG * NB;
            const int Wp = a.g.Wp;
            const bool skip = (a.dbg & 1) != 0;
            mbar_wait(wbar, 0);
            int s = 0, tl = 0; uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tl) {
                const int acc = tl & 1;
                const uint32_t aph = (uint32_t)(tl >> 1) & 1u;
                mbar_wait(tempty0 + 8 * acc, aph ^ 1u);
                const uint32_t dcol = tmem_base + (uint32_t)acc * NB;
                if (KS > 0) {
                    // one stage holds all of K: 9*KS MMAs, descriptor offsets are immediates
                    mbar_wait(full0 + 8 * s, ph);
                    tc_fence_after();
                    const uint32_t a_lo = a_lo0 + (uint32_t)s * a_stage;
                    if (NBT != 0 && !skip && (a.dbg & 56)) {
                        // timing probes (see GemmArgs::dbg); compiled into the 16- / 32-wide instantiations only -- in
                        // the generic-width ones the second unrolled loop cost 40-80 registers and a resident CTA
                        const uint32_t idesc3 = make_idesc(3 * NB, 0, 0);
#pragma unroll
                        for (int tap = 0; tap < 9; ++tap) {
                            if ((a.dbg & 32) && tap % 3) continue;
                            const uint32_t at = a_lo + ((a.dbg & 8) ? 0u : (uint32_t)((tap / 3 - 1) * Wp + (tap % 3 - 1)));
                            const uint32_t bt = b_lo0 + (uint32_t)tap * b_tap;
                            const uint32_t dc = (a.dbg & 32) ? tmem_base + (uint32_t)acc * 3 * NB
                                              : ((a.dbg & 16) && (tap & 1) ? tmem_base + (uint32_t)(acc ^ 1) * NB : dcol);
#pragma unroll
                            for (int ks = 0; ks < (KS ? KS : 1); ++ks)
                                if (leader) tc_mma2(dc, at + (uint32_t)ks * a_kstep, d_hi, bt + (uint32_t)ks * b_kstep, d_hi,
                                                    (a.dbg & 32) ? idesc3 : idesc, (tap | ks) ? 1u : 0u);
                        }
                    } else if (!skip) {
#pragma unroll
                        for (int tap = 0; tap < 9; ++tap) {
                            const uint32_t at = a_lo + (uint32_t)((tap / 3 - 1) * Wp + (tap % 3 - 1));
                            const uint32_t bt = b_lo0 + (uint32_t)tap * b_tap;
#pragma unroll
                            for (int ks = 0; ks < (KS ? KS : 1); ++ks)
                                if (leader) tc_mma2(dcol, at + (uint32_t)ks * a_kstep, d_hi, bt + (uint32_t)ks * b_kstep, d_hi,
                                                    idesc, (tap | ks) ? 1u : 0u);
                        }
                    }
                    if (leader) tc_commit(empty0 + 8 * s);      // smem stage reusable once the MMAs retire
                    if (++s == a.nstage) { s = 0; ph ^= 1u; }
                } else {
                    for (int ci = 0; ci < a.n_kc; ++ci) {
                        const int kg0 = ci * a.KC, ksteps = min(a.KC, KG - kg0) >> 1;
                        mbar_wait(full0 + 8 * s, ph);
                        tc_fence_after();
                        const uint32_t a_lo = a_lo0 + (uint32_t)s * a_stage;
                        const uint32_t b_lo = b_lo0 + (uint32_t)kg0 * NB;
                        if (!skip) {
                            if (a.ntaps == 9) {
#pragma unroll
                                for (int tap = 0; tap < 9; ++tap) {
                                    uint32_t at = a_lo + (uint32_t)((tap / 3 - 1) * Wp + (tap % 3 - 1));
                                    uint32_t bt = b_lo + (uint32_t)tap * b_tap;
#pragma unroll 1
                                    for (int kk = 0; kk < ksteps; ++kk, at += a_kstep, bt += b_kstep) {
                                        const uint32_t accf = tap ? 1u : (uint32_t)((kk | ci) != 0);
                                        if (leader) tc_mma2(dcol, at, d_hi, bt, d_hi, idesc, accf);
                                    }
                                }
                            } else {
                                uint32_t at = a_lo, bt = b_lo;
#pragma unroll 1
                                for (int kk = 0; kk < ksteps; ++kk, at += a_kstep, bt += b_kstep) {
                                    const uint32_t accf = (uint32_t)((kk | ci) != 0);
                                    if (leader) tc_mma2(dcol, at, d_hi, bt, d_hi, idesc, accf);
                                }
                            }
                        }
                        if (leader) tc_commit(empty0 + 8 * s);
                        if (++s == a.nstage) { s = 0; ph ^= 1u; }
                    }
                }
                if (leader) tc_commit(tfull0 + 8 * acc);        // accumulator ready for the epilogue
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------ epilogue (warps 2..5)
        const int quad = warp & 3;                       // TMEM lane quadrant this warp may read
        const int m = quad * 32 + lane;
        float* wstat = sstat + (size_t)(warp - 2) * 2 * NB;
        constexpr int NR = (NBT && EPI) ? NBT : 1;
        float r1[NR], r2[NR];                            // running BN sums of this thread's rows (fast epilogues)
#pragma unroll
        for (int i = 0; i < NR; ++i) { r1[i] = 0.f; r2[i] = 0.f; }
        const __nv_bfloat16* lin = a.red.lin;
        // mode-2 contribution of 8 columns [cc, cc+8) of out0: dv = the values as stored (bf16-rounded)
        auto red8 = [&](int cc, const float* dv, const float* lv, float* a1, float* a2) {
            const float4* sc4 = reinterpret_cast<const float4*>(sred + cc);
            const float4* sh4 = reinterpret_cast<const float4*>(sred + a.N0 + cc);
            const float4* mu4 = reinterpret_cast<const float4*>(sred + 2 * a.N0 + cc);
            float sc[8], sh[8], mu[8];
            *reinterpret_cast<float4*>(sc) = sc4[0]; *reinterpret_cast<float4*>(sc + 4) = sc4[1];
            *reinterpret_cast<float4*>(sh) = sh4[0]; *reinterpret_cast<float4*>(sh + 4) = sh4[1];
            *reinterpret_cast<float4*>(mu) = mu4[0]; *reinterpret_cast<float4*>(mu + 4) = mu4[1];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float dy = fmaf(sc[j], lv[j], sh[j]) > 0.f ? dv[j] : 0.f;
                a1[j] += dy;
                a2[j] = fmaf(dy, lv[j] - mu[j], a2[j]);      // centred: no cancellation against mean * sum dy'
            }
        };
        // generic epilogue of one 16-column chunk: bias, store (bf16 / fp32 planes or fp32 row-major), sums
        auto finish_chunk = [&](int c, float (&v)[16], int q, int p, bool inrange, bool valid) {
            const float4* b4 = reinterpret_cast<const float4*>(sbias + c);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 b = b4[i];
                v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
            }
            const int col = n0 + c;
            float s1[16], s2[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) { s1[i] = 0.f; s2[i] = 0.f; }
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int cc = col + hh * 8;
                void* base; int accf, kgp;
                if (cc < a.N0) { base = a.out0; accf = a.acc0; kgp = cc >> 3; }
                else { base = a.out1; accf = a.acc1; kgp = (cc - a.N0) >> 3; }
                float o[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o[i] = v[hh * 8 + i];
                if (a.out_mode == 0) {
                    __nv_bfloat16* d = plane_row((__nv_bfloat16*)base, kgp, a.g.P, p);
                    if (accf && inrange) { float t[8]; Row8<__nv_bfloat16>::load(d, t);
#pragma unroll
                        for (int i = 0; i < 8; ++i) { o[i] += t[i]; v[hh * 8 + i] = o[i]; } }   // sums see the accumulated value
                    const uint4 u = pack_bf16x8(o);
                    if (inrange) *reinterpret_cast<uint4*>(d) = u;
                    if (stats_mode == 2 && valid && cc < a.N0) {
                        float dv[8], lv[8];
                        unpack_bf16x8(u, dv);
                        Row8<__nv_bfloat16>::load(plane_row(lin, kgp, a.g.P, p), lv);
                        red8(cc, dv, lv, s1 + hh * 8, s2 + hh * 8);
                    }
                } else if (inrange) {
                    if (a.out_mode == 1) {
                        float* d = plane_row((float*)base, kgp, a.g.P, p);
                        if (accf) { float t[8]; Row8<float>::load(d, t);
#pragma unroll
                            for (int i = 0; i < 8; ++i) { o[i] += t[i]; v[hh * 8 + i] = o[i]; } }
                        Row8<float>::store(d, o);
                    } else {
                        // fp32 row-major [row][ld]: logits of the fully-connected heads
                        const int ld = cc < a.N0 ? a.ld0 : a.ld1;
                        Row8<float>::store((float*)base + (size_t)q * ld + kgp * 8, o);
                    }
                }
            }
            if (stats_mode == 1 && valid) {
#pragma unroll
                for (int i = 0; i < 16; ++i) { s1[i] = v[i]; s2[i] = v[i] * v[i]; }
            }
            if (stats_mode) {                           // generic epilogue: one warp reduction per chunk
                float t1 = warp_colsum16(s1, lane);
                float t2 = warp_colsum16(s2, lane);
                if (lane < 16) { wstat[c + lane] += t1; wstat[NB + c + lane] += t2; }
            }
        };
        // fast epilogues: the row's position inside its image block (r = q mod S) advances by a constant
        // per tile, so validity costs one multiply-high per tile instead of two divisions with fix-ups;
        // mode 2 requests the rows of `lin` one tile ahead (their latency would sit on the per-tile
        // critical path of the epilogue otherwise)
        const int S_ = a.g.S, Wp_ = a.g.Wp;
        const int dq = 128 * (int)gridDim.x;
        int dr = 0, rq = 0, qrun = (int)blockIdx.x * 128 + m;
        auto valid_of = [&](int q_, int r_) {
            const int hr = (int)__umulhi((uint32_t)r_, a.g.mWp);     // exact: r < S << 2^32 / Wp
            return q_ < rows && r_ >= Wp_ && r_ != hr * Wp_;
        };
        uint4 lnext[NR / 8 ? NR / 8 : 1];
        auto fetch_lin = [&](int q_, bool v_) {
#pragma unroll
            for (int j = 0; j < NR / 8; ++j) {
                lnext[j] = make_uint4(0u, 0u, 0u, 0u);
                if (v_ && n0 + j * 8 < a.N0)
                    lnext[j] = __ldg(reinterpret_cast<const uint4*>(plane_row(lin, (n0 >> 3) + j, a.g.P, a.g.G + q_)));
            }
        };
        bool vrun = false;
        if (FAST && NBT) {
            dr = dq - (int)__umulhi((uint32_t)dq, a.g.mS) * S_;
            if (dr < 0) dr += S_; else if (dr >= S_) dr -= S_;
            rq = qrun - (int)__umulhi((uint32_t)qrun, a.g.mS) * S_;
            if (rq < 0) rq += S_; else if (rq >= S_) rq -= S_;
            vrun = stats_mode ? valid_of(qrun, rq) : false;
            if (EPI == 2) fetch_lin(qrun, vrun);
        }
        int it = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const int acc = it & 1;
            const uint32_t aph = (uint32_t)(it >> 1) & 1u;
            const int q = tile * 128 + m;
            const int p = a.g.G + q;
            const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)acc * NB;
            bool valid, inrange = q < rows && !(a.dbg & 2);
            if (FAST && NBT) {
                valid = vrun;
                uint4 lrow[NR / 8 ? NR / 8 : 1];
                if (EPI == 2) {
#pragma unroll
                    for (int j = 0; j < NR / 8; ++j) lrow[j] = lnext[j];
                }
                // next tile of this CTA
                qrun += dq; rq += dr;
                if (rq >= S_) rq -= S_;
                if (stats_mode) vrun = valid_of(qrun, rq);
                if (EPI == 2) fetch_lin(qrun, vrun);
                mbar_wait(tfull0 + 8 * acc, aph);
                tc_fence_after();
#pragma unroll
                for (int ci = 0; ci < NR / 16; ++ci) {
                    float v[16];
                    tc_ld16(taddr + ci * 16, v);
                    if (ci == NR / 16 - 1) {             // accumulator drained: hand it back before the math
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(tempty0 + 8 * acc);
                    }
                    if (a.bias) {
                        const float4* b4 = reinterpret_cast<const float4*>(sbias + ci * 16);
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float4 b = b4[i];
                            v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
                        }
                    }
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int cl = ci * 16 + hh * 8, cc = n0 + cl;
                        const bool to0 = cc < a.N0;
                        __nv_bfloat16* d = to0 ? plane_row((__nv_bfloat16*)a.out0, cc >> 3, a.g.P, p)
                                               : plane_row((__nv_bfloat16*)a.out1, (cc - a.N0) >> 3, a.g.P, p);
                        const uint4 u = pack_bf16x8(v + hh * 8);
                        if (inrange) *reinterpret_cast<uint4*>(d) = u;
                        if (EPI == 2 && valid && to0) {
                            float dv[8], lv[8];
                            unpack_bf16x8(u, dv);
                            unpack_bf16x8(lrow[cl >> 3], lv);
                            red8(cc, dv, lv, r1 + cl, r2 + cl);
                        }
                    }
                    if (EPI == 1 && stats_mode == 1 && valid) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            r1[ci * 16 + i] += v[i];
                            r2[ci * 16 + i] = fmaf(v[i], v[i], r2[ci * 16 + i]);
                        }
                    }
                }
            } else if (NBT) {
                int n_, h_, w_;
                valid = stats_mode ? row_valid(a.g, q, n_, h_, w_) : false;
                mbar_wait(tfull0 + 8 * acc, aph);
                tc_fence_after();
#pragma unroll
                for (int ci = 0; ci < NBT / 16; ++ci) {
                    float v[16];
                    tc_ld16(taddr + ci * 16, v);
                    if (ci == NBT / 16 - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(tempty0 + 8 * acc);
                    }
                    finish_chunk(ci * 16, v, q, p, inrange, valid);
                }
            } else {
                int n_, h_, w_;
                valid = stats_mode ? row_valid(a.g, q, n_, h_, w_) : false;
                mbar_wait(tfull0 + 8 * acc, aph);
                tc_fence_after();
                for (int c = 0; c < NB; c += 16) {
                    float v[16];
                    tc_ld16(taddr + c, v);
                    finish_chunk(c, v, q, p, inrange, valid);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty0 + 8 * acc);
            }
        }
        if (NBT && FAST && stats_mode) {
#pragma unroll
            for (int ci = 0; ci < NR / 16; ++ci) {
                float t1 = warp_colsum16(r1 + (NR > 1 ? ci * 16 : 0), lane);
                float t2 = warp_colsum16(r2 + (NR > 1 ? ci * 16 : 0), lane);
                if (lane < 16) { wstat[ci * 16 + lane] = t1; wstat[NB + ci * 16 + lane] = t2; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (a.stats) {
        for (int i = threadIdx.x; i < 2 * NB; i += kThreads) {
            const int which = i / NB, j = i % NB;
            float t = 0.f;
            for (int w = 0; w < 4; ++w) t += sstat[(size_t)w * 2 * NB + which * NB + j];
            a.stats[((size_t)blockIdx.x * 2 + which) * a.N + n0 + j] = t;
        }
    }
    if (stats_mode == 1 && a.bn.acc && a.bn.defer) {
        mpnn_acc_only(a.bn.acc, a.N, n0, NB, [&](int i) {
            return sstat[i] + sstat[2 * NB + i] + sstat[4 * NB + i] + sstat[6 * NB + i]; });
    } else if (stats_mode == 1 && a.bn.acc) {
        const bool last = mpnn_acc_and_ticket(a.bn.acc, a.N, n0, NB, gridDim.x * gridDim.y, [&](int i) {
            return sstat[i] + sstat[2 * NB + i] + sstat[4 * NB + i] + sstat[6 * NB + i]; });
        if (last) mpnn_bn_fwd_finalize_last(a.bn, a.N);
    } else if (stats_mode == 2) {
        // only the columns of out0 carry sums; CTAs whose slice lies in out1 just draw their ticket
        int nbe = a.N0 - n0;
        nbe = nbe < 0 ? 0 : (nbe > NB ? NB : nbe);
        const bool last = mpnn_acc_and_ticket(a.red.f.acc, a.N0, n0, nbe, gridDim.x * gridDim.y, [&](int i) {
            const int k = (i / nbe) * NB + i % nbe;
            return sstat[k] + sstat[2 * NB + k] + sstat[4 * NB + k] + sstat[6 * NB + k]; });
        if (last) mpnn_bn_bwd_finalize_last(a.red.f, a.red.mr, a.N0);
    }
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

// ---------------------------------------------------------------------------
// bring-up probe: one CTA, operands copied verbatim into shared memory
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128, 1)
umma_selftest_kernel(const uint8_t* __restrict__ A, int a_bytes, int a_off, const uint8_t* __restrict__ Bm,
                     int b_bytes, float* __restrict__ D, int N, int K, int a_mn, int b_mn,
                     int lbo_a, int sbo_a, int lbo_b, int sbo_b) {
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* sA = smem;
    uint8_t* sB = smem + ((a_bytes + 127) & ~127);
    uint64_t* bar = reinterpret_cast<uint64_t*>(sB + ((b_bytes + 127) & ~127));
    uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < a_bytes / 16; i += blockDim.x)
        reinterpret_cast<uint4*>(sA)[i] = reinterpret_cast<const uint4*>(A)[i];
    for (int i = threadIdx.x; i < b_bytes / 16; i += blockDim.x)
        reinterpret_cast<uint4*>(sB)[i] = reinterpret_cast<const uint4*>(Bm)[i];
    const uint32_t ncols = tmem_cols_pow2(N);
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(slot)), "r"(ncols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy smem writes -> async proxy
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *slot;
    if (threadIdx.x == 0) {
        const uint32_t idesc = make_idesc(N, a_mn, b_mn);
        for (int k = 0; k < K / 16; ++k) {
            const uint64_t ad = make_desc(smem_u32(sA) + a_off + (uint32_t)k * 2 * lbo_a, lbo_a, sbo_a);
            const uint64_t bd = make_desc(smem_u32(sB) + (uint32_t)k * 2 * lbo_b, lbo_b, sbo_b);
            tc_mma(tmem_base, ad, bd, idesc, k > 0);
        }
        tc_commit(smem_u32(bar));
    }
    mbar_wait(smem_u32(bar), 0);
    tc_fence_after();
    const int m = warp * 32 + lane;
    for (int c = 0; c < N; c += 16) {
        float v[16];
        tc_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + c, v);
#pragma unroll
        for (int i = 0; i < 16; ++i) D[(size_t)m * N + c + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(ncols) : "memory");
    }
}

}  // namespace

// bwd (optional): fused BN-backward reduction on out0, see BwdRed.  lin/ss/mr belong to the BatchNorm
// whose output gradient out0 is; requires 9 taps, bf16 planes out, no accumulation into out0.
int mpnn_stencil_gemm_umma(const void* A0, int K0, const void* A1, int K1, const void* Wp, int ntaps,
                           const float* bias, void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                           Geom g, float* stats, int stats_cap, int* n_parts, int out_dtype,
                           const mpnn_bn_fuse* bn, const mpnn_bn_bwd_epi* bwd, const int* count, cudaStream_t st) {
    const int N = N0 + N1;
    MPNN_REQUIRE(K0 % 16 == 0 && K1 % 16 == 0, "stencil_gemm(tcgen05): K0=%d K1=%d must be multiples of 16", K0, K1);
    MPNN_REQUIRE(N % 16 == 0 && N0 % 16 == 0, "stencil_gemm(tcgen05): N0=%d N1=%d must be multiples of 16", N0, N1);
    MPNN_REQUIRE(ntaps == 1 || ntaps == 9, "stencil_gemm(tcgen05): ntaps=%d (1 or 9)", ntaps);
    MPNN_REQUIRE(!bwd || (!bn && !stats && !acc0 && ntaps == 9 && out_dtype == MPNN_BF16 && N0 > 0),
                 "stencil_gemm(tcgen05): fused BN-backward sums need a plain 9-tap bf16 data gradient");
    MPNN_REQUIRE(!bwd || (bwd->lin && bwd->ss && bwd->mr && bwd->f.acc && bwd->f.sums),
                 "stencil_gemm(tcgen05): incomplete mpnn_bn_bwd_epi");
    MPNN_REQUIRE(!count || (!bwd && !bn && !stats), "stencil_gemm(tcgen05): a counted launch computes no statistics");
    const int KG = (K0 + K1) / 8;
    static const int tune_halo8 = getenv("MPNN_TUNE_HALO8") ? atoi(getenv("MPNN_TUNE_HALO8")) : 0;
    static const int tune_per_sm = getenv("MPNN_TUNE_PER_SM") ? atoi(getenv("MPNN_TUNE_PER_SM")) : 0;
    static const int tune_nstage = getenv("MPNN_TUNE_NSTAGE") ? atoi(getenv("MPNN_TUNE_NSTAGE")) : 0;
    static const int tune_dbg = getenv("MPNN_TUNE_DBG") ? atoi(getenv("MPNN_TUNE_DBG")) : 0;
    static const int tune_generic = getenv("MPNN_TUNE_GENERIC") ? atoi(getenv("MPNN_TUNE_GENERIC")) : 0;
    int halo = ntaps == 9 ? g.Wp + 1 : 0;
    if (tune_halo8) halo = (halo + 7) & ~7;
    const int rowsA = 128 + 2 * halo;
    // planes per pipeline stage: all of K when that is small (convs), else ~32 KB slices (wide FC inputs)
    int KC = KG;
    if ((size_t)rowsA * 16 * KG > 40 * 1024) {
        KC = (int)((32 * 1024) / ((size_t)rowsA * 16)) & ~1;
        if (KC < 2) KC = 2;
    }
    const size_t stage = (size_t)rowsA * 16 * KC;
    const size_t kMax = 227 * 1024 - 1024;
    const size_t red_bytes = bwd ? (size_t)12 * N0 : 0;        // staged scale / shift / mean of the BN behind out0
    int split = 0, nstage = 0, NB = 0;
    auto try_split = [&](int s) {            // N in s slices of NB columns, if the resident weights fit
        NB = N / s;
        if (NB > 256) return false;
        size_t w = ((size_t)ntaps * KG * NB * 16 + 127) & ~(size_t)127;
        size_t fixed = w + 256 + (size_t)9 * NB * 4 + red_bytes;
        if (fixed + 2 * stage > kMax) return false;
        split = s;
        nstage = (int)((kMax - fixed) / stage);
        if (nstage > 4) nstage = 4;
        if (tune_nstage && nstage > tune_nstage) nstage = tune_nstage;
        return true;
    };
    for (int s = 1; s <= 8; s *= 2)
        if (N % (16 * s) || try_split(s)) break;
    // N = 48 or 80 (a head GEMM [W_leaf | W_r1] with a 32- or 64-wide router) has no power-of-two split into 16-wide
    // slices: when the whole N does not fit, fall back to the smallest other divisor (3 or 5 slices of 16 at F = 2048)
    for (int s = 3; split == 0 && s <= 16; ++s)
        if (N % (16 * s) == 0) try_split(s);
    MPNN_REQUIRE(split > 0, "stencil_gemm(tcgen05): K=%d N=%d does not fit shared memory", K0 + K1, N);
    // fully-connected data gradients at small batches (one or two row tiles, N = 256 .. 2048 outputs): the slice
    // width above leaves a handful of CTAs, each walking up to 16 accumulator chunks through the generic epilogue
    // (15 us for 128 x 2048 outputs at K = 32).  While the grid is below one CTA per SM, halve the slices.
    static const int tune_fcsplit = getenv("MPNN_TUNE_FC_SPLIT") ? atoi(getenv("MPNN_TUNE_FC_SPLIT")) : 1;
    // (MPNN_TUNE_CONV_SPLIT=1: the same for the 3x3 convs -- measured with the statistics riding on the conv launch it
    //  lost 2 %: every slice re-reads the input tile and adds a round of fp64 atomics; off by default)
    static const int tune_convsplit = getenv("MPNN_TUNE_CONV_SPLIT") ? atoi(getenv("MPNN_TUNE_CONV_SPLIT")) : 0;
    if ((ntaps == 1 && tune_fcsplit) || (ntaps == 9 && tune_convsplit && !bwd)) {
        const int nt = ceil_div(g.rows, 128);
        while ((long long)nt * split * 2 <= 148 && NB % 64 == 0 && (N0 == 0 || N0 % (NB / 2) == 0)) { split *= 2; NB /= 2; }
    }
    size_t w = ((size_t)ntaps * KG * NB * 16 + 127) & ~(size_t)127;
    // CTAs per SM by shared memory, TMEM columns (alloc blocks when exhausted) and registers.  The kernel
    // is latency-bound per CTA, so residency beats pipeline depth: take the deepest ring that still gives
    // the largest number of resident CTAs (e.g. 64-channel layers: 2 stages x 2 CTAs instead of 4 x 1).
    int ncols = 32;
    while (ncols < 2 * NB) ncols <<= 1;
    int cap = 512 / ncols;
    if (cap > 4) cap = 4;
    if (NB == 32 && cap > 2) cap = 2;                            // register budgets of the instantiations
    if (NB == 16 && bwd && cap > 3) cap = 3;
    // the generic-width instantiations need ~108 registers: two CTAs per SM are resident (ncu: occupancy limit 2 by
    // registers); a grid sized for three ran as 1.5 waves
    const int n_kc_ = ceil_div(KG, KC);
    const int ks = (ntaps == 9 && n_kc_ == 1) ? KG / 2 : 0;
    const bool fast_ok = !tune_generic && out_dtype == MPNN_BF16 && !acc0 && !acc1 && !stats;
    if (NB != 16 && NB != 32 && cap > 2) cap = 2;
    if (tune_per_sm && cap > tune_per_sm) cap = tune_per_sm;
    if (cap < 1) cap = 1;
    size_t smem = 0;
    int per_sm = 0;
    for (int ns = nstage; ns >= 2; --ns) {
        const size_t sm_ns = w + (size_t)ns * stage + 256 + (size_t)9 * NB * 4 + red_bytes;
        int fit = (int)((227 * 1024) / (sm_ns + 1024));
        if (fit > cap) fit = cap;
        if (fit < 1) fit = 1;
        if (fit > per_sm) { per_sm = fit; smem = sm_ns; nstage = ns; }
    }
    GemmArgs a;
    a.dbg = tune_dbg;
    a.bn = mpnn_bn_fuse{};
    if (bn) a.bn = *bn;
    a.red = BwdRed{};
    if (bwd) { a.red.lin = (const __nv_bfloat16*)bwd->lin; a.red.ss = bwd->ss; a.red.mr = bwd->mr; a.red.f = bwd->f; }
    a.stats_mode = (stats || bn) ? 1 : (bwd ? 2 : 0);
    a.A0 = (const __nv_bfloat16*)A0; a.A1 = (const __nv_bfloat16*)A1; a.Wp = (const __nv_bfloat16*)Wp;
    a.bias = bias; a.out0 = out0; a.out1 = out1; a.stats = stats; a.g = g;
    a.K0 = K0; a.K1 = K1; a.N = N; a.N0 = N0; a.NB = NB; a.ntaps = ntaps; a.acc0 = acc0; a.acc1 = acc1;
    a.out_mode = out_dtype == MPNN_BF16 ? 0 : (out_dtype == MPNN_F32 ? 1 : 2);
    a.ld0 = N0; a.ld1 = N1;
    a.n_tiles = ceil_div(g.rows, 128); a.nstage = nstage;
    a.rowsA = rowsA; a.halo = halo; a.KC = KC; a.n_kc = ceil_div(KG, KC);
    a.count = count;
    MPNN_REQUIRE(a.out_mode != 2 || (!acc0 && !acc1 && !stats && !bn), "stencil_gemm: row-major output cannot accumulate");
    int gx = 148 * per_sm / split;
    if (gx > a.n_tiles) gx = a.n_tiles;
    if (stats && gx > stats_cap) gx = stats_cap;
    if (gx < 1) gx = 1;
    if (n_parts) *n_parts = stats ? gx : 0;
    // kernel table: [slice width 16 / 32 / generic][K steps 0 (generic loop), 1..4][epilogue kind]; the counted
    // instantiations (live batch from device memory) exist for the epilogues without sums only
    typedef void (*Kern)(const GemmArgs);
    static const Kern generic[2][3] = {{stencil_gemm_umma_kernel<16, 0, 0>, stencil_gemm_umma_kernel<32, 0, 0>,
                                        stencil_gemm_umma_kernel<0, 0, 0>},
                                       {stencil_gemm_umma_kernel<16, 0, 0, true>, stencil_gemm_umma_kernel<32, 0, 0, true>,
                                        stencil_gemm_umma_kernel<0, 0, 0, true>}};
    // [0] forward, [1] fused BN-backward sums, [2] forward, counted
    static const Kern fast16[3][2] = {{stencil_gemm_umma_kernel<16, 1, 1>, stencil_gemm_umma_kernel<16, 2, 1>},
                                      {stencil_gemm_umma_kernel<16, 1, 2>, stencil_gemm_umma_kernel<16, 2, 2>},
                                      {stencil_gemm_umma_kernel<16, 1, 1, true>, stencil_gemm_umma_kernel<16, 2, 1, true>}};
    static const Kern fast32[3][4] = {{stencil_gemm_umma_kernel<32, 1, 1>, stencil_gemm_umma_kernel<32, 2, 1>,
                                       stencil_gemm_umma_kernel<32, 3, 1>, stencil_gemm_umma_kernel<32, 4, 1>},
                                      {stencil_gemm_umma_kernel<32, 1, 2>, stencil_gemm_umma_kernel<32, 2, 2>,
                                       stencil_gemm_umma_kernel<32, 3, 2>, stencil_gemm_umma_kernel<32, 4, 2>},
                                      {stencil_gemm_umma_kernel<32, 1, 1, true>, stencil_gemm_umma_kernel<32, 2, 1, true>,
                                       stencil_gemm_umma_kernel<32, 3, 1, true>, stencil_gemm_umma_kernel<32, 4, 1, true>}};
    // generic slice width (N >= 48), generic epilogue, unrolled issue loop for the K of the 32..128-channel layers
    static const Kern wide[2][5] = {{stencil_gemm_umma_kernel<0, 2, 0>, stencil_gemm_umma_kernel<0, 3, 0>,
                                     stencil_gemm_umma_kernel<0, 4, 0>, stencil_gemm_umma_kernel<0, 6, 0>,
                                     stencil_gemm_umma_kernel<0, 8, 0>},
                                    {stencil_gemm_umma_kernel<0, 2, 0, true>, stencil_gemm_umma_kernel<0, 3, 0, true>,
                                     stencil_gemm_umma_kernel<0, 4, 0, true>, stencil_gemm_umma_kernel<0, 6, 0, true>,
                                     stencil_gemm_umma_kernel<0, 8, 0, true>}};
    const int c = count ? 1 : 0;
    const int e = bwd ? 1 : 2 * c;
    Kern kern = generic[c][NB == 16 ? 0 : (NB == 32 ? 1 : 2)];
    if (fast_ok && NB == 16 && ks >= 1 && ks <= 2) kern = fast16[e][ks - 1];
    if (fast_ok && NB == 32 && ks >= 1 && ks <= 4) kern = fast32[e][ks - 1];
    if (!tune_generic && NB != 16 && NB != 32) {
        const int wi = ks == 2 ? 0 : ks == 3 ? 1 : ks == 4 ? 2 : ks == 6 ? 3 : ks == 8 ? 4 : -1;
        if (wi >= 0) kern = wide[c][wi];
    }
    // the > 48 KB dynamic shared memory opt-in is a per-device function attribute
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64 || !attr_set[dev]) {
        constexpr int nk = 6 + 3 * 2 + 3 * 4 + 2 * 5;
        Kern all[nk];
        int k = 0;
        for (int i = 0; i < 2; ++i) for (int j = 0; j < 3; ++j) all[k++] = generic[i][j];
        for (int i = 0; i < 3; ++i) for (int j = 0; j < 2; ++j) all[k++] = fast16[i][j];
        for (int i = 0; i < 3; ++i) for (int j = 0; j < 4; ++j) all[k++] = fast32[i][j];
        for (int i = 0; i < 2; ++i) for (int j = 0; j < 5; ++j) all[k++] = wide[i][j];
        for (int i = 0; i < nk; ++i) {
            cudaError_t e2 = cudaFuncSetAttribute(all[i], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMax);   // + static smem stays under 227 KB
            if (e2 != cudaSuccess) { mpnn_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e2)); return MPNN_ERR_CUDA; }
            // without this the driver picks the L1 / shared-memory split heuristically and may leave room for fewer
            // CTAs per SM than the grid was sized for (ncu: occupancy limit 2 by shared memory where 3 x 68 KB fit;
            // the persistent grid then ran as 1.5 waves)
            if (!getenv("MPNN_TUNE_NO_CARVEOUT")) cudaFuncSetAttribute(all[i], cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        }
        if (dev >= 0 && dev < 64) attr_set[dev] = true;
    }
    static const int tune_occ = getenv("MPNN_TUNE_OCC") ? atoi(getenv("MPNN_TUNE_OCC")) : 0;
    if (tune_occ) {      // tuning aid: clamp the persistent grid to what the occupancy calculator reports
        int occ = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, smem) == cudaSuccess && occ >= 1 && occ < per_sm) {
            int g2 = 148 * occ / split;
            if (g2 < 1) g2 = 1;
            if (gx > g2) gx = g2;
            if (n_parts && stats) *n_parts = gx;
        }
    }
    cudaError_t le = mpnn_launch_pdl(kern, dim3(gx, split), dim3(kThreads), smem, st, a);
    if (le != cudaSuccess) { mpnn_set_error("stencil_gemm_umma launch: %s", cudaGetErrorString(le)); return MPNN_ERR_CUDA; }
    return mpnn_check_launch("stencil_gemm_umma");
}

extern "C" int mpnn_umma_selftest(const void* A, int a_bytes, int a_off, const void* Bm, int b_bytes,
                                  float* D, int N, int K, int a_mn_major, int b_mn_major,
                                  int lbo_a, int sbo_a, int lbo_b, int sbo_b, void* stream) {
    MPNN_REQUIRE(N % 16 == 0 && N >= 16 && N <= 256 && K % 16 == 0, "umma_selftest: N=%d K=%d", N, K);
    MPNN_REQUIRE(a_bytes % 16 == 0 && b_bytes % 16 == 0 && a_off % 16 == 0, "umma_selftest: alignment");
    size_t smem = ((a_bytes + 127) & ~127) + ((b_bytes + 127) & ~127) + 64;
    MPNN_REQUIRE(smem <= 200 * 1024, "umma_selftest: operands too large");
    cudaError_t e = cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) { mpnn_set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return MPNN_ERR_CUDA; }
    umma_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(
        (const uint8_t*)A, a_bytes, a_off, (const uint8_t*)Bm, b_bytes, D, N, K, a_mn_major, b_mn_major,
        lbo_a, sbo_a, lbo_b, sbo_b);
    return mpnn_check_launch("umma_selftest");
}
