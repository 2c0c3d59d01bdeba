// Routing: per-example walk of the sink tree (policy softmax, epsilon floor,
// first-max argmax, child probabilities), its backward (actor expectation
// gradient / critic cost regression), per-node batch moments for TALR, and
// path compaction + image gather / scatter-add.
// Reference: lib/net_types.py:108-131 (actor), :193-243 (critic), :24-27 (TALR).
#include "common.cuh"
#include "../../include/mpnn.h"

#define RT_MAXS 8   // max sinks per switch

// softmax(r / tau) and the first-max argmax of r.  All loops are fully unrolled
// over RT_MAXS with a `j < ns` predicate so the small arrays stay in registers
// (statically indexed); callers must index `sm` the same way.
__device__ __forceinline__ int route_softmax(const float* r, int ns, float tau, float (&sm)[RT_MAXS]) {
    float mx = -INFINITY, mr = -INFINITY;
    int dec = 0;
#pragma unroll
    for (int j = 0; j < RT_MAXS; ++j) {
        sm[j] = 0.f;
        if (j < ns) {
            float v = r[j];
            if (v > mr) { mr = v; dec = j; }          // first maximal index (tf.argmax)
            sm[j] = v / tau;
            mx = fmaxf(mx, sm[j]);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < RT_MAXS; ++j)
        if (j < ns) { sm[j] = expf(sm[j] - mx); s += sm[j]; }
    const float inv = 1.f / s;
#pragma unroll
    for (int j = 0; j < RT_MAXS; ++j) sm[j] *= inv;
    return dec;
}

__device__ __forceinline__ float pick(const float (&v)[RT_MAXS], int idx) {
    float out = 0.f;
#pragma unroll
    for (int j = 0; j < RT_MAXS; ++j) out = (j == idx) ? v[j] : out;
    return out;
}

// the same with the arrays sized for the widest switch of the net (block-uniform, 2 / 4 / 8): a 2-sink chain
// does not pay for 8 predicated slots per step of the walk
template <int NS>
__device__ __forceinline__ int route_softmax_t(const float* r, int ns, float tau, float (&sm)[NS]) {
    float mx = -INFINITY, mr = -INFINITY;
    int dec = 0;
#pragma unroll
    for (int j = 0; j < NS; ++j) {
        sm[j] = 0.f;
        if (j < ns) {
            float v = r[j];
            if (v > mr) { mr = v; dec = j; }          // first maximal index (tf.argmax)
            sm[j] = v / tau;
            mx = fmaxf(mx, sm[j]);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NS; ++j)
        if (j < ns) { sm[j] = expf(sm[j] - mx); s += sm[j]; }
    const float inv = 1.f / s;
#pragma unroll
    for (int j = 0; j < NS; ++j) sm[j] *= inv;
    return dec;
}

template <int NS>
__device__ __forceinline__ float pick_t(const float (&v)[NS], int idx) {
    float out = 0.f;
#pragma unroll
    for (int j = 0; j < NS; ++j) out = (j == idx) ? v[j] : out;
    return out;
}

__global__ void route_fwd_kernel(const int* __restrict__ parent, const int* __restrict__ sink_idx,
                                 const int* __restrict__ n_sinks, const float* __restrict__ floor_,
                                 const int* __restrict__ sw, int n_nodes,
                                 const float* const* __restrict__ R, const float* __restrict__ hyp, int B,
                                 float* __restrict__ p_tr, float* __restrict__ p_ev, int* __restrict__ dec) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float tau = hyp[MPNN_HYP_TAU], eps = hyp[MPNN_HYP_EPS];
    p_tr[b] = 1.f; p_ev[b] = 1.f;
    for (int i = 1; i < n_nodes; ++i) {
        int par = parent[i];
        int ns = n_sinks[par];
        float pt = p_tr[(size_t)par * B + b], pe = p_ev[(size_t)par * B + b];
        if (ns >= 2) {
            float sm[RT_MAXS];
            int slot = sw[par];
            int d = route_softmax(R[slot] + (size_t)b * ns, ns, tau, sm);
            int si = sink_idx[i];
            if (si == 0 && dec) dec[(size_t)slot * B + b] = d;
            pt = (pt - eps * floor_[par]) * pick(sm, si) + eps * floor_[i];
            pe = pe * (d == si ? 1.f : 0.f);
        }
        p_tr[(size_t)i * B + b] = pt;
        p_ev[(size_t)i * B + b] = pe;
    }
}


// ---- staged variants ---------------------------------------------------------------------------------
// The walk is a chain of small dependent steps per example; in the kernels above every step goes through
// global memory (tree tables, pointer tables, the per-node running values), i.e. ~n_nodes x several L2
// round trips back to back.  For trees of up to RT_STAGED_MAX nodes the tables are staged in shared memory
// once per CTA, the per-example running values live in a shared-memory column per thread, and the
// per-example inputs are fetched up front with independent loads.  Same arithmetic, same order.
#define RT_STAGED_MAX 32
#define RT_T 64
struct RtTables {
    int *parent, *sink_idx, *n_sinks, *sw, *err, *child;
    float *floor_, *ops;
    const float** Rn;          // per node: logits of its router (switches only)
    float** dRn;
    const float** cen;         // per node: c_err / d_cor vectors of its classifier (leaves only)
    const float** dcn;
    float* col;                // [ncol][n][RT_T]
};
static size_t rt_smem_bytes(int n, int ncol) {
    return (size_t)n * (5 * 4 + RT_MAXS * 4 + 2 * 4 + 4 * 8) + (size_t)ncol * n * RT_T * 4 + 64;
}
__device__ __forceinline__ RtTables rt_carve(unsigned char* sm, int n, int ncol) {
    RtTables t;
    t.Rn = reinterpret_cast<const float**>(sm);  sm += (size_t)n * 8;
    t.dRn = reinterpret_cast<float**>(sm);       sm += (size_t)n * 8;
    t.cen = reinterpret_cast<const float**>(sm); sm += (size_t)n * 8;
    t.dcn = reinterpret_cast<const float**>(sm); sm += (size_t)n * 8;
    t.parent = reinterpret_cast<int*>(sm);   sm += (size_t)n * 4;
    t.sink_idx = reinterpret_cast<int*>(sm); sm += (size_t)n * 4;
    t.n_sinks = reinterpret_cast<int*>(sm);  sm += (size_t)n * 4;
    t.sw = reinterpret_cast<int*>(sm);       sm += (size_t)n * 4;
    t.err = reinterpret_cast<int*>(sm);      sm += (size_t)n * 4;
    t.child = reinterpret_cast<int*>(sm);    sm += (size_t)n * RT_MAXS * 4;
    t.floor_ = reinterpret_cast<float*>(sm); sm += (size_t)n * 4;
    t.ops = reinterpret_cast<float*>(sm);    sm += (size_t)n * 4;
    t.col = reinterpret_cast<float*>(sm);
    return t;
}

__device__ __forceinline__ void rt_prefetch(const void* p) { asm volatile("prefetch.global.L1 [%0];" :: "l"(p)); }

template <int NS>
__device__ __forceinline__ void route_fwd_walk(const RtTables& t, int n_nodes, const float* __restrict__ hyp, int B,
                                               float* __restrict__ p_tr, float* __restrict__ p_ev,
                                               int* __restrict__ dec) {
    const int tid = threadIdx.x;
    const int b = blockIdx.x * RT_T + tid;
    if (b >= B) return;
    const float tau = hyp[MPNN_HYP_TAU], eps = hyp[MPNN_HYP_EPS];
    for (int i = 0; i < n_nodes; ++i)                        // every router's logits of this example: in flight together
        if (t.Rn[i]) rt_prefetch(t.Rn[i] + (size_t)b * t.n_sinks[i]);
    float* pt_c = t.col + tid;                               // [n][RT_T] columns of this thread
    float* pe_c = t.col + (size_t)n_nodes * RT_T + tid;
    pt_c[0] = 1.f; pe_c[0] = 1.f;
    p_tr[b] = 1.f; p_ev[b] = 1.f;
    // siblings share their parent's softmax: evaluate it once, when the first sink (sink_idx 0) comes up
    float sm[NS];
    int d = 0, sm_of = -1;
    for (int i = 1; i < n_nodes; ++i) {
        const int par = t.parent[i], ns = t.n_sinks[par];
        float pt = pt_c[par * RT_T], pe = pe_c[par * RT_T];
        if (ns >= 2) {
            const int si = t.sink_idx[i];
            if (sm_of != par) {
                d = route_softmax_t<NS>(t.Rn[par] + (size_t)b * ns, ns, tau, sm);
                sm_of = par;
                if (dec) dec[(size_t)t.sw[par] * B + b] = d;
            }
            pt = (pt - eps * t.floor_[par]) * pick_t<NS>(sm, si) + eps * t.floor_[i];
            pe = pe * (d == si ? 1.f : 0.f);
        }
        pt_c[i * RT_T] = pt; pe_c[i * RT_T] = pe;
        p_tr[(size_t)i * B + b] = pt;
        p_ev[(size_t)i * B + b] = pe;
    }
}

__global__ void __launch_bounds__(RT_T)
route_fwd_staged_kernel(const int* __restrict__ parent, const int* __restrict__ sink_idx,
                        const int* __restrict__ n_sinks, const float* __restrict__ floor_,
                        const int* __restrict__ sw, int n_nodes,
                        const float* const* __restrict__ R, const float* __restrict__ hyp, int B,
                        float* __restrict__ p_tr, float* __restrict__ p_ev, int* __restrict__ dec) {
    extern __shared__ __align__(16) unsigned char rt_sm[];
    const RtTables t = rt_carve(rt_sm, n_nodes, 2);
    const int tid = threadIdx.x;
    __shared__ int s_nsmax;
    if (tid == 0) s_nsmax = 0;
    __syncthreads();
    for (int i = tid; i < n_nodes; i += RT_T) {
        t.parent[i] = i ? parent[i] : 0; t.sink_idx[i] = sink_idx[i]; t.n_sinks[i] = n_sinks[i];
        t.sw[i] = sw[i]; t.floor_[i] = floor_[i];
        t.Rn[i] = n_sinks[i] >= 2 ? R[sw[i]] : nullptr;
        atomicMax(&s_nsmax, n_sinks[i]);
    }
    __syncthreads();
    if (s_nsmax <= 2)      route_fwd_walk<2>(t, n_nodes, hyp, B, p_tr, p_ev, dec);
    else if (s_nsmax <= 4) route_fwd_walk<4>(t, n_nodes, hyp, B, p_tr, p_ev, dec);
    else                   route_fwd_walk<RT_MAXS>(t, n_nodes, hyp, B, p_tr, p_ev, dec);
}

extern "C" int mpnn_route_fwd(const int* parent, const int* sink_idx, const int* n_sinks,
                              const float* floor_, const int* sw, int n_nodes,
                              const float* const* R, const float* hyp, int B,
                              float* p_tr, float* p_ev, int* dec, void* stream) {
    MPNN_REQUIRE(n_nodes >= 1 && B >= 1 && hyp, "route_fwd: args");
    if (n_nodes <= RT_STAGED_MAX)
        route_fwd_staged_kernel<<<ceil_div(B, RT_T), RT_T, rt_smem_bytes(n_nodes, 2), (cudaStream_t)stream>>>(
            parent, sink_idx, n_sinks, floor_, sw, n_nodes, R, hyp, B, p_tr, p_ev, dec);
    else
        route_fwd_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(
            parent, sink_idx, n_sinks, floor_, sw, n_nodes, R, hyp, B, p_tr, p_ev, dec);
    return mpnn_check_launch("route_fwd");
}

__global__ void route_bwd_kernel(const int* parent, const int* sink_idx,
                                 const int* n_sinks, const int* child,
                                 const float* floor_, const int* sw,
                                 const float* ops, const int* err, int n_nodes,
                                 const float* const* R, const float* hyp, int B,
                                 const float* p_tr, const float* p_ev,
                                 const float* const* c_err, const float* const* d_cor,
                                 const float* k_cpt,
                                 int critic, float k_dec, float k_cre, int optimistic, int use_cls_err,
                                 float* const* dR, float* scratch,
                                 float* c_data) {
    int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float invB = 1.f / (float)B;
    const float tau = hyp[MPNN_HYP_TAU], eps = hyp[MPNN_HYP_EPS];
    const float kc = k_cpt ? k_cpt[b] : hyp[MPNN_HYP_KCPT];
    float* gp = scratch;                              // [n_nodes][B]
    float* cev = scratch + (size_t)n_nodes * B;       // critic
    float* cop = scratch + (size_t)2 * n_nodes * B;   // critic
    float total = 0.f;
    if (!critic) {
        for (int i = 0; i < n_nodes; ++i) {
            float ce = err[i] >= 0 ? c_err[err[i]][b] : 0.f;
            float local = ce + kc * ops[i];
            gp[(size_t)i * B + b] = local * invB;
            total += p_tr[(size_t)i * B + b] * local;
        }
        for (int i = n_nodes - 1; i >= 1; --i) {
            int par = parent[i];
            int ns = n_sinks[par];
            float g = gp[(size_t)i * B + b];
            if (ns >= 2) {
                float sm[RT_MAXS];
                route_softmax(R[sw[par]] + (size_t)b * ns, ns, tau, sm);
                g *= pick(sm, sink_idx[i]);
            }
            gp[(size_t)par * B + b] += g;
        }
        for (int i = 0; i < n_nodes; ++i) {
            int ns = n_sinks[i];
            if (ns < 2) continue;
            const float* r = R[sw[i]] + (size_t)b * ns;
            float sm[RT_MAXS], gs[RT_MAXS];
            route_softmax(r, ns, tau, sm);
            float pt = p_tr[(size_t)i * B + b];
            float dot = 0.f, r2 = 0.f;
#pragma unroll
            for (int j = 0; j < RT_MAXS; ++j) {
                gs[j] = 0.f;
                if (j < ns) {
                    gs[j] = gp[(size_t)child[i * RT_MAXS + j] * B + b] * (pt - eps * floor_[i]);
                    dot = fmaf(sm[j], gs[j], dot);
                    r2 = fmaf(r[j], r[j], r2);
                }
            }
            float* out = dR[sw[i]] + (size_t)b * ns;
#pragma unroll
            for (int j = 0; j < RT_MAXS; ++j)
                if (j < ns) out[j] = sm[j] * (gs[j] - dot) / tau + pt * k_dec * 2.f * r[j] * invB;
            total += pt * k_dec * r2;
        }
    } else {
        for (int i = n_nodes - 1; i >= 0; --i) {
            int ns = n_sinks[i];
            float ce;
            if (use_cls_err) ce = err[i] >= 0 ? 1.f - d_cor[err[i]][b] : 0.f;
            else ce = err[i] >= 0 ? c_err[err[i]][b] : 0.f;
            float base = ce + kc * ops[i];
            float pt = p_tr[(size_t)i * B + b];
            float cre = 0.f;
            if (ns < 2) {
                float e = base, o = base;
                for (int j = 0; j < ns; ++j) {
                    int ch = child[i * RT_MAXS + j];
                    e += cev[(size_t)ch * B + b]; o += cop[(size_t)ch * B + b];
                }
                cev[(size_t)i * B + b] = e; cop[(size_t)i * B + b] = o;
            } else {
                const float* r = R[sw[i]] + (size_t)b * ns;
                float sm[RT_MAXS];
                int d = route_softmax(r, ns, tau, sm);
                float mn = INFINITY;
                float* out = dR[sw[i]] + (size_t)b * ns;
                for (int j = 0; j < ns; ++j) {
                    int ch = child[i * RT_MAXS + j];
                    float ev = cev[(size_t)ch * B + b], op = cop[(size_t)ch * B + b];
                    mn = fminf(mn, op);
                    float tgt = optimistic ? op : ev;
                    float dlt = r[j] + tgt;
                    cre = fmaf(dlt, dlt, cre);
                    out[j] = pt * invB * k_cre * 2.f * dlt;
                }
                cre *= k_cre;
                cev[(size_t)i * B + b] = base + cev[(size_t)child[i * RT_MAXS + d] * B + b];
                cop[(size_t)i * B + b] = base + mn;
            }
            float ce_true = err[i] >= 0 ? c_err[err[i]][b] : 0.f;
            total += pt * (ce_true + cre);
        }
    }
    if (c_data) c_data[b] = total;
}


template <int NS>
__device__ __forceinline__ void route_bwd_walk(const RtTables& t, int n_nodes, const float* __restrict__ hyp, int B,
                                               const float* __restrict__ p_tr, const float* __restrict__ k_cpt,
                                               int critic, float k_dec, float k_cre, int optimistic, int use_cls_err,
                                               float* __restrict__ c_data) {
    const int tid = threadIdx.x, n = n_nodes;
    const int b = blockIdx.x * RT_T + tid;
    if (b >= B) return;
    const float invB = 1.f / (float)B;
    const float tau = hyp[MPNN_HYP_TAU], eps = hyp[MPNN_HYP_EPS];
    const float kc = k_cpt ? k_cpt[b] : hyp[MPNN_HYP_KCPT];
    const size_t cs = (size_t)n * RT_T;
    float* pt_c = t.col + tid;                 // p_tr of every node
    float* ce_c = t.col + cs + tid;            // c_err of every node (0 off the leaves)
    float* g_c = t.col + 2 * cs + tid;         // actor: dL/dp_tr; critic: c_ev
    float* o_c = t.col + 3 * cs + tid;         // critic: c_opt
    float* dc_c = t.col + 4 * cs + tid;        // critic with use_cls_err: 1 - d_cor
    // per-example inputs: independent loads, issued together
    for (int i = 0; i < n; ++i)
        if (t.Rn[i]) rt_prefetch(t.Rn[i] + (size_t)b * t.n_sinks[i]);
#pragma unroll 4
    for (int i = 0; i < n; ++i) {
        pt_c[i * RT_T] = p_tr[(size_t)i * B + b];
        ce_c[i * RT_T] = t.cen[i] ? t.cen[i][b] : 0.f;
        if (use_cls_err) dc_c[i * RT_T] = t.dcn[i] ? 1.f - t.dcn[i][b] : 0.f;
    }
    float total = 0.f;
    float sm[NS];
    int sm_of = -1, d = 0;
    if (!critic) {
        for (int i = 0; i < n; ++i) {
            const float local = ce_c[i * RT_T] + kc * t.ops[i];
            g_c[i * RT_T] = local * invB;
            total += pt_c[i * RT_T] * local;
        }
        for (int i = n - 1; i >= 1; --i) {
            const int par = t.parent[i], ns = t.n_sinks[par];
            float g = g_c[i * RT_T];
            if (ns >= 2) {
                if (sm_of != par) { route_softmax_t<NS>(t.Rn[par] + (size_t)b * ns, ns, tau, sm); sm_of = par; }
                g *= pick_t<NS>(sm, t.sink_idx[i]);
            }
            g_c[par * RT_T] += g;
        }
        for (int i = 0; i < n; ++i) {
            const int ns = t.n_sinks[i];
            if (ns < 2) continue;
            const float* r = t.Rn[i] + (size_t)b * ns;
            float gs[NS], rv[NS];
            route_softmax_t<NS>(r, ns, tau, sm);
            sm_of = i;
            const float pt = pt_c[i * RT_T];
            float dot = 0.f, r2 = 0.f;
#pragma unroll
            for (int j = 0; j < NS; ++j) {
                gs[j] = 0.f; rv[j] = 0.f;
                if (j < ns) {
                    rv[j] = r[j];
                    gs[j] = g_c[t.child[i * RT_MAXS + j] * RT_T] * (pt - eps * t.floor_[i]);
                    dot = fmaf(sm[j], gs[j], dot);
                    r2 = fmaf(rv[j], rv[j], r2);
                }
            }
            float* out = t.dRn[i] + (size_t)b * ns;
#pragma unroll
            for (int j = 0; j < NS; ++j)
                if (j < ns) out[j] = sm[j] * (gs[j] - dot) / tau + pt * k_dec * 2.f * rv[j] * invB;
            total += pt * k_dec * r2;
        }
    } else {
        for (int i = n - 1; i >= 0; --i) {
            const int ns = t.n_sinks[i];
            const float ce_true = ce_c[i * RT_T];
            const float ce = use_cls_err ? dc_c[i * RT_T] : ce_true;
            const float base = ce + kc * t.ops[i];
            const float pt = pt_c[i * RT_T];
            float cre = 0.f;
            if (ns < 2) {
                float e = base, o = base;
                for (int j = 0; j < ns; ++j) {
                    const int ch = t.child[i * RT_MAXS + j];
                    e += g_c[ch * RT_T]; o += o_c[ch * RT_T];
                }
                g_c[i * RT_T] = e; o_c[i * RT_T] = o;
            } else {
                const float* r = t.Rn[i] + (size_t)b * ns;
                d = route_softmax_t<NS>(r, ns, tau, sm);
                float mn = INFINITY;
                float* out = t.dRn[i] + (size_t)b * ns;
                for (int j = 0; j < ns; ++j) {
                    const int ch = t.child[i * RT_MAXS + j];
                    const float ev = g_c[ch * RT_T], op = o_c[ch * RT_T];
                    mn = fminf(mn, op);
                    const float tgt = optimistic ? op : ev;
                    const float dlt = r[j] + tgt;
                    cre = fmaf(dlt, dlt, cre);
                    out[j] = pt * invB * k_cre * 2.f * dlt;
                }
                cre *= k_cre;
                g_c[i * RT_T] = base + g_c[t.child[i * RT_MAXS + d] * RT_T];
                o_c[i * RT_T] = base + mn;
            }
            total += pt * (ce_true + cre);
        }
    }
    if (c_data) c_data[b] = total;
}

__global__ void __launch_bounds__(RT_T)
route_bwd_staged_kernel(const int* __restrict__ parent, const int* __restrict__ sink_idx,
                        const int* __restrict__ n_sinks, const int* __restrict__ child,
                        const float* __restrict__ floor_, const int* __restrict__ sw,
                        const float* __restrict__ ops, const int* __restrict__ err, int n_nodes,
                        const float* const* __restrict__ R, const float* __restrict__ hyp, int B,
                        const float* __restrict__ p_tr,
                        const float* const* __restrict__ c_err, const float* const* __restrict__ d_cor,
                        const float* __restrict__ k_cpt,
                        int critic, float k_dec, float k_cre, int optimistic, int use_cls_err,
                        float* const* __restrict__ dR, float* __restrict__ c_data) {
    extern __shared__ __align__(16) unsigned char rt_sm[];
    const RtTables t = rt_carve(rt_sm, n_nodes, 5);
    const int tid = threadIdx.x, n = n_nodes;
    __shared__ int s_nsmax;
    if (tid == 0) s_nsmax = 0;
    __syncthreads();
    for (int i = tid; i < n; i += RT_T) {
        t.parent[i] = i ? parent[i] : 0; t.sink_idx[i] = sink_idx[i]; t.n_sinks[i] = n_sinks[i];
        t.sw[i] = sw[i]; t.floor_[i] = floor_[i]; t.ops[i] = ops[i]; t.err[i] = err[i];
        const bool is_sw = n_sinks[i] >= 2;
        atomicMax(&s_nsmax, n_sinks[i]);
        t.Rn[i] = is_sw ? R[sw[i]] : nullptr;
        t.dRn[i] = is_sw ? dR[sw[i]] : nullptr;
        t.cen[i] = err[i] >= 0 ? c_err[err[i]] : nullptr;
        t.dcn[i] = (err[i] >= 0 && use_cls_err) ? d_cor[err[i]] : nullptr;
        for (int j = 0; j < RT_MAXS; ++j) t.child[i * RT_MAXS + j] = child[i * RT_MAXS + j];
    }
    __syncthreads();
    if (s_nsmax <= 2)
        route_bwd_walk<2>(t, n, hyp, B, p_tr, k_cpt, critic, k_dec, k_cre, optimistic, use_cls_err, c_data);
    else if (s_nsmax <= 4)
        route_bwd_walk<4>(t, n, hyp, B, p_tr, k_cpt, critic, k_dec, k_cre, optimistic, use_cls_err, c_data);
    else
        route_bwd_walk<RT_MAXS>(t, n, hyp, B, p_tr, k_cpt, critic, k_dec, k_cre, optimistic, use_cls_err, c_data);
}

extern "C" int mpnn_route_bwd(const int* parent, const int* sink_idx, const int* n_sinks, const int* child,
                              const float* floor_, const int* sw, const float* ops, const int* err,
                              int n_nodes, const float* const* R, const float* hyp, int B,
                              const float* p_tr, const float* p_ev,
                              const float* const* c_err, const float* const* d_cor,
                              const float* k_cpt,
                              int critic, float k_dec, float k_cre, int optimistic, int use_cls_err,
                              float* const* dR, float* scratch, float* c_data, void* stream) {
    MPNN_REQUIRE(n_nodes >= 1 && B >= 1 && hyp, "route_bwd: args");
    if (n_nodes <= RT_STAGED_MAX)
        route_bwd_staged_kernel<<<ceil_div(B, RT_T), RT_T, rt_smem_bytes(n_nodes, 5), (cudaStream_t)stream>>>(
            parent, sink_idx, n_sinks, child, floor_, sw, ops, err, n_nodes, R, hyp, B, p_tr, c_err, d_cor,
            k_cpt, critic, k_dec, k_cre, optimistic, use_cls_err, dR, c_data);
    else
        route_bwd_kernel<<<ceil_div(B, 128), 128, 0, (cudaStream_t)stream>>>(
            parent, sink_idx, n_sinks, child, floor_, sw, ops, err, n_nodes, R, hyp, B, p_tr, p_ev, c_err, d_cor,
            k_cpt, critic, k_dec, k_cre, optimistic, use_cls_err, dR, scratch, c_data);
    return mpnn_check_launch("route_bwd");
}

// ------------------------------------------------------------- node moments
__global__ void node_moments_kernel(const float* __restrict__ p_tr, int B, float* __restrict__ stats) {
    const int i = blockIdx.x;
    float s2 = 0.f, s1 = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        float v = p_tr[(size_t)i * B + b];
        s2 = fmaf(v, v, s2); s1 += v;
    }
    __shared__ float red[2][8];
    s2 = warp_sum(s2); s1 = warp_sum(s1);
    if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s2; red[1][threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, c = 0.f;
        for (int w = 0; w < 8; ++w) { a += red[0][w]; c += red[1][w]; }
        stats[i * 2] = a / B;
        stats[i * 2 + 1] = c / B;
    }
}

extern "C" int mpnn_node_moments(const float* p_tr, int n_nodes, int B, float* stats, void* stream) {
    node_moments_kernel<<<n_nodes, 256, 0, (cudaStream_t)stream>>>(p_tr, B, stats);
    return mpnn_check_launch("node_moments");
}

// ---------------------------------------------------------- path compaction
// One CTA per node; ballot + warp/CTA prefix scan; order preserving.
__global__ void __launch_bounds__(1024)
compact_paths_kernel(const float* __restrict__ p_ev, int B, int* __restrict__ idx, int* __restrict__ count) {
    const int node = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ int wcount[32];
    __shared__ int base_s;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    for (int b0 = 0; b0 < B; b0 += 1024) {
        int b = b0 + threadIdx.x;
        bool take = b < B && p_ev[(size_t)node * B + b] > 0.5f;
        unsigned m = __ballot_sync(0xffffffffu, take);
        if (lane == 0) wcount[warp] = __popc(m);
        __syncthreads();
        int wbase = 0, tot = 0;
        for (int w = 0; w < 32; ++w) { int c = wcount[w]; if (w < warp) wbase += c; tot += c; }
        int base = base_s;
        if (take) idx[(size_t)node * B + base + wbase + __popc(m & ((1u << lane) - 1u))] = b;
        __syncthreads();
        if (threadIdx.x == 0) base_s = base + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) count[node] = base_s;
}

extern "C" int mpnn_compact_paths(const float* p_ev, int n_nodes, int B, int* idx, int* count, void* stream) {
    compact_paths_kernel<<<n_nodes, 1024, 0, (cudaStream_t)stream>>>(p_ev, B, idx, count);
    return mpnn_check_launch("compact_paths");
}

// --------------------------------------------------- gather / scatter-add
// Image blocks are S contiguous rows per plane, so both are row-vector copies.
template <typename T, bool SCATTER>
__global__ void move_images_kernel(const T* __restrict__ src, int Ps, const int* __restrict__ idx,
                                   const int* __restrict__ count, T* __restrict__ dst, int Pd,
                                   int KG, int S, int G) {
    const int n = *count;
    const long long total = (long long)KG * n * S;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        int r = i % S;
        long long t = i / S;
        int j = t % n;
        int kg = t / n;
        int img = idx[j];
        if (!SCATTER) {
            const uint4* s = reinterpret_cast<const uint4*>(plane_row(src, kg, Ps, G + img * S + r));
            uint4* d = reinterpret_cast<uint4*>(plane_row(dst, kg, Pd, G + j * S + r));
            d[0] = s[0];
            if (sizeof(T) == 4) d[1] = s[1];
        } else {
            float a[8], c[8];
            Row8<T>::load(plane_row(src, kg, Ps, G + j * S + r), a);
            T* d = plane_row(dst, kg, Pd, G + img * S + r);
            Row8<T>::load(d, c);
#pragma unroll
            for (int q = 0; q < 8; ++q) c[q] += a[q];
            Row8<T>::store(d, c);
        }
    }
}

template <bool SCATTER>
static int move_images(const void* src, int Bs, int Ps, const int* idx, const int* count,
                       void* dst, int Bd, int Pd, int C, int H, int W, int G, int dtype, void* stream) {
    MPNN_REQUIRE(C % 8 == 0, "gather/scatter: C=%d", C);
    int S = (H + 1) * (W + 1);
    int cap = SCATTER ? Bs : Bd;
    long long total = (long long)(C / 8) * cap * S;
    int grid = (int)((total + 255) / 256);
    if (grid > 148 * 16) grid = 148 * 16;
    if (grid < 1) grid = 1;
    MPNN_DISPATCH_DTYPE(dtype, (move_images_kernel<T, SCATTER><<<grid, 256, 0, (cudaStream_t)stream>>>(
        (const T*)src, Ps, idx, count, (T*)dst, Pd, C / 8, S, G)));
    return mpnn_check_launch(SCATTER ? "scatter_add_images" : "gather_images");
}

extern "C" int mpnn_gather_images(const void* src, int Bs, int Ps, const int* idx, const int* count,
                                  void* dst, int Bd, int Pd, int C, int H, int W, int G, int dtype, void* stream) {
    return move_images<false>(src, Bs, Ps, idx, count, dst, Bd, Pd, C, H, W, G, dtype, stream);
}
extern "C" int mpnn_scatter_add_images(const void* src, int Bs, int Ps, const int* idx, const int* count,
                                       void* dst, int Bd, int Pd, int C, int H, int W, int G, int dtype, void* stream) {
    return move_images<true>(src, Bs, Ps, idx, count, dst, Bd, Pd, C, H, W, G, dtype, stream);
}

// The per-example router feature alpha_cpt * k_cpt of the examples at one node of the compacted walk, in the
// node's compact order: into the fp32 `extra` vector of the CUDA-core heads and / or into the feature column of
// the tcgen05 heads (bf16 with round-to-nearest-even, the rounding of torch's fp32 -> bf16 copy_).
__global__ void __launch_bounds__(256)
gather_feature_kernel(const float* __restrict__ src, const int* __restrict__ orig, const int* __restrict__ count,
                      int n_max, float* __restrict__ dst, void* __restrict__ col, int col_stride, int col_dtype) {
    const int n = count ? min(*count, n_max) : n_max;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
        const float v = src[orig ? orig[j] : j];
        if (dst) dst[j] = v;
        if (col) {
            if (col_dtype == MPNN_BF16)
                static_cast<__nv_bfloat16*>(col)[(size_t)j * col_stride] = __float2bfloat16_rn(v);
            else
                static_cast<float*>(col)[(size_t)j * col_stride] = v;
        }
    }
}

extern "C" int mpnn_gather_feature(const float* src, const int* orig, const int* count, int n, float* dst,
                                   void* col, int col_stride, int col_dtype, void* stream) {
    MPNN_REQUIRE(n >= 0 && (col == nullptr || (col_stride >= 1 && (col_dtype == MPNN_F32 || col_dtype == MPNN_BF16))),
                 "gather_feature: n=%d col_stride=%d col_dtype=%d", n, col_stride, col_dtype);
    if (n == 0 || (dst == nullptr && col == nullptr)) return MPNN_OK;
    MPNN_REQUIRE(src, "gather_feature: NULL src");
    int grid = ceil_div(n, 256);
    if (grid > 148) grid = 148;
    gather_feature_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, orig, count, n, dst, col, col_stride, col_dtype);
    return mpnn_check_launch("gather_feature");
}

// ------------------------------------------------ per-switch compaction (compacted ev-mode evaluator)
// The reference evaluates every node on the whole batch and weights statistics with the one-hot p_ev
// (net_types.py:127-131, train-nets:117-130); in 'ev' mode an example only needs the nodes on its own
// path.  For one switch: dec[b] = first-max argmax of R[b][0..ns) over the n examples present at the
// switch, and for every sink the ascending list of positions (rows of the parent's compact batch) and
// of original example ids that chose it -- ballot + prefix scan, order preserving, one CTA.
__global__ void __launch_bounds__(1024)
route_compact_kernel(const float* __restrict__ R, int ldr, int ns, int n_max, const int* __restrict__ parent_orig,
                     int cap, int* __restrict__ dec, int* __restrict__ pos, int* __restrict__ orig,
                     int* __restrict__ count, const int* __restrict__ n_count) {
    const int n = n_count ? min(max(*n_count, 0), n_max) : n_max;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ int wcount[8][32];
    __shared__ int base_s[8];
    if (threadIdx.x < 8) base_s[threadIdx.x] = 0;
    __syncthreads();
    for (int b0 = 0; b0 < n; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        int d = -1;
        if (b < n) {
            float best = R[(size_t)b * ldr];
            d = 0;
            for (int i = 1; i < ns; ++i) {
                const float v = R[(size_t)b * ldr + i];
                if (v > best) { best = v; d = i; }           // strict: the first maximum wins (tf.argmax)
            }
            if (dec) dec[b] = d;
        }
        unsigned m[8];
        for (int s = 0; s < ns; ++s) {
            m[s] = __ballot_sync(0xffffffffu, d == s);
            if (lane == 0) wcount[s][warp] = __popc(m[s]);
        }
        __syncthreads();
        if (d >= 0) {
            int wbase = 0;
            for (int w = 0; w < warp; ++w) wbase += wcount[d][w];
            const int at = base_s[d] + wbase + __popc(m[d] & ((1u << lane) - 1u));
            pos[(size_t)d * cap + at] = b;
            orig[(size_t)d * cap + at] = parent_orig ? parent_orig[b] : b;
        }
        __syncthreads();
        if (threadIdx.x < ns) {
            int tot = 0;
            for (int w = 0; w < 32; ++w) tot += wcount[threadIdx.x][w];
            base_s[threadIdx.x] += tot;
        }
        __syncthreads();
    }
    if (threadIdx.x < ns) count[threadIdx.x] = base_s[threadIdx.x];
}

extern "C" int mpnn_route_compact_counted(const float* R, int ldr, int ns, int n, const int* parent_orig, int cap,
                                          int* dec, int* pos, int* orig, int* count, const int* n_count, void* stream) {
    MPNN_REQUIRE(R && pos && orig && count && ns >= 1 && ns <= 8 && n >= 0 && cap >= n && ldr >= ns,
                 "route_compact: ns=%d n=%d cap=%d ldr=%d", ns, n, cap, ldr);
    route_compact_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(R, ldr, ns, n, parent_orig, cap, dec, pos, orig, count,
                                                               n_count);
    return mpnn_check_launch("route_compact");
}

extern "C" int mpnn_route_compact(const float* R, int ldr, int ns, int n, const int* parent_orig, int cap,
                                  int* dec, int* pos, int* orig, int* count, void* stream) {
    return mpnn_route_compact_counted(R, ldr, ns, n, parent_orig, cap, dec, pos, orig, count, nullptr, stream);
}

// Leaf statistics of the examples routed to one Softmax + CrossEntropyError classifier: mpnn_leaf_stats_targets
// (heads.cu) with the labels as the correctness target.
extern "C" int mpnn_leaf_stats(const float* Z, int ldz, int n_cls, const float* y, const int* pos, const int* orig,
                               const int* count, int n, double* out, void* stream) {
    return mpnn_leaf_stats_targets(Z, ldz, n_cls, y, y, n_cls, pos, orig, count, n, out, stream);
}
