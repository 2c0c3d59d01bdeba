// Dense 'ev'-mode statistics of one chunk on the device (train-nets:111-130 summed over the chunk's examples,
// scripts/lib/desc.py:10-22): the per-example quantities the dense forward already holds in fp32 (p_ev, p_tr,
// d_cor, c_err, R, y) are turned into the fp64 terms of the host reduction and added to a running total.
//
// The reduction order is fixed by the capacity alone: CTA c owns rows [c*ROWS, (c+1)*ROWS), every thread of it sums
// whole columns over those rows in row order (no shuffles, no atomics), and the finishing kernel adds the CTAs'
// partials column by column in CTA order.  Two passes over the same data therefore give the same bits.
#include "common.cuh"
#include "../../include/mpnn.h"

namespace {

constexpr int ROWS = MPNN_STATS_ROWS;
constexpr int THREADS = 256;

struct StatsArgs {
    const mpnn_stats_desc* descs;
    int n_leaf, n_sw, n_cls;
    const float* y;
    const float* node_p_ev;
    const double* ops;
    int n_nodes, B, M;
    double* work;
    double* total;
    const int* count;
};

__device__ __forceinline__ int live_rows(const StatsArgs& a) {
    return a.count ? min(max(*a.count, 0), a.B) : a.B;
}

__global__ void __launch_bounds__(THREADS) stats_partials_kernel(StatsArgs a) {
    const int n = live_rows(a);
    const int r0 = blockIdx.x * ROWS;
    if (r0 >= n) return;                                  // the finishing kernel reads only CTAs with live rows
    const int r1 = min(r0 + ROWS, n);
    const int per_leaf = 4 + 2 * a.n_cls;
    const int leaf_cols = a.n_leaf * per_leaf;
    double* out = a.work + (size_t)blockIdx.x * a.M;
    for (int q = threadIdx.x; q < a.M; q += blockDim.x) {
        double s = 0.0;
        if (q < leaf_cols) {
            const int l = q / per_leaf, k = q - l * per_leaf;
            const mpnn_stats_desc d = a.descs[l];
            if (k == 2) {
                for (int r = r0; r < r1; ++r) s += (double)d.c_err[r];
            } else if (k == 3) {
                if (d.p_tr)
                    for (int r = r0; r < r1; ++r) s += (double)d.p_tr[r];
            } else {
                const bool cor = k == 0 || (k >= 4 && k < 4 + a.n_cls);
                const int c = k < 4 ? -1 : (cor ? k - 4 : k - 4 - a.n_cls);
                for (int r = r0; r < r1; ++r) {
                    const double pe = d.p_ev ? (double)d.p_ev[r] : 1.0;
                    const double dc = (double)d.d_cor[r];
                    double v = cor ? pe * dc : pe * (1.0 - dc);
                    if (c >= 0) v *= (double)a.y[(size_t)r * a.n_cls + c];
                    s += v;
                }
            }
        } else if (q < leaf_cols + a.n_sw) {
            const mpnn_stats_desc d = a.descs[a.n_leaf + (q - leaf_cols)];
            for (int r = r0; r < r1; ++r) {
                double x = 0.0;
                for (int i = 0; i < d.ns; ++i) x += fabs((double)d.R[(size_t)r * d.ns + i]);
                s += x / d.ns;
            }
        } else if (q == leaf_cols + a.n_sw) {              // acc: the leaves' p_ev * d_cor, in table order
            for (int r = r0; r < r1; ++r) {
                double x = 0.0;
                for (int l = 0; l < a.n_leaf; ++l) {
                    const mpnn_stats_desc& d = a.descs[l];
                    x += (d.p_ev ? (double)d.p_ev[r] : 1.0) * (double)d.d_cor[r];
                }
                s += x;
            }
        } else {                                           // moc: every node's p_ev * ops, in node order
            for (int r = r0; r < r1; ++r) {
                double x = 0.0;
                for (int i = 0; i < a.n_nodes; ++i)
                    x += (a.node_p_ev ? (double)a.node_p_ev[(size_t)i * a.B + r] : 1.0) * a.ops[i];
                s += x;
            }
        }
        out[q] = s;
    }
}

__global__ void __launch_bounds__(THREADS) stats_finish_kernel(StatsArgs a) {
    const int n = live_rows(a);
    const int ctas = (n + ROWS - 1) / ROWS;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.M || ctas == 0) return;
    double s = 0.0;
    for (int c = 0; c < ctas; ++c) s += a.work[(size_t)c * a.M + q];
    a.total[q] += s;
}

}  // namespace

extern "C" int mpnn_stats_accumulate(const mpnn_stats_desc* descs, int n_leaf, int n_sw, const float* y, int n_cls,
                                     const float* node_p_ev, const double* ops, int n_nodes, int B,
                                     double* work, double* total, const int* count, void* stream) {
    MPNN_REQUIRE(descs && y && ops && work && total && n_leaf >= 1 && n_sw >= 0 && n_cls >= 1 && n_nodes >= 1 && B >= 1,
                 "stats_accumulate: n_leaf=%d n_sw=%d n_cls=%d n_nodes=%d B=%d", n_leaf, n_sw, n_cls, n_nodes, B);
    const long long M = (long long)n_leaf * (4 + 2 * (long long)n_cls) + n_sw + 2;
    MPNN_REQUIRE(M < (1 << 30), "stats_accumulate: %lld totals", M);
    StatsArgs a{descs, n_leaf, n_sw, n_cls, y, node_p_ev, ops, n_nodes, B, (int)M, work, total, count};
    stats_partials_kernel<<<ceil_div(B, ROWS), THREADS, 0, (cudaStream_t)stream>>>(a);
    int rc = mpnn_check_launch("stats_accumulate");
    if (rc != MPNN_OK) return rc;
    stats_finish_kernel<<<ceil_div((int)M, THREADS), THREADS, 0, (cudaStream_t)stream>>>(a);
    return mpnn_check_launch("stats_accumulate");
}
