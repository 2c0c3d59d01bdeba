/* libmpnn_sm100 -- C ABI of the B200 (sm_100a) hot path of multipath-nn.
 *
 * The reference (MasonMcGill/multipath-nn) has no FFI boundary: its hot path
 * is a TensorFlow graph built by scripts/lib/layer_types.py and
 * scripts/lib/net_types.py and executed by `net.train.run(...)`
 * (scripts/train-nets:141-143) and `session.run(state_tensors)`
 * (scripts/lib/desc.py:17-18).  Each entry point below replaces the TF op
 * call sites named in its comment (paths relative to /root/reference/scripts).
 *
 * Conventions
 *   - every function returns 0 or a negative error code; mpnn_last_error()
 *     gives the text.  Nothing is allocated or freed on behalf of the caller.
 *   - all pointers are DEVICE pointers unless stated; `stream` is a
 *     cudaStream_t passed as void*.
 *   - activations use the "padded planes" layout
 *         T x[C/8][P][8],  row p = G + n*(H+1)*(W+1) + (h+1)*(W+1) + (w+1)
 *     (zero pad row/column 0 of every image block, G zero guard rows in
 *     front, >=192 behind).  dtype: 0 = fp32, 1 = bf16.  C is padded to a
 *     multiple of 8 (16 in bf16 mode).
 *   - feature matrices (inputs of fully-connected heads) use the same
 *     layout with one row per example: T x[F/8][Balloc][8].
 */
#ifndef MPNN_H
#define MPNN_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* Per-step scalars live in a small DEVICE float array `hyp` so that a captured
 * CUDA graph can be replayed with new values (net_types.py:139-145 feeds). */
enum { MPNN_HYP_LR = 0, MPNN_HYP_MU = 1, MPNN_HYP_TAU = 2, MPNN_HYP_EPS = 3,
       MPNN_HYP_KCPT = 4, MPNN_HYP_GSCALE = 5, MPNN_HYP_DRAW = 6 /* bits of a uint32: Dropout draw counter */,
       MPNN_HYP_COUNT = 8 };

const char* mpnn_last_error(void);
int mpnn_version(void);
/* 1 if the tcgen05 (bf16) kernels were compiled in */
int mpnn_has_umma(void);

/* ---- input / weight packing ------------------------------------------- */
/* ToPyramid (lib/layer_types.py:118-125): scale i of the pyramid is
 * x0[:, ::step, ::step, :] (legacy bilinear resize at integer factors).
 * x0 is NHWC fp32 (B,H0,W0,C0); writes the valid pixels of `planes`
 * (H = H0/step, W = W0/step, Cpad channels, extra channels zero). */
int mpnn_pack_input(const float* x0, int B, int H0, int W0, int C0, int step,
                    void* planes, int Cpad, int G, int P, int dtype, void* stream);
/* MultiscaleLLN (lib/layer_types.py:126-147) on the `step`-strided subsample of an RGB image (one pyramid
 * scale): out [B][H0/step][W0/step][3] fp32 = x / (local luminance / local density + eps), Gaussian window of
 * standard deviation sigma and half-width ceil(2 sigma).  Followed by mpnn_pack_input(out, ..., step = 1). */
int mpnn_lln(const float* x0, int B, int H0, int W0, int C0, int step, float sigma, float eps,
             float* out, void* stream);

/* HWIO fp32 conv weights (lib/layer_types.py:158-173) or (n_in,n_chan) FC
 * weights -> packed operand  Wp[tap][Ktot/8][Ntot][8].
 *   mode 0 (forward):  k = k_off + i, n = n_off + o, tap = t
 *   mode 1 (dgrad):    k = k_off + o, n = n_off + i, tap = ntaps-1-t
 * Elements not written (channel padding) must have been zeroed by the caller. */
int mpnn_pack_weights(const float* w, int ntaps, int I, int O, int mode,
                      int k_off, int Ktot, int n_off, int Ntot,
                      void* packed, int dtype, void* stream);

/* mode | 4: the RESIDUAL of the bf16 rounding, w - bf16(w), is packed instead of w ("lo" part of the bf16x3
 * precision mode, see mpnn_split_planes; "mid" part of the bf16x6 mode).
 * mode | 8: the residual of two roundings, w - bf16(w) - bf16(w - bf16(w)) ("lo" part of the bf16x6 mode, see
 * mpnn_split_planes3). */
/* the same for a whole table of tensors in one launch (device array of descriptors);
 * additionally mode 2: ((float*)packed)[n_off + o] = w[o], o < O (fp32 vector copy) */
typedef struct {
    const float* w; void* packed;
    int ntaps, I, O, mode, k_off, Ktot, n_off, Ntot;
} mpnn_pack_desc;
int mpnn_pack_weights_batched(const mpnn_pack_desc* descs, int n, int blocks_per_desc,
                              int dtype, void* stream);

/* fp32 planes -> (hi | lo) bf16 planes with x = hi + lo: src [C/8][P][8] fp32, dst [2*C/8][P][8] bf16, planes
 * [0, C/8) = bf16(x), planes [C/8, 2*C/8) = bf16(x - bf16(x)).  Operand format of the "bf16x3" precision mode:
 * a fp32 product is evaluated on the tensor cores as a_hi*b_hi + a_lo*b_hi + a_hi*b_lo (2^-16 relative) with
 * fp32 accumulation, i.e. mpnn_stencil_gemm with A0 = dst (2C channels), A1 = dst (its first C channels) and
 * weights packed as [hi; hi; lo] along K.  Carries the reference's fp32 arithmetic (lib/layer_types.py:106-107)
 * onto tcgen05 within the 1e-3 tolerance. */
int mpnn_split_planes(const float* src, int C, int P, void* dst, void* stream);

/* three-way split: dst [3*C/8][P][8] bf16 = (hi | mid | lo), hi = bf16(x), mid = bf16(x - hi), lo = bf16(x - hi - mid):
 * 24 significant bits.  Operand format of the "bf16x6" precision mode: a fp32 product is the six bf16 tensor-core
 * products a_h*b_h + a_m*b_h + a_l*b_h + a_h*b_m + a_m*b_m + a_h*b_l (every term of relative size >= 2^-16; what
 * is dropped is <= 2^-23) accumulated in fp32 -- two launches of K = 3C: A0 = dst (3C channels) against weights
 * [hi; hi; hi], then, accumulating, A0 = dst (first 2C channels), A1 = dst (first C) against [mid; mid; lo].
 * This is the tensor-core mode that meets the 1e-3 tolerance on gradients (lib/layer_types.py:106-107 in fp32). */
int mpnn_split_planes3(const float* src, int C, int P, void* dst, void* stream);

/* ---- training-batch augmentation (scripts/lib/data.py:24-34) -------------- */
/* x [N][H][W][C], y [N][n_cls] fp32: the training set resident on the device.  Per output example i
 * (all device int arrays of length B, drawn on the host in the reference's order):
 *   idx[i] sample, flip[i] horizontal mirror, (du[i], dv[i]) row / column shift; pixels shifted in
 *   from outside the image take the per-channel mean of the image.  Writes x_out [B][H][W][C],
 *   y_out [B][n_cls]. */
int mpnn_augment_batch(const float* x, const float* y, int N, int H, int W, int C, int n_cls,
                       const int* idx, const int* flip, const int* du, const int* dv, int B,
                       float* x_out, float* y_out, void* stream);

/* ---- stencil GEMM: tf.nn.conv2d SAME (lib/layer_types.py:106-107,181-185) */
/* out[p][n] = bias[n] + sum_tap sum_k A[p+off(tap)][k] * Wp[tap][k][n]
 * A = concat(A0 (K0 ch), A1 (K1 ch)); columns [0,N0) go to out0, [N0,N0+N1)
 * to out1.  ntaps = 9 (3x3) or 1.  impl: 0 = fp32 SIMT, 1 = tcgen05 (bf16).
 * out_dtype: 0 fp32 planes, 1 bf16 planes, 2 (tcgen05 only) fp32 ROW-MAJOR
 *   out0[row][N0], out1[row][N1] with row = p - G -- used with ntaps = 1,
 *   H = W = 0 (rows = B examples) for the fully-connected heads, whose wide K is
 *   streamed through the pipeline in 32 KB slices.
 * stats (optional): per-CTA partial sums over VALID pixels of out:
 *   stats[cta][0][n] = sum, stats[cta][1][n] = sum of squares; returns the
 *   number of partial rows written through *n_parts (host pointer).
 * Pad rows of the outputs are unspecified. acc0/acc1: add into out. */
int mpnn_stencil_gemm(const void* A0, int K0, const void* A1, int K1,
                      const void* Wp, int ntaps, const float* bias,
                      void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                      int B, int H, int W, int G, int P,
                      float* stats, int stats_cap, int* n_parts,
                      int dtype, int out_dtype, int impl, void* stream);

/* Train-mode BatchNorm statistics fused into their producer ("last CTA finalises").
 * acc: [2*C + 1] doubles, zeroed ONCE at allocation (the kernels leave it zeroed):
 * every CTA adds its partial sums with fp64 atomics and draws a ticket; the last
 * one converts the totals into ss = (gamma*rstd, beta - mean*gamma*rstd),
 * mr = (mean, rstd), updates the running averages (lib/layer_types.py:219-249)
 * and resets acc.  Replaces stats + mpnn_bn_finalize on the training path. */
typedef struct {
    double* acc;
    const float* gamma; const float* beta;
    float* m_avg; float* v_avg;      /* running moments (may be NULL) */
    float* ss; float* mr;            /* outputs, [2][C] each */
    double count;                    /* B*H*W */
    float d; float eps;
    int defer;                       /* 1: the producer only ADDS its partial sums into acc (no ticket, no finalisation, acc is
                                      * not reset: the caller zeroes it once per step); the constants are derived by the
                                      * consumer, mpnn_bn_relu_pool_fwd_acc -- takes the fence / ticket / last-CTA round trips
                                      * (3.4 us) off the dependent-launch chain */
    int reserved;
} mpnn_bn_fuse;
/* mpnn_stencil_gemm (9 taps, single output, no accumulate) + fused BN statistics of `out` */
int mpnn_conv_bn_stats(const void* A0, int K0, const void* A1, int K1,
                       const void* Wp, const float* bias, void* out, int N,
                       int B, int H, int W, int G, int P, const mpnn_bn_fuse* bn,
                       int dtype, int impl, void* stream);

/* the same with accumulation into `out` (acc != 0: out += conv, the statistics are those of the stored
 * values) and an output dtype chosen separately from the operand dtype (0 fp32 planes, 1 bf16 planes); bn may
 * be NULL (no statistics). */
int mpnn_conv_acc_bn_stats(const void* A0, int K0, const void* A1, int K1,
                           const void* Wp, const float* bias, void* out, int N, int acc,
                           int B, int H, int W, int G, int P, const mpnn_bn_fuse* bn,
                           int dtype, int out_dtype, int impl, void* stream);

/* weight gradient of the above:
 *   dW0[tap][k][n] += sum_p A0[p+off][k] * Gd[p][n]   (k < K0real, n < Nreal)
 *   dW1 likewise for A1;  dbias[n] += sum_p Gd[p][n]
 * dW0/dW1/dbias are fp32 HWIO gradient tensors ([tap][Kreal][Nreal]). */
int mpnn_stencil_wgrad(const void* A0, int K0, int K0real, float* dW0,
                       const void* A1, int K1, int K1real, float* dW1,
                       const void* Gd, int N, int Nreal, float* dbias, int ntaps,
                       int B, int H, int W, int G, int P,
                       int dtype, int impl, void* stream);

/* ---- BatchNorm + ReLU + max-pool (lib/layer_types.py:109-110,219-249,196-199) */
/* partial sums -> scale/shift.  train: batch mean / biased var over `count`
 * elements, EMA update of m_avg/v_avg with decay d; else uses the EMAs.
 * ss[0][c] = gamma*rstd, ss[1][c] = beta - mean*gamma*rstd,
 * mr[0][c] = mean, mr[1][c] = rstd. */
int mpnn_bn_finalize(const float* partials, int n_parts, int C, double count,
                     const float* gamma, const float* beta, float* m_avg, float* v_avg,
                     float d, float eps, int train, float* ss, float* mr, void* stream);
/* act = relu(ss0*lin+ss1) on valid pixels (skipped if act==NULL);
 * pooled = 2x2/2 max of lin, written in the (H/2,W/2) geometry (if !NULL);
 * feat[(h*W+w)*(C/8)+kg][n][8] = act (if !NULL; the LinTrans flatten order). */
int mpnn_bn_relu_pool_fwd(const void* lin, int C, int B, int H, int W, int G, int P,
                          const float* ss, void* act, void* pooled, int Pp,
                          void* feat, int Balloc, int dtype, void* stream);
/* mpnn_bn_relu_pool_fwd with the train-mode constants derived IN the kernel from the totals a producer launched with
 * bn->defer = 1 has accumulated in bn->acc: every thread recomputes scale / shift of its 8 channels (2 doubles each),
 * one CTA per plane writes bn->ss, bn->mr and updates the running moments (lib/layer_types.py:231-238). */
int mpnn_bn_relu_pool_fwd_acc(const void* lin, int C, int B, int H, int W, int G, int P,
                              const mpnn_bn_fuse* bn, void* act, void* pooled, int Pp,
                              void* feat, int Balloc, int dtype, void* stream);
/* backward, pass 1: partial sums of dy' and dy'*(x - mean) (dy' = relu-masked sum
 * of dAct and dFeat; centred so that nothing cancels against mean * sum dy'); *n_parts rows written. */
int mpnn_bn_bwd_reduce(const void* lin, const void* dAct, const void* dFeat, int Balloc,
                       const float* ss, const float* mr, int C,
                       int B, int H, int W, int G, int P,
                       float* partials, int cap, int* n_parts, int dtype, void* stream);
/* the same reduction with the finalisation fused (last CTA): writes sums[2][C] and adds
 * dgamma / dbeta; acc as in mpnn_bn_fuse.  Replaces bn_bwd_reduce + bn_bwd_finalize. */
typedef struct { double* acc; float* sums; float* dgamma; float* dbeta; } mpnn_bn_bwd_fuse;
int mpnn_bn_bwd_reduce_fused(const void* lin, const void* dAct, const void* dFeat, int Balloc,
                             const float* ss, const float* mr, int C,
                             int B, int H, int W, int G, int P,
                             const mpnn_bn_bwd_fuse* f, int dtype, void* stream);
/* Data gradient of a 3x3 conv with the BatchNorm-backward reduction of the layer BELOW fused into its
 * epilogue (tcgen05 path only; replaces mpnn_bn_bwd_reduce_fused over (lin, dAct) for that layer):
 *   out0[p][n] (n < N0) = dAct of the parent activation, out1 (N1 columns) = gradient wrt the pooled
 *   predecessor, as in mpnn_stencil_gemm(Gd, K, NULL, 0, Wp, 9, NULL, out0, N0, 0, out1, N1, 0, ...);
 *   with dy' = out0 * [ss0*lin + ss1 > 0] (lin, ss, mr: pre-BN output and constants of the parent's
 *   BatchNorm, N0 channels) the kernel accumulates sum dy' and sum dy'*(lin - mean) over the valid pixels and the
 *   last CTA writes f.sums / adds f.dgamma, f.dbeta exactly like mpnn_bn_bwd_reduce_fused.
 * TF autodiff of lib/layer_types.py:181-185 and :219-249. */
typedef struct {
    const void* lin; const float* ss; const float* mr;
    mpnn_bn_bwd_fuse f;
} mpnn_bn_bwd_epi;
int mpnn_conv_dgrad_bn_reduce(const void* Gd, int K, const void* Wp, void* out0, int N0, void* out1, int N1,
                              int B, int H, int W, int G, int P, const mpnn_bn_bwd_epi* epi,
                              int dtype, int impl, void* stream);

/* partials (from bn_bwd_reduce) hold sum dy' and sum dy'*(x - mean) per channel;
 * sums[0][c] = sum dy', sums[1][c] = sum dy'*xhat; dgamma += sums1, dbeta += sums0 */
int mpnn_bn_bwd_finalize(const float* partials, int n_parts, int C, const float* mr,
                         float* sums, float* dgamma, float* dbeta, void* stream);
/* backward, pass 2: dLin = ss0*(dy' - mean(dy') - xhat*mean(dy'*xhat))
 *                        + unpool(dPooled)   [argmax recomputed from lin]
 * ss==NULL: BN branch absent (dead scale) -> only the unpool term. */
int mpnn_bn_relu_pool_bwd(const void* lin, const void* dAct, const void* dFeat, int Balloc,
                          const void* dPooled, int Pp,
                          const float* ss, const float* mr, const float* sums, double count,
                          int C, int B, int H, int W, int G, int P,
                          void* dLin, float* dbias /* += column sums of dLin, or NULL */,
                          int dtype, void* stream);
#define MPNN_BN_SMALL_MAX_PIXELS 8192
/* small tensors (B*H*W <= MPNN_BN_SMALL_MAX_PIXELS, no pooled output): the train-mode statistics of `lin`
 * (lib/layer_types.py:219-249: batch moments, running-average update, scale / shift) AND mpnn_bn_relu_pool_fwd in
 * ONE launch -- replaces the statistics riding on the conv launch (mpnn_conv_bn_stats) for tensors whose conv would
 * otherwise end in a chain of atomics, a ticket and a last-CTA finalisation.  Writes ss / mr like mpnn_bn_finalize. */
int mpnn_bn_fwd_small(const void* lin, int C, int B, int H, int W, int G, int P,
                      const float* gamma, const float* beta, float* m_avg, float* v_avg,
                      float d, float eps, float* ss, float* mr,
                      void* act, void* feat, int Balloc, int dtype, void* stream);
/* small tensors (B*H*W <= MPNN_BN_SMALL_MAX_PIXELS, no pooling branch): mpnn_bn_bwd_reduce_fused and
 * mpnn_bn_relu_pool_bwd in ONE launch -- an 8-CTA cluster per 8-channel plane keeps its pixels in registers and
 * exchanges the per-channel sums through distributed shared memory.  sums (optional) / dgamma / dbeta as in
 * mpnn_bn_bwd_fuse; same results as the two-pass pair (fp64 sums across CTAs, fixed order). */
int mpnn_bn_bwd_small(const void* lin, const void* dAct, const void* dFeat, int Balloc,
                      const float* ss, const float* mr, int C, int B, int H, int W, int G, int P,
                      float* sums, float* dgamma, float* dbeta, double count,
                      void* dLin, float* dbias, int dtype, void* stream);

/* ---- heads: LinTrans / Softmax / CrossEntropyError (lib/layer_types.py:39-53,81-84,262-272) */
/* Z[b][j] = sum_f X[f][b] W[f][j] (+ extra[b]*W[F][j]) + bias[j] */
int mpnn_fc_fwd(const void* X, int F, int Balloc, int B, const float* W, const float* bias,
                const float* extra, int n, float* Z, int dtype, void* stream);
/* dX[f][b] = sum_j dZ0[b][j] W0[f][j] (+ dZ1 W1) */
int mpnn_fc_bwd_data(const float* dZ0, const float* W0, int n0,
                     const float* dZ1, const float* W1, int n1,
                     int F, int Balloc, int B, void* dX, int dtype, void* stream);
/* dW[f][j] += sum_b X[f][b] dZ[b][j]; dW[F][j] += sum_b extra[b] dZ[b][j]; db[j] += sum_b dZ[b][j] */
int mpnn_fc_bwd_weight(const void* X, int F, int Balloc, int B, const float* extra,
                       const float* dZ, int n, float* dW, float* db, int dtype, void* stream);
/* prob = softmax(Z); c_err = -sum y log(eps/n + (1-eps) prob); d_cor = [argmax prob == argmax y]
 * (first maximal index). */
int mpnn_softmax_ce_fwd(const float* Z, int ldz /* row stride of Z */, const float* y, int B, int n, float eps,
                        float* prob, float* c_err, float* d_cor, void* stream);
/* dZ[b][j] = coef[b]*coef_scale * d c_err[b] / d Z[b][j]   (coef==NULL -> 1).
 * Outputs (each optional): dZ fp32 [B][n]; dZp two bf16 planes [2][Balloc][8]
 * (columns >= n zero; operand of the tcgen05 head GEMMs); dbias += column sums. */
int mpnn_softmax_ce_bwd(const float* prob, const float* y, int B, int n, float eps,
                        const float* coef, float coef_scale, float* dZ,
                        void* dZp, int Balloc, float* dbias, void* stream);
/* SquaredError (lib/layer_types.py:255-260) on the LinTrans output x = Z: c_err = sum_j (x - y)^2,
 * d_cor = [argmax x == argmax y]; out [B][n] = dense copy of x (read by the backward).
 * Backward: dZ = coef*coef_scale * 2 (x - y), outputs as in mpnn_softmax_ce_bwd. */
int mpnn_squared_err_fwd(const float* Z, int ldz, const float* y, int B, int n,
                         float* out, float* c_err, float* d_cor, void* stream);
int mpnn_squared_err_bwd(const float* out, const float* y, int B, int n,
                         const float* coef, float coef_scale, float* dZ,
                         void* dZp, int Balloc, float* dbias, void* stream);
/* SuperclassCrossEntropyError (lib/layer_types.py:274-285): y_sup [B][n_sup] = y [B][n_cls] @ w_cls [n_cls][n_sup];
 * the loss is mpnn_softmax_ce_fwd / _bwd with y_sup in place of y and n = n_sup. */
int mpnn_superclass_targets(const float* y, const float* w_cls, int B, int n_cls, int n_sup,
                            float* y_sup, void* stream);

/* MaxPool (lib/layer_types.py:86-94), 2x2 window and step 2 -- with the reference's swapped (ksize, strides)
 * arguments the one configuration where window = `stride` and step = `supp` coincide -- on a padded-planes
 * tensor: out (planes at H/2 x W/2, Pp rows per plane) and / or feat, the flattened (h, w, c) feature layout
 * [F/8][Balloc][8] of the pooled tensor.  Backward: dx = (dout + dfeat) at the first maximum of each 2x2 block,
 * zero elsewhere (all of dx is written).  TF autodiff of tf.nn.max_pool. */
int mpnn_maxpool2_fwd(const void* x, int C, int B, int H, int W, int G, int P,
                      void* out, int Pp, void* feat, int Balloc, int dtype, void* stream);
int mpnn_maxpool2_bwd(const void* x, const void* dout, const void* dfeat, int Balloc,
                      int C, int B, int H, int W, int G, int P, int Pp, void* dx, int dtype, void* stream);
/* GlobalMaxPool (lib/layer_types.py:96-100): feat [C/8][Balloc][8] = max over the image, arg (int32, same shape)
 * = h * W + w of the first maximum; backward scatters dfeat to the recorded positions (all of dx is written). */
int mpnn_global_maxpool_fwd(const void* x, int C, int B, int H, int W, int G, int P,
                            void* feat, int* arg, int Balloc, int dtype, void* stream);
int mpnn_global_maxpool_bwd(const void* dfeat, const int* arg, int Balloc, int C, int B, int H, int W,
                            int G, int P, void* dx, int dtype, void* stream);

/* ActivityError (lib/layer_types.py:287-293): cost[b] = alpha * sum_{h,w,c} x^2 (a per-example c_mod);
 * backward: dx (+)= scale * coef[b] * x (scale = 2 alpha / B; coef = the node's p_tr row, NULL: 1;
 * acc = 0 writes dx on the image pixels, acc != 0 adds to it). */
int mpnn_activity_fwd(const void* x, int C, int B, int H, int W, int G, int P, float alpha,
                      float* cost, int dtype, void* stream);
int mpnn_activity_bwd(const void* x, int C, int B, int H, int W, int G, int P, const float* coef,
                      float scale, void* dx, int acc, int dtype, void* stream);

/* Dropout (lib/layer_types.py:212-217; tf.nn.dropout(x, keep), every mode): x *= m / keep in place, m from a
 * counter-based hash of (seed, hyp[MPNN_HYP_DRAW], NHWC element index) -- see csrc/activity.cu.  x is a planes
 * tensor (feat = 0) or its flattened feature copy [H*W*C/8][Balloc][8] (feat = 1): both see the same mask.
 * The backward pass is the same call on the gradient. */
int mpnn_dropout(void* x, int C, int B, int H, int W, int G, int P, int feat, int Balloc,
                 float keep, unsigned seed, const float* hyp, int dtype, void* stream);

/* Router tail (arch_and_hypers.py:45-49): BN -> ReLU -> FC(16) -> BN -> ReLU -> FC(ns)
 * applied to Z1 = output of the first router FC.  One CTA.
 * bn{1,2}: gamma,beta,m_avg,v_avg (C=16 each). save: >= 4*C floats (mean1,rstd1,mean2,rstd2). */
int mpnn_router_tail_fwd(const float* Z1, int B, int C,
                         const float* g1, const float* b1, float* m1, float* v1,
                         const float* W2, const float* bias2,
                         const float* g2, const float* b2, float* m2, float* v2,
                         const float* W3, const float* bias3, int ns,
                         float d, float eps, int train,
                         float* Z2, float* R, float* save, void* stream);
/* gradients are ACCUMULATED into dW*, db*, dg*, dbt*; dZ1 is written. */
int mpnn_router_tail_bwd(const float* Z1, const float* Z2, const float* dR, int B, int C, int ns,
                         const float* g1, const float* b1, const float* W2,
                         const float* g2, const float* b2, const float* W3,
                         const float* save,
                         float* dg1, float* dbt1, float* dW2, float* dbias2,
                         float* dg2, float* dbt2, float* dW3, float* dbias3,
                         float* dZ1, float* scratch /* >= 2*B*C */, void* stream);

/* All routers of a net in one launch (one CTA per router); descriptors are a
 * DEVICE array.  Semantics per element as in the two functions above. */
typedef struct {
    const float* Z1; const float* g1; const float* b1; float* m1; float* v1;
    const float* W2; const float* bias2; const float* g2; const float* b2; float* m2; float* v2;
    const float* W3; const float* bias3; float* Z2; float* R; float* save;
    int ns; int reserved;
} mpnn_router_fwd_desc;
int mpnn_router_tail_fwd_batched(const mpnn_router_fwd_desc* descs, int n, int B, int C,
                                 float d, float eps, int train, void* stream);
typedef struct {
    const float* Z1; const float* Z2; const float* dR;
    const float* g1; const float* b1; const float* W2; const float* g2; const float* b2;
    const float* W3; const float* save;
    float* dg1; float* dbt1; float* dW2; float* dbias2; float* dg2; float* dbt2; float* dW3; float* dbias3;
    float* dZ1; float* scratch;
    void* dZ1p;        /* optional: dZ1 also as two bf16 planes [2][Balloc][8] */
    float* dbias1;     /* optional: += column sums of dZ1 (bias of the first router FC) */
    int ns; int Balloc;
} mpnn_router_bwd_desc;
int mpnn_router_tail_bwd_batched(const mpnn_router_bwd_desc* descs, int n, int B, int C, void* stream);

/* tcgen05 weight gradient of the heads sharing one feature matrix X
 * ([F/8][Balloc][8] bf16; Balloc a multiple of 128), dZ as bf16 planes [N/8][Balloc][8]:
 *   dWa[f][j] += sum_b X[f][b] dZ[b][j]            (f < Fa, j < na)   LogReg
 *   dWb[f][j] += sum_b X[f][b] dZ[b][Nsplit + j]   (f < Fb, j < nb)   first router FC */
int mpnn_fc_wgrad(const void* X, int F, int Balloc, int B, const void* dZ, int N, int Nsplit,
                  float* dWa, int Fa, int na, float* dWb, int Fb, int nb, void* stream);

/* ---- routing (lib/net_types.py:108-131,193-243) ------------------------ */
/* Tree tables (device int/float arrays, nodes in preorder, node 0 = root):
 *   parent[i], sink_idx[i] (position among parent's sinks), n_sinks[i],
 *   floor[i] = n_leaves(i)/n_leaves(root) (multiplied by hyp[EPS] on device),
 *   sw[i] = switch slot or -1,
 *   ops[i] = n_ops + router.n_ops, err[i] = leaf slot or -1.
 * logits: R[slot] -> float* table (device array of pointers), each [B][n_sinks].
 * Outputs p_tr, p_ev: [n_nodes][B]; dec: [n_switch][B] int32 (argmax, first max). */
int mpnn_route_fwd(const int* parent, const int* sink_idx, const int* n_sinks,
                   const float* floor_, const int* sw, int n_nodes,
                   const float* const* R, const float* hyp, int B,
                   float* p_tr, float* p_ev, int* dec, void* stream);
/* Actor (critic=0): gradient of c_tot wrt router logits and per-leaf CE
 * coefficients (net_types.py:167-177):
 *   coef[slot][b] = p_tr[leaf][b]
 *   dR[slot][b][i] = d/dR of mean_b( sum_l p_tr(c_err + k_cpt ops) + sg(p_tr) k_dec |R|^2 )
 * Critic (critic=1; net_types.py:201-243,275-280): also computes c_ev/c_opt
 * bottom-up and dR = p_tr/B * 2 k_cre (R_i + target_i).
 *   c_err: table of per-leaf [B] arrays; d_cor likewise (use_cls_err).
 *   scratch: >= 3*n_nodes*B floats. */
int mpnn_route_bwd(const int* parent, const int* sink_idx, const int* n_sinks,
                   const int* child /* [n_nodes][8] child node per sink */,
                   const float* floor_, const int* sw, const float* ops, const int* err,
                   int n_nodes, const float* const* R, const float* hyp, int B,
                   const float* p_tr, const float* p_ev,
                   const float* const* c_err, const float* const* d_cor,
                   const float* k_cpt /* [B] or NULL -> hyp[KCPT] */,
                   int critic, float k_dec, float k_cre, int optimistic, int use_cls_err,
                   float* const* dR, float* scratch, float* c_data /* [B] per-example cost or NULL */,
                   void* stream);
/* per-node batch moments of p_tr: stats[i][0] = mean p_tr^2, stats[i][1] = mean p_tr */
int mpnn_node_moments(const float* p_tr, int n_nodes, int B, float* stats, void* stream);

/* Path compaction: for every node, the ascending list of examples with
 * p_ev == 1 (ballot + prefix scan); idx[node][B], count[node]. */
int mpnn_compact_paths(const float* p_ev, int n_nodes, int B, int* idx, int* count, void* stream);
/* gather / scatter-add whole image blocks between padded-planes tensors:
 * dst image j <- src image idx[j] (gather); dst image idx[j] += src image j (scatter). */
int mpnn_gather_images(const void* src, int Bs, int Ps, const int* idx, const int* count,
                       void* dst, int Bd, int Pd, int C, int H, int W, int G, int dtype, void* stream);
int mpnn_scatter_add_images(const void* src, int Bs, int Ps, const int* idx, const int* count,
                            void* dst, int Bd, int Pd, int C, int H, int W, int G, int dtype, void* stream);

/* ---- compacted ev-mode evaluation (statistics of scripts/lib/desc.py:10-36, train-nets:111-130) ----
 * One switch of the tree on the n examples present at it: dec[b] = first-max argmax of R[b][0..ns)
 * (R row-major, row stride ldr); for every sink s the ascending list of the rows of this compact batch
 * that chose it (pos[s][.]), their original example ids (orig[s][.] = parent_orig[pos] or pos itself when
 * parent_orig is NULL) and count[s].  pos / orig have row stride cap >= n.  dec may be NULL. */
int mpnn_route_compact(const float* R, int ldr, int ns, int n, const int* parent_orig, int cap,
                       int* dec, int* pos, int* orig, int* count, void* stream);
/* Statistics of one classifier over the examples routed to it: Z row-major logits of the parent's compact
 * batch (row stride ldz), y dense one-hot labels [B][n_cls] indexed by ORIGINAL example id; the examples are
 * rows pos[j] / ids orig[j], j < *count (count NULL -> j < n; pos / orig NULL -> identity).
 *   out[0] += #correct, out[1] += #incorrect, out[2 + c] += sum cor*y[c], out[2 + n_cls + c] += sum (1-cor)*y[c]
 * (p_cor, p_inc, p_cor_by_cls, p_inc_by_cls of train-nets:121-124 summed over the batch; out is double). */
int mpnn_leaf_stats(const float* Z, int ldz, int n_cls, const float* y, const int* pos, const int* orig,
                    const int* count, int n, double* out, void* stream);
/* Routed inference: the results of the examples that exit at one classifier.  Rows pos[j] of the logits Z
 * (row stride ldz) of the parent's compact batch, original ids orig[j], j < *count (count NULL -> j < n;
 * pos / orig NULL -> identity; the grid covers n, so *count <= n):
 *   prob[orig[j]][c] = softmax(Z[pos[j]])[c]     (c < n_cls <= 32; the same bits as mpnn_softmax_ce_fwd)
 *   cls[orig[j]]     = first argmax of that row of prob
 *   exit_id[orig[j]] = leaf,   ops[orig[j]] = path_ops
 * n == 0 is a no-op. */
int mpnn_leaf_emit(const float* Z, int ldz, int n_cls, const int* pos, const int* orig, const int* count, int n,
                   int leaf, double path_ops, float* prob, int* cls, int* exit_id, double* ops, void* stream);
/* The per-example router feature through the compaction: dst[j] = src[orig[j]] for j < *count (count NULL ->
 * j < n; orig NULL -> identity; dst may be NULL), and, when col != NULL, the same value into the strided column
 * col[j * col_stride] of dtype col_dtype (0 fp32, 1 bf16 rounded to nearest even, like torch's copy_). */
int mpnn_gather_feature(const float* src, const int* orig, const int* count, int n, float* dst,
                        void* col, int col_stride, int col_dtype, void* stream);

/* ---- optimiser: minimize_expectation + MomentumOptimizer (lib/net_types.py:24-37) */
/* For segment s covering theta[seg_start[s] : seg_start[s+1]):
 *   g = grad*hyp[GSCALE] + 2*seg_l2[s]*coef*theta,  coef = node mean p_tr (1 if node_stats==NULL)
 *   g *= seg_mult[s] / sqrt(node mean p_tr^2)       (TALR; skipped if !talr or node_stats==NULL)
 *   a = mu*a + g ; theta -= lr*a
 * seg_node[s] = preorder node index. */
int mpnn_talr_momentum_step(float* theta, const float* grad, float* accum, int n,
                            const int* seg_start, const int* seg_node, const float* seg_mult,
                            const float* seg_l2, int n_seg, const float* node_stats, int talr,
                            const float* hyp /* LR, MU, GSCALE */, void* stream);

/* ---- data-parallel gradient all-reduce (NCCL over NVLink / NVSwitch) ------------------------------
 * The reference is single-process (scripts/train-nets:159-164).  Data parallelism shards the batch over one
 * process per GPU; the one collective of a step sums the flat fp32 buffer [gradients | per-node TALR moments]
 * in place (the 1/world factor is applied by mpnn_talr_momentum_step through hyp[GSCALE]).
 *   comm      an ncclComm_t (as void*): either one the host application already owns, or one made here:
 *             rank 0 calls mpnn_comm_unique_id, ships the 128 bytes to the other ranks, then EVERY rank calls
 *             mpnn_comm_init_rank (collective; binds to the current CUDA device).
 * NCCL is resolved at run time from the copy already loaded in the process (else libnccl.so.2 /
 * $MPNN_NCCL_LIB); mpnn_nccl_version() returns 0 when none is available.  The launch is asynchronous on
 * `stream` and may be captured into a CUDA graph. */
int mpnn_nccl_version(void);
int mpnn_comm_unique_id(void* id128 /* host, 128 bytes */);
int mpnn_comm_init_rank(void** comm /* host, out */, int world, int rank, const void* id128 /* host */);
int mpnn_comm_destroy(void* comm);
int mpnn_allreduce_flat(void* comm, float* buf, long long n, void* stream);

/* ---- the data-parallel step tail as ONE kernel over NVLink peer memory ----------------------------------
 * Replaces mpnn_allreduce_flat + mpnn_talr_momentum_step (lib/net_types.py:24-37,96-97,178-181 on the batch
 * sharded over one process per GPU of a node): gradient reduce-scatter by peer loads, TALR + momentum on the
 * owned slice, all-gather of theta / momentum (and of the reduced gradient when write_back != 0) by peer
 * stores, two flag exchanges -- see csrc/p2p.cu.
 *   exchange buffer   one per rank, from mpnn_p2p_alloc (cudaMalloc, zero-filled):
 *                     [MPNN_P2P_FLAG_BYTES of flags | grad (g0 moments + n, padded to 4) | theta | accum],
 *                     the three vectors at 16-byte-aligned byte offsets off_*; identical layout on every rank.
 *   mapping           every rank exports its buffer (mpnn_p2p_export -> MPNN_P2P_HANDLE_BYTES, a
 *                     cudaIpcMemHandle_t), ships the handle to the other ranks of the node, and maps theirs with
 *                     mpnn_p2p_import; base[r] is rank r's buffer as seen from this process (base[rank]: local).
 *   the call          collective: every rank launches it once per step on its own stream (it may be captured
 *                     into a CUDA graph); seg_* / hyp / talr as in mpnn_talr_momentum_step, use_stats = the net
 *                     has per-node moments in grad[0:g0).  [lo, hi) is the range of parameters the call handles
 *                     (multiples of 4; hi <= 0: up to the end) and `channel` (0..3) the flag set it uses: a step
 *                     may issue the deep-stage parameters early, under the rest of the backward pass, and the
 *                     remainder at its end, on different channels.  Waits are bounded: a peer that never arrives
 *                     sets a status word (mpnn_p2p_status != 0) instead of hanging the device. */
#define MPNN_P2P_MAX 16
#define MPNN_P2P_HANDLE_BYTES 64
#define MPNN_P2P_FLAG_BYTES 4096
typedef struct {
    void* base[MPNN_P2P_MAX];
    int world, rank;
    long long off_grad, off_theta, off_accum;
    int g0, n;
} mpnn_p2p_desc;
int mpnn_p2p_alloc(void** ptr /* host, out */, long long bytes);
int mpnn_p2p_free(void* ptr);
int mpnn_p2p_export(void* ptr, void* handle64 /* host, out */);
int mpnn_p2p_import(const void* handle64 /* host */, void** ptr /* host, out */);
int mpnn_p2p_close(void* ptr);
int mpnn_p2p_status(const void* local_base, int* status /* host, out */);
int mpnn_allreduce_talr_p2p(const mpnn_p2p_desc* d /* host */, const int* seg_start, const int* seg_node,
                            const float* seg_mult, const float* seg_l2, int n_seg, int use_stats, int talr,
                            const float* hyp, int write_back, int lo, int hi, int channel, void* stream);

/* ---- counted launches: the live batch in device memory ------------------------------------------------------
 * Each entry point below is the one named without `_counted`, plus `count`: a DEVICE int holding the live batch m.
 * The batch argument B (n for mpnn_route_compact) becomes the capacity the grid is sized for; the call processes
 * the first min(*count, B) examples exactly as the uncounted call with batch m would (bit for bit: the launch
 * variants are chosen from the capacity and do the same per-row arithmetic), and writes nothing at or past them.
 * m = 0 is valid.  count == NULL is the uncounted call.  A stream-ordered walk whose batch sizes are produced on
 * the device (mpnn_route_compact's count) can so be launched, and captured into a CUDA graph, without reading
 * them back to the host.
 *   mpnn_stencil_gemm_counted: no statistics (stats == NULL).  Rows are pixels: q < m * (H+1)(W+1).
 *   mpnn_router_tail_fwd_batched_counted: train == 0 only (train-mode moments are batch statistics).
 *   mpnn_route_compact_counted: n_count is the count of the parent's compact batch (its `count` is the output). */
int mpnn_pack_input_counted(const float* x0, int B, int H0, int W0, int C0, int step,
                            void* planes, int Cpad, int G, int P, int dtype, const int* count, void* stream);
int mpnn_stencil_gemm_counted(const void* A0, int K0, const void* A1, int K1,
                              const void* Wp, int ntaps, const float* bias,
                              void* out0, int N0, int acc0, void* out1, int N1, int acc1,
                              int B, int H, int W, int G, int P,
                              float* stats, int stats_cap, int* n_parts,
                              int dtype, int out_dtype, int impl, const int* count, void* stream);
int mpnn_bn_relu_pool_fwd_counted(const void* lin, int C, int B, int H, int W, int G, int P,
                                  const float* ss, void* act, void* pooled, int Pp,
                                  void* feat, int Balloc, int dtype, const int* count, void* stream);
int mpnn_fc_fwd_counted(const void* X, int F, int Balloc, int B, const float* W, const float* bias,
                        const float* extra, int n, float* Z, int dtype, const int* count, void* stream);
int mpnn_router_tail_fwd_batched_counted(const mpnn_router_fwd_desc* descs, int n, int B, int C,
                                         float d, float eps, int train, const int* count, void* stream);
int mpnn_route_compact_counted(const float* R, int ldr, int ns, int n, const int* parent_orig, int cap,
                               int* dec, int* pos, int* orig, int* count, const int* n_count, void* stream);
/* mpnn_split_planes3 on the live images of a padded-planes tensor of geometry (B, H, W, G, P) and C channels: rows
 * [0, G + m*(H+1)*(W+1)) of each of the C/8 planes, m = min(*count, B), with the same bits as the whole-tensor call;
 * the rest of dst is not written, and m = 0 writes nothing.  Rows past the live images may keep a larger earlier
 * batch's values: the row after the last live image is a pad row, zero in src and dst, so no 3x3 conv of a live
 * image reads them.  Unlike the entry points above it takes the geometry (the uncounted call takes only P). */
int mpnn_split_planes3_counted(const float* src, int C, int B, int H, int W, int G, int P, void* dst,
                               const int* count, void* stream);

/* ---- tcgen05 bring-up probe (tests only) -------------------------------- */
/* D[128][N] = A[128][K] * B[N][K]^T through one CTA of tcgen05.mma; all
 * operands in the interleaved (no-swizzle) core-matrix layout. */
int mpnn_umma_selftest(const void* A, int a_bytes, int a_off, const void* Bm, int b_bytes,
                       float* D, int N, int K, int a_mn_major, int b_mn_major,
                       int lbo_a, int sbo_a, int lbo_b, int sbo_b, void* stream);

#ifdef __cplusplus
}
#endif
#endif
