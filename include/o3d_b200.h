/*
 * o3d_b200.h — C ABI of libo3d_b200.so (hand-written sm_100a kernels for the Open3DSOT hot path).
 *
 * Conventions (SURVEY.md §8b):
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`; the caller owns all buffers,
 *     including scratch and pre-zeroed gradient outputs — nothing is allocated inside;
 *   - float = IEEE fp32, indices = int32, tensors dense row-major in the shape given in the comment;
 *   - `stream` is a cudaStream_t passed as void*; kernels are only enqueued (no synchronisation), so
 *     every entry point may be captured into a CUDA graph;
 *   - no host-side state: what an entry point does depends on its arguments only.  The one exception
 *     is the process-wide force_mt switch of o3d_debug_set(), the library's only mutable global;
 *   - return value 0 = ok, <0 = argument / CUDA error; o3d_last_error() gives the text (thread-local);
 *   - no torch types anywhere.
 *
 * The first block mirrors, one to one, the nine pybind entry points of `pointnet2_ops._ext` that the
 * reference binds at pointnet2/utils/pointnet2_utils.py:17 and calls at :56,:92,:98,:125,:162,:184,:217,
 * :237,:268 (tensor layouts and result conventions identical).  The second block holds the fused
 * supersets used by the B200-native modules (channels-last activations).
 */
#ifndef O3D_B200_H
#define O3D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define O3D_B200_VERSION 100

int o3d_version(void);
const char* o3d_last_error(void);
int o3d_opt_threads(int work);  /* upstream cuda_utils.h opt_n_threads(): defines the FPS tie order */
int o3d_device_sms(void);

/* ------------------------------------------------------------------------------------------------
 * Block 1 — drop-in for pointnet2_ops._ext
 * ---------------------------------------------------------------------------------------------- */

/* _ext.furthest_point_sampling(xyz, npoint)            pointnet2_utils.py:56
 * xyz (B,N,3) f32 -> idx (B,npoint) i32. Starts at index 0, skips points with |p|^2 <= 1e-3,
 * ties resolved exactly as the upstream block reduction does.  N <= 16384.                      */
int o3d_fps(const float* xyz, int B, int N, int npoint, int32_t* idx, void* stream);

/* _ext.gather_points(features, idx)                    pointnet2_utils.py:92
 * features (B,C,N), idx (B,M) -> out (B,C,M)                                                    */
int o3d_gather(const float* features, const int32_t* idx, int B, int C, int N, int M, float* out, void* stream);

/* _ext.gather_points_grad(grad_out, idx, N)            pointnet2_utils.py:98
 * grad_out (B,C,M), idx (B,M) -> grad_features (B,C,N), MUST be zero-filled by the caller       */
int o3d_gather_grad(const float* grad_out, const int32_t* idx, int B, int C, int N, int M, float* grad_features,
                    void* stream);

/* _ext.ball_query(new_xyz, xyz, radius, nsample)       pointnet2_utils.py:268
 * new_xyz (B,M,3), xyz (B,N,3) -> idx (B,M,nsample): first nsample indices in ascending order with
 * d^2 < radius^2 (strict, fp32), remaining slots = first hit, no hit = 0.                        */
int o3d_ball_query(const float* new_xyz, const float* xyz, int B, int N, int M, float radius, int nsample,
                   int32_t* idx, void* stream);

/* _ext.group_points(features, idx)                     pointnet2_utils.py:217
 * features (B,C,N), idx (B,M,S) -> out (B,C,M,S)                                                */
int o3d_group(const float* features, const int32_t* idx, int B, int C, int N, int M, int S, float* out, void* stream);

/* _ext.group_points_grad(grad_out, idx, N)             pointnet2_utils.py:237
 * grad_out (B,C,M,S), idx (B,M,S) -> grad_features (B,C,N), zero-filled by the caller           */
int o3d_group_grad(const float* grad_out, const int32_t* idx, int B, int C, int N, int M, int S, float* grad_features,
                   void* stream);

/* _ext.three_nn(unknown, known)                        pointnet2_utils.py:125
 * unknown (B,n,3), known (B,m,3) -> dist2 (B,n,3) SQUARED distances, idx (B,n,3); ties -> lower index;
 * m < 3 leaves +inf / 0 in the unused slots (upstream 1e40 cast to float).                      */
int o3d_three_nn(const float* unknown, const float* known, int B, int n, int m, float* dist2, int32_t* idx,
                 void* stream);

/* _ext.three_interpolate(features, idx, weight)        pointnet2_utils.py:162
 * features (B,c,m), idx (B,n,3), weight (B,n,3) -> out (B,c,n)                                   */
int o3d_three_interpolate(const float* features, const int32_t* idx, const float* weight, int B, int c, int m, int n,
                          float* out, void* stream);

/* _ext.three_interpolate_grad(grad_out, idx, weight, m) pointnet2_utils.py:184
 * grad_out (B,c,n) -> grad_features (B,c,m), zero-filled by the caller                          */
int o3d_three_interpolate_grad(const float* grad_out, const int32_t* idx, const float* weight, int B, int c, int n,
                               int m, float* grad_features, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Block 2 — fused supersets (channels-last activations: a feature tensor is (B, N, C), so one
 * point's channel vector is one contiguous, 16-byte-aligned row; C % 4 == 0)
 * ---------------------------------------------------------------------------------------------- */

/* QueryAndGroup.forward in one kernel (pointnet2_utils.py:299-339): ball query + xyz grouping +
 * centre subtraction (+ /radius) + feature grouping + concat.
 *   xyz (B,N,3), new_xyz (B,M,3), feat_cl (B,N,C) or NULL (C=0)
 *   -> idx (B,M,S) (may be NULL), grouped_cl (B,M,S,C+4): [features(C) | dx dy dz | 0]
 * (the reference's channel order [xyz, features] is restored by the weight packing of the MLP).  */
int o3d_ballquery_group(const float* xyz, const float* new_xyz, const float* feat_cl, int B, int N, int M, int C,
                        float radius, int nsample, int normalize_xyz, int32_t* idx, float* grouped_cl, void* stream);

/* Backward of the grouping above w.r.t. features and (optionally) coordinates.
 *   grad_grouped_cl (B,M,S,C+4), idx (B,M,S)
 *   -> grad_feat_cl (B,N,C) += ..., grad_xyz (B,N,3) += ..., grad_new_xyz (B,M,3) -= sum_s ...
 * all three accumulated with fp32 reductions (pre-zeroed by caller; any may be NULL).            */
int o3d_ballquery_group_grad(const float* grad_grouped_cl, const int32_t* idx, int B, int N, int M, int C, int S,
                             float radius, int normalize_xyz, float* grad_feat_cl, float* grad_xyz,
                             float* grad_new_xyz, void* stream);

/* PointnetFPModule's three_nn + inverse-distance weights + three_interpolate in one kernel
 * (pointnet2_modules.py:187-195): unknown (B,n,3), known (B,m,3), known_feat_cl (B,m,c)
 *   -> out_cl (B,n,c), idx (B,n,3), weight (B,n,3)  (idx/weight kept for the backward)            */
int o3d_three_nn_interpolate(const float* unknown, const float* known, const float* known_feat_cl, int B, int n, int m,
                             int c, float* out_cl, int32_t* idx, float* weight, void* stream);
int o3d_three_nn_interpolate_grad(const float* grad_out_cl, const int32_t* idx, const float* weight, int B, int n, int m,
                                  int c, float* grad_known_feat_cl, void* stream);

/* BoxAwareXCorr grouping by an explicit (top-k) index list (models/head/xcorr.py:87-90), channels-last:
 * feat_cl (B,N,C), idx (B,L) -> out_cl (B,L,C); the gradient is accumulated into a pre-zeroed (B,N,C).   */
int o3d_group_rows(const float* feat_cl, const int32_t* idx, int B, int N, int L, int C, float* out_cl, void* stream);
int o3d_group_rows_grad(const float* grad_out_cl, const int32_t* idx, int B, int N, int L, int C, float* grad_feat_cl,
                        void* stream);

/* Cross-correlation front ends (models/head/xcorr.py).  The MLP + max-pool behind either of them is a lifted stack
 * (o3d_lift_t below), which also provides the gradient of the BoxAware grouping (indices carry no gradient).
 *
 * o3d_xcorr_boxaware_fwd — BoxAwareXCorr (xcorr.py:81-88: cdist + argsort + [:k]): template_bc (B,M,D), search_bc (B,N,D),
 *   D <= 16, k <= 8 -> idx (B,N,k): the k template points with the nearest box cloud per search point, nearest first,
 *   equal distances in ascending template order; squared distances by direct differences (see csrc/xcorr.cu).
 * o3d_xcorr_p2b_fwd — P2B_XCorr's cosine map (xcorr.py:37-38): tfeat_cl (B,n1,C), sfeat_cl (B,n2,C) channels-last
 *   -> sim (B,n2,n1) = <t_i / max(|t_i|, eps), s_j / max(|s_j|, eps)>; tnorm (B,n1) / snorm (B,n2) (nullable) keep the
 *   norms for the backward.
 * o3d_xcorr_p2b_bwd — dsim (B,n2,n1) -> d_tfeat_cl (B,n1,C), d_sfeat_cl (B,n2,C) (either may be NULL; plain stores).   */
int o3d_xcorr_boxaware_fwd(const float* template_bc, const float* search_bc, int B, int M, int N, int D, int k, int32_t* idx,
                           void* stream);
int o3d_xcorr_p2b_fwd(const float* tfeat_cl, const float* sfeat_cl, int B, int n1, int n2, int C, float eps, float* sim,
                      float* tnorm, float* snorm, void* stream);
int o3d_xcorr_p2b_bwd(const float* dsim, const float* sim, const float* tfeat_cl, const float* sfeat_cl, const float* tnorm,
                      const float* snorm, int B, int n1, int n2, int C, float eps, float* d_tfeat_cl, float* d_sfeat_cl,
                      void* stream);

/* ------------------------------------------------------------------------------------------------
 * Block 3 — point-wise MLP layers (SharedMLP / Seq of the reference: 1x1 conv + BatchNorm + ReLU
 * [+ max-pool over nsample / k / template points]; pointnet2/utils/pytorch_utils.py:12-37,68-121,
 * pointnet2_modules.py:64-73, models/head/xcorr.py:47-51,98-101).
 * Activations are channels-last matrices X[P, ld] (ld % 4 == 0, 16-byte aligned rows); weights are
 * zero-padded to multiples of 4 in both dimensions.  All statistics buffers are fp64, pre-zeroed.
 * ---------------------------------------------------------------------------------------------- */

/* Y[p,n] = sum_k A(X)[p,k] * wt[k,n] (+ bias[n]),  A(v) = relu?(v*in_scale[k] + in_shift[k]) (scale/shift nullable).
 * wt is the TRANSPOSED weight [K, ldw].  Optional outputs: y (raw pre-BN, nullable), sum / sumsq (per-channel
 * batch statistics), and for S > 0 the per-group (S consecutive positions; S | 128, S | P) ymax / ymin / arg
 * (argmax | argmin << 16), each [P/S, ldp].                                                        */
int o3d_pw_fwd(const float* x, int ldx, const float* in_scale, const float* in_shift, int in_relu, const float* wt,
               int ldw, const float* bias, int P, int K, int N, float* y, int ldy, double* sum, double* sumsq, int S,
               float* ymax, float* ymin, int32_t* arg, int ldp, void* stream);

/* The layer's output gradient is given implicitly as  dY = a*g + b + cc*y  (batch-norm backward; a == NULL -> dY = g)
 * with g either dense [P, ldg] or pooled: g[p,c] = (p % S == sel[p/S,c]) ? dpool[p/S,c] : 0.
 * dgrad: out[p,n] = sum_c dY[p,c] * w[c,n]; if yprev != NULL the previous layer's ReLU mask
 *        [yprev*pscale+pshift > 0] is applied and s1 += out, s2y += out*yprev are accumulated.      */
int o3d_pw_dgrad(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                 const float* dpool, const int32_t* sel, int S, int ldp, const float* w, int ldw, int P, int Cout,
                 int Cin, float* out, int ldo, const float* yprev, int ldyp, const float* pscale, const float* pshift,
                 int prelu, double* s1, double* s2y, void* stream);

/* wgrad: dw[m,n] += sum_p dY[p,m] * A(X)[p,n]   (dw pre-zeroed, [Cout, lddw], fp32 reductions)       */
int o3d_pw_wgrad(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                 const float* dpool, const int32_t* sel, int S, int ldp, const float* x, int ldx, const float* in_scale,
                 const float* in_shift, int in_relu, int P, int Cout, int Cin, float* dw, int lddw, void* stream);

/* BatchNorm bookkeeping (torch semantics: biased variance to normalise, unbiased for running_var, momentum
 * update, num_batches_tracked += 1): scale = gamma*invstd, shift = beta - mean*scale.               */
int o3d_bn_fwd_finalize(const double* sum, const double* sumsq, double count, const float* gamma, const float* beta,
                        float* running_mean, float* running_var, long long* num_batches_tracked, float momentum,
                        float eps, int training, int C, float* scale, float* shift, float* mean, float* invstd,
                        void* stream);
/* `training`: bit 0 = batch statistics were used; bit 1 = ACCUMULATE into dgamma / dbeta instead of overwriting them. */
int o3d_bn_bwd_finalize(const double* s1, const double* s2y, double count, const float* gamma, const float* mean,
                        const float* invstd, int training, int C, float* a, float* b, float* cc, float* dgamma,
                        float* dbeta, void* stream);

/* Pooled activation: out[g,c] = relu?(scale*ysel + shift), ysel = scale >= 0 ? ymax : ymin, sel = its position. */
int o3d_pool_finalize(const float* ymax, const float* ymin, const int32_t* arg, const float* scale, const float* shift,
                      int relu, int G, int C, int ldp, float* out, int ldo, int32_t* sel, float* ysel, void* stream);
int o3d_pool_bwd_prep(const float* dout, int ldd, const float* out, int ldo, const float* ysel, int relu, int G, int C,
                      int ldp, float* dpool, double* s1, double* s2y, void* stream);
/* Dense activation and its backward preparation (g = dout * [out > 0], s1 = sum g, s2y = sum g*y).   */
int o3d_act_apply(const float* y, int ldy, const float* scale, const float* shift, int relu, int P, int C, float* out,
                  int ldo, void* stream);
int o3d_dense_bwd_prep(const float* dout, int ldd, const float* out, int ldo, const float* y, int ldy, int relu, int P,
                       int C, float* g, int ldg, double* s1, double* s2y, void* stream);

/* Tensor-core (tcgen05 / TMEM, 3xTF32) variants of o3d_pw_fwd / o3d_pw_dgrad for >= 128 output channels and
 * K >= 32.  The weight operand is passed pre-tiled: o3d_pw_tc_pretile() rewrites a row-major matrix
 * w[rows, ldw] (rows = the GEMM's output channels, K contiguous) into per-(128-row tile, 32-wide k-block)
 * shared-memory images [hi | lo], K-major SWIZZLE_128B, that the kernel streams with cp.async.bulk.
 * forward:  rows = Cout, K = Cin   (w = the padded conv weight)
 * dgrad  :  rows = Cin,  K = Cout  (w = its transpose)                                                */
long long o3d_pw_tc_wtile_bytes(int rows, int K);
/* Measurement switch, process-wide and not synchronised: force_mt = 1 makes every tensor-core GEMM take one 128-channel
 * tile per CTA.  tc_debug must be 0; anything but (0, 0) and (0, 1) returns O3D_ERR_ARG and changes nothing.        */
int o3d_debug_set(int tc_debug, int force_mt);
int o3d_pw_tc_pretile(const float* w, int ldw, int rows, int K, void* wtiles, void* stream);
int o3d_pw_fwd_tc(const float* x, int ldx, const float* in_scale, const float* in_shift, int in_relu, const void* wtiles,
                  const float* bias, int P, int K, int N, float* y, int ldy, double* sum, double* sumsq, int S,
                  float* ymax, float* ymin, int32_t* arg, int ldp, void* stream);
int o3d_pw_dgrad_tc(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                    const float* dpool, const int32_t* sel, int S, int ldp, const void* wtiles_t, int P, int Cout,
                    int Cin, float* out, int ldo, const float* yprev, int ldyp, const float* pscale,
                    const float* pshift, int prelu, double* s1, double* s2y, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Block 4 — a whole MLP stack (SharedMLP / Seq) per call.  The descriptor carries the raw parameter
 * pointers of the reference modules in their checkpoint layout (weight [cout, cin] row-major, BN
 * gamma/beta/running stats); packing, per-layer GEMMs, BN bookkeeping, pooling and — backward —
 * BN-backward, wgrad, dgrad and un-packing of the gradients are all enqueued by one call.
 * ---------------------------------------------------------------------------------------------- */
#define O3D_MAX_LAYERS 8

/* "Lifted" first layer.  When the first 1x1 convolution of a stack acts on GROUPED rows — QueryAndGroup
 * (pointnet2_utils.py:317-329: [xyz(idx) - centre, features(idx)]), BoxAwareXCorr's top-k grouping (xcorr.py:87-90) or
 * P2B_XCorr's [similarity, template xyz, template feature] fusion tensor (xcorr.py:39-46) — its linearity lets the
 * feature part of the convolution run ONCE per source point instead of once per (centre, neighbour) position:
 *     Y0[p, c] = Z[row(p), c] + s[p][0] * u[0][c] + s[p][1] * u[1][c] + s[p][2] * u[2][c] + s[p][3] * u[3][c]
 *       Z = W0_f . source features  (zrows x C0, computed by an ordinary one-layer stack over the source points; optional)
 *       s = up to four per-position scalars with their weight columns u: the relative coordinates (dx, dy, dz) of a set
 *           abstraction layer — applied directly, in the reference's difference-then-multiply form — or P2B's cosine
 *           similarity (optional)
 * Neither the grouped tensor nor Y0 is written to memory: Y0 exists only inside the operand loaders / epilogues of
 * the next layer's GEMMs (tensor-core path), its batch statistics come from one gather pass, and the backward is a
 * scatter of dY0 into dZ / ds / du.  Layer 0 of the descriptor then carries only BatchNorm / ReLU (weight NULL).
 * row(p) = cloud(p) * rows_per_cloud + (ridx ? ridx[p] : p % ridx_mod),  cloud(p) = p / pos_per_cloud.             */
typedef struct o3d_lift_t {
    const float* z;        /* [zrows, ldz], ldz == round4(C0), or NULL (no gathered part)             */
    int ldz;
    const int32_t* ridx;   /* [P] source row of each position, local to its cloud, or NULL            */
    int ridx_mod;          /* used when ridx == NULL                                                  */
    int rows_per_cloud;    /* Z rows per cloud                                                        */
    int pos_per_cloud;     /* positions per cloud                                                     */
    int grp;               /* work unit of the gather / scatter passes: consecutive positions per thread (power of two
                              dividing P; the ball-query group size, so that first-hit padding merges)               */
    const float* s;        /* [P, 4] (unused columns zero) or NULL                                    */
    const float* u;        /* [4, ldz] (unused rows zero) or NULL                                     */
    /* backward outputs (NULL = not wanted), all zero-filled by the caller                           */
    float* d_z;            /* [zrows, ldz]   += scatter of dY0                                        */
    float* d_s;            /* [P, 4]         += dY0 . u[j]                                            */
    float* d_u;            /* [4, ldz]       += sum_p s[p][j] * dY0[p]                                */
} o3d_lift_t;

typedef struct o3d_stack_t {
    int n_layers;   /* 1..O3D_MAX_LAYERS */
    int P;          /* positions (rows of the channels-last input)                               */
    int K0;         /* input row length (multiple of 4, zero padded)                             */
    int S;          /* pooling group size over consecutive positions (0 = dense output)          */
    int training;   /* BatchNorm uses batch statistics and updates the running ones              */
    int use_tc;     /* tcgen05 3xTF32 kernels where the shape qualifies: bit 0 forward + dgrad, bit 1 wgrad;
                       other bits are rejected                                                   */
    int xyz_first;  /* layer-0 weight columns are [xyz(3) | features(c0)], input rows [features | dx dy dz 0] */
    int c0;         /* real feature channels of layer 0 when xyz_first                           */
    int dx_cols;    /* backward: only the first dx_cols input columns need a gradient (0 = all K0) */
    int cin[O3D_MAX_LAYERS], cout[O3D_MAX_LAYERS], relu[O3D_MAX_LAYERS], has_bn[O3D_MAX_LAYERS];
    float momentum[O3D_MAX_LAYERS], eps[O3D_MAX_LAYERS];
    const float* weight[O3D_MAX_LAYERS];
    const float* bias[O3D_MAX_LAYERS];
    const float* gamma[O3D_MAX_LAYERS];
    const float* beta[O3D_MAX_LAYERS];
    float* running_mean[O3D_MAX_LAYERS];
    float* running_var[O3D_MAX_LAYERS];
    long long* num_batches_tracked[O3D_MAX_LAYERS];
    /* backward outputs, same layouts as the parameters (NULL = not wanted) */
    float* d_weight[O3D_MAX_LAYERS];
    float* d_bias[O3D_MAX_LAYERS];
    float* d_gamma[O3D_MAX_LAYERS];
    float* d_beta[O3D_MAX_LAYERS];
    const o3d_lift_t* lift;   /* non-NULL: layer 0 is lifted (weight[0] == NULL, cout[0] = C0, K0 = round4(C0), x unused) */
    int accumulate;           /* backward: d_weight / d_bias / d_gamma / d_beta are ADDED to (the caller's persistent .grad buffers —
                                 saves one elementwise add per parameter and call); 0 = overwritten                            */
    const void* prepared;     /* non-NULL (inference only): parameter block filled by o3d_stack_prepare(); the forward then
                                 neither packs weights nor finalises BatchNorm                                            */
} o3d_stack_t;

long long o3d_stack_workspace_bytes(const o3d_stack_t* d, int backward);
/* Static-weight inference (the B=1 tracking loop): pack the weights / fold the running BN statistics once. */
long long o3d_stack_prepared_bytes(const o3d_stack_t* d);
int o3d_stack_prepare(const o3d_stack_t* d, void* block, void* stream);
/* out: [P or P/S, round4(cout_last)]; ws_fwd must stay alive (untouched) until the backward call. */
int o3d_stack_forward(const o3d_stack_t* d, const float* x, void* ws_fwd, float* out, int keep_for_backward,
                      void* stream);
/* dout: contiguous [rows, round4(cout_last)]; dx: [P, K0] or NULL (columns >= dx_cols are left undefined when
 * dx_cols > 0). */
int o3d_stack_backward(const o3d_stack_t* d, const float* x, const void* ws_fwd, void* ws_bwd, const float* out,
                       const float* dout, float* dx, void* stream);

/* A whole set-abstraction layer in ONE kernel, inference only (running BatchNorm statistics, no saved tensors): replaces the
 * body of _PointnetSAModuleBase.forward — QueryAndGroup (pointnet2/utils/pointnet2_utils.py:299-339), the SharedMLP and the
 * max-pool over nsample (pointnet2/utils/pointnet2_modules.py:58-76) — for one (grouper, mlp) scale.
 * d describes the SharedMLP in the reference's layout: xyz_first = 1, c0 = feature channels C, cin[0] = 3 + C, every cout <= 256,
 * C <= 288; P / K0 / S / training / lift are ignored.  o3d_sa_fused_prepare() packs the weights (pre-tiled TF32 hi | lo images) and
 * folds BatchNorm + bias into per-channel scale / shift once; `block` (o3d_sa_fused_prepared_bytes() bytes) then serves every call.
 * xyz [B, N, 3], new_xyz [B, M, 3], feat_cl [B, N, ldf] channels-last (NULL iff c0 == 0), out [B * M, ldo] channels-last,
 * idx (nullable) [B, M, nsample] receives the ball-query result.  nsample must divide 64 and M be a multiple of 64 / nsample. */
long long o3d_sa_fused_prepared_bytes(const o3d_stack_t* d);
int o3d_sa_fused_prepare(const o3d_stack_t* d, void* block, void* stream);
int o3d_sa_fused_forward(const o3d_stack_t* d, const void* block, const float* xyz, const float* new_xyz, const float* feat_cl,
                         int ldf, int B, int N, int M, float radius, int nsample, int normalize, float* out, int ldo, int32_t* idx,
                         void* stream);

/* Lifted first layer (o3d_lift_t), helpers used by o3d_stack_forward/backward.
 * o3d_lift_stats : gidx[p] = global Z row of position p; sum / sumsq (nullable) += per-channel batch statistics of Y0;
 *                  y0 (nullable) receives Y0 itself [P, C0] (the CUDA-core fallback reads it as an ordinary activation).
 * o3d_lift_scatter: dY0 = a*g + b + cc*Y0 (a == NULL: dY0 = g) scattered into lf->d_z / d_cc / d_s / d_u (see o3d_lift_t);
 *                  y0 NULL = re-gather Y0 from Z.                                                                          */
int o3d_lift_stats(const o3d_lift_t* lf, int P, int C0, int32_t* gidx, float* y0, double* sum, double* sumsq, void* stream);
int o3d_lift_scatter(const o3d_lift_t* lf, int P, int C0, const int32_t* gidx, const float* y0, const float* g, int ldg,
                     const float* a, const float* b, const float* cc, void* stream);

/* wgrad, wide tiles (up to 256 x 256 of dW per CTA, all of TMEM), split over positions; the per-split partial tiles go
 * to `part` (o3d_pw_wgrad_tc2_workspace_floats() floats) and a second kernel adds their sum into dw.              */
long long o3d_pw_wgrad_tc2_workspace_floats(void);
int o3d_pw_wgrad_tc2(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                     const float* dpool, const int32_t* sel, int S, int ldp, const float* x, int ldx,
                     const float* in_scale, const float* in_shift, int in_relu, int P, int Cout, int Cin, float* dw,
                     int lddw, float* part, long long part_floats, void* stream);

/* Adam over a flat fp32 parameter bucket (torch.optim.Adam semantics; the reference uses betas (0.5, 0.999),
 * eps 1e-6: models/base_model.py:28-36).  state = device float[2] {step count (incremented by the call), lr}.  */
int o3d_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float* state,
                  float beta1, float beta2, float eps, float weight_decay, void* stream);

/* Block 5 — box-frame crop of LiDAR scans (tracking frame loop and training-pair construction; replaces the host numpy of
 * datasets/points_utils.py generate_subwindow :223-254, cropAndCenterPC :102-124, crop_pc_axis_aligned :147-173).
 *   local[b,i,:] = R[b]^T (scans[frame[b],i,:] - center[b]);  keep[b,i] = i < count[frame[b]] && |local| < half[b] per axis
 * scans [F,N,3]; count [F] int64 or NULL (all N valid); frame [B] int64 or NULL (frame b = b); rot [B,9] row-major with
 * the box axes in its columns; half [B,3] = (l, w, h) * scale / 2 + offset.                                        */
int o3d_crop_box_frame(const float* scans, const long long* count, const long long* frame, const float* center,
                       const float* rot, const float* half, int B, int N, float* local, unsigned char* keep, void* stream);

/* Fixed-shape resampling of a masked candidate set (datasets/points_utils.py:24-40 regularize_pc, device form): per cloud,
 * n = #keep;  n >= size: the `size` kept candidates with the smallest keys u_perm, in ascending key order (a uniform draw
 * without replacement);  2 < n < size: draw i = the floor(u_pick[i] * n)-th kept candidate;  n <= 2: zeros.
 * points [B, N, 3], keep [B, N] (bytes, non-zero = kept), u_perm [B, N] and u_pick [B, size] uniform in [0, 1),
 * scratch [B, N] int32, out [B, size, 3], src [B, size] int64 (source index of every output point), n_out (nullable) [B] int64.
 * size <= 2048. */
int o3d_resample(const float* points, const unsigned char* keep, const float* u_perm, const float* u_pick, int B, int N, int size,
                 int32_t* scratch, float* out, long long* src, long long* n_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* O3D_B200_H */
