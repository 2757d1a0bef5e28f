// Host-side orchestration of a whole MLP stack (SharedMLP / Seq of the reference) in ONE C-ABI call per direction.
//
// Python dispatch cost dominated the first fused version (hundreds of tiny torch ops per step just to pad / transpose
// weights and slice workspaces), so the per-layer sequencing lives here: the caller hands over one descriptor with the
// raw parameter pointers of the reference modules (weights in their checkpoint layout), one workspace buffer, and gets
// every kernel of the stack enqueued on the stream: weight packing, per-layer GEMM (+tcgen05 variant), batch-norm
// finalisation, pooling / activation, and on the way back the BN-backward finalisation, wgrad, dgrad and the
// un-packing of the weight gradients into the checkpoint layout.  Nothing is allocated and nothing synchronises, so a
// stack can be captured into a CUDA graph.
#include <string.h>
#include "common.cuh"
#include "pwmlp_tc.cuh"
#include "../../include/o3d_b200.h"

namespace {

inline size_t al(size_t x) { return (x + 255) & ~(size_t)255; }
// channels handled by the tensor-core kernels: whole 128-tiles, or one partial tile for 64 <= c < 128; the rest
// (xyz / box-cloud extras of a first layer) goes through the exact CUDA-core kernel
inline int tc_main(int c) { return c >= 128 ? (c / 128) * 128 : (c >= 64 ? c : 0); }
inline int r4(int x) { return (x + 3) & ~3; }

// ---- weight packing -----------------------------------------------------------------------------------------
// src: [cout, cin] row-major (checkpoint layout).  dst wp: [Nw, K] zero padded; wt: [K, Nw] its transpose.
// xyz_first: src columns are [xyz(3) | feat(c0)] while the kernel rows are [feat(c0) | zeros | dx dy dz 0] (K = c0p + 4).
__device__ __forceinline__ int src_col(int k, int K, int cin, int xyz_first, int c0) {
    if (!xyz_first) return k < cin ? k : -1;
    if (k < c0) return 3 + k;             // feature columns
    if (k >= K - 4 && k < K - 1) return k - (K - 4);   // dx dy dz
    return -1;
}

// One kernel prepares everything a layer's GEMMs need from the checkpoint-layout weight:
//   wp [Nw, K] zero-padded (+ column re-ordering), wt [K, Nw] its transpose, the zero-padded bias, and — when the tensor-core
//   kernels take the layer — the pre-tiled hi|lo shared-memory images for the forward GEMM (rows = output channels) and
//   for the dgrad GEMM (rows = input channels); the image layout is the one documented at w_pretile_kernel (pwmlp_tc.cu).
// A thread owns 4 consecutive k of one (padded) row n.
__device__ __forceinline__ uint32_t tile_sw128(int r, int c) {
    return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u); }

struct PackLayer {
    const float* src; const float* bias; float* wp; float* wt; float* bias_p; uint8_t* tiles_f; uint8_t* tiles_b;
    int cout, cin, Nw, K, xyz_first, Km /* input channels tiled for dgrad */, Npad, Kpad /* iteration space */;
};
struct PackArgs { PackLayer l[O3D_MAX_LAYERS]; int c0; };

// all layers of a stack in one launch: blockIdx.y = layer
__global__ void pack_weight_kernel(const PackArgs args) {
    const PackLayer& L = args.l[blockIdx.y];
    const float* __restrict__ src = L.src;
    const float* __restrict__ bias = L.bias;
    float* __restrict__ wp = L.wp;
    float* __restrict__ wt = L.wt;
    float* __restrict__ bias_p = L.bias_p;
    uint8_t* __restrict__ tiles_f = L.tiles_f;
    uint8_t* __restrict__ tiles_b = L.tiles_b;
    const int cout = L.cout, cin = L.cin, Nw = L.Nw, K = L.K, xyz_first = L.xyz_first, c0 = args.c0, Km = L.Km, Npad = L.Npad,
              Kpad = L.Kpad;
    constexpr int TILE = 128 * 32 * 4;
    const int nkb_f = (K + 31) / 32;
    const int k4n = Kpad / 4;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (bias_p && i < Nw) bias_p[i] = i < cout ? bias[i] : 0.f;
    if (i >= Npad * k4n) return;
    const int n = i / k4n, k = (i % k4n) * 4;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (n < cout) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int sc = (k + j < K) ? src_col(k + j, K, cin, xyz_first, c0) : -1;
            if (sc >= 0) v[j] = src[(size_t)n * cin + sc];
        }
    }
    if (n < Nw && k < K) {
        *reinterpret_cast<float4*>(wp + (size_t)n * K + k) = make_float4(v[0], v[1], v[2], v[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) wt[(size_t)(k + j) * Nw + n] = v[j];
    }
    if (tiles_f && k < nkb_f * 32) {   // forward image: tile (n / 128, k / 32), row n % 128, 16-byte chunk (k % 32) / 4
        uint8_t* dst = tiles_f + ((size_t)(n >> 7) * nkb_f + (k >> 5)) * (2 * TILE) + tile_sw128(n & 127, (k & 31) >> 2);
        *reinterpret_cast<float4*>(dst) = make_float4(tf32_hi(v[0]), tf32_hi(v[1]), tf32_hi(v[2]), tf32_hi(v[3]));
        *reinterpret_cast<float4*>(dst + TILE) =
            make_float4(v[0] - tf32_hi(v[0]), v[1] - tf32_hi(v[1]), v[2] - tf32_hi(v[2]), v[3] - tf32_hi(v[3]));
    }
    if (tiles_b && n < ((Nw + 31) / 32) * 32) {   // dgrad image: rows = input channels k..k+3 (< Km), "K" index = n
        const int nkb_b = (Nw + 31) / 32;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int row = k + j;
            if (row >= ((Km + 127) / 128) * 128) continue;
            const float val = row < Km ? v[j] : 0.f;
            uint8_t* dst = tiles_b + ((size_t)(row >> 7) * nkb_b + (n >> 5)) * (2 * TILE) + tile_sw128(row & 127, (n & 31) >> 2) +
                           (n & 3) * 4;
            *reinterpret_cast<float*>(dst) = tf32_hi(val);
            *reinterpret_cast<float*>(dst + TILE) = val - tf32_hi(val);
        }
    }
}

struct UnpackLayer { const float* dwp; float* dst; int cout, cin, K, xyz_first; };
struct UnpackArgs { UnpackLayer l[O3D_MAX_LAYERS]; int c0; int accumulate; };

// padded / re-ordered weight gradients -> the checkpoint layout, all layers of a stack in one launch (blockIdx.y = layer)
__global__ void unpack_wgrad_kernel(const UnpackArgs args) {
    const UnpackLayer& L = args.l[blockIdx.y];
    const float* __restrict__ dwp = L.dwp;
    float* __restrict__ dst = L.dst;
    const int cout = L.cout, cin = L.cin, K = L.K, xyz_first = L.xyz_first, c0 = args.c0;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (!dst || i >= cout * K) return;
    const int n = i / K, k = i % K;
    const int sc = src_col(k, K, cin, xyz_first, c0);
    if (sc >= 0) {
        float* o = dst + (size_t)n * cin + sc;
        *o = args.accumulate ? *o + dwp[i] : dwp[i];
    }
}

__global__ void d2f_kernel(const double* __restrict__ src, int n, float* __restrict__ dst, int accumulate) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (accumulate ? dst[i] : 0.f) + (float)src[i];
}

// ---- workspace plan -------------------------------------------------------------------------------------------
struct Plan {
    int n, P, S, rows;
    bool lift, virt;     // layer 0 lifted (o3d_lift_t); virt: Y0 is never stored (the tensor-core kernels gather it)
    size_t gidx;         // [P] int32: global Z row of every position (forward workspace)
    int Nw[O3D_MAX_LAYERS], K[O3D_MAX_LAYERS];
    bool tc_f[O3D_MAX_LAYERS], tc_b[O3D_MAX_LAYERS];
    // forward (persisted) offsets
    size_t wp[O3D_MAX_LAYERS], wt[O3D_MAX_LAYERS], bias[O3D_MAX_LAYERS], y[O3D_MAX_LAYERS], vec[O3D_MAX_LAYERS],
        stat[O3D_MAX_LAYERS], tiles[O3D_MAX_LAYERS];
    size_t ymax, ymin, arg, sel, ysel, stat_all, stat_bytes, fwd_bytes, param_bytes;
    // backward (temporary) offsets
    size_t bstat, bstat_bytes, coef[O3D_MAX_LAYERS], dwp[O3D_MAX_LAYERS], btiles[O3D_MAX_LAYERS], dpool, gbuf[2], wpart, bwd_bytes;
    long long wpart_floats;
};

bool make_plan(const o3d_stack_t* d, Plan& p) {
    if (d->n_layers < 1 || d->n_layers > O3D_MAX_LAYERS || d->P < 0 || d->K0 < 4 || (d->K0 & 3) || (d->use_tc & ~3)) return false;
    p.n = d->n_layers; p.P = d->P; p.S = d->S;
    p.rows = d->S > 0 ? d->P / d->S : d->P;
    p.lift = d->lift != nullptr;
    p.virt = false;
    if (p.lift && (p.n < 2 || d->weight[0] != nullptr || (d->cout[0] & 3) || d->lift->ldz != d->cout[0] || d->bias[0])) return false;
    size_t o = 0;
    for (int l = 0; l < p.n; ++l) {
        p.Nw[l] = r4(d->cout[l]);
        p.K[l] = l == 0 ? (p.lift ? 0 : d->K0) : p.Nw[l - 1];
        // forward: also single, partly filled position tiles (P >= 16: the B = 1 tracking frame's 64 / 128-position head layers —
        // on the CUDA-core kernel such a layer is a 256-deep serial loop on two CTAs, 38 us; here one tile, 15 us)
        // (inference: also narrow output layers — 1 / 5 / 9 channels of the heads — as one partly filled channel tile)
        // (inference: any output width — e.g. the vote layer's 3 + 256 channels — as whole + one partly filled channel tile)
        p.tc_f[l] = (d->use_tc & 1) && (p.Nw[l] % 128 == 0 || p.Nw[l] == 64 || !d->training) && p.K[l] >= 32 &&
                    d->P >= (d->training ? 128 : 16) &&
                    !(l == d->n_layers - 1 && d->S > 0 && 64 % d->S != 0);
        p.tc_b[l] = (d->use_tc & 1) && p.K[l] >= 64 && p.Nw[l] >= 32 && d->P >= 128;
    }
    if (p.lift) {
        // Y0 stays virtual when all three GEMMs of layer 1 run on the tensor cores over whole 32-channel k-blocks
        const bool tcw1 = (d->use_tc & 2) && p.Nw[1] >= 64 && p.K[1] >= 64 && d->P >= 4096;
        // (inference: no weight-gradient kernel will run, so its size floor P >= 4096 does not apply)
        p.virt = p.tc_f[1] && p.tc_b[1] && (tcw1 || !d->training) && tc_main(p.K[1]) == p.K[1] && p.K[1] % 32 == 0;
    }
    // statistics block first (one memset)
    p.stat_all = o;
    for (int l = 0; l < p.n; ++l) { p.stat[l] = o; o += al(sizeof(double) * 2 * p.Nw[l]); }
    for (int l = 0; l < p.n; ++l) { p.vec[l] = o; o += al(sizeof(float) * 4 * p.Nw[l]); }   // zeroed together with the stats
    p.stat_bytes = o - p.stat_all;
    for (int l = 0; l < p.n; ++l) {
        p.wp[l] = o; o += al(sizeof(float) * (size_t)p.Nw[l] * p.K[l]);
        p.wt[l] = o; o += al(sizeof(float) * (size_t)p.Nw[l] * p.K[l]);
        p.bias[l] = o; o += al(sizeof(float) * p.Nw[l]);
        p.tiles[l] = o; if (p.tc_f[l]) o += al((size_t)o3d_pw_tc_wtile_bytes(p.Nw[l], p.K[l]));
        p.btiles[l] = o; if (p.tc_b[l]) o += al((size_t)o3d_pw_tc_wtile_bytes(tc_main(p.K[l]), p.Nw[l]));
    }
    p.param_bytes = o;       // everything above depends on the parameters only (eval mode): o3d_stack_prepare() fills it once
    for (int l = 0; l < p.n; ++l) {
        p.y[l] = o; if (!(l == 0 && p.virt)) o += al(sizeof(float) * (size_t)p.P * p.Nw[l]);
    }
    p.gidx = o; if (p.lift && d->lift->z) o += al(sizeof(int32_t) * (size_t)p.P);
    const size_t gsz = al(sizeof(float) * (size_t)p.rows * p.Nw[p.n - 1]);
    p.ymax = o; o += p.S > 0 ? gsz : 0;
    p.ymin = o; o += p.S > 0 ? gsz : 0;
    p.arg = o; o += p.S > 0 ? gsz : 0;
    p.sel = o; o += p.S > 0 ? gsz : 0;
    p.ysel = o; o += p.S > 0 ? gsz : 0;
    p.fwd_bytes = o;
    // backward
    o = 0;
    p.bstat = o;
    for (int l = 0; l < p.n; ++l) o += al(sizeof(double) * 2 * p.Nw[l]);
    size_t maxk = 0;
    for (int l = 0; l < p.n; ++l) { p.coef[l] = o; o += al(sizeof(float) * 5 * p.Nw[l]); }
    for (int l = 0; l < p.n; ++l) { p.dwp[l] = o; o += al(sizeof(float) * (size_t)p.Nw[l] * p.K[l]); }
    p.bstat_bytes = o;                      // sums | BN-backward coefficients | padded weight gradients: one memset
    for (int l = 0; l < p.n; ++l) {
        if ((size_t)p.K[l] > maxk) maxk = p.K[l];
    }
    size_t maxn = 0;
    for (int l = 0; l < p.n; ++l) if ((size_t)p.Nw[l] > maxn) maxn = p.Nw[l];
    if (maxn > maxk) maxk = maxn;
    p.dpool = o; o += p.S > 0 ? gsz : 0;
    for (int i = 0; i < 2; ++i) { p.gbuf[i] = o; o += al(sizeof(float) * (size_t)p.P * maxk); }
    p.wpart = o;
    p.wpart_floats = 0;
    if ((d->use_tc & 2) && d->P >= 4096) {
        p.wpart_floats = o3d_pw_wgrad_tc2_workspace_floats();
        o += al(sizeof(float) * (size_t)p.wpart_floats);
    }
    p.bwd_bytes = o;
    return true;
}

inline double* stat_sum(const Plan& p, uint8_t* ws, int l) { return reinterpret_cast<double*>(ws + p.stat[l]); }
template <class T> inline T* at(uint8_t* ws, size_t off) { return reinterpret_cast<T*>(ws + off); }
template <class T> inline const T* at(const uint8_t* ws, size_t off) { return reinterpret_cast<const T*>(ws + off); }

// every layer's padded weights, transposes, bias and pre-tiled images: one launch
int pack_params(const o3d_stack_t* d, const Plan& p, uint8_t* ws, int keep_for_backward, cudaStream_t st) {
        PackArgs pa{};
        pa.c0 = d->c0;
        int work_max = 0;
        for (int l = 0; l < p.n; ++l) {
            const int Nw = p.Nw[l], K = p.K[l];
            PackLayer& q = pa.l[l];
            q.src = d->weight[l]; q.bias = d->bias[l];
            q.wp = at<float>(ws, p.wp[l]); q.wt = at<float>(ws, p.wt[l]);
            q.bias_p = d->bias[l] ? at<float>(ws, p.bias[l]) : nullptr;
            q.tiles_f = p.tc_f[l] ? ws + p.tiles[l] : nullptr;
            q.tiles_b = (p.tc_b[l] && keep_for_backward) ? ws + p.btiles[l] : nullptr;
            q.cout = d->cout[l]; q.cin = d->cin[l]; q.Nw = Nw; q.K = K; q.xyz_first = l == 0 ? d->xyz_first : 0;
            q.Km = tc_main(K);
            q.Npad = Nw; q.Kpad = K;
            if (l == 0 && p.lift) { q.Npad = 0; q.bias_p = nullptr; q.tiles_f = q.tiles_b = nullptr; }   // no weight: nothing to pack
            if (q.tiles_f) { q.Npad = ((Nw + 127) / 128) * 128; q.Kpad = ((K + 31) / 32) * 32; }
            if (q.tiles_b) {
                if (q.Npad < ((Nw + 31) / 32) * 32) q.Npad = ((Nw + 31) / 32) * 32;
                if (q.Kpad < ((q.Km + 127) / 128) * 128) q.Kpad = ((q.Km + 127) / 128) * 128;
            }
            const int work = q.Npad * (q.Kpad / 4);
            if (work > work_max) work_max = work;
        }
        pack_weight_kernel<<<dim3((work_max + 255) / 256, p.n), 256, 0, st>>>(pa);
        O3D_CHECK_LAUNCH("o3d_stack_forward: pack_weight");
    return O3D_OK;
}

}  // namespace

extern "C" long long o3d_stack_workspace_bytes(const o3d_stack_t* d, int backward) {
    Plan p;
    if (!d || !make_plan(d, p)) return -1;
    return (long long)(backward ? p.bwd_bytes : p.fwd_bytes);
}

extern "C" long long o3d_stack_prepared_bytes(const o3d_stack_t* d) {
    Plan p;
    if (!d || !make_plan(d, p)) return -1;
    return (long long)p.param_bytes;
}

// Inference with static weights: pack the weights and fold the running BatchNorm statistics ONCE into `block`
// (o3d_stack_prepared_bytes() bytes); a descriptor whose `prepared` points at it skips both in every forward call.
// The block depends on the layer shapes AND on P's size class (which layers take the tensor-core path): prepare per shape.
extern "C" int o3d_stack_prepare(const o3d_stack_t* d, void* block, void* stream) {
    O3D_REQUIRE(d && block, O3D_ERR_ARG, "o3d_stack_prepare: null pointer");
    O3D_REQUIRE(!d->training, O3D_ERR_ARG, "o3d_stack_prepare: eval mode only (train-mode BatchNorm needs the batch)");
    Plan p;
    O3D_REQUIRE(make_plan(d, p), O3D_ERR_ARG, "o3d_stack_prepare: bad stack description");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)block;
    O3D_CUDA(cudaMemsetAsync(ws + p.stat_all, 0, p.stat_bytes, st), "o3d_stack_prepare: memset");
    if (int rc = pack_params(d, p, ws, 0, st)) return rc;
    for (int l = 0; l < p.n; ++l) {
        if (!d->has_bn[l]) continue;
        const int Nw = p.Nw[l];
        float* vec = at<float>(ws, p.vec[l]);
        if (int rc = o3d_bn_fwd_finalize(nullptr, nullptr, (double)p.P, d->gamma[l], d->beta[l], d->running_mean[l], d->running_var[l],
                                         nullptr, d->momentum[l], d->eps[l], 0, d->cout[l], vec, vec + Nw, vec + 2 * Nw, vec + 3 * Nw,
                                         stream))
            return rc;
    }
    return O3D_OK;
}

extern "C" int o3d_stack_forward(const o3d_stack_t* d, const float* x, void* ws_fwd, float* out, int keep_for_backward,
                                 void* stream) {
    O3D_REQUIRE(d && (x || d->lift) && ws_fwd && out, O3D_ERR_ARG, "o3d_stack_forward: null pointer");
    Plan p;
    O3D_REQUIRE(make_plan(d, p), O3D_ERR_ARG, "o3d_stack_forward: bad stack description");
    O3D_REQUIRE(p.S == 0 || (128 % p.S == 0 && p.P % p.S == 0), O3D_ERR_ARG, "o3d_stack_forward: group size %d", p.S);
    if (p.P == 0) return O3D_OK;
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* ws = (uint8_t*)ws_fwd;
    // Parameter block (padded / transposed / pre-tiled weights, BN scale / shift): per call in the workspace, or — inference
    // with static weights — the block o3d_stack_prepare() filled once (no packing, no BN finalisation per call).
    const bool prepared = d->prepared != nullptr;
    O3D_REQUIRE(!prepared || (!d->training && !keep_for_backward), O3D_ERR_ARG, "o3d_stack_forward: a prepared block is for inference only");
    uint8_t* wsp = prepared ? (uint8_t*)d->prepared : ws;
    if (!prepared) {
        O3D_CUDA(cudaMemsetAsync(ws + p.stat_all, 0, p.stat_bytes, st), "o3d_stack_forward: memset");   // statistics + BN vectors
        if (int rc = pack_params(d, p, wsp, keep_for_backward, st)) return rc;
    }
    const float* cur = x;
    int cur_ld = d->K0;
    const float *in_scale = nullptr, *in_shift = nullptr;
    int in_relu = 0;
    const int L = p.n - 1;
    for (int l = 0; l < p.n; ++l) {
        const int Nw = p.Nw[l], K = p.K[l], cout = d->cout[l];
        float* wt = at<float>(wsp, p.wt[l]);
        float* bias = d->bias[l] ? at<float>(wsp, p.bias[l]) : nullptr;
        const bool last = l == L, pool = last && p.S > 0;
        const bool keep_y = !last || keep_for_backward || !pool;
        float* y = keep_y ? at<float>(ws, p.y[l]) : nullptr;
        const bool stats = d->training && d->has_bn[l];
        double* sum = stats ? stat_sum(p, wsp, l) : nullptr;
        double* sumsq = stats ? sum + Nw : nullptr;
        float* ymax = pool ? at<float>(ws, p.ymax) : nullptr;
        float* ymin = pool ? at<float>(ws, p.ymin) : nullptr;
        int32_t* arg = pool ? at<int32_t>(ws, p.arg) : nullptr;
        int rc;
        if (l == 0 && p.lift) {
            // lifted layer: one gather pass = row indices + batch statistics (+ Y0 itself on the CUDA-core fallback)
            rc = o3d_lift_stats(d->lift, p.P, Nw, at<int32_t>(ws, p.gidx), p.virt ? nullptr : y, sum, sumsq, stream);
        } else if (l == 1 && p.virt) {
            rc = pw_fwd_tc_lift(d->lift, at<int32_t>(ws, p.gidx), in_scale, in_shift, in_relu, wsp + p.tiles[l], bias, p.P, K, cout,
                                y, Nw, sum, sumsq, pool ? p.S : 0, ymax, ymin, arg, Nw, 0, stream);
        } else if (p.tc_f[l]) {
            // snake order: layer 0 starts where the grouping kernel finished (the end), layer 1 where layer 0 finished, ...
            void* tiles = wsp + p.tiles[l];
            rc = pw_fwd_tc(cur, cur_ld, in_scale, in_shift, in_relu, tiles, bias, p.P, K, cout, y, Nw, sum, sumsq, pool ? p.S : 0,
                           ymax, ymin, arg, Nw, (l & 1) == 0, stream);
        } else {
            rc = o3d_pw_fwd(cur, cur_ld, in_scale, in_shift, in_relu, wt, Nw, bias, p.P, K, cout, y, Nw, sum, sumsq,
                            pool ? p.S : 0, ymax, ymin, arg, Nw, stream);
        }
        if (rc) return rc;
        float* vec = at<float>(wsp, p.vec[l]);
        float *sc = nullptr, *sh = nullptr;
        if (d->has_bn[l]) {
            sc = vec; sh = vec + Nw;
            if (!prepared)      // prepared: scale / shift of the running statistics are already in the block
            rc = o3d_bn_fwd_finalize(sum, sumsq, (double)p.P, d->gamma[l], d->beta[l], d->running_mean[l], d->running_var[l],
                                     d->training ? d->num_batches_tracked[l] : nullptr, d->momentum[l], d->eps[l],
                                     d->training, cout, sc, sh, vec + 2 * Nw, vec + 3 * Nw, stream);
            if (rc) return rc;
        }
        if (last) {
            if (pool) {
                rc = o3d_pool_finalize(ymax, ymin, arg, sc, sh, d->relu[l], p.rows, Nw, Nw, out, Nw,
                                       keep_for_backward ? at<int32_t>(ws, p.sel) : nullptr,
                                       keep_for_backward ? at<float>(ws, p.ysel) : nullptr, stream);
            } else if (d->has_bn[l] || d->relu[l]) {
                rc = o3d_act_apply(y, Nw, sc, sh, d->relu[l], p.P, Nw, out, Nw, stream);
            } else {
                O3D_CUDA(cudaMemcpyAsync(out, y, sizeof(float) * (size_t)p.P * Nw, cudaMemcpyDeviceToDevice, st),
                         "o3d_stack_forward: copy out");
                rc = O3D_OK;
            }
            if (rc) return rc;
        }
        cur = y; cur_ld = Nw; in_scale = sc; in_shift = sh; in_relu = d->relu[l];
    }
    return O3D_OK;
}

extern "C" int o3d_stack_backward(const o3d_stack_t* d, const float* x, const void* ws_fwd, void* ws_bwd, const float* out,
                                  const float* dout, float* dx, void* stream) {
    O3D_REQUIRE(d && (x || d->lift) && ws_fwd && ws_bwd && out && dout, O3D_ERR_ARG, "o3d_stack_backward: null pointer");
    Plan p;
    O3D_REQUIRE(make_plan(d, p), O3D_ERR_ARG, "o3d_stack_backward: bad stack description");
    if (p.P == 0) return O3D_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const uint8_t* wf = (const uint8_t*)ws_fwd;
    uint8_t* wb = (uint8_t*)ws_bwd;
    O3D_CUDA(cudaMemsetAsync(wb + p.bstat, 0, p.bstat_bytes, st), "o3d_stack_backward: memset");
    auto s1 = [&](int l) { size_t o = p.bstat; for (int i = 0; i < l; ++i) o += al(sizeof(double) * 2 * p.Nw[i]); return at<double>(wb, o); };
    const int L = p.n - 1;
    const int NwL = p.Nw[L];
    const float* yL = at<float>(wf, p.y[L]);
    const float* g = nullptr;      // dense gradient entering layer l's BN/ReLU
    float* dpool = nullptr;
    int rc;
    if (p.S > 0) {
        dpool = at<float>(wb, p.dpool);
        rc = o3d_pool_bwd_prep(dout, NwL, out, NwL, at<float>(wf, p.ysel), d->relu[L], p.rows, NwL, NwL, dpool, s1(L),
                               s1(L) + NwL, stream);
        if (rc) return rc;
    } else if (d->has_bn[L] || d->relu[L]) {
        float* gb = at<float>(wb, p.gbuf[0]);
        rc = o3d_dense_bwd_prep(dout, NwL, out, NwL, yL, NwL, d->relu[L], p.P, NwL, gb, NwL, s1(L), s1(L) + NwL, stream);
        if (rc) return rc;
        g = gb;
    } else {
        g = dout;
        if (d->bias[L]) {
            rc = o3d_dense_bwd_prep(dout, NwL, nullptr, 0, nullptr, 0, 0, p.P, NwL, nullptr, 0, s1(L), nullptr, stream);
            if (rc) return rc;
        }
    }
    int gsel = (g == at<float>(wb, p.gbuf[0])) ? 1 : 0;   // next free ping-pong buffer
    for (int l = L; l >= 0; --l) {
        const int Nl = p.Nw[l], K = p.K[l], cout = d->cout[l];
        float* coef = at<float>(wb, p.coef[l]);
        const float *a = nullptr, *b = nullptr, *cc = nullptr;
        const float* vec = at<float>(wf, p.vec[l]);
        if (d->has_bn[l]) {
            rc = o3d_bn_bwd_finalize(s1(l), s1(l) + Nl, (double)p.P, d->gamma[l], vec + 2 * Nl, vec + 3 * Nl,
                                     (d->training ? 1 : 0) | (d->accumulate ? 2 : 0),
                                     cout, coef, coef + Nl, coef + 2 * Nl, d->d_gamma[l], d->d_beta[l], stream);
            if (rc) return rc;
            a = coef; b = coef + Nl; cc = coef + 2 * Nl;
            if (d->d_bias[l] && !d->accumulate)      // BN removes the mean: the bias gradient is zero (nothing to add when accumulating)
                O3D_CUDA(cudaMemsetAsync(d->d_bias[l], 0, sizeof(float) * cout, st), "d_bias");
        } else if (d->d_bias[l]) {
            d2f_kernel<<<(cout + 127) / 128, 128, 0, st>>>(s1(l), cout, d->d_bias[l], d->accumulate);
        }
        if (l == 0 && p.lift) {
            // the lifted layer has no GEMM: dY0 = a*g + b + cc*Y0 is scattered into dZ / dcc / ds / du
            const o3d_lift_t* lf = d->lift;
            if (lf->d_z || lf->d_s || lf->d_u) {
                rc = o3d_lift_scatter(lf, p.P, Nl, at<int32_t>(wf, p.gidx), p.virt ? nullptr : at<float>(wf, p.y[0]), g, Nl, a, b,
                                      cc, stream);
                if (rc) return rc;
            }
            break;
        }
        const bool pooled = (l == L && p.S > 0);
        const float* gl = pooled ? nullptr : g;
        const float* yl = a ? at<float>(wf, p.y[l]) : nullptr;
        const float* dpl = pooled ? dpool : nullptr;
        const int32_t* sel = pooled ? at<int32_t>(wf, p.sel) : nullptr;
        const int Sg = pooled ? p.S : 0;
        // input operand of this layer
        const float* xin = l == 0 ? x : at<float>(wf, p.y[l - 1]);
        const float* pvec = l == 0 ? nullptr : at<float>(wf, p.vec[l - 1]);
        const int Kp = K;
        const float* psc = (l > 0 && d->has_bn[l - 1]) ? pvec : nullptr;
        const float* psh = (l > 0 && d->has_bn[l - 1]) ? pvec + Kp : nullptr;
        const int prelu = l > 0 ? d->relu[l - 1] : 0;
        if (l > 0 || dx) {
            float* gout = l > 0 ? at<float>(wb, p.gbuf[gsel]) : dx;
            const bool mask = l > 0 && (d->has_bn[l - 1] || d->relu[l - 1]);
            const bool want = l > 0 && (d->has_bn[l - 1] || d->bias[l - 1] != nullptr);
            const float* yprev = mask ? at<float>(wf, p.y[l - 1]) : nullptr;
            double* ps1 = want ? s1(l - 1) : nullptr;
            double* ps2 = want ? s1(l - 1) + K : nullptr;
            if (l == 1 && p.virt) {
                rc = pw_dgrad_tc_lift(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, wf + p.btiles[l], p.P, Nl, K, gout, K, d->lift,
                                      at<int32_t>(wf, p.gidx), psc, psh, prelu, ps1, ps2, stream);
            } else if (p.tc_b[l]) {
                // tensor cores on the first floor(K/128)*128 input channels, exact CUDA-core kernel on the ragged tail
                // (the xyz / box-cloud extras of a first layer)
                const int Km = tc_main(K);
                const void* tiles = wf + p.btiles[l];   // written by the forward pass's pack kernel
                rc = o3d_pw_dgrad_tc(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, tiles, p.P, Nl, Km, gout, K, yprev, K, psc, psh,
                                     prelu, ps1, ps2, stream);
                if (rc) return rc;
                // the ragged tail of a first layer holds (dx,dy,dz,0): skipped when the caller needs no coordinate gradient
                const bool tail_wanted = !(l == 0 && d->dx_cols > 0 && d->dx_cols <= Km);
                if (K > Km && tail_wanted)
                    rc = o3d_pw_dgrad(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, at<float>(wf, p.wp[l]) + Km, K, p.P, Nl, K - Km,
                                      gout + Km, K, yprev ? yprev + Km : nullptr, K, psc ? psc + Km : nullptr,
                                      psh ? psh + Km : nullptr, prelu, ps1 ? ps1 + Km : nullptr, ps2 ? ps2 + Km : nullptr, stream);
            } else {
                rc = o3d_pw_dgrad(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, at<float>(wf, p.wp[l]), K, p.P, Nl, K, gout, K,
                                  yprev, K, psc, psh, prelu, ps1, ps2, stream);
            }
            if (rc) return rc;
            g = gout;
            gsel ^= 1;
        }
        if (d->d_weight[l]) {
            float* dwp = at<float>(wb, p.dwp[l]);
            const bool tcw = (d->use_tc & 2) && Nl >= 64 && K >= 64 && p.P >= 4096;
            // every tensor-core weight gradient goes through the split-K kernel whose partial tiles are summed by a second kernel
            // in a fixed order (deterministic)
            if (l == 1 && p.virt) {
                rc = pw_wgrad_tc_lift(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, d->lift, at<int32_t>(wf, p.gidx), psc, psh, prelu, p.P,
                                      Nl, K, dwp, K, at<float>(wb, p.wpart), p.wpart_floats, stream);
            } else if (tcw) {
                // tensor-core part: the first floor(K/128)*128 input channels; ragged tail (xyz / box-cloud extras)
                // goes through the exact CUDA-core kernel on the remaining columns
                const int Kmain = tc_main(K);
                rc = o3d_pw_wgrad_tc2(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, xin, K, psc, psh, prelu, p.P, Nl, Kmain, dwp, K,
                                      at<float>(wb, p.wpart), p.wpart_floats, stream);
                if (rc) return rc;
                if (K > Kmain)
                    rc = o3d_pw_wgrad(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, xin + Kmain, K, psc ? psc + Kmain : nullptr,
                                      psh ? psh + Kmain : nullptr, prelu, p.P, Nl, K - Kmain, dwp + Kmain, K, stream);
            } else {
                rc = o3d_pw_wgrad(gl, Nl, yl, Nl, a, b, cc, dpl, sel, Sg, Nl, xin, K, psc, psh, prelu, p.P, Nl, K, dwp, K, stream);
            }
            if (rc) return rc;
        }
    }
    {
        UnpackArgs ua{};
        ua.c0 = d->c0;
        ua.accumulate = d->accumulate;
        int work_max = 0;
        for (int l = 0; l < p.n; ++l) {
            UnpackLayer& q = ua.l[l];
            q.dwp = at<float>(wb, p.dwp[l]); q.dst = d->d_weight[l];
            q.cout = d->cout[l]; q.cin = d->cin[l]; q.K = p.K[l]; q.xyz_first = l == 0 ? d->xyz_first : 0;
            if (q.dst && q.cout * q.K > work_max) work_max = q.cout * q.K;
        }
        if (work_max > 0) {
            unpack_wgrad_kernel<<<dim3((work_max + 255) / 256, p.n), 256, 0, st>>>(ua);
            O3D_CHECK_LAUNCH("o3d_stack_backward: unpack_wgrad");
        }
    }
    return O3D_OK;
}
