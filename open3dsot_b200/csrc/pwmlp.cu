// Point-wise (1x1-conv) MLP layers with batch-norm statistics, ReLU and group pooling fused into the GEMMs.
//
// Replaces the reference's SharedMLP / Seq stacks — cuDNN 1x1 conv + BatchNorm(train) + ReLU + max-pool over
// materialised (B,C,npoint,nsample) tensors — pointnet2/utils/pytorch_utils.py:12-37,68-121,300-339 as driven by
// pointnet2/utils/pointnet2_modules.py:64-73, models/head/xcorr.py:47-51,98-101 and models/head/rpn.py:48-60.
//
// Layout: activations are channels-last matrices  X[P, ld]  (P = B*npoint*nsample positions, one 16-byte aligned
// row per position).  A layer is  Y = A(X) * Wt (+bias)  with A = the previous layer's BN-affine + ReLU applied
// while the operand tile is loaded (so normalised activations are never written), and the epilogue
//   * writes the raw pre-BN output Y once,
//   * accumulates the per-channel batch statistics (sum, sum of squares; fp32 partials -> fp64 atomics),
//   * optionally reduces max / min (+ first arg) over each group of S consecutive positions — the SA max-pool
//     over nsample, the BoxAware max over k, the P2B max over template points — so the pooled tensor of the LAST
//     layer is produced without another pass (min is kept because gamma/sigma may be negative).
// Backward uses the same GEMM core twice per layer:
//   dgrad  D = dY * W           epilogue: g_prev = D * [z_prev > 0], sums of g_prev and g_prev*y_prev
//   wgrad  dW = dY^T * A(X)     split over P, fp32 RED into dW
// with  dY = a*g + b + c*Y  (the batch-norm backward, per-channel a,b,c from bn_bwd_finalize) evaluated in the
// operand loader, so dY is never materialised either.
//
// This file is the exact-fp32 CUDA-core implementation (128 x {64,128} x 16 tiles, 256 threads, 8x8 or 4x8
// register blocks, register-prefetch double buffering).  It is the numerical ground truth for the tensor-core
// (tcgen05, 3xTF32) variant in pwmlp_tc.cu, which shares these loaders' semantics and the epilogue contract.
#include "common.cuh"
#include "../../include/o3d_b200.h"

namespace {

constexpr int BM = 128;   // positions per tile (fwd/dgrad) or output-channel rows (wgrad)
constexpr int BK = 16;
constexpr int NT = 256;   // threads
constexpr int AS_LD = BK + 4;  // As[m][k] row stride (floats): 80 B keeps float4 alignment

struct ActIn {  // position-major operand:  v = x[p, k];  v = v*scale[k] + shift[k] (if scale);  v = max(v,0) (if relu)
    const float* x;
    int ld;
    const float* scale;
    const float* shift;
    int relu;
};

struct DyIn {  // dY[p, c] = a[c]*g[p,c] + b[c] + cc[c]*y[p,c]      (a == nullptr -> dY = g)
    const float* g;      // dense g [P, ldg]                          (mode 0)
    int ldg;
    const float* y;      // raw pre-BN output of this layer [P, ldy]
    int ldy;
    const float* a;
    const float* b;
    const float* cc;
    const float* dpool;  // pooled mode: g[p,c] = (p % S == sel[p/S, c]) ? dpool[p/S, c] : 0      [G, ldp]
    const int32_t* sel;
    int S;
    int ldp;
};

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// Operand loads are split in two so that the register-prefetch double buffering really overlaps memory latency with the
// FMA loop: fetch_*() issues only address-independent global loads (clamped, always in range) BEFORE the tile's math,
// finish_*() applies the per-channel transform (and the range mask) AFTER it, right before the st.shared.
struct ActRaw { float4 v; };
struct DyRaw { float4 g, y; };

__device__ __forceinline__ ActRaw fetch_act(const ActIn& in, int p, int P, int k, int K) {
    ActRaw r;
    r.v = ld4(in.x + (size_t)(p < P ? p : P - 1) * in.ld + (k < K ? k : 0));
    return r;
}
__device__ __forceinline__ float4 finish_act(const ActIn& in, const ActRaw& r, int p, int P, int k, int K) {
    if (!(p < P && k < K)) return make_float4(0.f, 0.f, 0.f, 0.f);
    float4 v = r.v;
    if (in.scale) {
        const float4 s = ld4(in.scale + k), t = ld4(in.shift + k);
        v.x = fmaf(v.x, s.x, t.x); v.y = fmaf(v.y, s.y, t.y); v.z = fmaf(v.z, s.z, t.z); v.w = fmaf(v.w, s.w, t.w);
    }
    if (in.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
    return v;
}
__device__ __forceinline__ DyRaw fetch_dy(const DyIn& in, int p, int P, int c, int C) {
    DyRaw r;
    const int pp = p < P ? p : P - 1, cc = c < C ? c : 0;
    if (in.dpool) {
        const int grp = pp / in.S, s = pp - grp * in.S;
        const int4 sl = __ldg(reinterpret_cast<const int4*>(in.sel + (size_t)grp * in.ldp + cc));
        const float4 d = ld4(in.dpool + (size_t)grp * in.ldp + cc);
        r.g = make_float4(sl.x == s ? d.x : 0.f, sl.y == s ? d.y : 0.f, sl.z == s ? d.z : 0.f, sl.w == s ? d.w : 0.f);
    } else {
        r.g = ld4(in.g + (size_t)pp * in.ldg + cc);
    }
    r.y = in.a ? ld4(in.y + (size_t)pp * in.ldy + cc) : make_float4(0.f, 0.f, 0.f, 0.f);
    return r;
}
__device__ __forceinline__ float4 finish_dy(const DyIn& in, const DyRaw& r, int p, int P, int c, int C) {
    if (!(p < P && c < C)) return make_float4(0.f, 0.f, 0.f, 0.f);
    float4 v = r.g;
    if (in.a) {
        const float4 a = ld4(in.a + c), b = ld4(in.b + c), cc = ld4(in.cc + c);
        v.x = fmaf(a.x, v.x, fmaf(cc.x, r.y.x, b.x)); v.y = fmaf(a.y, v.y, fmaf(cc.y, r.y.y, b.y));
        v.z = fmaf(a.z, v.z, fmaf(cc.z, r.y.z, b.z)); v.w = fmaf(a.w, v.w, fmaf(cc.w, r.y.w, b.w));
    }
    return v;
}

__device__ __forceinline__ void prefetch_act(const ActIn& in, int p0, int rows, int P) {
    if (p0 < P) o3d_prefetch_l2(in.x + (size_t)p0 * in.ld, (size_t)min(rows, P - p0) * in.ld * sizeof(float));
}
__device__ __forceinline__ void prefetch_dy(const DyIn& in, int p0, int rows, int P) {
    if (p0 >= P) return;
    const size_t n = (size_t)min(rows, P - p0);
    if (!in.dpool) o3d_prefetch_l2(in.g + (size_t)p0 * in.ldg, n * in.ldg * sizeof(float));
    if (in.a) o3d_prefetch_l2(in.y + (size_t)p0 * in.ldy, n * in.ldy * sizeof(float));
    if (in.dpool) {   // pooled-gradient tables of the groups these rows belong to
        const int g0 = p0 / in.S, g1 = (p0 + (int)n - 1) / in.S;
        const size_t bytes = (size_t)(g1 - g0 + 1) * in.ldp * sizeof(float);
        o3d_prefetch_l2(in.dpool + (size_t)g0 * in.ldp, bytes);
        o3d_prefetch_l2(in.sel + (size_t)g0 * in.ldp, bytes);
    }
}

// ------------------------------------------------------------------------------------------------------------
// Shared-memory plan (dynamic):  main loop  As[2][BM*AS_LD] | Bs[2][BK*(BN+4)]   (or A2s[2][BK*(BM+4)] for wgrad)
//                                epilogue   Cs[BM][BN+4]  (aliases the main-loop buffers)  + red[NT/(BN/4)][BN][2]
template <int BN>
struct Cfg {
    static constexpr int TX = BN / 8;         // threads along N (each owns 4 + 4 columns)
    static constexpr int TY = NT / TX;        // threads along M
    static constexpr int TM = BM / TY;        // rows per thread (8 for BN=128, 4 for BN=64)
    static constexpr int BS_LD = BN + 4;
    static constexpr int CS_LD = BN + 4;
    static constexpr int A2_LD = BM + 4;
    static constexpr size_t MAIN_FLOATS = 2 * BM * AS_LD + 2 * BK * BS_LD;
    static constexpr size_t MAIN2_FLOATS = 2 * BK * A2_LD + 2 * BK * BS_LD;
    static constexpr size_t EPI_FLOATS = (size_t)BM * CS_LD + (size_t)(NT / (BN / 4)) * BN * 2;  // Cs + red[RL][BN][2]
    static constexpr size_t SMEM_BYTES =
        4 * (EPI_FLOATS > MAIN_FLOATS ? (EPI_FLOATS > MAIN2_FLOATS ? EPI_FLOATS : MAIN2_FLOATS)
                                      : (MAIN_FLOATS > MAIN2_FLOATS ? MAIN_FLOATS : MAIN2_FLOATS));
};

// acc[i][j] += sum_k A[m_i][k] * B[k][n_j] over one BK tile; A stored [m][k].
template <int BN>
__device__ __forceinline__ void mma_tile_mk(const float* __restrict__ As, const float* __restrict__ Bs, int ty, int tx,
                                            float (&acc)[Cfg<BN>::TM][8]) {
    constexpr int TM = Cfg<BN>::TM;
    constexpr int BS_LD = Cfg<BN>::BS_LD;
#pragma unroll
    for (int kk = 0; kk < BK; kk += 4) {
        float4 a[TM];
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] = *reinterpret_cast<const float4*>(As + (ty * TM + i) * AS_LD + kk);
#pragma unroll
        for (int k4 = 0; k4 < 4; ++k4) {
            const float4 b0 = *reinterpret_cast<const float4*>(Bs + (kk + k4) * BS_LD + tx * 4);
            const float4 b1 = *reinterpret_cast<const float4*>(Bs + (kk + k4) * BS_LD + BN / 2 + tx * 4);
#pragma unroll
            for (int i = 0; i < TM; ++i) {
                const float av = k4 == 0 ? a[i].x : k4 == 1 ? a[i].y : k4 == 2 ? a[i].z : a[i].w;
                acc[i][0] = fmaf(av, b0.x, acc[i][0]); acc[i][1] = fmaf(av, b0.y, acc[i][1]);
                acc[i][2] = fmaf(av, b0.z, acc[i][2]); acc[i][3] = fmaf(av, b0.w, acc[i][3]);
                acc[i][4] = fmaf(av, b1.x, acc[i][4]); acc[i][5] = fmaf(av, b1.y, acc[i][5]);
                acc[i][6] = fmaf(av, b1.z, acc[i][6]); acc[i][7] = fmaf(av, b1.w, acc[i][7]);
            }
        }
    }
}

// Same, A stored [k][m] (wgrad).
template <int BN>
__device__ __forceinline__ void mma_tile_km(const float* __restrict__ A2, const float* __restrict__ Bs, int ty, int tx,
                                            float (&acc)[Cfg<BN>::TM][8]) {
    constexpr int TM = Cfg<BN>::TM;
    constexpr int BS_LD = Cfg<BN>::BS_LD;
    constexpr int A2_LD = Cfg<BN>::A2_LD;
#pragma unroll
    for (int k = 0; k < BK; ++k) {
        float a[TM];
#pragma unroll
        for (int i = 0; i < TM; i += 4) {
            const float4 t = *reinterpret_cast<const float4*>(A2 + k * A2_LD + ty * TM + i);
            a[i] = t.x; a[i + 1] = t.y; a[i + 2] = t.z; a[i + 3] = t.w;
        }
        const float4 b0 = *reinterpret_cast<const float4*>(Bs + k * BS_LD + tx * 4);
        const float4 b1 = *reinterpret_cast<const float4*>(Bs + k * BS_LD + BN / 2 + tx * 4);
#pragma unroll
        for (int i = 0; i < TM; ++i) {
            acc[i][0] = fmaf(a[i], b0.x, acc[i][0]); acc[i][1] = fmaf(a[i], b0.y, acc[i][1]);
            acc[i][2] = fmaf(a[i], b0.z, acc[i][2]); acc[i][3] = fmaf(a[i], b0.w, acc[i][3]);
            acc[i][4] = fmaf(a[i], b1.x, acc[i][4]); acc[i][5] = fmaf(a[i], b1.y, acc[i][5]);
            acc[i][6] = fmaf(a[i], b1.z, acc[i][6]); acc[i][7] = fmaf(a[i], b1.w, acc[i][7]);
        }
    }
}

// B tile loader: Bsrc is row-major [K, ldb] (n contiguous); tile rows k0..k0+15, columns n0..n0+BN-1.
template <int BN>
struct BLoad {
    static constexpr int V = BK * BN / 4 / NT;  // float4 per thread: 2 (BN=128) or 1 (BN=64)
    float4 r[V];
    __device__ __forceinline__ void load(const float* __restrict__ Bsrc, int ldb, int K, int N, int k0, int n0, int tid) {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const int id = tid + v * NT;
            const int k = id / (BN / 4), n = (id % (BN / 4)) * 4;
            r[v] = (k0 + k < K && n0 + n < N) ? ld4(Bsrc + (size_t)(k0 + k) * ldb + n0 + n) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    __device__ __forceinline__ void store(float* Bs, int tid) const {
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const int id = tid + v * NT;
            const int k = id / (BN / 4), n = (id % (BN / 4)) * 4;
            *reinterpret_cast<float4*>(Bs + k * Cfg<BN>::BS_LD + n) = r[v];
        }
    }
};

template <int BN>
__device__ __forceinline__ void stage_acc(float* Cs, const float (&acc)[Cfg<BN>::TM][8], int ty, int tx) {
    constexpr int TM = Cfg<BN>::TM;
    constexpr int LD = Cfg<BN>::CS_LD;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        *reinterpret_cast<float4*>(Cs + (ty * TM + i) * LD + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        *reinterpret_cast<float4*>(Cs + (ty * TM + i) * LD + BN / 2 + tx * 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
    }
}

// Column sums over the staged tile: every thread owns the same 4 columns in all its rows (NT % (BN/4) == 0), partial
// sums go through red[8][BN][2] and leave as one fp64 atomic per column and statistic.
template <int BN>
__device__ __forceinline__ void reduce_cols(float* red, const float (&s1)[4], const float (&s2)[4], int tid, int n0,
                                            int Nw, double* __restrict__ o1, double* __restrict__ o2) {
    constexpr int C4 = BN / 4;
    constexpr int RL = NT / C4;  // row lanes: 8 (BN=128) or 16 (BN=64)
    const int c4 = tid % C4, rl = tid / C4;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        red[(rl * BN + c4 * 4 + j) * 2 + 0] = s1[j];
        red[(rl * BN + c4 * 4 + j) * 2 + 1] = s2[j];
    }
    __syncthreads();
    if (tid < BN && n0 + tid < Nw) {
        float t1 = 0.f, t2 = 0.f;
#pragma unroll
        for (int r = 0; r < RL; ++r) {
            t1 += red[(r * BN + tid) * 2 + 0];
            t2 += red[(r * BN + tid) * 2 + 1];
        }
        atomicAdd(o1 + n0 + tid, (double)t1);
        atomicAdd(o2 + n0 + tid, (double)t2);
    }
}

// ------------------------------------------------------------------------------------------------------------
// Forward:  Y[p, n] = sum_k A(X)[p,k] * Wt[k, n] (+ bias[n])
struct FwdEpi {
    float* y; int ldy;           // raw output (may be nullptr when only pooling is wanted)
    const float* bias;           // nullable
    double* sum; double* sumsq;  // nullable: batch statistics
    int S;                       // group size for pooling (0 = none)
    float* ymax; float* ymin;    // [G, ldp]
    int32_t* arg;                // [G, ldp]: argmax | argmin << 16
    int ldp;
};

template <int BN>
__global__ void __launch_bounds__(NT, 2)
    pw_fwd_kernel(ActIn ain, const float* __restrict__ Wt, int ldw, int P, int K, int N, int Nw, FwdEpi ep) {
    using C = Cfg<BN>;
    extern __shared__ __align__(16) float smem[];
    float* As = smem;
    float* Bs = smem + 2 * BM * AS_LD;
    const int tid = threadIdx.x, tx = tid % C::TX, ty = tid / C::TX;
    const int p0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    if (tid == 0 && blockIdx.y == 0 && K > 32) prefetch_act(ain, p0, BM, P);   // whole rows -> L2 once, contiguously

    float acc[C::TM][8];
#pragma unroll
    for (int i = 0; i < C::TM; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    // A tile: 128 rows x 16 k = 512 float4 -> 2 per thread: row = id/4, kv = (id%4)*4
    ActRaw ra[2];
    BLoad<BN> rb;
    const int nk = (K + BK - 1) / BK;
    auto load_tiles = [&](int kt) {
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int id = tid + v * NT;
            ra[v] = fetch_act(ain, p0 + id / 4, P, kt * BK + (id % 4) * 4, K);
        }
        rb.load(Wt, ldw, K, N, kt * BK, n0, tid);
    };
    auto store_tiles = [&](int buf, int kt) {
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int id = tid + v * NT;
            *reinterpret_cast<float4*>(As + buf * BM * AS_LD + (id / 4) * AS_LD + (id % 4) * 4) =
                finish_act(ain, ra[v], p0 + id / 4, P, kt * BK + (id % 4) * 4, K);
        }
        rb.store(Bs + buf * BK * C::BS_LD, tid);
    };
    load_tiles(0);
    store_tiles(0, 0);
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) load_tiles(kt + 1);
        mma_tile_mk<BN>(As + buf * BM * AS_LD, Bs + buf * BK * C::BS_LD, ty, tx, acc);
        if (kt + 1 < nk) store_tiles(buf ^ 1, kt + 1);
        __syncthreads();
    }

    // ---- epilogue through the staged tile
    float* Cs = smem;
    float* red = smem + BM * C::CS_LD;
    stage_acc<BN>(Cs, acc, ty, tx);
    __syncthreads();
    constexpr int C4 = BN / 4;
    const int c4 = tid % C4, rl = tid / C4;
    const int col = n0 + c4 * 4;
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ep.bias && col < Nw) bv = ld4(ep.bias + col);
    for (int r = rl; r < BM; r += NT / C4) {
        float4 v = *reinterpret_cast<float4*>(Cs + r * C::CS_LD + c4 * 4);
        v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
        if (ep.bias) *reinterpret_cast<float4*>(Cs + r * C::CS_LD + c4 * 4) = v;  // pooling below reads biased values
        if (p0 + r < P && col < Nw) {
            if (ep.y) *reinterpret_cast<float4*>(ep.y + (size_t)(p0 + r) * ep.ldy + col) = v;
            s1[0] += v.x; s1[1] += v.y; s1[2] += v.z; s1[3] += v.w;
            s2[0] = fmaf(v.x, v.x, s2[0]); s2[1] = fmaf(v.y, v.y, s2[1]);
            s2[2] = fmaf(v.z, v.z, s2[2]); s2[3] = fmaf(v.w, v.w, s2[3]);
        }
    }
    if (ep.sum) reduce_cols<BN>(red, s1, s2, tid, n0, Nw, ep.sum, ep.sumsq);
    if (ep.S > 0) {
        __syncthreads();
        const int groups = BM / ep.S;
        for (int it = tid; it < groups * BN; it += NT) {
            const int gi = it / BN, c = it % BN;
            const int prow = p0 + gi * ep.S;
            if (prow >= P || n0 + c >= Nw) continue;
            float mx = -INFINITY, mn = INFINITY;
            int ax = 0, an = 0;
            for (int s = 0; s < ep.S; ++s) {
                const float v = Cs[(gi * ep.S + s) * C::CS_LD + c];
                if (v > mx) { mx = v; ax = s; }
                if (v < mn) { mn = v; an = s; }
            }
            const size_t o = (size_t)(prow / ep.S) * ep.ldp + n0 + c;
            ep.ymax[o] = mx; ep.ymin[o] = mn; ep.arg[o] = ax | (an << 16);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------
// dgrad:  D[p, n] = sum_c dY[p, c] * W[c, n]       (c over this layer's outputs, n over its inputs)
// epilogue (mask mode): g_prev = D * [yprev*scale+shift > 0]; sums of g_prev and g_prev*yprev; write g_prev.
struct DgradEpi {
    float* out; int ldo;                 // g_prev (or plain D) [P, ldo]
    const float* yprev; int ldyp;        // raw pre-BN output of the previous layer (mask mode), nullable
    const float* scale; const float* shift;  // previous layer's BN affine (nullable -> mask on yprev itself)
    int relu;                            // previous layer has ReLU
    double* s1; double* s2y;             // nullable
};

template <int BN>
__global__ void __launch_bounds__(NT, 2)
    pw_dgrad_kernel(DyIn din, const float* __restrict__ W, int ldw, int P, int K /*Cout*/, int N /*Cin*/, int Nw,
                    DgradEpi ep) {
    using C = Cfg<BN>;
    extern __shared__ __align__(16) float smem[];
    float* As = smem;
    float* Bs = smem + 2 * BM * AS_LD;
    const int tid = threadIdx.x, tx = tid % C::TX, ty = tid / C::TX;
    const int p0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    if (tid == 0 && blockIdx.y == 0 && K > 32) prefetch_dy(din, p0, BM, P);
    float acc[C::TM][8];
#pragma unroll
    for (int i = 0; i < C::TM; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    DyRaw ra[2];
    BLoad<BN> rb;
    const int nk = (K + BK - 1) / BK;
    auto load_tiles = [&](int kt) {
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int id = tid + v * NT;
            ra[v] = fetch_dy(din, p0 + id / 4, P, kt * BK + (id % 4) * 4, K);
        }
        rb.load(W, ldw, K, N, kt * BK, n0, tid);
    };
    auto store_tiles = [&](int buf, int kt) {
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int id = tid + v * NT;
            *reinterpret_cast<float4*>(As + buf * BM * AS_LD + (id / 4) * AS_LD + (id % 4) * 4) =
                finish_dy(din, ra[v], p0 + id / 4, P, kt * BK + (id % 4) * 4, K);
        }
        rb.store(Bs + buf * BK * C::BS_LD, tid);
    };
    load_tiles(0);
    store_tiles(0, 0);
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) load_tiles(kt + 1);
        mma_tile_mk<BN>(As + buf * BM * AS_LD, Bs + buf * BK * C::BS_LD, ty, tx, acc);
        if (kt + 1 < nk) store_tiles(buf ^ 1, kt + 1);
        __syncthreads();
    }
    float* Cs = smem;
    float* red = smem + BM * C::CS_LD;
    stage_acc<BN>(Cs, acc, ty, tx);
    __syncthreads();
    constexpr int C4 = BN / 4;
    const int c4 = tid % C4, rl = tid / C4;
    const int col = n0 + c4 * 4;
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ep.scale && col < Nw) { sc = ld4(ep.scale + col); sh = ld4(ep.shift + col); }
    for (int r = rl; r < BM; r += NT / C4) {
        if (p0 + r >= P || col >= Nw) continue;
        float4 v = *reinterpret_cast<float4*>(Cs + r * C::CS_LD + c4 * 4);
        if (ep.yprev) {
            const float4 y = ld4(ep.yprev + (size_t)(p0 + r) * ep.ldyp + col);
            if (ep.relu) {
                v.x = fmaf(y.x, sc.x, sh.x) > 0.f ? v.x : 0.f; v.y = fmaf(y.y, sc.y, sh.y) > 0.f ? v.y : 0.f;
                v.z = fmaf(y.z, sc.z, sh.z) > 0.f ? v.z : 0.f; v.w = fmaf(y.w, sc.w, sh.w) > 0.f ? v.w : 0.f;
            }
            s2[0] = fmaf(v.x, y.x, s2[0]); s2[1] = fmaf(v.y, y.y, s2[1]);
            s2[2] = fmaf(v.z, y.z, s2[2]); s2[3] = fmaf(v.w, y.w, s2[3]);
        }
        s1[0] += v.x; s1[1] += v.y; s1[2] += v.z; s1[3] += v.w;
        *reinterpret_cast<float4*>(ep.out + (size_t)(p0 + r) * ep.ldo + col) = v;
    }
    if (ep.s1) reduce_cols<BN>(red, s1, s2, tid, n0, Nw, ep.s1, ep.s2y);
}

// ------------------------------------------------------------------------------------------------------------
// wgrad:  dW[m, n] += sum_p dY[p, m] * A(X)[p, n]   over this CTA's slice of positions (grid.z), fp32 RED.
template <int BN>
__global__ void __launch_bounds__(NT, 2)
    pw_wgrad_kernel(DyIn din, ActIn ain, int P, int M /*Cout*/, int N /*Cin (padded)*/, int chunk, float* __restrict__ dW,
                    int lddw) {
    using C = Cfg<BN>;
    extern __shared__ __align__(16) float smem[];
    float* A2 = smem;
    float* Bs = smem + 2 * BK * C::A2_LD;
    const int tid = threadIdx.x, tx = tid % C::TX, ty = tid / C::TX;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    const int pbeg = blockIdx.z * chunk, pend = min(P, pbeg + chunk);
    if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0) {   // one CTA per position slice streams its rows into L2
        prefetch_dy(din, pbeg, pend - pbeg, pend);
        prefetch_act(ain, pbeg, pend - pbeg, pend);
    }
    float acc[C::TM][8];
#pragma unroll
    for (int i = 0; i < C::TM; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    // A2 tile: 16 positions x 128 m = 512 float4 (2 / thread); B tile: 16 positions x BN (V / thread)
    constexpr int VB = BK * BN / 4 / NT;
    DyRaw ra[2];
    ActRaw rb[VB];
    const int nk = (pend - pbeg + BK - 1) / BK;
    auto load_tiles = [&](int kt) {
        const int pk = pbeg + kt * BK;
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int id = tid + v * NT;
            ra[v] = fetch_dy(din, pk + id / 32, pend, m0 + (id % 32) * 4, M);
        }
#pragma unroll
        for (int v = 0; v < VB; ++v) {
            const int id = tid + v * NT;
            rb[v] = fetch_act(ain, pk + id / (BN / 4), pend, n0 + (id % (BN / 4)) * 4, N);
        }
    };
    auto store_tiles = [&](int buf, int kt) {
        const int pk = pbeg + kt * BK;
#pragma unroll
        for (int v = 0; v < 2; ++v) {
            const int id = tid + v * NT;
            *reinterpret_cast<float4*>(A2 + buf * BK * C::A2_LD + (id / 32) * C::A2_LD + (id % 32) * 4) =
                finish_dy(din, ra[v], pk + id / 32, pend, m0 + (id % 32) * 4, M);
        }
#pragma unroll
        for (int v = 0; v < VB; ++v) {
            const int id = tid + v * NT;
            *reinterpret_cast<float4*>(Bs + buf * BK * C::BS_LD + (id / (BN / 4)) * C::BS_LD + (id % (BN / 4)) * 4) =
                finish_act(ain, rb[v], pk + id / (BN / 4), pend, n0 + (id % (BN / 4)) * 4, N);
        }
    };
    if (nk > 0) {
        load_tiles(0);
        store_tiles(0, 0);
    }
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) load_tiles(kt + 1);
        mma_tile_km<BN>(A2 + buf * BK * C::A2_LD, Bs + buf * BK * C::BS_LD, ty, tx, acc);
        if (kt + 1 < nk) store_tiles(buf ^ 1, kt + 1);
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < C::TM; ++i) {
        const int m = m0 + ty * C::TM + i;
        if (m >= M) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int n = n0 + h * (BN / 2) + tx * 4;
            if (n < N)
                atomicAdd(reinterpret_cast<float4*>(dW + (size_t)m * lddw + n),
                          make_float4(acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]));
        }
    }
}

// Forward layer with a handful of input columns (an xyz-only first layer, K <= 8) and no pooling: the tiled kernel spends
// its time on empty k-tiles, this one is a single streaming pass — thread = (4 output channels, every R-th position), the
// K x 4 weight block lives in registers, rows are stored as coalesced float4, batch statistics go through registers ->
// shared memory -> one fp64 RED per channel and block.
template <int KQ>
__global__ void __launch_bounds__(256, 2)
    pw_fwd_skinny_kernel(ActIn ain, const float* __restrict__ Wt, int ldw, int P, int K, int Nw, int LQ, int chunk, FwdEpi ep) {
    __shared__ float red[2][256 * 4];
    const int tid = threadIdx.x;
    const int n0 = blockIdx.y * 256;
    const int cq = tid % LQ, r = tid / LQ, R = 256 / LQ;
    const int n = n0 + cq * 4;
    const bool on = n < Nw;
    float4 w[4 * KQ];
#pragma unroll
    for (int k = 0; k < 4 * KQ; ++k) w[k] = (on && k < K) ? ld4(Wt + (size_t)k * ldw + n) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 bv = (on && ep.bias) ? ld4(ep.bias + n) : make_float4(0.f, 0.f, 0.f, 0.f);
    float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
    const int pbeg = blockIdx.x * chunk, pend = min(P, pbeg + chunk);
    constexpr int U = 4;
    for (int p = pbeg + r; p < pend; p += U * R) {
        ActRaw x[U][KQ];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int q = 0; q < KQ; ++q) x[u][q] = fetch_act(ain, p + u * R, pend, q * 4, K);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int pp = p + u * R;
            if (pp >= pend || !on) continue;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int q = 0; q < KQ; ++q) {
                const float4 xv = finish_act(ain, x[u][q], pp, pend, q * 4, K);
                const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 ww = w[q * 4 + j];
                    acc.x = fmaf(xx[j], ww.x, acc.x); acc.y = fmaf(xx[j], ww.y, acc.y);
                    acc.z = fmaf(xx[j], ww.z, acc.z); acc.w = fmaf(xx[j], ww.w, acc.w);
                }
            }
            acc.x += bv.x; acc.y += bv.y; acc.z += bv.z; acc.w += bv.w;
            if (ep.y) *reinterpret_cast<float4*>(ep.y + (size_t)pp * ep.ldy + n) = acc;
            s1.x += acc.x; s1.y += acc.y; s1.z += acc.z; s1.w += acc.w;
            s2.x = fmaf(acc.x, acc.x, s2.x); s2.y = fmaf(acc.y, acc.y, s2.y);
            s2.z = fmaf(acc.z, acc.z, s2.z); s2.w = fmaf(acc.w, acc.w, s2.w);
        }
    }
    if (!ep.sum) return;
    for (int i = tid; i < 2 * 256 * 4; i += 256) (&red[0][0])[i] = 0.f;
    __syncthreads();
    if (on) {
        const float a1[4] = {s1.x, s1.y, s1.z, s1.w}, a2[4] = {s2.x, s2.y, s2.z, s2.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            atomicAdd(&red[0][cq * 4 + i], a1[i]);
            atomicAdd(&red[1][cq * 4 + i], a2[i]);
        }
    }
    __syncthreads();
    for (int i = tid; i < 256; i += 256) {
        if (n0 + i < Nw) {
            atomicAdd(ep.sum + n0 + i, (double)red[0][i]);
            atomicAdd(ep.sumsq + n0 + i, (double)red[1][i]);
        }
    }
}

template <int KQ>
int launch_fwd_skinny(const ActIn& ain, const float* wt, int ldw, int P, int K, int Nw, const FwdEpi& ep, cudaStream_t st) {
    const int slabs = (Nw + 255) / 256;
    const int mq = (std::min(Nw, 256) + 3) / 4;
    const int LQ = mq <= 16 ? 16 : (mq <= 32 ? 32 : 64);
    const int R = 256 / LQ;
    int want = (4 * o3d_num_sms() + slabs - 1) / slabs;
    int chunk = (P + want - 1) / want;
    chunk = ((chunk + 4 * R - 1) / (4 * R)) * (4 * R);
    const int nx = (P + chunk - 1) / chunk;
    pw_fwd_skinny_kernel<KQ><<<dim3(nx, slabs), 256, 0, st>>>(ain, wt, ldw, P, K, Nw, LQ, chunk, ep);
    O3D_CHECK_LAUNCH("o3d_pw_fwd (skinny)");
    return O3D_OK;
}

// wgrad for a handful of input columns — an xyz-only first layer, or the (dx, dy, dz, 0) / box-cloud extras behind the
// tensor-core part of a first layer:  dW[m, n] += sum_p dY[p, m] * A(X)[p, n],  n < 4*NQ <= 12.
// No tiles: one streaming pass over dY (the only operand of any size), thread = (4 output channels, every R-th position),
// U positions of raw loads in flight per thread, block-level reduction through shared-memory REDs.
template <int NQ, int U>
__global__ void __launch_bounds__(256, 2)
    pw_wgrad_skinny_kernel(DyIn din, ActIn ain, int P, int M, int N, int LQ /*threads per position row*/, int chunk,
                           float* __restrict__ dW, int lddw) {
    __shared__ float red[256 * 4 * NQ];                  // [256 channels][4*NQ columns]
    const int tid = threadIdx.x;
    for (int i = tid; i < 256 * 4 * NQ; i += 256) red[i] = 0.f;
    __syncthreads();
    const int m0 = blockIdx.y * 256;
    const int cq = tid % LQ, r = tid / LQ, R = 256 / LQ;
    const int m = m0 + cq * 4;
    const int pbeg = blockIdx.x * chunk, pend = min(P, pbeg + chunk);
    float acc[4][4 * NQ];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4 * NQ; ++j) acc[i][j] = 0.f;
    // per-thread constants: the BN-backward coefficients of this thread's 4 channels and the input prologue of the few
    // columns (left inside finish_*() the compiler re-loads them for every position)
    const bool on = m < M;
    float4 ca = make_float4(1.f, 1.f, 1.f, 1.f), cb = make_float4(0.f, 0.f, 0.f, 0.f), ccf = cb;
    if (on && din.a) { ca = ld4(din.a + m); cb = ld4(din.b + m); ccf = ld4(din.cc + m); }
    float4 xs[NQ], xt[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) {
        xs[q] = make_float4(1.f, 1.f, 1.f, 1.f);
        xt[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ain.scale && q * 4 < N) { xs[q] = ld4(ain.scale + q * 4); xt[q] = ld4(ain.shift + q * 4); }
    }
    for (int p = pbeg + r; p < pend; p += U * R) {
        DyRaw d[U];
        ActRaw x[U][NQ];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            d[u] = fetch_dy(din, p + u * R, pend, m, M);
#pragma unroll
            for (int q = 0; q < NQ; ++q) x[u][q] = fetch_act(ain, p + u * R, pend, q * 4, N);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!(on && p + u * R < pend)) continue;          // outside the slice / channel range: contributes nothing
            float4 v = d[u].g;
            if (din.a) {
                const float4 yy = d[u].y;
                v.x = fmaf(ca.x, v.x, fmaf(ccf.x, yy.x, cb.x)); v.y = fmaf(ca.y, v.y, fmaf(ccf.y, yy.y, cb.y));
                v.z = fmaf(ca.z, v.z, fmaf(ccf.z, yy.z, cb.z)); v.w = fmaf(ca.w, v.w, fmaf(ccf.w, yy.w, cb.w));
            }
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                if (q * 4 >= N) continue;
                float4 xv = x[u][q].v;
                if (ain.scale) {
                    xv.x = fmaf(xv.x, xs[q].x, xt[q].x); xv.y = fmaf(xv.y, xs[q].y, xt[q].y);
                    xv.z = fmaf(xv.z, xs[q].z, xt[q].z); xv.w = fmaf(xv.w, xs[q].w, xt[q].w);
                }
                if (ain.relu) { xv.x = fmaxf(xv.x, 0.f); xv.y = fmaxf(xv.y, 0.f); xv.z = fmaxf(xv.z, 0.f); xv.w = fmaxf(xv.w, 0.f); }
                const float xx[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][q * 4 + j] = fmaf(vv[i], xx[j], acc[i][q * 4 + j]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4 * NQ; ++j) atomicAdd(&red[(cq * 4 + i) * 4 * NQ + j], acc[i][j]);
    __syncthreads();
    for (int i = tid; i < 256 * 4 * NQ; i += 256) {
        const int mm = m0 + i / (4 * NQ), n = i % (4 * NQ);
        if (mm < M && n < N) atomicAdd(dW + (size_t)mm * lddw + n, red[i]);
    }
}

template <int NQ, int U>
int launch_wgrad_skinny(const DyIn& din, const ActIn& ain, int P, int Cout, int Cin, float* dw, int lddw, cudaStream_t st) {
    const int slabs = (Cout + 255) / 256;
    const int mq = (std::min(Cout, 256) + 3) / 4;
    const int LQ = mq <= 16 ? 16 : (mq <= 32 ? 32 : 64);
    const int R = 256 / LQ;
    int want = (2 * o3d_num_sms() + slabs - 1) / slabs;
    int chunk = (P + want - 1) / want;
    chunk = ((chunk + U * R - 1) / (U * R)) * (U * R);
    const int nx = (P + chunk - 1) / chunk;
    pw_wgrad_skinny_kernel<NQ, U><<<dim3(nx, slabs), 256, 0, st>>>(din, ain, P, Cout, Cin, LQ, chunk, dw, lddw);
    O3D_CHECK_LAUNCH("o3d_pw_wgrad (skinny)");
    return O3D_OK;
}

// ------------------------------------------------------------------------------------------------------------
// Small per-channel kernels
__global__ void bn_fwd_finalize_kernel(const double* __restrict__ sum, const double* __restrict__ sumsq, double count,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       float* __restrict__ rmean, float* __restrict__ rvar, long long* __restrict__ nbt,
                                       float momentum, float eps, int training, int C, float* __restrict__ scale,
                                       float* __restrict__ shift, float* __restrict__ mean, float* __restrict__ invstd) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0 && training && nbt) *nbt += 1;
    if (c >= C) return;
    float mu, istd;
    if (training) {
        const double m = sum[c] / count;
        double var = sumsq[c] / count - m * m;
        if (var < 0.0) var = 0.0;
        mu = (float)m;
        istd = (float)(1.0 / sqrt(var + (double)eps));
        if (rmean) {
            const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
            rmean[c] = (1.f - momentum) * rmean[c] + momentum * mu;
            rvar[c] = (1.f - momentum) * rvar[c] + momentum * (float)unbiased;
        }
    } else {
        mu = rmean[c];
        istd = 1.0f / sqrtf(rvar[c] + eps);
    }
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    const float sc = g * istd;
    scale[c] = sc;
    shift[c] = b - mu * sc;
    mean[c] = mu;
    invstd[c] = istd;
}

// from s1 = sum g, s2y = sum g*y:  dgamma, dbeta and the coefficients of dY = a*g + b + cc*y
__global__ void bn_bwd_finalize_kernel(const double* __restrict__ s1, const double* __restrict__ s2y, double count,
                                       const float* __restrict__ gamma, const float* __restrict__ mean,
                                       const float* __restrict__ invstd, int training, int C, float* __restrict__ a,
                                       float* __restrict__ b, float* __restrict__ cc, float* __restrict__ dgamma,
                                       float* __restrict__ dbeta) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const double mu = mean[c], istd = invstd[c], g = gamma ? gamma[c] : 1.0;
    const double sum_g = s1[c];
    const double sum_gx = (s2y[c] - mu * sum_g) * istd;  // sum g * xhat
    const bool acc = (training & 2) != 0;          // bit 1: accumulate into dgamma / dbeta (caller-owned .grad buffers)
    training &= 1;
    if (dgamma) dgamma[c] = (acc ? dgamma[c] : 0.f) + (float)sum_gx;
    if (dbeta) dbeta[c] = (acc ? dbeta[c] : 0.f) + (float)sum_g;
    const double aa = g * istd;
    if (training) {
        const double c2 = -aa * istd * sum_gx / count;
        a[c] = (float)aa;
        cc[c] = (float)c2;
        b[c] = (float)(-aa * sum_g / count - c2 * mu);
    } else {
        a[c] = (float)aa;
        cc[c] = 0.f;
        b[c] = 0.f;
    }
}

// pooled output: out[g,c] = act(scale*ysel + shift), ysel = scale >= 0 ? ymax : ymin; sel = matching arg
__global__ void pool_finalize_kernel(const float* __restrict__ ymax, const float* __restrict__ ymin,
                                     const int32_t* __restrict__ arg, const float* __restrict__ scale,
                                     const float* __restrict__ shift, int relu, long long total, int C, int ldp,
                                     float* __restrict__ out, int ldo, int32_t* __restrict__ sel,
                                     float* __restrict__ ysel) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long g = i / C;
    const int c = (int)(i % C);
    const float sc = scale ? scale[c] : 1.f, sh = shift ? shift[c] : 0.f;
    const size_t o = (size_t)g * ldp + c;
    const bool pos = sc >= 0.f;
    const float y = pos ? ymax[o] : ymin[o];
    float v = fmaf(y, sc, sh);
    if (relu) v = fmaxf(v, 0.f);
    out[(size_t)g * ldo + c] = v;
    if (sel) sel[o] = pos ? (arg[o] & 0xFFFF) : (arg[o] >> 16);
    if (ysel) ysel[o] = y;
}

// Row-streaming helpers of the two "prep" kernels below: block = 128 channels x 4 row lanes, every thread walks its rows
// four at a time (independent loads first), the 4 row lanes are combined through shared memory, one fp64 RED per channel
// and block.
constexpr int PREP_LANES = 4, PREP_UNROLL = 4;
__device__ __forceinline__ void prep_reduce(float t1, float t2, int c, int C, double* s1, double* s2y) {
    __shared__ float red[2][PREP_LANES][128];
    red[0][threadIdx.y][threadIdx.x] = t1;
    red[1][threadIdx.y][threadIdx.x] = t2;
    __syncthreads();
    if (threadIdx.y == 0 && c < C) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int l = 0; l < PREP_LANES; ++l) { a += red[0][l][threadIdx.x]; b += red[1][l][threadIdx.x]; }
        if (s1) atomicAdd(s1 + c, (double)a);
        if (s2y) atomicAdd(s2y + c, (double)b);
    }
}

// backward of the pooled activation: dpool = dout * [out > 0] (if relu); column sums of dpool and dpool*ysel
__global__ void __launch_bounds__(128 * PREP_LANES)
    pool_bwd_prep_kernel(const float* __restrict__ dout, int ldd, const float* __restrict__ out, int ldo,
                         const float* __restrict__ ysel, int relu, int G, int C, int ldp, float* __restrict__ dpool,
                         double* __restrict__ s1, double* __restrict__ s2y) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    const int cc = c < C ? c : C - 1;
    float t1 = 0.f, t2 = 0.f;
    const int step = gridDim.y * PREP_LANES;
    for (int g0 = blockIdx.y * PREP_LANES + threadIdx.y; g0 < G; g0 += step * PREP_UNROLL) {
        float d[PREP_UNROLL], o[PREP_UNROLL], ys[PREP_UNROLL];
#pragma unroll
        for (int u = 0; u < PREP_UNROLL; ++u) {
            const int g = min(g0 + u * step, G - 1);
            d[u] = dout[(size_t)g * ldd + cc];
            o[u] = relu ? out[(size_t)g * ldo + cc] : 1.f;
            ys[u] = ysel[(size_t)g * ldp + cc];
        }
#pragma unroll
        for (int u = 0; u < PREP_UNROLL; ++u) {
            const int g = g0 + u * step;
            if (g >= G || c >= C) continue;
            const float v = (relu && !(o[u] > 0.f)) ? 0.f : d[u];
            dpool[(size_t)g * ldp + c] = v;
            t1 += v;
            t2 = fmaf(v, ys[u], t2);
        }
    }
    prep_reduce(t1, t2, c, C, s1, s1 ? s2y : nullptr);
}

// dense activation (no pooling): out = act(scale*y + shift)
__global__ void act_apply_kernel(const float* __restrict__ y, int ldy, const float* __restrict__ scale,
                                 const float* __restrict__ shift, int relu, long long total, int C,
                                 float* __restrict__ out, int ldo) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const long long p = i / C;
    const int c = (int)(i % C);
    float v = y[(size_t)p * ldy + c];
    if (scale) v = fmaf(v, scale[c], shift[c]);
    if (relu) v = fmaxf(v, 0.f);
    out[(size_t)p * ldo + c] = v;
}

// dense backward prep: g = dout * [out > 0] (if relu); column sums of g and g*y (y nullable -> only s1)
__global__ void __launch_bounds__(128 * PREP_LANES)
    dense_bwd_prep_kernel(const float* __restrict__ dout, int ldd, const float* __restrict__ out, int ldo,
                          const float* __restrict__ y, int ldy, int relu, int P, int C, float* __restrict__ g, int ldg,
                          double* __restrict__ s1, double* __restrict__ s2y) {
    const int c = blockIdx.x * 128 + threadIdx.x;
    const int cc = c < C ? c : C - 1;
    float t1 = 0.f, t2 = 0.f;
    const int step = gridDim.y * PREP_LANES;
    for (int p0 = blockIdx.y * PREP_LANES + threadIdx.y; p0 < P; p0 += step * PREP_UNROLL) {
        float d[PREP_UNROLL], o[PREP_UNROLL], yy[PREP_UNROLL];
#pragma unroll
        for (int u = 0; u < PREP_UNROLL; ++u) {
            const int p = min(p0 + u * step, P - 1);
            d[u] = dout[(size_t)p * ldd + cc];
            o[u] = relu ? out[(size_t)p * ldo + cc] : 1.f;
            yy[u] = y ? y[(size_t)p * ldy + cc] : 0.f;
        }
#pragma unroll
        for (int u = 0; u < PREP_UNROLL; ++u) {
            const int p = p0 + u * step;
            if (p >= P || c >= C) continue;
            const float v = (relu && !(o[u] > 0.f)) ? 0.f : d[u];
            if (g) g[(size_t)p * ldg + c] = v;
            t1 += v;
            t2 = fmaf(v, yy[u], t2);
        }
    }
    prep_reduce(t1, t2, c, C, s1, s2y);
}

template <typename Kern>
int set_smem(Kern k, size_t bytes, const char* name) {
    if (bytes > 48 * 1024) O3D_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes), name);
    return O3D_OK;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace

// ============================================================================================================
extern "C" int o3d_pw_fwd(const float* x, int ldx, const float* in_scale, const float* in_shift, int in_relu,
                          const float* wt, int ldw, const float* bias, int P, int K, int N, float* y, int ldy,
                          double* sum, double* sumsq, int S, float* ymax, float* ymin, int32_t* arg, int ldp,
                          void* stream) {
    O3D_REQUIRE(x && wt, O3D_ERR_ARG, "o3d_pw_fwd: null pointer");
    O3D_REQUIRE(P >= 0 && K >= 4 && N >= 1, O3D_ERR_ARG, "o3d_pw_fwd: bad sizes P=%d K=%d N=%d", P, K, N);
    O3D_REQUIRE((K & 3) == 0 && (ldx & 3) == 0 && (ldw & 3) == 0 && (y == nullptr || (ldy & 3) == 0), O3D_ERR_ARG,
                "o3d_pw_fwd: K and leading dimensions must be multiples of 4 (K=%d ldx=%d ldw=%d ldy=%d)", K, ldx, ldw, ldy);
    O3D_REQUIRE(aligned16(x) && aligned16(wt) && aligned16(y) && aligned16(in_scale) && aligned16(in_shift) && aligned16(bias),
                O3D_ERR_ALIGN, "o3d_pw_fwd: pointers must be 16-byte aligned");
    O3D_REQUIRE(S == 0 || (BM % S == 0 && P % S == 0 && ymax && ymin && arg && (ldp & 3) == 0), O3D_ERR_ARG,
                "o3d_pw_fwd: group size S=%d must divide 128 and P, and pooled buffers are required", S);
    if (P == 0) return O3D_OK;
    const int Nw = (N + 3) & ~3;  // writable columns (pad columns of Y receive the zero-padded product)
    O3D_REQUIRE(ldw >= Nw && (y == nullptr || ldy >= Nw), O3D_ERR_ARG, "o3d_pw_fwd: ldw/ldy smaller than padded N");
    ActIn ain{x, ldx, in_scale, in_shift, in_relu};
    FwdEpi ep{y, ldy, bias, sum, sumsq, S, ymax, ymin, arg, ldp};
    cudaStream_t st = (cudaStream_t)stream;
    if (K <= 8 && S == 0 && P >= 4096) {
        if (K <= 4) return launch_fwd_skinny<1>(ain, wt, ldw, P, K, Nw, ep, st);
        return launch_fwd_skinny<2>(ain, wt, ldw, P, K, Nw, ep, st);
    }
    if (Nw <= 64) {
        if (int e = set_smem(pw_fwd_kernel<64>, Cfg<64>::SMEM_BYTES, "o3d_pw_fwd")) return e;
        dim3 grid((P + BM - 1) / BM, (Nw + 63) / 64);
        pw_fwd_kernel<64><<<grid, NT, Cfg<64>::SMEM_BYTES, st>>>(ain, wt, ldw, P, K, Nw, Nw, ep);
    } else {
        if (int e = set_smem(pw_fwd_kernel<128>, Cfg<128>::SMEM_BYTES, "o3d_pw_fwd")) return e;
        dim3 grid((P + BM - 1) / BM, (Nw + 127) / 128);
        pw_fwd_kernel<128><<<grid, NT, Cfg<128>::SMEM_BYTES, st>>>(ain, wt, ldw, P, K, Nw, Nw, ep);
    }
    O3D_CHECK_LAUNCH("o3d_pw_fwd");
    return O3D_OK;
}

static DyIn make_dy(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                    const float* dpool, const int32_t* sel, int S, int ldp) {
    DyIn d;
    d.g = g; d.ldg = ldg; d.y = y; d.ldy = ldy; d.a = a; d.b = b; d.cc = cc;
    d.dpool = dpool; d.sel = sel; d.S = S > 0 ? S : 1; d.ldp = ldp;
    return d;
}

extern "C" int o3d_pw_dgrad(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b,
                            const float* cc, const float* dpool, const int32_t* sel, int S, int ldp, const float* w,
                            int ldw, int P, int Cout, int Cin, float* out, int ldo, const float* yprev, int ldyp,
                            const float* pscale, const float* pshift, int prelu, double* s1, double* s2y,
                            void* stream) {
    O3D_REQUIRE((g || dpool) && w && out, O3D_ERR_ARG, "o3d_pw_dgrad: null pointer");
    O3D_REQUIRE((Cout & 3) == 0 && (Cin & 3) == 0 && (ldw & 3) == 0 && (ldo & 3) == 0, O3D_ERR_ARG,
                "o3d_pw_dgrad: channel counts / leading dimensions must be multiples of 4");
    O3D_REQUIRE(a == nullptr || y != nullptr, O3D_ERR_ARG, "o3d_pw_dgrad: BN coefficients need y");
    if (P == 0) return O3D_OK;
    DyIn din = make_dy(g, ldg, y, ldy, a, b, cc, dpool, sel, S, ldp);
    DgradEpi ep{out, ldo, yprev, ldyp, pscale, pshift, prelu, s1, s2y};
    cudaStream_t st = (cudaStream_t)stream;
    if (Cin <= 64) {
        if (int e = set_smem(pw_dgrad_kernel<64>, Cfg<64>::SMEM_BYTES, "o3d_pw_dgrad")) return e;
        dim3 grid((P + BM - 1) / BM, (Cin + 63) / 64);
        pw_dgrad_kernel<64><<<grid, NT, Cfg<64>::SMEM_BYTES, st>>>(din, w, ldw, P, Cout, Cin, Cin, ep);
    } else {
        if (int e = set_smem(pw_dgrad_kernel<128>, Cfg<128>::SMEM_BYTES, "o3d_pw_dgrad")) return e;
        dim3 grid((P + BM - 1) / BM, (Cin + 127) / 128);
        pw_dgrad_kernel<128><<<grid, NT, Cfg<128>::SMEM_BYTES, st>>>(din, w, ldw, P, Cout, Cin, Cin, ep);
    }
    O3D_CHECK_LAUNCH("o3d_pw_dgrad");
    return O3D_OK;
}

extern "C" int o3d_pw_wgrad(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b,
                            const float* cc, const float* dpool, const int32_t* sel, int S, int ldp, const float* x,
                            int ldx, const float* in_scale, const float* in_shift, int in_relu, int P, int Cout,
                            int Cin, float* dw, int lddw, void* stream) {
    O3D_REQUIRE((g || dpool) && x && dw, O3D_ERR_ARG, "o3d_pw_wgrad: null pointer");
    O3D_REQUIRE((Cout & 3) == 0 && (Cin & 3) == 0 && (lddw & 3) == 0 && (ldx & 3) == 0, O3D_ERR_ARG,
                "o3d_pw_wgrad: channel counts / leading dimensions must be multiples of 4");
    if (P == 0) return O3D_OK;
    DyIn din = make_dy(g, ldg, y, ldy, a, b, cc, dpool, sel, S, ldp);
    ActIn ain{x, ldx, in_scale, in_shift, in_relu};
    cudaStream_t st = (cudaStream_t)stream;
    if (Cin <= 12 && P >= 4096) {
        if (Cin <= 4) return launch_wgrad_skinny<1, 4>(din, ain, P, Cout, Cin, dw, lddw, st);
        if (Cin <= 8) return launch_wgrad_skinny<2, 2>(din, ain, P, Cout, Cin, dw, lddw, st);
        return launch_wgrad_skinny<3, 2>(din, ain, P, Cout, Cin, dw, lddw, st);
    }
    const int mt = (Cout + BM - 1) / BM;
    const int bn = Cin <= 64 ? 64 : 128;
    const int ntile = (Cin + bn - 1) / bn;
    // split P so that the grid covers ~4 waves of the SMs, in multiples of BK positions
    int want = (4 * o3d_num_sms() + mt * ntile - 1) / (mt * ntile);
    int chunk = (P + want - 1) / want;
    chunk = ((chunk + BK - 1) / BK) * BK;
    if (chunk < 4 * BK) chunk = 4 * BK;
    const int nz = (P + chunk - 1) / chunk;
    O3D_REQUIRE(nz <= 65535, O3D_ERR_ARG, "o3d_pw_wgrad: too many position slices");
    dim3 grid(mt, ntile, nz);
    if (bn == 64) {
        if (int e = set_smem(pw_wgrad_kernel<64>, Cfg<64>::SMEM_BYTES, "o3d_pw_wgrad")) return e;
        pw_wgrad_kernel<64><<<grid, NT, Cfg<64>::SMEM_BYTES, st>>>(din, ain, P, Cout, Cin, chunk, dw, lddw);
    } else {
        if (int e = set_smem(pw_wgrad_kernel<128>, Cfg<128>::SMEM_BYTES, "o3d_pw_wgrad")) return e;
        pw_wgrad_kernel<128><<<grid, NT, Cfg<128>::SMEM_BYTES, st>>>(din, ain, P, Cout, Cin, chunk, dw, lddw);
    }
    O3D_CHECK_LAUNCH("o3d_pw_wgrad");
    return O3D_OK;
}

extern "C" int o3d_bn_fwd_finalize(const double* sum, const double* sumsq, double count, const float* gamma,
                                   const float* beta, float* running_mean, float* running_var,
                                   long long* num_batches_tracked, float momentum, float eps, int training, int C,
                                   float* scale, float* shift, float* mean, float* invstd, void* stream) {
    O3D_REQUIRE(scale && shift && mean && invstd && C >= 1, O3D_ERR_ARG, "o3d_bn_fwd_finalize: null pointer");
    O3D_REQUIRE(training ? (sum && sumsq) : (running_mean && running_var), O3D_ERR_ARG,
                "o3d_bn_fwd_finalize: statistics missing");
    bn_fwd_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        sum, sumsq, count, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, training, C, scale,
        shift, mean, invstd);
    O3D_CHECK_LAUNCH("o3d_bn_fwd_finalize");
    return O3D_OK;
}

extern "C" int o3d_bn_bwd_finalize(const double* s1, const double* s2y, double count, const float* gamma,
                                   const float* mean, const float* invstd, int training, int C, float* a, float* b,
                                   float* cc, float* dgamma, float* dbeta, void* stream) {
    O3D_REQUIRE(s1 && s2y && mean && invstd && a && b && cc, O3D_ERR_ARG, "o3d_bn_bwd_finalize: null pointer");
    bn_bwd_finalize_kernel<<<(C + 127) / 128, 128, 0, (cudaStream_t)stream>>>(s1, s2y, count, gamma, mean, invstd,
                                                                                training, C, a, b, cc, dgamma, dbeta);
    O3D_CHECK_LAUNCH("o3d_bn_bwd_finalize");
    return O3D_OK;
}

extern "C" int o3d_pool_finalize(const float* ymax, const float* ymin, const int32_t* arg, const float* scale,
                                 const float* shift, int relu, int G, int C, int ldp, float* out, int ldo, int32_t* sel,
                                 float* ysel, void* stream) {
    O3D_REQUIRE(ymax && ymin && arg && out, O3D_ERR_ARG, "o3d_pool_finalize: null pointer");
    const long long total = (long long)G * C;
    if (total == 0) return O3D_OK;
    pool_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        ymax, ymin, arg, scale, shift, relu, total, C, ldp, out, ldo, sel, ysel);
    O3D_CHECK_LAUNCH("o3d_pool_finalize");
    return O3D_OK;
}

extern "C" int o3d_pool_bwd_prep(const float* dout, int ldd, const float* out, int ldo, const float* ysel, int relu,
                                 int G, int C, int ldp, float* dpool, double* s1, double* s2y, void* stream) {
    O3D_REQUIRE(dout && out && ysel && dpool, O3D_ERR_ARG, "o3d_pool_bwd_prep: null pointer");
    if (G == 0) return O3D_OK;
    int gy = (G + PREP_LANES * PREP_UNROLL - 1) / (PREP_LANES * PREP_UNROLL);   // one unrolled pass per thread ...
    const int cap = 4 * o3d_num_sms() / ((C + 127) / 128);                       // ... up to ~4 blocks per SM
    if (gy > cap) gy = cap;
    if (gy < 1) gy = 1;
    dim3 grid((C + 127) / 128, gy);
    pool_bwd_prep_kernel<<<grid, dim3(128, PREP_LANES), 0, (cudaStream_t)stream>>>(dout, ldd, out, ldo, ysel, relu, G, C, ldp, dpool, s1,
                                                                  s2y);
    O3D_CHECK_LAUNCH("o3d_pool_bwd_prep");
    return O3D_OK;
}

extern "C" int o3d_act_apply(const float* y, int ldy, const float* scale, const float* shift, int relu, int P, int C,
                             float* out, int ldo, void* stream) {
    O3D_REQUIRE(y && out, O3D_ERR_ARG, "o3d_act_apply: null pointer");
    const long long total = (long long)P * C;
    if (total == 0) return O3D_OK;
    act_apply_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(y, ldy, scale, shift, relu,
                                                                                         total, C, out, ldo);
    O3D_CHECK_LAUNCH("o3d_act_apply");
    return O3D_OK;
}

extern "C" int o3d_dense_bwd_prep(const float* dout, int ldd, const float* out, int ldo, const float* y, int ldy,
                                  int relu, int P, int C, float* g, int ldg, double* s1, double* s2y, void* stream) {
    O3D_REQUIRE(dout, O3D_ERR_ARG, "o3d_dense_bwd_prep: null pointer");
    O3D_REQUIRE(!relu || out, O3D_ERR_ARG, "o3d_dense_bwd_prep: relu mask needs the forward output");
    if (P == 0) return O3D_OK;
    int gy = (P + PREP_LANES * PREP_UNROLL - 1) / (PREP_LANES * PREP_UNROLL);
    const int cap = 4 * o3d_num_sms() / ((C + 127) / 128);
    if (gy > cap) gy = cap;
    if (gy < 1) gy = 1;
    dim3 grid((C + 127) / 128, gy);
    dense_bwd_prep_kernel<<<grid, dim3(128, PREP_LANES), 0, (cudaStream_t)stream>>>(dout, ldd, out, ldo, y, ldy, relu, P, C, g, ldg, s1,
                                                                   s2y);
    O3D_CHECK_LAUNCH("o3d_dense_bwd_prep");
    return O3D_OK;
}
