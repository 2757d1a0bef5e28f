// Furthest point sampling for sm_100a.
//
// Replaces `_ext.furthest_point_sampling` (reference call site pointnet2/utils/pointnet2_utils.py:56;
// upstream kernel furthest_point_sampling_kernel<block> in pointnet2_ops, see oracle/pointnet2_ops_ref.c).
//
// Design: one persistent CTA per cloud (the npoint-long dependency chain is the only serial axis, the
// batch is the only parallel one).  The cloud lives in registers: every thread owns PPT points
// (x,y,z, running min-distance) for the whole kernel; coordinates are also staged once in shared
// memory so the winner's xyz can be broadcast with one LDS.  Each iteration is
//   PPT x (3 FSUB + FMUL + 2 FFMA + FMNMX + compare)  ->  warp REDUX.max / REDUX.min
//   -> one STS per warp -> ONE __syncthreads (double-buffered slots) -> LDS + REDUX.max/min
// i.e. no shared-memory tree and no global `temp` array (upstream: 9 barrier levels + B*N floats in HBM).
//
// Bit-exactness.  Upstream's result depends on its reduction tree: thread t scans k = t, t+block, ...
// with a strict '>' (lowest k wins inside a thread) and the shared-memory tree keeps the LEFT operand
// on ties, which makes the winner among equal distances the one with the smallest
//     prio(k) = bitrev_{log2 block}(k mod block) * ceil(N/block) + (k div block),   block = opt_n_threads(N).
// We therefore take the arg-max over the total order (distance desc, prio asc); any reduction shape then
// yields upstream's index.  Distances use the same contraction nvcc applies upstream (common.cuh o3d_sq3).
// Points with x^2+y^2+z^2 <= 1e-3 (compared in double, as upstream's float-vs-double-literal test does)
// never update and never win; if no point is eligible the index is 0.
#include "common.cuh"
#include "../../include/o3d_b200.h"

namespace {

struct FpsParams {
    int N, npoint;
    int block_ref;   // opt_n_threads(N) of the upstream launch (defines the tie order)
    int log2_block;  // log2(block_ref)
    int cnt;         // ceil(N / block_ref)
};

__device__ __forceinline__ uint32_t fps_bitrev(uint32_t t, int log2_block) {
    return log2_block == 0 ? 0u : (__brev(t) >> (32 - log2_block));
}

template <int THREADS, int PPT>
__global__ void __launch_bounds__(THREADS) fps_kernel(const float* __restrict__ xyz, int32_t* __restrict__ idx,
                                                      FpsParams prm) {
    extern __shared__ __align__(16) float s_xyz[];  // 3*N floats, then block_ref*cnt uint16: priority -> point index
    constexpr int NW = THREADS / 32;
    __shared__ uint32_t s_key[2][NW];
    __shared__ uint32_t s_pri[2][NW];

    const int N = prm.N, npoint = prm.npoint;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* __restrict__ p = xyz + (size_t)blockIdx.x * N * 3;
    int32_t* __restrict__ out = idx + (size_t)blockIdx.x * npoint;

    uint16_t* s_dec = reinterpret_cast<uint16_t*>(s_xyz + 3 * N);   // decode table: a winner's priority -> its index (one LDS instead
                                                                   // of a runtime integer division + modulo + bit reversal per iteration)
    for (int i = tid; i < 3 * N; i += THREADS) s_xyz[i] = p[i];
    __syncthreads();

    float px[PPT], py[PPT], pz[PPT], td[PPT];
    uint32_t pri[PPT];
#pragma unroll
    for (int i = 0; i < PPT; ++i) {
        const int k = tid + i * THREADS;
        px[i] = py[i] = pz[i] = 0.f;
        td[i] = 1e10f;
        pri[i] = 0xFFFFFFFFu;  // 0xFFFFFFFF marks "never a candidate"
        if (k < N) {
            px[i] = s_xyz[k * 3 + 0];
            py[i] = s_xyz[k * 3 + 1];
            pz[i] = s_xyz[k * 3 + 2];
            const float mag = o3d_sq3(px[i], py[i], pz[i]);
            if (!((double)mag <= 1e-3)) {
                pri[i] = fps_bitrev((uint32_t)(k % prm.block_ref), prm.log2_block) * (uint32_t)prm.cnt +
                         (uint32_t)(k / prm.block_ref);
                s_dec[pri[i]] = (uint16_t)k;        // N <= 16384; priorities of eligible points are distinct and < block_ref * cnt
            }
        }
    }
    __syncthreads();

    int old = 0;
    if (tid == 0) out[0] = 0;

    for (int j = 1; j < npoint; ++j) {
        const float x1 = s_xyz[old * 3 + 0], y1 = s_xyz[old * 3 + 1], z1 = s_xyz[old * 3 + 2];
        // per-point keys first (independent), then a pairwise tournament: the dependent compare chain is log2(PPT) deep
        uint32_t ck[PPT], cp[PPT];  // key 0 == "no candidate" (upstream: best = -1, besti = 0)
#pragma unroll
        for (int i = 0; i < PPT; ++i) {
            const float d = o3d_dist2(px[i], py[i], pz[i], x1, y1, z1);
            const float d2 = fminf(d, td[i]);
            const bool live = pri[i] != 0xFFFFFFFFu;
            td[i] = live ? d2 : td[i];
            ck[i] = live ? __float_as_uint(d2) + 1u : 0u;  // d2 >= +0 -> bit pattern is monotone
            cp[i] = pri[i];
        }
#pragma unroll
        for (int w = 1; w < PPT; w <<= 1) {
#pragma unroll
            for (int i = 0; i + w < PPT; i += 2 * w) {
                const bool take = ck[i + w] > ck[i] || (ck[i + w] == ck[i] && cp[i + w] < cp[i]);
                ck[i] = take ? ck[i + w] : ck[i];
                cp[i] = take ? cp[i + w] : cp[i];
            }
        }
        const uint32_t bk = ck[0], bp = cp[0];
        const uint32_t wm = __reduce_max_sync(0xFFFFFFFFu, bk);
        const uint32_t wp = __reduce_min_sync(0xFFFFFFFFu, bk == wm ? bp : 0xFFFFFFFFu);
        const int buf = j & 1;
        if (lane == 0) {
            s_key[buf][warp] = wm;
            s_pri[buf][warp] = wp;
        }
        __syncthreads();
        const uint32_t k2 = lane < NW ? s_key[buf][lane] : 0u;
        const uint32_t p2 = lane < NW ? s_pri[buf][lane] : 0xFFFFFFFFu;
        const uint32_t m2 = __reduce_max_sync(0xFFFFFFFFu, k2);
        const uint32_t q2 = __reduce_min_sync(0xFFFFFFFFu, k2 == m2 ? p2 : 0xFFFFFFFFu);
        old = m2 == 0u ? 0 : (int)s_dec[q2];
        if (tid == 0) out[j] = old;
    }
}

template <int THREADS, int PPT>
int launch_fps(const float* xyz, int B, int32_t* idx, const FpsParams& prm, cudaStream_t st) {
    const size_t smem = (size_t)prm.N * 3 * sizeof(float) + (size_t)prm.block_ref * prm.cnt * sizeof(uint16_t);
    if (smem > 48 * 1024)
        O3D_CUDA(cudaFuncSetAttribute(fps_kernel<THREADS, PPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem),
                 "o3d_fps: smem attribute");
    fps_kernel<THREADS, PPT><<<B, THREADS, smem, st>>>(xyz, idx, prm);
    O3D_CHECK_LAUNCH("o3d_fps");
    return O3D_OK;
}

}  // namespace

extern "C" int o3d_fps(const float* xyz, int B, int N, int npoint, int32_t* idx, void* stream) {
    O3D_REQUIRE(xyz && idx, O3D_ERR_ARG, "o3d_fps: null pointer");
    O3D_REQUIRE(B >= 0 && N >= 1 && npoint >= 0, O3D_ERR_ARG, "o3d_fps: bad sizes B=%d N=%d npoint=%d", B, N, npoint);
    O3D_REQUIRE(N <= 16384, O3D_ERR_ARG, "o3d_fps: N=%d exceeds the supported 16384 points per cloud", N);
    if (B == 0 || npoint == 0) return O3D_OK;
    FpsParams prm;
    prm.N = N;
    prm.npoint = npoint;
    prm.block_ref = o3d_opt_n_threads(N);
    prm.log2_block = 0;
    while ((1 << prm.log2_block) < prm.block_ref) ++prm.log2_block;
    prm.cnt = (N + prm.block_ref - 1) / prm.block_ref;
    cudaStream_t st = (cudaStream_t)stream;
    // measured on B200 (48 clouds): 128 threads x 8 points = 1,170 cycles per iteration at N = 1024; spreading the points over
    // more warps shortens the per-thread chain (the second-level reduction handles up to 32 warps in one step)
    if (N <= 128) return launch_fps<128, 1>(xyz, B, idx, prm, st);
    if (N <= 256) return launch_fps<128, 2>(xyz, B, idx, prm, st);
    // measured, N = 1024 -> 512 (cycles per iteration at 1965 MHz): 128 x 8: 1,170 (round 1) | 256 x 4: 660 | 512 x 2: 427 | 1024 x 1:
    // tried, slower; no time recorded;  N = 512 -> 256: 256 x 2: 330 | 512 x 1: 338.  Tried and dropped: a (x, y, z, index) float4 decode table
    // (one 16-byte LDS instead of the index lookup + three dependent coordinate loads): 512 x 2 went from 107 us to 145 us;
    // the block-level arg-max as one 64-bit shared-memory atomicMax of (key << 32 | ~priority) per warp instead of three of the
    // four warp reductions: 64-bit shared atomics compile to an LDS + ATOMS.CAS retry loop, and resampled clouds are full of
    // exact duplicates (ties -> many lanes enter it): 110 -> 233 us.
    if (N <= 512) return launch_fps<256, 2>(xyz, B, idx, prm, st);
    if (N <= 1024) return launch_fps<512, 2>(xyz, B, idx, prm, st);
    if (N <= 2048) return launch_fps<256, 8>(xyz, B, idx, prm, st);
    if (N <= 4096) return launch_fps<256, 16>(xyz, B, idx, prm, st);
    if (N <= 8192) return launch_fps<512, 16>(xyz, B, idx, prm, st);
    return launch_fps<512, 32>(xyz, B, idx, prm, st);
}
