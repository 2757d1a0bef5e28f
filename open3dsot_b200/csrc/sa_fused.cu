// A whole PointNet++ set-abstraction layer in ONE kernel — inference (static weights, running BatchNorm statistics).
//
// Replaces, for eval-mode forward passes, the body of _PointnetSAModuleBase.forward (pointnet2/utils/pointnet2_modules.py:58-76):
//   QueryAndGroup (ball_query + 2x group_points + centre subtraction [+ /radius] + cat, pointnet2_utils.py:299-339),
//   the SharedMLP (conv1x1 + BatchNorm(running stats) + ReLU, pt_utils.py) and the max-pool over nsample (F.max_pool2d).
// The training path (stack.cu: lifted first layer, batch statistics, saved tensors for the backward) keeps its multi-kernel
// form; this kernel is what the B = 1 tracking loop and model.eval() forward passes run.
//
// One CTA owns 64 positions = 64 / nsample neighbouring centres of one cloud and carries them through every layer:
//   A. the cloud's coordinates are staged into shared memory, one warp per centre runs the ball query (same code and order
//      as ball_query.cu) and keeps idx[64] and (dx, dy, dz)[64] in shared memory;
//   B. the 64 neighbour feature rows are gathered (coalesced 128-byte segments), split into TF32 hi / lo parts and stored as
//      the K-major SWIZZLE_128B activation operand (k-blocks of 32 channels: hi [64 x 128 B] | lo [64 x 128 B]);
//   C. per layer, the MMA warp issues 3xTF32 tcgen05.mma (M = 128 output channels, N = 64 positions, K = 8) over all
//      k-blocks, weights arriving as pre-tiled hi | lo images (o3d_sa_fused_prepare) through a bulk-copy ring that runs
//      ahead across layers; accumulators live in TMEM (64 columns per 128-channel tile).  The eight epilogue warps read them
//      back (tcgen05.ld), add the coordinate term of the first layer W0[:, 0:3] . (dx, dy, dz) with plain FMAs (exact fp32 —
//      the same split as the training path's lifted first layer), apply the folded BatchNorm + ReLU and write the result, hi /
//      lo split, over the activation operand IN PLACE: the layer's output never leaves the SM;
//   D. the last layer's epilogue max-pools over each centre's nsample positions in registers and stores one channels-last
//      row per centre.
// HBM / L2 traffic per CTA: the cloud's coordinates, 64 feature rows, the weight images, 64 / nsample output rows.
//
//   warps 0-7: query / gather / epilogue (warp % 4 = the TMEM lane quarter it may read) | 8: MMA issuer, TMEM alloc |
//   9: weight streamer
#include <type_traits>
#include "common.cuh"
#include "ball_query.cuh"
#include "tc_ptx.cuh"
#include "../../include/o3d_b200.h"

namespace {

constexpr int SF_POS = 64;                  // positions per CTA
constexpr int SF_THREADS = 320;
constexpr int SF_ACT_KB = 2 * SF_POS * 128; // bytes per activation k-block: hi | lo
constexpr int SF_WTILE = 2 * TILE_BYTES;    // one weight tile (128 channels x 32 k): hi | lo
constexpr int SF_MAX_SLOTS = 6;
constexpr int SF_MISC = 128 + SF_POS * 4 + SF_POS * 16;   // barriers + TMEM slot | idx | rel
constexpr uint32_t SF_TMEM_COLS = 128;      // two 128-channel tiles x 64 positions

__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t a, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_v4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}

struct SfLayer {
    int cout, n_mt, nkb, relu, mma;
    uint32_t vec_off;      // floats from the block start: scale[n_mt * 128] | shift[n_mt * 128]
};
struct SfParams {
    int n, Cp, ldf, N, M, S, BM;
    float radius, radius2;
    int normalize;
    int act_bytes, nslot;
    uint32_t wx_off;       // floats: W0's coordinate columns, [3][n_mt0 * 128]
    uint32_t tiles_off;    // bytes: weight tiles in consumption order (layer, channel tile, k-block)
    SfLayer l[O3D_MAX_LAYERS];
};

__global__ void __launch_bounds__(SF_THREADS, 2)
    sa_fused_kernel(const SfParams prm, const uint8_t* __restrict__ block, const float* __restrict__ xyz,
                    const float* __restrict__ new_xyz, const float* __restrict__ feat, float* __restrict__ out, int ldo,
                    int32_t* __restrict__ idx_out) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* act = smem;
    uint8_t* ring = smem + prm.act_bytes;
    uint8_t* misc = ring + prm.nslot * SF_WTILE;
    uint64_t* full = reinterpret_cast<uint64_t*>(misc);       // [SF_MAX_SLOTS] weight tile landed
    uint64_t* empty = full + SF_MAX_SLOTS;                    // [SF_MAX_SLOTS] MMAs reading the slot retired
    uint64_t* act_ready = empty + SF_MAX_SLOTS;               // activation operand of the next layer written (256 arrivals)
    uint64_t* layer_done = act_ready + 1;                     // every MMA of the layer retired
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(layer_done + 1);
    int32_t* s_idx = reinterpret_cast<int32_t*>(misc + 128);
    float4* s_rel = reinterpret_cast<float4*>(misc + 128 + SF_POS * 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nslot = prm.nslot;
    const bool mma0 = prm.l[0].mma != 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < SF_MAX_SLOTS; ++s) {
            o3d_mbar_init(full + s, 1);
            o3d_mbar_init(empty + s, 1);
        }
        o3d_mbar_init(act_ready, 256);
        o3d_mbar_init(layer_done, 1);
        o3d_fence_mbar_init();
    }
    if (warp == 8) tmem_alloc(tmem_slot, SF_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 8) {
        // ===================================================== MMA issuer
        const uint32_t idesc = make_idesc(TC_M, SF_POS);
        int slot = 0, phase = 0, ar = 0;
        for (int l = 0; l < prm.n; ++l) {
            const SfLayer& L = prm.l[l];
            if (!L.mma) continue;
            o3d_mbar_wait(act_ready, ar);
            ar ^= 1;
            tc_fence_after();
            for (int mt = 0; mt < L.n_mt; ++mt) {
                for (int kb = 0; kb < L.nkb; ++kb) {
                    o3d_mbar_wait(full + slot, phase);
                    tc_fence_after();
                    if (lane == 0) {
                        const uint32_t wb = o3d_smem_u32(ring + slot * SF_WTILE);
                        const uint32_t ab = o3d_smem_u32(act + kb * SF_ACT_KB);
                        const uint64_t whi = make_desc(wb), wlo = make_desc(wb + TILE_BYTES);
                        const uint64_t xhi = make_desc(ab), xlo = make_desc(ab + SF_ACT_KB / 2);
                        const uint32_t d_tmem = tmem_base + (uint32_t)(mt * SF_POS);
#pragma unroll
                        for (int ks = 0; ks < TC_K / 8; ++ks) {
                            const uint64_t adv = (uint64_t)((ks * 32) >> 4);   // +32 bytes along K inside the 128-byte swizzle row
                            umma_tf32(d_tmem, wlo + adv, xhi + adv, idesc, (kb | ks) != 0);
                            umma_tf32(d_tmem, whi + adv, xlo + adv, idesc, 1u);
                            umma_tf32(d_tmem, whi + adv, xhi + adv, idesc, 1u);
                        }
                        umma_commit(empty + slot);
                        if (mt == L.n_mt - 1 && kb == L.nkb - 1) umma_commit(layer_done);
                    }
                    __syncwarp();
                    if (++slot == nslot) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 9) {
        // ===================================================== weight streamer: runs ahead of the MMA warp, across layers
        if (lane == 0) {
            const uint8_t* src = block + prm.tiles_off;
            int slot = 0, phase = 0;
            for (int l = 0; l < prm.n; ++l) {
                const SfLayer& L = prm.l[l];
                if (!L.mma) continue;
                for (int t = 0; t < L.n_mt * L.nkb; ++t) {
                    o3d_mbar_wait(empty + slot, phase ^ 1);
                    o3d_mbar_expect_tx(full + slot, SF_WTILE);
                    o3d_bulk_g2s(ring + slot * SF_WTILE, src, SF_WTILE, full + slot);
                    src += SF_WTILE;
                    if (++slot == nslot) { slot = 0; phase ^= 1; }
                }
            }
        }
    } else {
        // ===================================================== query / gather / epilogue (256 threads)
        const int tid = threadIdx.x;
        const int S = prm.S, N = prm.N, M = prm.M;
        const int cpc = SF_POS / S;                     // centres of this CTA
        const int g0 = blockIdx.x * cpc;                // first centre, global over B * M (M % cpc == 0: one cloud per CTA)
        const int b = g0 / M;
        // ---- A. ball query
        float* s_xyz = reinterpret_cast<float*>(act);
        const float* cloud = xyz + (size_t)b * N * 3;
        for (int i = tid; i < 3 * N; i += 256) s_xyz[i] = __ldg(cloud + i);
        asm volatile("bar.sync 1, 256;" ::: "memory");
        for (int ci = warp; ci < cpc; ci += 8) {
            const int g = g0 + ci;
            int32_t* o = s_idx + ci * S;
            if (g < prm.BM) {
                const float* c = new_xyz + (size_t)g * 3;
                const float cx = __ldg(c), cy = __ldg(c + 1), cz = __ldg(c + 2);
                warp_ball_query(s_xyz, N, cx, cy, cz, prm.radius2, S, o, lane);
                __syncwarp();
                for (int i = lane; i < S; i += 32) {
                    const int k = o[i];
                    float dx = __fsub_rn(s_xyz[k * 3 + 0], cx), dy = __fsub_rn(s_xyz[k * 3 + 1], cy),
                          dz = __fsub_rn(s_xyz[k * 3 + 2], cz);
                    if (prm.normalize) {
                        dx = __fdiv_rn(dx, prm.radius);
                        dy = __fdiv_rn(dy, prm.radius);
                        dz = __fdiv_rn(dz, prm.radius);
                    }
                    s_rel[ci * S + i] = make_float4(dx, dy, dz, 0.f);
                    if (idx_out) idx_out[(size_t)g * S + i] = k;
                }
            } else {
                for (int i = lane; i < S; i += 32) {
                    o[i] = 0;
                    s_rel[ci * S + i] = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            __syncwarp();
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // idx / rel complete; the staged coordinates are dead from here on
        // ---- B. gather the feature rows into the activation operand
        if (mma0) {
            const int chunk = tid & 7, r0 = tid >> 3;    // rows r0 and r0 + 32, 16-byte chunk `chunk` of every k-block
            const float* f0 = feat + ((size_t)b * N + s_idx[r0]) * prm.ldf + chunk * 4;
            const float* f1 = feat + ((size_t)b * N + s_idx[r0 + 32]) * prm.ldf + chunk * 4;
            const uint32_t o0 = sw128(r0, chunk), o1 = sw128(r0 + 32, chunk);
            const int nkb = prm.l[0].nkb;
            for (int kb0 = 0; kb0 < nkb; kb0 += 4) {
                float4 v0[4], v1[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int k = (kb0 + j) * 32 + chunk * 4;
                    const bool on = kb0 + j < nkb && k < prm.Cp;
                    v0[j] = on ? ld4g(f0 + (kb0 + j) * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
                    v1[j] = on ? ld4g(f1 + (kb0 + j) * 32) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (kb0 + j >= nkb) break;
                    const uint32_t hi = o3d_smem_u32(act) + (uint32_t)((kb0 + j) * SF_ACT_KB);
                    const uint32_t lo = hi + SF_ACT_KB / 2;
                    sts_v4(hi + o0, hi_part(v0[j]));
                    sts_v4(lo + o0, lo_part(v0[j]));
                    sts_v4(hi + o1, hi_part(v1[j]));
                    sts_v4(lo + o1, lo_part(v1[j]));
                }
            }
            o3d_fence_proxy_async();
            o3d_mbar_arrive(act_ready);
        }
        // ---- C / D. per layer: accumulators -> (+ coordinate term) -> BatchNorm + ReLU -> next operand | max-pool
        // (the inner loop is issue-bound — 8 K..16 K outputs per layer on 8 warps — so everything that does not depend on the
        //  column is hoisted: shared-space addresses with compile-time offsets, the XOR swizzle as 8 per-thread constants,
        //  shift / mask instead of division by nsample, one instantiation per (first, last, has-MMA) combination)
        const int q = warp & 3, half = warp >> 2;
        const float* vecs = reinterpret_cast<const float*>(block);
        const uint32_t act_s = o3d_smem_u32(act), rel_s = o3d_smem_u32(s_rel);
        const int logS = 31 - __clz(S);                 // nsample divides 64: a power of two
        uint32_t xo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) xo[i] = (uint32_t)(((lane >> 2) ^ i) << 4) + (uint32_t)(i * 128);
        int ld_phase = 0;
        for (int l = 0; l < prm.n; ++l) {
            const SfLayer& L = prm.l[l];
            const bool last = l == prm.n - 1;
            const bool wide = L.n_mt == 2;
            const bool all_cols = wide || S > 32;       // one warp walks all 64 columns (a pooling group never spans two warps)
            const int m = wide ? half : 0;
            const int kb_out = m * 4 + q;               // the k-block of the next operand this warp's 32 channels form
            // channels past the layer's width are padding: nothing reads them
            const bool work = (wide || S <= 32 || half == 0) && (last ? kb_out * 32 < L.cout : kb_out < prm.l[l + 1].nkb);
            const int col0 = all_cols ? 0 : half * 32, ncol = all_cols ? 64 : 32;
            const int chl = kb_out * 32 + lane;         // this thread's output channel
            float sc = 0.f, sh = 0.f, wx0 = 0.f, wx1 = 0.f, wx2 = 0.f;
            if (work) {
                sc = __ldg(vecs + L.vec_off + chl);
                sh = __ldg(vecs + L.vec_off + L.n_mt * 128 + chl);
                if (l == 0) {
                    const float* wx = vecs + prm.wx_off;
                    const int ldw = L.n_mt * 128;
                    wx0 = __ldg(wx + chl);
                    wx1 = __ldg(wx + ldw + chl);
                    wx2 = __ldg(wx + 2 * ldw + chl);
                }
            }
            const float floor_v = L.relu ? 0.f : -INFINITY;
            if (L.mma) {
                o3d_mbar_wait(layer_done, ld_phase);
                ld_phase ^= 1;
                tc_fence_after();
            }
            if (work) {
                const uint32_t dst_s = act_s + (uint32_t)(kb_out * SF_ACT_KB + (lane & 3) * 4);
                const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(m * SF_POS);
                const bool out_on = chl < ldo;
                const bool real = chl < L.cout;
                auto run = [&](auto first_, auto last_, auto mma_) {
                    constexpr bool FIRST = decltype(first_)::value, LAST = decltype(last_)::value, MMA = decltype(mma_)::value;
                    float mx = -INFINITY;
                    for (int cc = col0; cc < col0 + ncol; cc += 16) {
                        uint32_t r[16];
                        if constexpr (MMA) tmem_ld16(t_addr + (uint32_t)cc, r);
                        const uint32_t rowbase = dst_s + (uint32_t)((cc >> 3) * 1024);
                        const uint32_t relbase = rel_s + (uint32_t)(cc * 16);
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float a = MMA ? __uint_as_float(r[j]) : 0.f;
                            if constexpr (FIRST) {
                                const float4 rel = lds_v4(relbase + j * 16);
                                a = fmaf(wx2, rel.z, fmaf(wx1, rel.y, fmaf(wx0, rel.x, a)));
                            }
                            const float v = fmaxf(fmaf(a, sc, sh), floor_v);
                            if constexpr (!LAST) {
                                const uint32_t off = rowbase + (uint32_t)((j >> 3) * 1024) + xo[j & 7];
                                const float h = hi1(v);
                                sts_f32(off, h);
                                sts_f32(off + SF_ACT_KB / 2, v - h);
                            } else {
                                mx = fmaxf(mx, v);
                                if (((cc + j + 1) & (S - 1)) == 0) {
                                    const int g = g0 + ((cc + j) >> logS);
                                    if (out_on && g < prm.BM) out[(size_t)g * ldo + chl] = real ? mx : 0.f;
                                    mx = -INFINITY;
                                }
                            }
                        }
                    }
                };
                using T = std::true_type;
                using F = std::false_type;
                if (l == 0) {
                    if (L.mma) { if (last) run(T{}, T{}, T{}); else run(T{}, F{}, T{}); }
                    else { if (last) run(T{}, T{}, F{}); else run(T{}, F{}, F{}); }
                } else {
                    if (last) run(F{}, T{}, T{}); else run(F{}, F{}, T{});
                }
            }
            if (!last) {
                o3d_fence_proxy_async();
                tc_fence_before();
                o3d_mbar_arrive(act_ready);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        tmem_dealloc(tmem_base, SF_TMEM_COLS);
    }
}

// ---- parameter block ------------------------------------------------------------------------------------------------
struct SfPackLayer {
    const float *w, *bias, *gamma, *beta, *mean, *var;
    float eps;
    int cout, cin, col0 /* first source column of the tiled part */, kreal /* tiled source columns */, nkb, n_mt, has_bn, mma;
    uint32_t vec_off;
    size_t tile_off;
};
struct SfPackArgs { SfPackLayer l[O3D_MAX_LAYERS]; uint32_t wx_off; };

// blockIdx.y = layer; a thread owns 4 consecutive k of one (padded) output channel
__global__ void sa_fused_pack_kernel(const SfPackArgs args, uint8_t* __restrict__ block) {
    const SfPackLayer& L = args.l[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int rows = L.n_mt * 128;
    float* vec = reinterpret_cast<float*>(block) + L.vec_off;
    if (i < rows) {
        float sc = 0.f, sh = 0.f;
        if (i < L.cout) {
            sc = 1.f;
            if (L.has_bn) {
                const float istd = 1.0f / sqrtf(L.var[i] + L.eps);
                sc = (L.gamma ? L.gamma[i] : 1.f) * istd;
                sh = (L.beta ? L.beta[i] : 0.f) - L.mean[i] * sc;
            }
            if (L.bias) sh = fmaf(sc, L.bias[i], sh);
        }
        vec[i] = sc;
        vec[rows + i] = sh;
        if (blockIdx.y == 0) {
            float* wx = reinterpret_cast<float*>(block) + args.wx_off;
#pragma unroll
            for (int j = 0; j < 3; ++j) wx[j * rows + i] = i < L.cout ? L.w[(size_t)i * L.cin + j] : 0.f;
        }
    }
    if (!L.mma) return;
    const int k4n = L.nkb * 8;
    if (i >= rows * k4n) return;
    const int n = i / k4n, k = (i % k4n) * 4;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (n < L.cout) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (k + j < L.kreal) v[j] = L.w[(size_t)n * L.cin + L.col0 + k + j];
    }
    uint8_t* dst = block + L.tile_off + ((size_t)(n >> 7) * L.nkb + (k >> 5)) * SF_WTILE + sw128(n & 127, (k & 31) >> 2);
    *reinterpret_cast<float4*>(dst) = make_float4(hi1(v[0]), hi1(v[1]), hi1(v[2]), hi1(v[3]));
    *reinterpret_cast<float4*>(dst + TILE_BYTES) = make_float4(v[0] - hi1(v[0]), v[1] - hi1(v[1]), v[2] - hi1(v[2]), v[3] - hi1(v[3]));
}

struct SfPlan {
    SfParams prm;
    size_t tile_off[O3D_MAX_LAYERS];
    size_t bytes;
    int max_kb;
};

// d: the SA layer's SharedMLP as a stack description — xyz_first = 1, c0 = feature channels, K0 = round4(c0) + 4 (unused here)
bool sf_plan(const o3d_stack_t* d, SfPlan& p) {
    if (!d || d->n_layers < 1 || d->n_layers > O3D_MAX_LAYERS || !d->xyz_first || d->c0 < 0) return false;
    SfParams& q = p.prm;
    q.n = d->n_layers;
    const int C = d->c0;
    if (d->cin[0] != C + 3 || C > 288) return false;     // 9 k-blocks of input features: 144 KB operand + a two-slot weight ring
    q.Cp = (C + 3) & ~3;
    size_t off = 0;   // floats
    p.max_kb = 0;
    for (int l = 0; l < q.n; ++l) {
        SfLayer& L = q.l[l];
        L.cout = d->cout[l];
        if (L.cout < 1 || L.cout > 256) return false;
        if (l > 0 && d->cin[l] != d->cout[l - 1]) return false;
        if (d->has_bn[l] && (!d->running_mean[l] || !d->running_var[l])) return false;
        L.n_mt = (L.cout + 127) / 128;
        L.relu = d->relu[l];
        const int kreal = l == 0 ? C : d->cout[l - 1];
        L.nkb = (kreal + 31) / 32;
        L.mma = L.nkb > 0;
        L.vec_off = (uint32_t)off;
        off += 2 * (size_t)L.n_mt * 128;
        if (L.nkb > p.max_kb) p.max_kb = L.nkb;        // the operand buffer holds the k-blocks a layer reads
    }
    q.wx_off = (uint32_t)off;
    off += 3 * (size_t)q.l[0].n_mt * 128;
    size_t bytes = (off * sizeof(float) + 1023) & ~(size_t)1023;
    q.tiles_off = (uint32_t)bytes;
    for (int l = 0; l < q.n; ++l) {
        p.tile_off[l] = bytes;
        if (q.l[l].mma) bytes += (size_t)q.l[l].n_mt * q.l[l].nkb * SF_WTILE;
    }
    p.bytes = bytes;
    return true;
}

}  // namespace

extern "C" long long o3d_sa_fused_prepared_bytes(const o3d_stack_t* d) {
    SfPlan p;
    if (!sf_plan(d, p)) return -1;
    return (long long)p.bytes;
}

extern "C" int o3d_sa_fused_prepare(const o3d_stack_t* d, void* block, void* stream) {
    O3D_REQUIRE(d && block, O3D_ERR_ARG, "o3d_sa_fused_prepare: null pointer");
    SfPlan p;
    O3D_REQUIRE(sf_plan(d, p), O3D_ERR_ARG, "o3d_sa_fused_prepare: this SharedMLP does not fit the fused layer (see o3d_sa_fused_forward)");
    SfPackArgs a{};
    a.wx_off = p.prm.wx_off;
    int work_max = 0;
    for (int l = 0; l < p.prm.n; ++l) {
        const SfLayer& L = p.prm.l[l];
        SfPackLayer& q = a.l[l];
        O3D_REQUIRE(d->weight[l], O3D_ERR_ARG, "o3d_sa_fused_prepare: layer %d has no weight", l);
        q.w = d->weight[l]; q.bias = d->bias[l]; q.gamma = d->gamma[l]; q.beta = d->beta[l];
        q.mean = d->running_mean[l]; q.var = d->running_var[l]; q.eps = d->eps[l];
        q.cout = L.cout; q.cin = d->cin[l];
        q.col0 = l == 0 ? 3 : 0;
        q.kreal = l == 0 ? d->c0 : d->cout[l - 1];
        q.nkb = L.nkb; q.n_mt = L.n_mt; q.has_bn = d->has_bn[l]; q.mma = L.mma;
        q.vec_off = L.vec_off; q.tile_off = p.tile_off[l];
        int work = L.n_mt * 128 * (L.nkb > 0 ? L.nkb * 8 : 1);
        if (work > work_max) work_max = work;
    }
    sa_fused_pack_kernel<<<dim3((work_max + 255) / 256, p.prm.n), 256, 0, (cudaStream_t)stream>>>(a, (uint8_t*)block);
    O3D_CHECK_LAUNCH("o3d_sa_fused_prepare");
    return O3D_OK;
}

extern "C" int o3d_sa_fused_forward(const o3d_stack_t* d, const void* block, const float* xyz, const float* new_xyz,
                                    const float* feat_cl, int ldf, int B, int N, int M, float radius, int nsample, int normalize,
                                    float* out, int ldo, int32_t* idx, void* stream) {
    O3D_REQUIRE(d && block && xyz && new_xyz && out, O3D_ERR_ARG, "o3d_sa_fused_forward: null pointer");
    SfPlan p;
    O3D_REQUIRE(sf_plan(d, p), O3D_ERR_ARG, "o3d_sa_fused_forward: SharedMLP outside the fused layer's range (<= 256 channels per layer)");
    O3D_REQUIRE(B >= 0 && N >= 1 && M >= 0, O3D_ERR_ARG, "o3d_sa_fused_forward: bad sizes B=%d N=%d M=%d", B, N, M);
    O3D_REQUIRE(nsample >= 1 && SF_POS % nsample == 0 && M % (SF_POS / nsample) == 0, O3D_ERR_ARG,
                "o3d_sa_fused_forward: nsample=%d must divide %d and npoint=%d be a multiple of %d", nsample, SF_POS, M,
                SF_POS / (nsample > 0 && SF_POS % nsample == 0 ? nsample : 1));
    O3D_REQUIRE((d->c0 == 0) == (feat_cl == nullptr), O3D_ERR_ARG, "o3d_sa_fused_forward: features / c0 mismatch");
    O3D_REQUIRE(!feat_cl || (ldf >= p.prm.Cp && (ldf & 3) == 0 && (reinterpret_cast<uintptr_t>(feat_cl) & 15) == 0), O3D_ERR_ARG,
                "o3d_sa_fused_forward: feature rows must be 16-byte aligned with ldf >= round4(c0)");
    const int last = p.prm.n - 1;
    O3D_REQUIRE(ldo >= p.prm.l[last].cout, O3D_ERR_ARG, "o3d_sa_fused_forward: ldo=%d < %d output channels", ldo, p.prm.l[last].cout);
    if (B == 0 || M == 0) return O3D_OK;
    SfParams prm = p.prm;
    prm.ldf = ldf; prm.N = N; prm.M = M; prm.S = nsample; prm.BM = B * M;
    prm.radius = radius; prm.radius2 = radius * radius; prm.normalize = normalize;
    int act = p.max_kb * SF_ACT_KB;
    const int cloud = ((N * 12 + 1023) / 1024) * 1024;
    if (act < cloud) act = cloud;
    if (act < SF_ACT_KB) act = SF_ACT_KB;
    prm.act_bytes = act;
    const int budget = 227 * 1024 - 1024 - SF_MISC - act;
    int nslot = budget / SF_WTILE;
    if (nslot > SF_MAX_SLOTS) nslot = SF_MAX_SLOTS;
    int tiles = 0;
    for (int l = 0; l < prm.n; ++l) tiles += prm.l[l].mma ? prm.l[l].n_mt * prm.l[l].nkb : 0;
    if (nslot > tiles && tiles >= 2) nslot = tiles;       // a short stack needs no deeper ring: leaves room for a second CTA per SM
    O3D_REQUIRE(nslot >= 2, O3D_ERR_ARG, "o3d_sa_fused_forward: N=%d points per cloud do not fit the shared-memory staging", N);
    const int cpc = SF_POS / nsample;
    const int grid = (B * M) / cpc;
    if (grid > o3d_num_sms()) {       // more CTAs than SMs: a shallower ring lets two CTAs share an SM (228 KB, 1 KB reserved per CTA)
        const int fit = (113 * 1024 - 1024 - SF_MISC - act) / SF_WTILE;
        if (fit >= 2 && fit < nslot) nslot = fit;
    }
    prm.nslot = nslot;
    const int smem = 1024 + act + nslot * SF_WTILE + SF_MISC;
    O3D_CUDA(cudaFuncSetAttribute(sa_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem), "o3d_sa_fused_forward: smem attribute");
    sa_fused_kernel<<<grid, SF_THREADS, smem, (cudaStream_t)stream>>>(prm, (const uint8_t*)block, xyz, new_xyz, feat_cl, out, ldo, idx);
    O3D_CHECK_LAUNCH("o3d_sa_fused_forward");
    return O3D_OK;
}
