// Tensor-core (tcgen05 / TMEM) implementation of the point-wise MLP forward and data-gradient GEMMs, 3xTF32.
//
// Same contract as pw_fwd_kernel / pw_dgrad_kernel in pwmlp.cu (which remain the exact-fp32 ground truth and
// serve the shapes this kernel does not take: K < 32, ragged channel tails, very small P).
//
//   D[ch, pos] = sum_k  Wmat[ch, k] * Act[pos, k]          ch tile = 128 (UMMA M), pos tile = 128 (UMMA N)
//
// with Act produced on the fly from global memory (forward: relu(bn(Y_prev)); dgrad: dY = a*g + b + c*Y) and split
// into a TF32 "hi" part (the fp32 word with its 13 low mantissa bits cleared) and a "lo" part
// (x - hi, exact), so that   Whi*Xhi + Wlo*Xhi + Whi*Xlo   carries ~21 mantissa bits — fp32-grade accuracy, which
// the 1e-4 parity bar needs and a single TF32 pass (10 bits) cannot give.
//
// Roles of pw_tc_kernel (576 threads = 18 warps, one persistent CTA per SM, all roles walk the same static tile sequence):
//   warp 0        allocates TMEM (double-buffered accumulators: 2 x MT x 128 fp32 columns) and, one elected lane, issues
//                 tcgen05.mma.cta_group::1.kind::tf32 (M128 N128 K8), 12 per 32-channel k-block and channel tile, committing
//                 each stage back to the producers and each finished tile to the epilogue through mbarriers
//   warp 1        one lane streams the pre-tiled, pre-swizzled weight images (hi|lo, 32 KB per k-block and channel tile,
//                 written once per call by stack.cu's pack kernel) with cp.async.bulk (UBLKCP) onto the stage's "full"
//                 barrier, and asks for the next position tile's rows with cp.async.bulk.prefetch.L2
//   warps 4-11    epilogue: tcgen05.ld 32 lanes x 16 columns; lane = output channel, columns = positions, so the batch
//                 statistics, the group max/min/arg and the ReLU-mask sums are plain per-thread loops and every global
//                 store of a warp is one coalesced 128-byte line (MT = 2: one warp group per channel tile;
//                 MT = 1: the two groups split the columns)
//   warps 2,3,12-17  operand producers (256 threads, 4 neighbouring rows each): coalesced 16-byte loads issued one
//                 k-block ahead ("raw-first"), transform, hi/lo split, 128B-swizzled st.shared, fence.proxy.async, arrive
// Shared memory: MT = 1: 3 stages x (W 32K | X 32K) = 192 KB;  MT = 2: 2 stages x (W 64K | X 32K) = 192 KB; K-major
// SWIZZLE_128B tiles.  The wgrad kernel further down has its own role table.
#include "common.cuh"
#include "lift.cuh"
#include "pwmlp_tc.cuh"
#include "tc_ptx.cuh"
#include "../../include/o3d_b200.h"

namespace {

// ---- operand descriptions (same semantics as ActIn / DyIn in pwmlp.cu) --------------------------------------
// `prep(k)` fetches the per-channel coefficients of the thread's 4 channels once per k-block; `row(p)` then costs one
// (forward) or two (dgrad) 16-byte loads.
struct TcAct {
    static constexpr int DEPTH = 2;   // items (k-blocks) of raw loads a producer thread keeps in flight
    const float* x; int ld; const float* scale; const float* shift; int relu;
    struct Coef { float4 s, t; bool on; };
    // raw operand rows of one thread for one k-block: rows p0 + i * stride, i < R
    template <int R> struct Batch { float4 v[R]; };
    __device__ __forceinline__ Coef prep(int k, int K) const {
        Coef c;
        c.on = k < K;
        c.s = make_float4(1.f, 1.f, 1.f, 1.f);
        c.t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c.on && scale) { c.s = ld4g(scale + k); c.t = ld4g(shift + k); }
        return c;
    }
    // unconditional, always-in-range loads (clamped indices): nothing here depends on loaded data, so the whole batch is
    // issued back to back and is in flight together; masking and the transform happen in finish()
    template <int R>
    __device__ __forceinline__ void fetch(Batch<R>& b, int p0, int stride, int P, int k, int K) const {
        const int kk = k < K ? k : 0;
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const int p = p0 + i * stride;
            b.v[i] = ld4g(x + (size_t)(p < P ? p : P - 1) * ld + kk);
        }
    }
    template <int R>
    __device__ __forceinline__ float4 finish(const Batch<R>& b, const Coef& c, int i, int p, int P) const {
        float4 v = b.v[i];
        if (!(c.on && p < P)) return make_float4(0.f, 0.f, 0.f, 0.f);
        if (scale) { v.x = fmaf(v.x, c.s.x, c.t.x); v.y = fmaf(v.y, c.s.y, c.t.y); v.z = fmaf(v.z, c.s.z, c.t.z); v.w = fmaf(v.w, c.s.w, c.t.w); }
        if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        return v;
    }
    __device__ __forceinline__ void prefetch_rows(int p0, int rows, int P) const {   // full rows p0 .. p0+rows-1 -> L2
        if (p0 < P) o3d_prefetch_l2(x + (size_t)p0 * ld, (size_t)min(rows, P - p0) * ld * sizeof(float));
    }
};

// Lifted first layer as an operand (include/o3d_b200.h: o3d_lift_t): row p of the "activation matrix" is
//     relu(bn(Y0[p])),  Y0[p, k] = Z[gidx[p], k] + sum_j s[p][j] * u[j][k]
// gathered from the (L2-resident) source-point matrix Z — the grouped tensor and Y0 itself are never stored.
// Same interface as TcAct; loads stay "raw-first": gidx -> Z row (two dependent loads; the row indices are fetched one call
// ahead), the s.u terms / BN / ReLU happen in finish().
struct TcLift {
    static constexpr int DEPTH = 1;
    LiftView lv; const float* scale; const float* shift; int relu;
    int la;   // positions between two consecutive fetches of a thread (wgrad: the k-block length; 0: same rows again, next k-block)
    struct Coef { float4 s, t, u0, u1, u2, u3; bool on; };
    // nrow / tag: row indices fetched ahead for the NEXT call (tag = its p0 + 1, 0 = none), so that only a thread's first
    // k-block of a slice / position tile pays the dependent gidx -> Z load chain
    template <int R> struct Batch { float4 v[R]; float4 sv[R]; int nrow[R]; int tag; };
    __device__ __forceinline__ Coef prep(int k, int K) const {
        Coef c;
        c.on = k < K;
        c.s = make_float4(1.f, 1.f, 1.f, 1.f);
        c.t = c.u0 = c.u1 = c.u2 = c.u3 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c.on && scale) { c.s = ld4g(scale + k); c.t = ld4g(shift + k); }
        if (c.on && lv.u) { c.u0 = ld4g(lv.u + k); c.u1 = ld4g(lv.u + lv.ldz + k); c.u2 = ld4g(lv.u + 2 * lv.ldz + k); c.u3 = ld4g(lv.u + 3 * lv.ldz + k); }
        return c;
    }
    template <int R>
    __device__ __forceinline__ void fetch(Batch<R>& b, int p0, int stride, int P, int k, int K) const {
        const int kk = k < K ? k : 0;
        if (lv.z) {
            int row[R];
            if (b.tag == p0 + 1) {
#pragma unroll
                for (int i = 0; i < R; ++i) row[i] = b.nrow[i];
            } else if (R == 4 && stride == 1 && (p0 & 3) == 0 && p0 + 3 < P) {
                const int4 r4 = __ldg(reinterpret_cast<const int4*>(lv.gidx + p0));
                row[0] = r4.x; row[R > 1 ? 1 : 0] = r4.y; row[R > 2 ? 2 : 0] = r4.z; row[R > 3 ? 3 : 0] = r4.w;
            } else {
#pragma unroll
                for (int i = 0; i < R; ++i) {
                    const int p = p0 + i * stride;
                    row[i] = __ldg(lv.gidx + (p < P ? p : P - 1));
                }
            }
#pragma unroll
            for (int i = 0; i < R; ++i) b.v[i] = ld4g(lv.z + (size_t)row[i] * lv.ldz + kk);
            if (la == 0) {
#pragma unroll
                for (int i = 0; i < R; ++i) b.nrow[i] = row[i];
                b.tag = p0 + 1;
            } else {
                const int pn = p0 + la;
#pragma unroll
                for (int i = 0; i < R; ++i) {
                    const int p = pn + i * stride;
                    b.nrow[i] = __ldg(lv.gidx + (p < P ? p : P - 1));
                }
                b.tag = pn + 1;
            }
        }
        if (lv.s) {
#pragma unroll
            for (int i = 0; i < R; ++i) {
                const int p = p0 + i * stride;
                b.sv[i] = ld4g(lv.s + (size_t)(p < P ? p : P - 1) * 4);
            }
        }
    }
    template <int R>
    __device__ __forceinline__ float4 finish(const Batch<R>& b, const Coef& c, int i, int p, int P) const {
        const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!(c.on && p < P)) return zero;
        float4 v = lift_val4(lv.z ? b.v[i] : zero, lv.s ? b.sv[i] : zero, c.u0, c.u1, c.u2, c.u3);
        if (scale) { v.x = fmaf(v.x, c.s.x, c.t.x); v.y = fmaf(v.y, c.s.y, c.t.y); v.z = fmaf(v.z, c.s.z, c.t.z); v.w = fmaf(v.w, c.s.w, c.t.w); }
        if (relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        return v;
    }
    __device__ __forceinline__ void prefetch_rows(int p0, int rows, int P) const {   // index / scalar slices; Z itself lives in L2
        if (p0 >= P) return;
        const size_t n = (size_t)min(rows, P - p0);
        if (lv.z) o3d_prefetch_l2(lv.gidx + p0, n * sizeof(int32_t));
        if (lv.s) o3d_prefetch_l2(lv.s + (size_t)p0 * 4, n * 16);
    }
};

struct TcDy {
    static constexpr int DEPTH = 1;   // 32 raw registers per item: no room for a second one under the 96-register cap
    const float* g; int ldg; const float* y; int ldy; const float* a; const float* b; const float* cc;
    const float* dpool; const int32_t* sel; int S; int ldp;
    int sh;   // S == 1 << sh (pooling group sizes are powers of two on this path)
    struct Coef { float4 a, b, c; bool on; };
    // raw operand rows of one thread for one k-block: rows p0 + i * stride, i < R (R >= 2).
    // Pooled gradient: when all R rows fall into one pooling group — the usual case, a thread's rows are neighbours — the
    // two [G, ldp] tables are read ONCE (g[0] = dpool entry, g[1] = bit pattern of sel) and the per-row select moves to
    // finish(); selecting inside fetch() would make every row wait for its own table load before the next row's loads go out.
    template <int R> struct Batch { float4 g[R]; float4 y[R]; bool shared; };
    __device__ __forceinline__ Coef prep(int k, int K) const {
        Coef c;
        c.on = k < K;
        c.a = make_float4(1.f, 1.f, 1.f, 1.f);
        c.b = c.c = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c.on && a) { c.a = ld4g(a + k); c.b = ld4g(b + k); c.c = ld4g(cc + k); }
        return c;
    }
    template <int R>
    __device__ __forceinline__ void fetch(Batch<R>& bt, int p0, int stride, int P, int k, int K) const {
        const int kk = k < K ? k : 0;
        bt.shared = false;
        if (dpool) {
            const int pf = p0 < P ? p0 : P - 1;
            const int pe = p0 + (R - 1) * stride;
            const int pl = pe < P ? pe : P - 1;
            if (R >= 2 && (pf >> sh) == (pl >> sh)) {   // the two tables live in g[0], g[1]
                bt.shared = true;
                const size_t go = (size_t)(pf >> sh) * ldp + kk;
                bt.g[0] = ld4g(dpool + go);
                const int4 sl = __ldg(reinterpret_cast<const int4*>(sel + go));
                bt.g[R >= 2 ? 1 : 0] = make_float4(__int_as_float(sl.x), __int_as_float(sl.y), __int_as_float(sl.z), __int_as_float(sl.w));
            } else {
#pragma unroll
                for (int i = 0; i < R; ++i) {
                    const int p = p0 + i * stride, pp = p < P ? p : P - 1;
                    const int s = pp & (S - 1);
                    const size_t go = (size_t)(pp >> sh) * ldp + kk;
                    const int4 sl = __ldg(reinterpret_cast<const int4*>(sel + go));
                    const float4 d = ld4g(dpool + go);
                    bt.g[i] = make_float4(sl.x == s ? d.x : 0.f, sl.y == s ? d.y : 0.f, sl.z == s ? d.z : 0.f, sl.w == s ? d.w : 0.f);
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < R; ++i) {
                const int p = p0 + i * stride;
                bt.g[i] = ld4g(g + (size_t)(p < P ? p : P - 1) * ldg + kk);
            }
        }
#pragma unroll
        for (int i = 0; i < R; ++i) {
            const int p = p0 + i * stride;
            bt.y[i] = a ? ld4g(y + (size_t)(p < P ? p : P - 1) * ldy + kk) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    template <int R>
    __device__ __forceinline__ float4 finish(const Batch<R>& bt, const Coef& c, int i, int p, int P) const {
        if (!(c.on && p < P)) return make_float4(0.f, 0.f, 0.f, 0.f);
        float4 v = bt.g[i];
        if (bt.shared) {
            const int s = p & (S - 1);
            const float4 d = bt.g[0], sl = bt.g[R >= 2 ? 1 : 0];
            v = make_float4(__float_as_int(sl.x) == s ? d.x : 0.f, __float_as_int(sl.y) == s ? d.y : 0.f,
                            __float_as_int(sl.z) == s ? d.z : 0.f, __float_as_int(sl.w) == s ? d.w : 0.f);
        }
        if (a) {
            const float4 yy = bt.y[i];
            v.x = fmaf(c.a.x, v.x, fmaf(c.c.x, yy.x, c.b.x)); v.y = fmaf(c.a.y, v.y, fmaf(c.c.y, yy.y, c.b.y));
            v.z = fmaf(c.a.z, v.z, fmaf(c.c.z, yy.z, c.b.z)); v.w = fmaf(c.a.w, v.w, fmaf(c.c.w, yy.w, c.b.w));
        }
        return v;
    }
    __device__ __forceinline__ void prefetch_rows(int p0, int rows, int P) const {
        if (p0 >= P) return;
        const size_t n = (size_t)min(rows, P - p0);
        if (!dpool) o3d_prefetch_l2(g + (size_t)p0 * ldg, n * ldg * sizeof(float));
        if (a) o3d_prefetch_l2(y + (size_t)p0 * ldy, n * ldy * sizeof(float));
        if (dpool) {   // the [G, ldp] tables of the groups these rows belong to: without this every k-block of a tile starts
                       // with a cold miss on a new 128-byte line of each table
            const int g0 = p0 >> sh, g1 = (p0 + (int)n - 1) >> sh;
            const size_t bytes = (size_t)(g1 - g0 + 1) * ldp * sizeof(float);
            o3d_prefetch_l2(dpool + (size_t)g0 * ldp, bytes);
            o3d_prefetch_l2(sel + (size_t)g0 * ldp, bytes);
        }
    }
};

// ---- epilogues: thread = one output channel `ch`, called once per 32-position column group ------------------
// LD: compile-time row stride of y (0 = use the runtime ldy)
template <int LD>
struct TcFwdEpi {
    float* y; int ldy; const float* bias; double* sum; double* sumsq;
    int S, log2S; float* ymax; float* ymin; int32_t* arg; int ldp;
    // per-thread running state (fp32 inside a 32-position group, fp64 across groups and tiles)
    float bv, mx, mn; int ax, an; double d1, d2;
    __device__ __forceinline__ void begin(int ch, int Nw) {
        d1 = d2 = 0.0;
        bv = (bias && ch < Nw) ? bias[ch] : 0.f;
        mx = -INFINITY; mn = INFINITY; ax = an = 0;
    }
    __device__ __forceinline__ void prefetch(int, int, int, int) {}
    __device__ __forceinline__ const int32_t* lift_gidx() const { return nullptr; }
    __device__ __forceinline__ const float* lift_s() const { return nullptr; }
    __device__ __forceinline__ void set_tile(const int32_t*, const float4*) {}
    // Fast path = a full group of 16 positions that lies inside one pooling group (S >= 16, the set-abstraction case):
    // no per-element range or group-boundary test, the max / min / first-arg scan is local to the 16 values and is merged
    // into the running (mx, ax, mn, an) of the pooling group with two compares.  Everything else takes the element-wise path.
    __device__ __forceinline__ void group(const uint32_t (&r)[16], int ch, int Nw, int pbase, int P) {
        if (ch >= Nw) return;
        float s1 = 0.f, s2 = 0.f;
        const int smask = S - 1;
        float* yp = y ? y + (size_t)pbase * ldy + ch : nullptr;
        if (pbase + 16 <= P && (S == 0 || S >= 16)) {
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]) + bv;
            if (yp) {
                const size_t st = LD ? (size_t)LD : (size_t)ldy;   // compile-time stride -> immediate store offsets
#pragma unroll
                for (int j = 0; j < 16; ++j) yp[j * st] = v[j];
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                s1 += v[j];
                s2 = fmaf(v[j], v[j], s2);
            }
            if (S > 0) {
                float gm = v[0], gn = v[0];
                int ga = 0, gb = 0;
#pragma unroll
                for (int j = 1; j < 16; ++j) {
                    if (v[j] > gm) { gm = v[j]; ga = j; }
                    if (v[j] < gn) { gn = v[j]; gb = j; }
                }
                const int s0 = pbase & smask;
                if (s0 == 0) { mx = gm; ax = ga; mn = gn; an = gb; }
                else {
                    if (gm > mx) { mx = gm; ax = s0 + ga; }
                    if (gn < mn) { mn = gn; an = s0 + gb; }
                }
                if (s0 + 16 == S) {
                    const size_t o = (size_t)(pbase >> log2S) * ldp + ch;
                    ymax[o] = mx; ymin[o] = mn; arg[o] = ax | (an << 16);
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                if (pbase + j >= P) break;
                const float v = __uint_as_float(r[j]) + bv;
                if (yp) yp[(size_t)j * ldy] = v;
                s1 += v;
                s2 = fmaf(v, v, s2);
                if (S > 0) {
                    const int s = (pbase + j) & smask;
                    if (s == 0) { mx = -INFINITY; mn = INFINITY; ax = an = 0; }
                    if (v > mx) { mx = v; ax = s; }
                    if (v < mn) { mn = v; an = s; }
                    if (s == smask) {
                        const size_t o = (size_t)((pbase + j) >> log2S) * ldp + ch;
                        ymax[o] = mx; ymin[o] = mn; arg[o] = ax | (an << 16);
                    }
                }
            }
        }
        d1 += (double)s1;
        d2 += (double)s2;
    }
    __device__ __forceinline__ void end(int ch, int Nw) {
        if (sum && ch < Nw) {
            atomicAdd(sum + ch, d1);
            atomicAdd(sumsq + ch, d2);
        }
    }
};

// LD: compile-time row stride shared by out and yprev (0 = use the runtime ldo / ldyp)
// LIFT: the previous layer is a lifted one (its raw output is re-evaluated from Z / s.u); a separate instantiation so that the
// ordinary dgrad kernels carry none of its state
template <int LD, bool LIFT = false>
struct TcDgradEpi {
    float* out; int ldo; const float* yprev; int ldyp; const float* scale; const float* shift; int relu;
    double* s1g; double* s2y;
    LiftView lv;             // lv.z / lv.s set: the previous layer's raw output is the lifted Y0 (re-evaluated, never stored)
    float sc, sh; double d1, d2;
    float yv[16];
    float u0, u1, u2, u3; const int32_t* gs; const float4* ss;   // lifted: this thread's u[j][ch]; the tile's gidx / s slices staged in shared memory
    __device__ __forceinline__ bool lifted() const { return LIFT; }
    __device__ __forceinline__ void begin(int ch, int Nw) {
        d1 = d2 = 0.0;
        sc = (scale && ch < Nw) ? scale[ch] : 1.f;
        sh = (shift && ch < Nw) ? shift[ch] : 0.f;
        if constexpr (LIFT) {
            const bool on = lv.u && ch < Nw;
            u0 = on ? lv.u[ch] : 0.f; u1 = on ? lv.u[lv.ldz + ch] : 0.f; u2 = on ? lv.u[2 * lv.ldz + ch] : 0.f; u3 = on ? lv.u[3 * lv.ldz + ch] : 0.f;
            gs = nullptr;
        }
    }
    __device__ __forceinline__ const int32_t* lift_gidx() const { return LIFT ? lv.gidx : nullptr; }
    __device__ __forceinline__ const float* lift_s() const { return LIFT ? lv.s : nullptr; }
    __device__ __forceinline__ void set_tile(const int32_t* g, const float4* s4) { if constexpr (LIFT) { gs = g; ss = s4; } }
    // lifted yprev: `col` = first column of the group inside the tile (index into the staged gidx slice)
    __device__ __forceinline__ void prefetch_lift(int ch, int pbase, int col, int P) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float z = lv.z ? __ldg(lv.z + (size_t)gs[col + j] * lv.ldz + ch) : 0.f;
            const float4 sv = lv.s ? ss[col + j] : make_float4(0.f, 0.f, 0.f, 0.f);
            yv[j] = lift_val(z, sv, u0, u1, u2, u3);
        }
    }
    // (an L2 prefetch of these rows one tile ahead was measured: 7-15 % slower, it competes with the loader's own window)
    // issue the previous layer's raw outputs for this column group before waiting on TMEM (independent loads)
    __device__ __forceinline__ void prefetch(int ch, int Nw, int pbase, int P) {
        if (ch >= Nw) return;
        if constexpr (LIFT) { prefetch_lift(ch, pbase, pbase & (TC_N - 1), P); return; }
        if (!yprev) return;
        if (pbase + 16 <= P) {
            const float* yp = yprev + (size_t)pbase * ldyp + ch;
            const size_t st = LD ? (size_t)LD : (size_t)ldyp;
#pragma unroll
            for (int j = 0; j < 16; ++j) yv[j] = __ldg(yp + j * st);
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const int pj = min(pbase + j, P - 1);      // clamped: the load is unconditional, group() masks by range
                yv[j] = __ldg(yprev + (size_t)pj * ldyp + ch);
            }
        }
    }
    __device__ __forceinline__ void group(const uint32_t (&r)[16], int ch, int Nw, int pbase, int P) {
        if (ch >= Nw) return;
        float s1 = 0.f, s2 = 0.f;
        float* op = out + (size_t)pbase * ldo + ch;
        if (pbase + 16 <= P) {          // full group: no per-element range test
            float v[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
            if (yprev || lifted()) {
                if (relu) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = fmaf(yv[j], sc, sh) > 0.f ? v[j] : 0.f;
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) s2 = fmaf(v[j], yv[j], s2);
            }
            const size_t st = LD ? (size_t)LD : (size_t)ldo;       // compile-time stride -> immediate store offsets
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                s1 += v[j];
                op[j * st] = v[j];
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                if (pbase + j >= P) break;
                float v = __uint_as_float(r[j]);
                if (yprev || lifted()) {
                    if (relu && !(fmaf(yv[j], sc, sh) > 0.f)) v = 0.f;
                    s2 = fmaf(v, yv[j], s2);
                }
                s1 += v;
                op[(size_t)j * ldo] = v;
            }
        }
        d1 += (double)s1;
        d2 += (double)s2;
    }
    __device__ __forceinline__ void end(int ch, int Nw) {
        if (s1g && ch < Nw) {
            atomicAdd(s1g + ch, d1);
            atomicAdd(s2y + ch, d2);
        }
    }
};

// ------------------------------------------------------------------------------------------------------------
// MT = number of 128-channel tiles one CTA accumulates for the same 128 positions (1 or 2).  With MT = 2 the
// activation tile is produced once for 256 output channels: producer and epilogue work per MMA halve.
//   warps: 0 MMA issuer (+TMEM alloc) | 1 weight streamer | 4-7, 8-11 epilogue | 2,3,12-17 producers   (576 threads)
//   MT=2: epilogue warps 4-7 own channel tile 0, warps 8-11 tile 1 (all 128 columns each)
//   MT=1: warps 4-7 take columns 0-63, warps 8-11 columns 64-127 of the single tile
template <int MT> struct TcCfg {
    static constexpr int STAGES = MT == 2 ? 2 : 3;
    static constexpr int STAGE_BYTES_ = (2 * MT + 2) * TILE_BYTES;      // MT x (Whi|Wlo) | Xhi | Xlo
    static constexpr int SMEM = STAGES * STAGE_BYTES_ + 1024 + 256 + 1024 + 4096;   // + alignment | barriers | gidx + s slices (lifted dgrad)
    static constexpr uint32_t TMEM = MT == 2 ? 512 : 256;
};
constexpr int TC2_THREADS = 576;   // 18 warps: 0 MMA | 1 weights | 2,3,12-17 producers | 4-11 epilogue

template <int MT, class BLoad, class Epi>
__global__ void __launch_bounds__(TC2_THREADS, 1)
    pw_tc_kernel(BLoad bl, const uint8_t* __restrict__ wtiles, int P, int K, int Nw, int nkb, Epi epi, int rev) {
    using C = TcCfg<MT>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES_);
    uint64_t* full = bars;                        // [STAGES]  producers + weight copy -> MMA
    uint64_t* empty = bars + C::STAGES;           // [STAGES]  MMA (tcgen05.commit) -> producers
    uint64_t* tfull = bars + 2 * C::STAGES;       // [2]       MMA -> epilogue
    uint64_t* tempty = bars + 2 * C::STAGES + 2;  // [2]       epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * C::STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int mt0 = blockIdx.y * MT;              // first 128-channel tile of this CTA
    const int n_ptiles = (P + TC_N - 1) / TC_N;
    // `rev`: walk the position tiles from the last to the first.  Consecutive layers alternate the direction, so a layer
    // starts on the part of its input that the previous kernel touched last and that is still resident in the 126 MB L2.
    auto tile_of = [&](int t) { return rev ? n_ptiles - 1 - t : t; };

    if (threadIdx.x == 0) {
        for (int s = 0; s < C::STAGES; ++s) {
            o3d_mbar_init(full + s, 256 + 1);
            o3d_mbar_init(empty + s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            o3d_mbar_init(tfull + a, 1);
            o3d_mbar_init(tempty + a, 256);
        }
        o3d_fence_mbar_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, C::TMEM);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================================================== MMA issuer
        const uint32_t idesc = make_idesc(TC_M, TC_N);
        int stage = 0, phase = 0, acc = 0, aphase = 0;
        for (int t = blockIdx.x; t < n_ptiles; t += gridDim.x) {
            o3d_mbar_wait(tempty + acc, aphase ^ 1);
            tc_fence_after();
            for (int kb = 0; kb < nkb; ++kb) {
                o3d_mbar_wait(full + stage, phase);
                tc_fence_after();
                if (lane == 0) {
                    const uint32_t sb = o3d_smem_u32(smem + stage * C::STAGE_BYTES_);
                    const uint64_t xhi = make_desc(sb + 2 * MT * TILE_BYTES), xlo = make_desc(sb + (2 * MT + 1) * TILE_BYTES);
#pragma unroll
                    for (int m = 0; m < MT; ++m) {
                        const uint32_t d_tmem = tmem_base + (uint32_t)((acc * MT + m) * TC_N);
                        const uint64_t whi = make_desc(sb + 2 * m * TILE_BYTES), wlo = make_desc(sb + (2 * m + 1) * TILE_BYTES);
#pragma unroll
                        for (int ks = 0; ks < TC_K / 8; ++ks) {
                            const uint64_t adv = (uint64_t)((ks * 32) >> 4);   // +32 bytes along K inside the 128B swizzle row
                            umma_tf32(d_tmem, wlo + adv, xhi + adv, idesc, (kb | ks) != 0);
                            umma_tf32(d_tmem, whi + adv, xlo + adv, idesc, 1u);
                            umma_tf32(d_tmem, whi + adv, xhi + adv, idesc, 1u);
                        }
                    }
                    umma_commit(empty + stage);                           // frees the stage when these MMAs retire
                    if (kb == nkb - 1) umma_commit(tfull + acc);          // accumulators complete -> epilogue
                }
                __syncwarp();
                if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
            }
            if (++acc == 2) { acc = 0; aphase ^= 1; }
        }
    } else if (warp == 1) {
        // ===================================================== weight-tile streamer (bulk copy engine)
        if (lane == 0) {
            int stage = 0, phase = 0;
            if ((int)blockIdx.x < n_ptiles) {
                bl.prefetch_rows(tile_of(blockIdx.x) * TC_N, TC_N, P);
            }
            for (int t = blockIdx.x; t < n_ptiles; t += gridDim.x) {
                if (t + (int)gridDim.x < n_ptiles) {
                    bl.prefetch_rows(tile_of(t + (int)gridDim.x) * TC_N, TC_N, P);   // next tile of this CTA -> L2
                }
                for (int kb = 0; kb < nkb; ++kb) {
                    o3d_mbar_wait(empty + stage, phase ^ 1);
                    o3d_mbar_expect_tx(full + stage, MT * 2 * TILE_BYTES);
#pragma unroll
                    for (int m = 0; m < MT; ++m)
                        o3d_bulk_g2s(smem + stage * C::STAGE_BYTES_ + 2 * m * TILE_BYTES,
                                     wtiles + ((size_t)(mt0 + m) * nkb + kb) * (2 * TILE_BYTES), 2 * TILE_BYTES, full + stage);
                    if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp >= 4 && warp < 12) {
        // ===================================================== epilogue (8 warps)
        const int q = warp & 3;                       // TMEM lane quarter this warp may access
        const int grp = (warp - 4) >> 2;              // 0: warps 4-7, 1: warps 8-11
        const int m = MT == 2 ? grp : 0;              // channel tile inside the CTA
        const int cg0 = MT == 2 ? 0 : grp * 4, cg1 = MT == 2 ? 8 : grp * 4 + 4;   // 16-column groups to handle
        const int ch = (mt0 + m) * TC_M + q * 32 + lane;
        epi.begin(ch, Nw);
        int acc = 0, aphase = 0;
        int32_t* gsm = reinterpret_cast<int32_t*>(smem + C::STAGES * C::STAGE_BYTES_ + 256);   // [2][TC_N] row indices
        float4* ssm = reinterpret_cast<float4*>(smem + C::STAGES * C::STAGE_BYTES_ + 256 + 1024);   // [2][TC_N] per-position scalars
        for (int t = blockIdx.x; t < n_ptiles; t += gridDim.x) {
            const int pt0 = tile_of(t) * TC_N;
            {
                // lifted previous layer: stage the tile's 128 row indices (warps 4-7) and per-position scalars (warps 8-11) once,
                // all 8 epilogue warps read them; the named barrier of tile t+1 orders the re-use of the slices by tile t+2
                const int32_t* gi = epi.lift_gidx();
                const float* si = epi.lift_s();
                if (gi || si) {
                    const int pp = min(pt0 + q * 32 + lane, P - 1);
                    if (gi && grp == 0) gsm[acc * TC_N + q * 32 + lane] = __ldg(gi + pp);
                    if (si && grp == 1) ssm[acc * TC_N + q * 32 + lane] = ld4g(si + (size_t)pp * 4);
                    asm volatile("bar.sync 1, 256;" ::: "memory");
                    epi.set_tile(gsm + acc * TC_N, ssm + acc * TC_N);
                }
            }
            epi.prefetch(ch, Nw, pt0 + cg0 * 16, P);
            o3d_mbar_wait(tfull + acc, aphase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((acc * MT + m) * TC_N);
#pragma unroll 1
            for (int cg = cg0; cg < cg1; ++cg) {
                uint32_t r[16];
                tmem_ld16(taddr + cg * 16, r);
                epi.group(r, ch, Nw, pt0 + cg * 16, P);
                if (cg + 1 < cg1) epi.prefetch(ch, Nw, pt0 + (cg + 1) * 16, P);
            }
            tc_fence_before();
            o3d_mbar_arrive(tempty + acc);
            if (++acc == 2) { acc = 0; aphase ^= 1; }
        }
        epi.end(ch, Nw);
    } else {
        // ===================================================== activation-operand producers (8 warps, 256 threads)
        // Per k-block: [raw rows of kb already in registers] -> wait for the stage -> transform, hi/lo split, swizzled
        // st.shared -> fence + arrive -> issue the raw loads of kb+1 (all back to back, nothing depends on them until
        // the next iteration, so they fly while the MMA warp works through the stages ahead).
        const int pw = warp < 4 ? warp - 2 : warp - 10;   // producer warp 0..7
        const int pt = pw * 32 + lane;                    // 0..255
        const int chunk = pt & 7;                         // 16-byte chunk (4 channels) inside the 128-byte row
        const int row0 = (pt >> 3) * 4;                   // 4 neighbouring rows row0 + i, i < 4 (one pooling group)
        int stage = 0, phase = 0;
        // The (tile, k-block) nest is walked as one flat sequence of items so that the raw loads of the items ahead — also
        // when they belong to the next position tile — are in flight while the current one is being stored.  A loader with
        // DEPTH == 2 (the forward operand: 16 raw registers per item) keeps two items in flight per thread: one k-block
        // of loads per thread does not cover the memory latency at two pipeline stages (tensor pipe 61 % busy).
        struct Cur { int t, kb, p0; };
        auto advance = [&](Cur& c) {
            if (++c.kb == nkb) {
                c.kb = 0;
                c.t += gridDim.x;
                if (c.t < n_ptiles) c.p0 = tile_of(c.t) * TC_N;
            }
        };
        using Batch4 = typename BLoad::template Batch<4>;
        auto issue = [&](Batch4& r, typename BLoad::Coef& cf, const Cur& c) {
            if (c.t >= n_ptiles) return;
            const int k = c.kb * TC_K + chunk * 4;
            cf = bl.prep(k, K);
            bl.fetch(r, c.p0 + row0, 1, P, k, K);
        };
        auto emit = [&](const Batch4& r, const typename BLoad::Coef& cf, const Cur& c) {
            o3d_mbar_wait(empty + stage, phase ^ 1);
            uint8_t* xhi = smem + stage * C::STAGE_BYTES_ + 2 * MT * TILE_BYTES;
            uint8_t* xlo = xhi + TILE_BYTES;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float4 v = bl.finish(r, cf, i, c.p0 + row0 + i, P);
                const uint32_t off = sw128(row0 + i, chunk);
                *reinterpret_cast<float4*>(xhi + off) = hi_part(v);
                *reinterpret_cast<float4*>(xlo + off) = lo_part(v);
            }
            o3d_fence_proxy_async();              // generic-proxy stores -> visible to the tensor core (async proxy)
            o3d_mbar_arrive(full + stage);
            if (++stage == C::STAGES) { stage = 0; phase ^= 1; }
        };
        Cur c0{(int)blockIdx.x, 0, 0};
        if (c0.t < n_ptiles) c0.p0 = tile_of(c0.t) * TC_N;
        Batch4 r0{};      // value-initialised: TcLift keeps a look-ahead tag in the batch
        typename BLoad::Coef f0 = bl.prep(chunk * 4, K);
        issue(r0, f0, c0);
        if constexpr (BLoad::DEPTH == 2 && MT == 2) {   // measured: +5 % on the 256-channel layers, -8 % on the narrow ones
            Cur c1 = c0;
            if (c1.t < n_ptiles) advance(c1);
            Batch4 r1{};
            typename BLoad::Coef f1 = f0;
            issue(r1, f1, c1);
            while (c0.t < n_ptiles) {
                emit(r0, f0, c0);
                c0 = c1;
                advance(c0);                      // two items ahead of the one just stored
                issue(r0, f0, c0);
                if (c1.t >= n_ptiles) break;
                emit(r1, f1, c1);
                c1 = c0;
                if (c1.t < n_ptiles) advance(c1);
                issue(r1, f1, c1);
            }
        } else {
            while (c0.t < n_ptiles) {
                emit(r0, f0, c0);
                advance(c0);
                issue(r0, f0, c0);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, C::TMEM);
    }
}

// ------------------------------------------------------------------------------------------------------------
// wgrad on the tensor core:  dW[m, n] += sum_p dY[p, m] * X[p, n]  over this CTA's slice of positions.
// Both operands are position-major in global memory (channels contiguous), i.e. "MN-major" for a GEMM whose K is the
// position index.  For 32-bit (tf32) MN-major operands the tensor core accepts exactly one shared-memory layout,
// SWIZZLE_128B_BASE32B (cute::UMMA::Layout_MN_SW128_32B_Atom): atoms of 4 positions x 32 channels (512 B; one
// position = one 128-byte row), the 32-byte chunk index XOR-ed with (position % 4).  The producers copy coalesced
// float4 rows straight into it — no transposition — and the instruction descriptor marks A and B as MN-major.
__host__ __device__ constexpr uint32_t make_idesc_mn(int M, int N) {
    return make_idesc(M, N) | (1u << 15) | (1u << 16);
}
// L2 prefetch of one CTA's slice of position rows, paced by the MMA warp's progress (rows consumed, published in shared
// memory): at most WINDOW rows ahead.  Prefetching the whole slice up front asks for several hundred MB across the grid —
// more than the 126 MB L2 — and the lines are evicted again before their k-block comes up (measured: DRAM reads 1.7x the
// algorithmic bytes with a 384-row window, L2 hit rate 11 %).
template <class LA, class LB>
__device__ __forceinline__ void paced_prefetch(const LA& da, const LB& xb, int pbeg, int pend, volatile int* progress) {
    constexpr int CH = 32, WINDOW = 4 * CH;   // 148 CTAs x 3 operands x 128 rows x <= 1 KB stays well inside the L2
    int issued = pbeg;
    while (issued < pend) {
        const int target = pbeg + *progress + WINDOW;
        if (issued < target) {
            da.prefetch_rows(issued, CH, pend);
            xb.prefetch_rows(issued, CH, pend);
            issued += CH;
        } else {
            __nanosleep(256);
        }
    }
}

// Wide tiles: one CTA accumulates a (128*MH) x (128*NH) block of dW (MH*NH accumulators = up to all 512 TMEM columns) over
// its slice of positions, 16 positions per stage.  Against a 128 x 128 tile per CTA with fp32 REDs into dW (the kernel this
// one replaced) every loaded activation row feeds twice as many MMAs, which halves the L2->SM traffic per FLOP — the limiter
// of that kernel — and the split-K partial tiles are written with plain coalesced stores into a workspace and summed in a
// fixed order by a second kernel instead of 65k float REDs per CTA: deterministic, and measured 0.7 % faster over the step.
//   operand tile [16 positions x 128*H channels], MN-major SWIZZLE_128B_BASE32B: atom(cb, pq) at (cb + 4*H*pq) * 512
//   descriptor (channel half h, k-step ks): start = tile + h*2048 + ks*2*SBO, LBO = 512, SBO = 4*H*512
// positions per pipeline stage: each producer thread must keep >= 2 float4 per operand in flight, or the bytes in flight per SM
// (512 threads x 32 B at 16 positions x 128 channels) cap the kernel near 2.3 TB/s — measured on the 128 x 128 kernel at the SA1
// shapes (ncu, profiles/r2_step_dram_final.txt: 278 us for 629 MB); the single-accumulator variant therefore takes 32 positions
template <int MH, int NH> constexpr int wg2_k() { return MH * NH == 1 ? 32 : 16; }
constexpr int WG2_STAGES = 3;
constexpr int WG2_THREADS = 576;   // warps: 0 MMA | 1 prefetch | 2-17 producers (4-11 also run the epilogue)

template <int MH, int NH> struct Wg2Cfg {
    static constexpr int K = wg2_k<MH, NH>();
    static constexpr int A_BYTES = K * 128 * MH * 4;            // one of hi / lo
    static constexpr int B_BYTES = K * 128 * NH * 4;
    static constexpr int STAGE = 2 * A_BYTES + 2 * B_BYTES;
    static constexpr int SMEM = WG2_STAGES * STAGE + 1024 + 256;
    static constexpr uint32_t TMEM = (MH * NH * 128) <= 128 ? 128 : ((MH * NH * 128) <= 256 ? 256 : 512);
};

__device__ __forceinline__ uint64_t make_desc_mn2(uint32_t smem_addr, int H) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)(512 >> 4) << 16;
    d |= (uint64_t)((4 * H * 512) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)1 << 61;
    return d;
}
template <int H>
__device__ __forceinline__ uint32_t sw_mn2(int p_local, int c4) {   // c4 = float4 index along the 128*H channels
    const int cb = c4 >> 3, c32 = (c4 & 7) >> 1, half = c4 & 1, j0 = p_local & 3;
    return (uint32_t)((cb + 4 * H * (p_local >> 2)) * 512 + j0 * 128 + ((c32 ^ j0) << 5) + (half << 4));
}

template <int MH, int NH, class XB>
__global__ void __launch_bounds__(WG2_THREADS, 1)
    pw_wgrad_tc2_kernel(TcDy da, XB xb, int P, int M, int N, int chunk, float* __restrict__ part) {
    using C = Wg2Cfg<MH, NH>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + WG2_STAGES * C::STAGE);
    uint64_t* full = bars;
    uint64_t* empty = bars + WG2_STAGES;
    uint64_t* tfull = bars + 2 * WG2_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * WG2_STAGES + 1);
    volatile int* progress = reinterpret_cast<volatile int*>(tmem_slot + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = blockIdx.z * 128 * MH, n0 = blockIdx.y * 128 * NH;
    const int pbeg = blockIdx.x * chunk, pend = min(P, pbeg + chunk);
    constexpr int WG2_K = C::K;
    const int nkb = pend > pbeg ? (pend - pbeg + WG2_K - 1) / WG2_K : 0;
    auto kpos = [&](int i) { return pbeg + i * WG2_K; };

    if (threadIdx.x == 0) {
        for (int s = 0; s < WG2_STAGES; ++s) {
            o3d_mbar_init(full + s, 512);
            o3d_mbar_init(empty + s, 1);
        }
        o3d_mbar_init(tfull, 1);
        *progress = 0;
        o3d_fence_mbar_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, C::TMEM);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        const uint32_t idesc = make_idesc_mn(TC_M, TC_N);
        int stage = 0, phase = 0;
        for (int kb = 0; kb < nkb; ++kb) {
            o3d_mbar_wait(full + stage, phase);
            tc_fence_after();
            if (lane == 0) {
                const uint32_t sb = o3d_smem_u32(smem + stage * C::STAGE);
                const uint32_t a_hi = sb, a_lo = sb + C::A_BYTES, b_hi = sb + 2 * C::A_BYTES, b_lo = b_hi + C::B_BYTES;
#pragma unroll
                for (int ks = 0; ks < WG2_K / 8; ++ks) {
                    const uint32_t ao = ks * 2 * (4 * MH * 512), bo = ks * 2 * (4 * NH * 512);
#pragma unroll
                    for (int mh = 0; mh < MH; ++mh)
#pragma unroll
                        for (int nh = 0; nh < NH; ++nh) {
                            const uint32_t d_tmem = tmem_base + (uint32_t)((mh * NH + nh) * 128);
                            const uint64_t ahi = make_desc_mn2(a_hi + mh * 2048 + ao, MH), alo = make_desc_mn2(a_lo + mh * 2048 + ao, MH);
                            const uint64_t bhi = make_desc_mn2(b_hi + nh * 2048 + bo, NH), blo = make_desc_mn2(b_lo + nh * 2048 + bo, NH);
                            umma_tf32(d_tmem, alo, bhi, idesc, (kb | ks) != 0);
                            umma_tf32(d_tmem, ahi, blo, idesc, 1u);
                            umma_tf32(d_tmem, ahi, bhi, idesc, 1u);
                        }
                }
                umma_commit(empty + stage);
                if (kb == nkb - 1) umma_commit(tfull);
                *progress = (kb + 1) * WG2_K;
            }
            __syncwarp();
            if (++stage == WG2_STAGES) { stage = 0; phase ^= 1; }
        }
    } else if (warp == 1) {
        if (lane == 0) paced_prefetch(da, xb, pbeg, pend, progress);
    } else {
        // producers (16 warps, 2-17): every thread serves both operands, raw loads first
        const int pt = threadIdx.x - 64;                                // 0..511
        constexpr int CA = 32 * MH, CB = 32 * NH;                       // float4 per position row
        constexpr int RA = WG2_K * CA / 512, RB = WG2_K * CB / 512;     // float4 per thread per stage (1 or 2)
        const int ca4 = pt % CA, pa0 = pt / CA, sa = 512 / CA;          // A: rows pa0 + sa*i
        const int cb4 = pt % CB, pb0 = pt / CB, sbs = 512 / CB;
        const TcDy::Coef cfa = da.prep(m0 + ca4 * 4, M);
        const typename XB::Coef cfb = xb.prep(n0 + cb4 * 4, N);
        TcDy::Batch<RA> ra = {};
        typename XB::template Batch<RB> rb = {};
        auto fetch = [&](int kb) {
            da.fetch(ra, kpos(kb) + pa0, sa, pend, m0 + ca4 * 4, M);
            xb.fetch(rb, kpos(kb) + pb0, sbs, pend, n0 + cb4 * 4, N);
        };
        int stage = 0, phase = 0;
        if (nkb > 0) fetch(0);
        for (int kb = 0; kb < nkb; ++kb) {
            o3d_mbar_wait(empty + stage, phase ^ 1);
            uint8_t* a_hi = smem + stage * C::STAGE;
            uint8_t* a_lo = a_hi + C::A_BYTES;
            uint8_t* b_hi = a_hi + 2 * C::A_BYTES;
            uint8_t* b_lo = b_hi + C::B_BYTES;
#pragma unroll
            for (int i = 0; i < RA; ++i) {
                const int pl = pa0 + sa * i;
                const float4 v = da.finish(ra, cfa, i, kpos(kb) + pl, pend);
                const uint32_t off = sw_mn2<MH>(pl, ca4);
                *reinterpret_cast<float4*>(a_hi + off) = hi_part(v);
                *reinterpret_cast<float4*>(a_lo + off) = lo_part(v);
            }
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                const int pl = pb0 + sbs * i;
                const float4 v = xb.finish(rb, cfb, i, kpos(kb) + pl, pend);
                const uint32_t off = sw_mn2<NH>(pl, cb4);
                *reinterpret_cast<float4*>(b_hi + off) = hi_part(v);
                *reinterpret_cast<float4*>(b_lo + off) = lo_part(v);
            }
            o3d_fence_proxy_async();
            o3d_mbar_arrive(full + stage);
            if (kb + 1 < nkb) fetch(kb + 1);
            if (++stage == WG2_STAGES) { stage = 0; phase ^= 1; }
        }
        if (warp >= 4 && warp < 12) {
            // epilogue: partial tile -> workspace part[split][m][n] (plain coalesced stores; zeros when this slice is empty)
            const int q = warp & 3, grp = (warp - 4) >> 2;                 // grp 0: warps 4-7, 1: warps 8-11
            const int Mt = 128 * MH * (int)gridDim.z, Nt = 128 * NH * (int)gridDim.y;
            float* __restrict__ out = part + (size_t)blockIdx.x * Mt * Nt;
            if (nkb > 0) {
                o3d_mbar_wait(tfull, 0);
                tc_fence_after();
            }
            for (int t = grp; t < MH * NH; t += 2) {                       // accumulators shared between the two warp groups
                const int mh = t / NH, nh = t % NH;
                const int row = m0 + mh * 128 + q * 32 + lane;
                float* __restrict__ orow = out + (size_t)row * Nt + n0 + nh * 128;
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(t * 128);
    #pragma unroll 1
                for (int cg = 0; cg < 8; ++cg) {
                    uint32_t r[16];
                    if (nkb > 0) {
                        tmem_ld16(taddr + cg * 16, r);
                    } else {
    #pragma unroll
                        for (int j = 0; j < 16; ++j) r[j] = 0u;
                    }
    #pragma unroll
                    for (int j = 0; j < 16; j += 4)
                        *reinterpret_cast<float4*>(orow + cg * 16 + j) =
                            make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]), __uint_as_float(r[j + 3]));
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, C::TMEM);
    }
}

// dW[m, n] (+)= sum over splits of part[s][m][n]   (Mt x Nt partial tiles -> the M x N corner of dW)
// 8 lanes share one float4 of output (each sums every 8th split, then a 3-step shuffle tree): 8x more loads in flight.
__global__ void __launch_bounds__(256)
    wgrad_reduce_kernel(const float* __restrict__ part, int splits, int Mt, int Nt, int M, int N, float* __restrict__ dW,
                        int lddw) {
    const int sub = threadIdx.x & 7;
    const int n4 = (blockIdx.x * 32 + (threadIdx.x >> 3)) * 4, m = blockIdx.y;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n4 < N && m < M) {
        const float* p = part + (size_t)m * Nt + n4;
        for (int s = sub; s < splits; s += 8) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(p + (size_t)s * Mt * Nt));
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
    }
#pragma unroll
    for (int o = 4; o >= 1; o >>= 1) {
        acc.x += __shfl_xor_sync(0xFFFFFFFFu, acc.x, o); acc.y += __shfl_xor_sync(0xFFFFFFFFu, acc.y, o);
        acc.z += __shfl_xor_sync(0xFFFFFFFFu, acc.z, o); acc.w += __shfl_xor_sync(0xFFFFFFFFu, acc.w, o);
    }
    if (sub == 0 && n4 < N && m < M) {
        float* o = dW + (size_t)m * lddw + n4;
        o[0] += acc.x;
        if (n4 + 1 < N) o[1] += acc.y;
        if (n4 + 2 < N) o[2] += acc.z;
        if (n4 + 3 < N) o[3] += acc.w;
    }
}

// Pre-tile a weight matrix W[rows, ld] (rows = UMMA M channels, k contiguous) into the per-(m_tile, k-block) shared-memory
// images the kernel bulk-copies: [hi 16 KB | lo 16 KB], K-major SWIZZLE_128B, zero padded.
__global__ void w_pretile_kernel(const float* __restrict__ W, int ld, int rows, int K, int nkb, uint8_t* __restrict__ out) {
    const int m_tile = blockIdx.y, kb = blockIdx.x;
    uint8_t* dst = out + ((size_t)m_tile * nkb + kb) * (2 * TILE_BYTES);
    for (int id = threadIdx.x; id < TC_M * 8; id += blockDim.x) {
        const int r = id >> 3, c = id & 7;
        const int row = m_tile * TC_M + r, k = kb * TC_K + c * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row < rows && k < K) v = *reinterpret_cast<const float4*>(W + (size_t)row * ld + k);
        const uint32_t off = sw128(r, c);
        *reinterpret_cast<float4*>(dst + off) = hi_part(v);
        *reinterpret_cast<float4*>(dst + TILE_BYTES + off) = lo_part(v);
    }
}

// o3d_debug_set(0, 1): every tensor-core GEMM takes one 128-channel tile per CTA (MT = 1), for measuring the MT = 2 choice.
// The library's only mutable global.
int g_tc_force_mt = 0;
inline int ilog2_exact(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

template <int MT, class BLoad, class Epi>
int launch_tc_mt(BLoad bl, const uint8_t* wtiles, int P, int K, int Nw, Epi epi, int rev, cudaStream_t st, const char* name) {
    auto kern = pw_tc_kernel<MT, BLoad, Epi>;
    O3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<MT>::SMEM), name);
    const int mt = (Nw + TC_M - 1) / TC_M;
    const int gy = (mt + MT - 1) / MT;
    const int nkb = (K + TC_K - 1) / TC_K;
    const int n_ptiles = (P + TC_N - 1) / TC_N;
    int gx = o3d_num_sms() / gy;
    if (gx < 1) gx = 1;
    if (gx > n_ptiles) gx = n_ptiles;
    kern<<<dim3(gx, gy), TC2_THREADS, TcCfg<MT>::SMEM, st>>>(bl, wtiles, P, K, Nw, nkb, epi, rev);
    O3D_CHECK_LAUNCH(name);
    return O3D_OK;
}

// Nw must be a multiple of 128 when more than one channel tile exists with MT = 2 (weight tiles are read pairwise).
// ... and only when there are enough position tiles to fill the machine: a B = 1 tracking frame has <= 32 of them, and two
// CTAs per tile (MT = 1, each streaming half of the weight image) finish a layer in 10.8 us instead of 14.9 us (measured).
inline bool tc_two_tiles(int Nw, int P = 1 << 30) {
    const int mt = (Nw + TC_M - 1) / TC_M, n_ptiles = (P + TC_N - 1) / TC_N;
    return mt % 2 == 0 && g_tc_force_mt != 1 && (long long)n_ptiles * mt > o3d_num_sms();
}

// MTMASK: which MT variants this (loader, epilogue) pair is instantiated for (bit 0: MT = 1, bit 1: MT = 2)
template <int MTMASK, class BLoad, class Epi>
int launch_tc(BLoad bl, const uint8_t* wtiles, int P, int K, int Nw, Epi epi, int rev, cudaStream_t st, const char* name) {
    if constexpr ((MTMASK & 2) != 0) {
        if (tc_two_tiles(Nw, P)) return launch_tc_mt<2>(bl, wtiles, P, K, Nw, epi, rev, st, name);
    }
    if constexpr ((MTMASK & 1) != 0) {
        if (!tc_two_tiles(Nw, P)) return launch_tc_mt<1>(bl, wtiles, P, K, Nw, epi, rev, st, name);
    }
    o3d_set_error("%s: no kernel variant for %d output channels", name, Nw);
    return O3D_ERR_ARG;
}

template <int LD, int MTMASK, class BLoad>
int launch_fwd(const BLoad& bl, const void* wtiles, const float* bias, int P, int K, int Nw, float* y, int ldy, double* sum,
               double* sumsq, int S, float* ymax, float* ymin, int32_t* arg, int ldp, int rev, cudaStream_t st) {
    TcFwdEpi<LD> ep{};
    ep.y = y; ep.ldy = ldy; ep.bias = bias; ep.sum = sum; ep.sumsq = sumsq;
    ep.S = S; ep.ymax = ymax; ep.ymin = ymin; ep.arg = arg; ep.ldp = ldp;
    ep.log2S = 0;
    while ((1 << ep.log2S) < S) ++ep.log2S;
    return launch_tc<MTMASK>(bl, (const uint8_t*)wtiles, P, K, Nw, ep, rev, st, "o3d_pw_fwd_tc");
}

// the usual activation widths get a compile-time row stride (immediate store offsets in the epilogue)
template <class BLoad>
int dispatch_fwd(const BLoad& bl, const void* wtiles, const float* bias, int P, int K, int N, float* y, int ldy, double* sum,
                 double* sumsq, int S, float* ymax, float* ymin, int32_t* arg, int ldp, int rev, cudaStream_t st) {
    const int Nw = (N + 3) & ~3;
    const bool two = tc_two_tiles(Nw, P);
#define O3D_FWD_ARGS bl, wtiles, bias, P, K, Nw, y, ldy, sum, sumsq, S, ymax, ymin, arg, ldp, rev, st
    if (ldy == 64 && !two) return launch_fwd<64, 1>(O3D_FWD_ARGS);
    if (ldy == 128 && !two) return launch_fwd<128, 1>(O3D_FWD_ARGS);
    if (ldy == 256 && two) return launch_fwd<256, 2>(O3D_FWD_ARGS);
    return launch_fwd<0, 3>(O3D_FWD_ARGS);
#undef O3D_FWD_ARGS
}

template <int LD, int MTMASK, bool LIFT = false>
int launch_dgrad(const TcDy& bl, const void* wtiles_t, int P, int Cout, int Cin, float* out, int ldo, const float* yprev,
                 int ldyp, const float* pscale, const float* pshift, int prelu, double* s1, double* s2y, cudaStream_t st,
                 const LiftView* lv = nullptr) {
    if constexpr (!LIFT) {
        if (lv) return launch_dgrad<LD, MTMASK, true>(bl, wtiles_t, P, Cout, Cin, out, ldo, yprev, ldyp, pscale, pshift, prelu, s1, s2y,
                                                      st, lv);
    }
    TcDgradEpi<LD, LIFT> ep{};
    if (lv) ep.lv = *lv;
    ep.out = out; ep.ldo = ldo; ep.yprev = yprev; ep.ldyp = ldyp; ep.scale = pscale; ep.shift = pshift; ep.relu = prelu;
    ep.s1g = s1; ep.s2y = s2y;
    // GEMM: D[cin, pos] = sum_cout Wt[cin, cout] * dY[pos, cout]  ->  "K" = Cout, "Nw" = Cin; always walks forward
    return launch_tc<MTMASK>(bl, (const uint8_t*)wtiles_t, P, Cout, Cin, ep, 0, st, "o3d_pw_dgrad_tc");
}

}  // namespace

extern "C" int o3d_debug_set(int tc_debug, int force_mt) {
    O3D_REQUIRE(tc_debug == 0 && (force_mt == 0 || force_mt == 1), O3D_ERR_ARG,
                "o3d_debug_set(%d, %d): tc_debug must be 0 (the profiling switches no longer exist), force_mt 0 or 1", tc_debug,
                force_mt);
    g_tc_force_mt = force_mt;
    return O3D_OK;
}

extern "C" long long o3d_pw_tc_wtile_bytes(int rows, int K) {
    const long long mt = (rows + TC_M - 1) / TC_M, nkb = (K + TC_K - 1) / TC_K;
    return mt * nkb * 2 * TILE_BYTES;
}

extern "C" int o3d_pw_tc_pretile(const float* w, int ldw, int rows, int K, void* wtiles, void* stream) {
    O3D_REQUIRE(w && wtiles, O3D_ERR_ARG, "o3d_pw_tc_pretile: null pointer");
    O3D_REQUIRE((K & 3) == 0 && (ldw & 3) == 0, O3D_ERR_ARG, "o3d_pw_tc_pretile: K and ldw must be multiples of 4");
    O3D_REQUIRE(((uintptr_t)wtiles & 15) == 0 && ((uintptr_t)w & 15) == 0, O3D_ERR_ALIGN, "o3d_pw_tc_pretile: alignment");
    const int mt = (rows + TC_M - 1) / TC_M, nkb = (K + TC_K - 1) / TC_K;
    w_pretile_kernel<<<dim3(nkb, mt), 256, 0, (cudaStream_t)stream>>>(w, ldw, rows, K, nkb, (uint8_t*)wtiles);
    O3D_CHECK_LAUNCH("o3d_pw_tc_pretile");
    return O3D_OK;
}

int pw_fwd_tc(const float* x, int ldx, const float* in_scale, const float* in_shift, int in_relu, const void* wtiles,
              const float* bias, int P, int K, int N, float* y, int ldy, double* sum, double* sumsq, int S, float* ymax,
              float* ymin, int32_t* arg, int ldp, int rev, void* stream) {
    O3D_REQUIRE(x && wtiles, O3D_ERR_ARG, "o3d_pw_fwd_tc: null pointer");
    O3D_REQUIRE(P >= 0 && K >= 4 && N >= 1 && (K & 3) == 0 && (ldx & 3) == 0, O3D_ERR_ARG, "o3d_pw_fwd_tc: bad sizes");
    O3D_REQUIRE(S == 0 || (P % S == 0 && 64 % S == 0 && ymax && ymin && arg), O3D_ERR_ARG,
                "o3d_pw_fwd_tc: pooling group size must divide 64 and P");
    if (P == 0) return O3D_OK;
    const TcAct bl{x, ldx, in_scale, in_shift, in_relu};
    return dispatch_fwd(bl, wtiles, bias, P, K, N, y, ldy, sum, sumsq, S, ymax, ymin, arg, ldp, rev, (cudaStream_t)stream);
}

extern "C" int o3d_pw_fwd_tc(const float* x, int ldx, const float* in_scale, const float* in_shift, int in_relu,
                             const void* wtiles, const float* bias, int P, int K, int N, float* y, int ldy, double* sum,
                             double* sumsq, int S, float* ymax, float* ymin, int32_t* arg, int ldp, void* stream) {
    return pw_fwd_tc(x, ldx, in_scale, in_shift, in_relu, wtiles, bias, P, K, N, y, ldy, sum, sumsq, S, ymax, ymin, arg, ldp, 0,
                     stream);
}

namespace {
int dgrad_tc_impl(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                  const float* dpool, const int32_t* sel, int S, int ldp, const void* wtiles_t, int P, int Cout, int Cin,
                  float* out, int ldo, const float* yprev, int ldyp, const float* pscale, const float* pshift, int prelu,
                  double* s1, double* s2y, void* stream, const LiftView* lv) {
    O3D_REQUIRE((g || dpool) && wtiles_t && out, O3D_ERR_ARG, "o3d_pw_dgrad_tc: null pointer");
    O3D_REQUIRE((Cout & 3) == 0 && (Cin & 3) == 0, O3D_ERR_ARG, "o3d_pw_dgrad_tc: channel counts must be multiples of 4");
    if (P == 0) return O3D_OK;
    TcDy bl{g, ldg, y, ldy, a, b, cc, dpool, sel, S > 0 ? S : 1, ldp, ilog2_exact(S > 0 ? S : 1)};
    cudaStream_t st = (cudaStream_t)stream;
    const bool two = tc_two_tiles(Cin, P);
    const int ld = (!yprev || ldyp == ldo) ? ldo : 0;   // one compile-time stride serves both out and yprev
#define O3D_DG_ARGS bl, wtiles_t, P, Cout, Cin, out, ldo, yprev, ldyp, pscale, pshift, prelu, s1, s2y, st, lv
    if (ld == 64 && !two) return launch_dgrad<64, 1>(O3D_DG_ARGS);
    if (ld == 128 && !two) return launch_dgrad<128, 1>(O3D_DG_ARGS);
    if (ld == 256 && two) return launch_dgrad<256, 2>(O3D_DG_ARGS);
    return launch_dgrad<0, 3>(O3D_DG_ARGS);
#undef O3D_DG_ARGS
}
}  // namespace

extern "C" int o3d_pw_dgrad_tc(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b,
                               const float* cc, const float* dpool, const int32_t* sel, int S, int ldp,
                               const void* wtiles_t, int P, int Cout, int Cin, float* out, int ldo, const float* yprev,
                               int ldyp, const float* pscale, const float* pshift, int prelu, double* s1, double* s2y,
                               void* stream) {
    return dgrad_tc_impl(g, ldg, y, ldy, a, b, cc, dpool, sel, S, ldp, wtiles_t, P, Cout, Cin, out, ldo, yprev, ldyp, pscale,
                         pshift, prelu, s1, s2y, stream, nullptr);
}

namespace {
template <int MH, int NH, class XB>
int launch_wgrad2(const TcDy& da, const XB& xb, int P, int Cout, int Cin, float* dw, int lddw, float* part,
                  long long part_floats, cudaStream_t st) {
    using C = Wg2Cfg<MH, NH>;
    auto kern = pw_wgrad_tc2_kernel<MH, NH, XB>;
    O3D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM), "o3d_pw_wgrad_tc2");
    const int mt = (Cout + 128 * MH - 1) / (128 * MH), nt = (Cin + 128 * NH - 1) / (128 * NH);
    const int Mt = mt * 128 * MH, Nt = nt * 128 * NH;
    int splits = o3d_num_sms() / (mt * nt);
    if (splits < 1) splits = 1;
    const long long cap = part_floats / ((long long)Mt * Nt);
    if (splits > cap) splits = (int)cap;
    // small problems (the heads: a few thousand positions): every split writes and the reduction re-reads a whole Mt x Nt partial
    // tile (256 KB for 256 x 256), so 148 splits of ~40 positions each move 77 MB for a 6,144-position layer — more than the
    // layer itself.  At least 128 positions per split (512 was measured and is worse: the split's pipeline is a serial chain of
    // k-blocks, 0.75 us each, and a dozen CTAs cannot hide it).
    const int by_size = (P + 127) / 128;
    if (splits > by_size) splits = by_size;
    O3D_REQUIRE(splits >= 1, O3D_ERR_ARG, "o3d_pw_wgrad_tc2: workspace too small");
    int chunk = (P + splits - 1) / splits;
    chunk = ((chunk + C::K - 1) / C::K) * C::K;
    splits = (P + chunk - 1) / chunk;
    kern<<<dim3(splits, nt, mt), WG2_THREADS, C::SMEM, st>>>(da, xb, P, Cout, Cin, chunk, part);
    O3D_CHECK_LAUNCH("o3d_pw_wgrad_tc2");
    dim3 rg((Cin / 4 + 31) / 32, Cout);
    wgrad_reduce_kernel<<<rg, 256, 0, st>>>(part, splits, Mt, Nt, Cout, Cin, dw, lddw);
    O3D_CHECK_LAUNCH("o3d_pw_wgrad_tc2: reduce");
    return O3D_OK;
}
template <class XB>
int dispatch_wgrad2(const TcDy& da, const XB& xb, int P, int Cout, int Cin, float* dw, int lddw, float* part,
                    long long part_floats, cudaStream_t st) {
    const bool m2 = Cout > 128, n2 = Cin > 128;
    if (m2 && n2) return launch_wgrad2<2, 2>(da, xb, P, Cout, Cin, dw, lddw, part, part_floats, st);
    if (m2) return launch_wgrad2<2, 1>(da, xb, P, Cout, Cin, dw, lddw, part, part_floats, st);
    if (n2) return launch_wgrad2<1, 2>(da, xb, P, Cout, Cin, dw, lddw, part, part_floats, st);
    return launch_wgrad2<1, 1>(da, xb, P, Cout, Cin, dw, lddw, part, part_floats, st);
}
inline TcLift make_tclift(const o3d_lift_t* lf, const int32_t* gidx, const float* scale, const float* shift, int relu) {
    return TcLift{LiftView{lf->z, lf->ldz, lf->z ? gidx : nullptr, lf->s, lf->u}, scale, shift, relu, 0};
}
}  // namespace

extern "C" long long o3d_pw_wgrad_tc2_workspace_floats(void) {
    return (long long)o3d_num_sms() * 256 * 256;   // splits * Mt * Nt never exceeds (#SMs / tiles) * tiles * 256 * 256
}

extern "C" int o3d_pw_wgrad_tc2(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b,
                                const float* cc, const float* dpool, const int32_t* sel, int S, int ldp, const float* x,
                                int ldx, const float* in_scale, const float* in_shift, int in_relu, int P, int Cout,
                                int Cin, float* dw, int lddw, float* part, long long part_floats, void* stream) {
    O3D_REQUIRE((g || dpool) && x && dw && part, O3D_ERR_ARG, "o3d_pw_wgrad_tc2: null pointer");
    O3D_REQUIRE((Cout & 3) == 0 && (Cin & 3) == 0 && (ldx & 3) == 0 && (lddw & 3) == 0, O3D_ERR_ARG,
                "o3d_pw_wgrad_tc2: channel counts / leading dimensions must be multiples of 4");
    if (P == 0) return O3D_OK;
    TcDy da{g, ldg, y, ldy, a, b, cc, dpool, sel, S > 0 ? S : 1, ldp, ilog2_exact(S > 0 ? S : 1)};
    TcAct xb{x, ldx, in_scale, in_shift, in_relu};
    return dispatch_wgrad2(da, xb, P, Cout, Cin, dw, lddw, part, part_floats, (cudaStream_t)stream);
}

// ---- lifted first layer (o3d_lift_t): the next layer's GEMMs read Y0 through TcLift / the lifted dgrad epilogue ----------
int pw_fwd_tc_lift(const o3d_lift_t* lf, const int32_t* gidx, const float* in_scale, const float* in_shift, int in_relu,
                   const void* wtiles, const float* bias, int P, int K, int N, float* y, int ldy, double* sum, double* sumsq,
                   int S, float* ymax, float* ymin, int32_t* arg, int ldp, int rev, void* stream) {
    O3D_REQUIRE(lf && (gidx || !lf->z) && wtiles, O3D_ERR_ARG, "pw_fwd_tc_lift: null pointer");
    O3D_REQUIRE(P >= 0 && K >= 32 && N >= 1 && (K & 3) == 0 && lf->ldz == K, O3D_ERR_ARG, "pw_fwd_tc_lift: bad sizes");
    O3D_REQUIRE(S == 0 || (P % S == 0 && 64 % S == 0 && ymax && ymin && arg), O3D_ERR_ARG,
                "pw_fwd_tc_lift: pooling group size must divide 64 and P");
    if (P == 0) return O3D_OK;
    const TcLift bl = make_tclift(lf, gidx, in_scale, in_shift, in_relu);
    return dispatch_fwd(bl, wtiles, bias, P, K, N, y, ldy, sum, sumsq, S, ymax, ymin, arg, ldp, rev, (cudaStream_t)stream);
}

// dgrad whose input side is a lifted first layer: the ReLU mask and the BatchNorm-backward sums use Y0 gathered from Z
int pw_dgrad_tc_lift(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                     const float* dpool, const int32_t* sel, int S, int ldp, const void* wtiles_t, int P, int Cout, int Cin,
                     float* out, int ldo, const o3d_lift_t* lf, const int32_t* gidx, const float* pscale, const float* pshift,
                     int prelu, double* s1, double* s2y, void* stream) {
    O3D_REQUIRE(lf && (gidx || !lf->z) && (lf->z || lf->s) && lf->ldz == Cin, O3D_ERR_ARG, "pw_dgrad_tc_lift: lift descriptor");
    const LiftView lv{lf->z, lf->ldz, lf->z ? gidx : nullptr, lf->s, lf->u};
    return dgrad_tc_impl(g, ldg, y, ldy, a, b, cc, dpool, sel, S, ldp, wtiles_t, P, Cout, Cin, out, ldo, nullptr, 0, pscale,
                         pshift, prelu, s1, s2y, stream, &lv);
}

int pw_wgrad_tc_lift(const float* g, int ldg, const float* y, int ldy, const float* a, const float* b, const float* cc,
                     const float* dpool, const int32_t* sel, int S, int ldp, const o3d_lift_t* lf, const int32_t* gidx,
                     const float* in_scale, const float* in_shift, int in_relu, int P, int Cout, int Cin, float* dw, int lddw,
                     float* part, long long part_floats, void* stream) {
    O3D_REQUIRE((g || dpool) && lf && (gidx || !lf->z) && dw && part, O3D_ERR_ARG, "pw_wgrad_tc_lift: null pointer");
    O3D_REQUIRE((Cout & 3) == 0 && (Cin & 3) == 0 && lf->ldz == Cin && (lddw & 3) == 0, O3D_ERR_ARG,
                "pw_wgrad_tc_lift: channel counts / leading dimensions");
    if (P == 0) return O3D_OK;
    TcDy da{g, ldg, y, ldy, a, b, cc, dpool, sel, S > 0 ? S : 1, ldp, ilog2_exact(S > 0 ? S : 1)};
    TcLift xb = make_tclift(lf, gidx, in_scale, in_shift, in_relu);
    xb.la = (Cout > 128 || Cin > 128) ? 16 : 32;      // a producer thread's next fetch lies one k-block of positions further
    return dispatch_wgrad2(da, xb, P, Cout, Cin, dw, lddw, part, part_floats, (cudaStream_t)stream);
}
