// tcgen05 kernels for one hidden block  Linear -> LayerNorm -> ReLU -> Dropout  (st_interp.py:659-666).
//
//   layer_fwd_kernel : z = A W^T on the tensor cores (TF32 in, FP32 accumulate in TMEM); A is either
//                      the previous block's activation image (bulk-copied HBM->SMEM) or, for block 1,
//                      the basis features [X|phi|psi] generated slab by slab straight into the
//                      swizzled SMEM operand (the N x K basis matrix never exists in HBM).
//                      Epilogue: bias + LayerNorm + ReLU + dropout (+ output head + loss) from TMEM.
//   layer_bwd_kernel : recomputes z the same way (=> recomputes the basis), forms dh = dz_next W_next
//                      in a second TMEM accumulator (or from the head), applies the dropout/ReLU/
//                      LayerNorm backward and writes the dz image + bias/LN/head gradients.
//   wgrad_kernel     : dW += dz^T A, reduction over rows, both operands MN-major from the same images.
//
// One CTA = one tile of TM rows: TM = 128 (128 TMEM lanes) or, for the forward and the x_img backward, TM = 64 (an
// M = 64 MMA, whose accumulator fills lanes 0-15 of each 32-lane quarter).  The operand images stay in 128-row slab
// tiles either way: a 64-row CTA i owns rows (i & 1) * 64 .. +63 of image tile i >> 1.  Worker warps 0 .. 4*CG-1
// (operand generation and epilogue): warp w owns TMEM lane quarter q = w & 3 (the hardware ties a warp to lanes
// 32*(w%4)..) and column group cg = w >> 2, i.e. thread = (row, 1/CG of the columns); at TM = 64 the two half-warps
// take alternate 32-column chunks, so thread = (row, 1/(2 CG) of the columns).  Then one producer warp (bulk copies)
// and one MMA issuer warp (one elected thread).  CG = 4 for latency (few tiles), CG = 2 with two CTAs per SM for
// throughput.  TM = 64 is for batches that fit in one wave of 64-row tiles: twice the SMs, half the rows per CTA.
// Blocks wider than MAX_N (up to MAX_W) run the wide forms, CG = 4 with 2 stages forward and 2 stages backward: two
// MMAs per K slab fill one accumulator of up to 512 tensor-memory columns.
#pragma once
#include "common.cuh"

namespace stdadk {

constexpr int WG_NSTAGE = 2;                  // wgrad: 2 stages of 96 KB
constexpr int RED_STRIDE = 4 + STDADK_MAX_Q;   // per (cg, row) scratch: four LayerNorm partials + Q head partials
__host__ __device__ constexpr int n_work(int cg) { return 128 * cg; }
__host__ __device__ constexpr int n_threads(int cg) { return 128 * cg + 64; }
__device__ __forceinline__ void worker_barrier(int nw) { asm volatile("bar.sync 1, %0;" ::"r"(nw) : "memory"); }

// Worker-thread geometry of a TM-row tile (see the header).  The column loops of the epilogues run over the WARP's
// chunks (wc, and at TM = 64 also wc + 32), so every tcgen05.ld and shuffle is executed by the whole warp; a thread's
// own chunk is c0 = wc + chunk_off, which at TM = 64 can lie at n_pad when n_pad is an odd multiple of 32.
template <int TM>
struct TileGeo {
    static_assert(TM == 128 || TM == 64, "tile height");
    static constexpr int ROWS_PER_WARP = TM / 4;                 // rows of a lane quarter
    static constexpr int WARP_COLS = TM == 128 ? 32 : 64;        // columns one warp covers per step of its loop
    __device__ static int row(int q4, int lane) { return q4 * ROWS_PER_WARP + (TM == 128 ? lane : (lane & 15)); }
    __device__ static int chunk_off(int lane) { return TM == 128 ? 0 : (lane >> 4) * 32; }
    // column group of the thread, 0 .. groups-1, in the order LayerNorm partials are combined
    __device__ static int group(int cg, int lane) { return TM == 128 ? cg : 2 * cg + (lane >> 4); }
    __host__ __device__ static constexpr int groups(int cg) { return TM == 128 ? cg : 2 * cg; }
};
// accumulator columns [wc, wc + 32) (TM = 128), or [wc, wc + 32) for half-warp 0 and [wc + 32, wc + 64) for half-warp 1
template <int TM>
__device__ __forceinline__ void acc_ld(uint32_t taddr, float (&v)[32]) {
    if (TM == 128) tmem_ld32(taddr, v);
    else tmem_ld16x2<32>(taddr, v);
}
// warp_transpose_sum within each half-warp: on return lane l holds the column sums of indices 2 (l & 15) and +1
__device__ __forceinline__ float2 halfwarp_transpose_sum(float (&v)[32], int lane) {
#pragma unroll
    for (int off = 8, n = 16; off >= 1; off >>= 1, n >>= 1) {
        bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < n; ++i) {
            float send = upper ? v[i] : v[i + n];
            float keep = upper ? v[i + n] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return make_float2(v[0], v[1]);
}
// Column sums of a 32-column chunk over the rows of the warp, added into cs[c0 ..]; skipped for chunks at n_pad.
template <int TM>
__device__ __forceinline__ void colsum_chunk(float* cs, int c0, bool cvalid, float (&v)[32], int lane) {
    if (TM == 128) {
        const float s = warp_transpose_sum(v, lane);
        atomicAdd(&cs[c0 + lane], s);
    } else {
        const float2 s = halfwarp_transpose_sum(v, lane);
        if (cvalid) {
            atomicAdd(&cs[c0 + 2 * (lane & 15)], s.x);
            atomicAdd(&cs[c0 + 2 * (lane & 15) + 1], s.y);
        }
    }
}

// ---------------------------------------------------------------- shared-memory carve-up
struct SmemPlan {
    uint32_t a_off, b_off, bar_off, tmem_off, vec_off, headw_off, knots_off, tknots_off, colsum_off, red_off, keep_off,
        total;
};
// tab_chunks > 0 (forward kernel of block 1): the knot tables are the chunk-indexed SoA tables of gen_basis_slab_soa
// (64 bytes per 4-feature chunk) instead of the knots4 / tknots2 copies.
__host__ __device__ inline SmemPlan plan_smem(int n_pad, int q, int k_s, int k_t, bool bwd, int cg = 1, int ns = 2,
                                              int tab_chunks = 0) {
    SmemPlan s;
    uint32_t o = 0;
    s.a_off = o; o += ns * SLAB_BYTES;
    s.b_off = o; o += ns * (uint32_t)n_pad * 128u;
    s.bar_off = o; o += 128;
    s.tmem_off = o; o += 16;
    s.vec_off = o; o += 4u * n_pad * 4u;                 // per column (bias, gamma, beta, -)
    s.headw_off = o; o += (uint32_t)(q > 0 ? (q * n_pad + STDADK_MAX_Q) * 4 : 0);
    o = (o + 15u) & ~15u;
    s.knots_off = o; o += tab_chunks > 0 ? (uint32_t)tab_chunks * 64u : (uint32_t)k_s * 16u;
    s.tknots_off = o; o += tab_chunks > 0 ? 0u : (uint32_t)k_t * 8u;
    o = (o + 15u) & ~15u;
    s.colsum_off = o; o += bwd ? (uint32_t)((3 + q) * n_pad + STDADK_MAX_Q) * 4u : 0u;
    s.red_off = s.a_off;   // epilogue scratch reuses the operand stages, which are dead once the last MMA committed
    (void)cg;
    s.keep_off = o;        // layer_fwd's keep bits (fwd_keep_bytes), when the launch has them, go last
    s.total = o + 1024;                                   // slack for manual 1024-byte alignment
    return s;
}

struct FwdK {
    BasisP basis;
    PointsP pts;
    LayerP L;
    HeadP head;
    const float* a_img;
    const float* a_img_lo;      // tf32x3 residual images (NULL in TF32 mode)
    const float* addend;
    float* out_img;
    float* out_img_lo;
    float* x_img;
    float* feat_img;
    float* stats;
    int has_head, k_slabs, n_pad, tmem_cols;
    unsigned int thresh16;
    float drop_scale;
    int n_tiles, passes;        // passes: 1 (TF32) or 3 (tf32x3)
    uint32_t keep_off;          // blocks 2+ at TM = 64, dropout, a settled step counter: offset of the keep bits
                                // formed before the wait (fwd_keep_bytes at sp.keep_off), else 0
    unsigned long long* dbg;    // optional phase timers of -DSTDADK_PF_DEBUG builds (stdadk_debug_counters, or in a
                                // training step stdadk_debug_step_counters), else NULL
};
// Keep bits that the one-wave forward of block 2+ (TM = 64, CG = 4) forms before its wait: one word per worker thread
// and chunk of its column loop, in shared memory behind the rest of the plan (sp.keep_off)
__host__ __device__ constexpr uint32_t fwd_keep_bytes(int n_pad) {
    return (uint32_t)n_work(4) * 4u * (uint32_t)((n_pad + 4 * 64 - 1) / (4 * 64));
}
// Development aid: globaltimer nanoseconds between the phases of a tile's life, summed over CTAs by one worker thread
// (dbg[0..4] and dbg[9..10] phase sums, dbg[5..7] waits of single threads, dbg[8] = CTAs).  Production builds carry
// none of it.
#ifdef STDADK_PF_DEBUG
#define FWD_T(slot)                                                       \
    do {                                                                  \
        if (P.dbg && tid == 0) {                                          \
            unsigned long long now_;                                      \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now_));      \
            atomicAdd(P.dbg + (slot), now_ - t_prev_);                    \
            t_prev_ = now_;                                               \
        }                                                                 \
    } while (0)
#define FWD_WAIT(slot, stmt)                                               \
    do {                                                                   \
        unsigned long long w0_ = 0, w1_;                                   \
        if (P.dbg) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(w0_)); \
        stmt;                                                              \
        if (P.dbg) {                                                       \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(w1_));        \
            atomicAdd(P.dbg + (slot), w1_ - w0_);                          \
        }                                                                  \
    } while (0)
#else
#define FWD_T(slot)
#define FWD_WAIT(slot, stmt) stmt
#endif

struct BwdK {
    BasisP basis;
    PointsP pts;
    LayerP L;
    HeadP head;
    const float* a_img;
    const float* a_img_lo;
    const float* addend;
    const float* x_img;
    const float* stats;
    const float* dz_next_img;
    const float* dz_next_img_lo;
    const float* wt_next_img;
    const float* wt_next_img_lo;
    float* dz_img;
    float* dz_img_lo;
    float* d_bias;
    float* d_gamma;
    float* d_beta;
    float* d_head_w;
    float* d_head_b;
    int has_head, k_slabs, k_slabs2, n_pad, tmem_cols, passes;
    int step_settled, x_settled;  // stdadk_bwd_args.settled bits (x-image backward only, else 0)
#ifdef STDADK_PF_DEBUG
    unsigned long long* dbg;    // phase stamps (STEP_T)
#endif
    unsigned int thresh16;
    float drop_scale;
};

// Four consecutive features [f, f+4) of the first Linear layer's input row -> one TF32 16-byte chunk.
// Fast paths: the chunk lies entirely in the spatial block (one LDS.128 per knot, support test, value only where
// d2 < theta'^2) or entirely in the temporal block; the generic per-feature path handles block boundaries.
template <int FN>
__device__ __forceinline__ float4 spatial_chunk(const float4* kp, float x, float y, bool lo) {
    float d2[4], th2[4], ith[4];
    bool in = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const float4 kn = kp[e];
        const float dx = x - kn.x, dy = y - kn.y;
        d2[e] = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
        th2[e] = kn.z;
        ith[e] = kn.w;
        in |= d2[e] < th2[e];
    }
    // the 32 rows of a warp are neighbours when the points are ordered (grids, sorted sites): most chunks are then
    // outside every row's support and cost one vote instead of four evaluations
    if (FN != STDADK_GAUSSIAN && !__any_sync(__activemask(), in)) return make_float4(0.f, 0.f, 0.f, 0.f);
    float o[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) o[e] = tf32_part(phi_from_d2<FN>(d2[e], th2[e], ith[e]), lo);
    return make_float4(o[0], o[1], o[2], o[3]);
}
// `lo` (tf32x3 mode): the chunk of the residual image, tf32(v - tf32(v)), instead of tf32(v).
__device__ __forceinline__ float4 feature_chunk(const BasisP& B, const float4* sk, const float2* st, int f, float x,
                                                float y, float t, const float* xrow, bool lo = false) {
    const int s0 = B.p_cov, s1 = B.p_cov + B.k_s, t1 = s1 + B.k_t;
    if (f >= s0 && f + 4 <= s1) {
        const float4* kp = sk + (f - s0);
        if (B.fn == STDADK_WENDLAND) return spatial_chunk<STDADK_WENDLAND>(kp, x, y, lo);
        if (B.fn == STDADK_TRIANGULAR) return spatial_chunk<STDADK_TRIANGULAR>(kp, x, y, lo);
        return spatial_chunk<STDADK_GAUSSIAN>(kp, x, y, lo);
    }
    if (f >= s1 && f + 4 <= t1) {
        const float2* tp = st + (f - s1);
        float o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            float2 tk = tp[e];
            o[e] = tf32_part(psi_eval(t, tk.x, tk.y), lo);
        }
        return make_float4(o[0], o[1], o[2], o[3]);
    }
    if (f >= t1) return make_float4(0.f, 0.f, 0.f, 0.f);
    return make_float4(tf32_part(feature_value(B, sk, st, f + 0, x, y, t, xrow), lo),
                       tf32_part(feature_value(B, sk, st, f + 1, x, y, t, xrow), lo),
                       tf32_part(feature_value(B, sk, st, f + 2, x, y, t, xrow), lo),
                       tf32_part(feature_value(B, sk, st, f + 3, x, y, t, xrow), lo));
}

// ---- chunk-indexed tables of the forward generator.  Entry ci (64 bytes) describes features [4 ci, 4 ci + 4) when they
// are all spatial (cx[4], cy[4], theta'^2[4], 1/theta'[4]) or all temporal (c[4], 1/bw[4], -, -): structure-of-arrays,
// so that one LDS.128 fills a register quad that the packed FP32 instructions (two values per issue slot) consume
// directly.  Mixed chunks (block boundaries, at most three per row) go through feature_value on the global tables.
__device__ __forceinline__ int chunk_kind(const BasisP& B, int f) {
    const int s0 = B.p_cov, s1 = s0 + B.k_s, t1 = s1 + B.k_t;
    if (f >= s0 && f + 4 <= s1) return 0;
    if (f >= s1 && f + 4 <= t1) return 1;
    if (f >= t1) return 2;
    return 3;
}
__device__ __forceinline__ void build_chunk_tables(const BasisP& B, float4* tab, int n_chunks, int tid, int nt) {
    for (int ci = tid; ci < n_chunks; ci += nt) {
        const int f = 4 * ci, kind = chunk_kind(B, f);
        float4* g = tab + 4 * ci;
        if (kind == 0) {
            const float4* kp = B.knots + (f - B.p_cov);
            const float4 k0 = kp[0], k1 = kp[1], k2 = kp[2], k3 = kp[3];
            g[0] = make_float4(k0.x, k1.x, k2.x, k3.x);
            g[1] = make_float4(k0.y, k1.y, k2.y, k3.y);
            g[2] = make_float4(k0.z, k1.z, k2.z, k3.z);
            g[3] = make_float4(k0.w, k1.w, k2.w, k3.w);
        } else if (kind == 1) {
            const float2* tp = B.tknots + (f - B.p_cov - B.k_s);
            const float2 t0 = tp[0], t1 = tp[1], t2 = tp[2], t3 = tp[3];
            g[0] = make_float4(t0.x, t1.x, t2.x, t3.x);
            g[1] = make_float4(t0.y, t1.y, t2.y, t3.y);
        }
    }
}
// Same arithmetic, operation by operation, as spatial_chunk / phi_from_d2 (the packed instructions round like the
// scalar ones), so the operand is bit-identical to what the backward and the prediction kernels regenerate.
// NC consecutive chunks at once: NC x 4 independent evaluations in flight per thread (a worker warp runs one dependent
// chain per chunk otherwise, and with ~4 worker warps per scheduler the LDS / MUFU latencies were exposed: ncu showed
// 10.7 cycles per issued instruction per warp), one support vote for the group.
template <int FN, bool LO, int NC>
__device__ __forceinline__ void spatial_chunks_soa(const float4* g, float2 xx, float2 yy, float4 (&out)[NC]) {
    constexpr bool lo = LO;
    float2 d2a[NC], d2b[NC];
    float4 th2[NC], ith[NC];
    bool in = false;
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const float4 cx = g[4 * k], cy = g[4 * k + 1];
        th2[k] = g[4 * k + 2];
        ith[k] = g[4 * k + 3];
        const float2 dxa = sub2(xx, make_float2(cx.x, cx.y)), dxb = sub2(xx, make_float2(cx.z, cx.w));
        const float2 dya = sub2(yy, make_float2(cy.x, cy.y)), dyb = sub2(yy, make_float2(cy.z, cy.w));
        // the sums stay scalar: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 (seen in SASS, CUDA 12.9),
        // which would change d2 -- and with it the support predicate -- in the last bit
        const float2 pxa = mul2(dxa, dxa), pya = mul2(dya, dya), pxb = mul2(dxb, dxb), pyb = mul2(dyb, dyb);
        d2a[k] = make_float2(__fadd_rn(pxa.x, pya.x), __fadd_rn(pxa.y, pya.y));
        d2b[k] = make_float2(__fadd_rn(pxb.x, pyb.x), __fadd_rn(pxb.y, pyb.y));
        in |= (d2a[k].x < th2[k].x) | (d2a[k].y < th2[k].y) | (d2b[k].x < th2[k].z) | (d2b[k].y < th2[k].w);
    }
    if (FN == STDADK_GAUSSIAN) {
        const float2 kk = make_float2(-0.72134752044448170f, -0.72134752044448170f);
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            const float2 ia = make_float2(ith[k].x, ith[k].y), ib = make_float2(ith[k].z, ith[k].w);
            const float2 ea = mul2(kk, mul2(mul2(d2a[k], ia), ia)), eb = mul2(kk, mul2(mul2(d2b[k], ib), ib));
            out[k] = make_float4(tf32_part(ex2_approx(ea.x), lo), tf32_part(ex2_approx(ea.y), lo),
                                 tf32_part(ex2_approx(eb.x), lo), tf32_part(ex2_approx(eb.y), lo));
        }
        return;
    }
    // ordered points (grids, sorted sites): most chunks are outside every row's support -> one vote, no evaluation
    if (!__any_sync(__activemask(), in)) {
#pragma unroll
        for (int k = 0; k < NC; ++k) out[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        return;
    }
    const float2 one = make_float2(1.0f, 1.0f);
#pragma unroll
    for (int k = 0; k < NC; ++k) {
        const float2 qa = make_float2(rsqrt_approx(fmaxf(d2a[k].x, 1e-30f)), rsqrt_approx(fmaxf(d2a[k].y, 1e-30f)));
        const float2 qb = make_float2(rsqrt_approx(fmaxf(d2b[k].x, 1e-30f)), rsqrt_approx(fmaxf(d2b[k].y, 1e-30f)));
        const float2 ra = mul2(mul2(d2a[k], qa), make_float2(ith[k].x, ith[k].y));
        const float2 rb = mul2(mul2(d2b[k], qb), make_float2(ith[k].z, ith[k].w));
        float2 ua = sub2(one, ra), ub = sub2(one, rb);
        ua = make_float2(fmaxf(ua.x, 0.0f), fmaxf(ua.y, 0.0f));
        ub = make_float2(fmaxf(ub.x, 0.0f), fmaxf(ub.y, 0.0f));
        float2 va = ua, vb = ub;
        if (FN == STDADK_WENDLAND) {
            const float2 c35 = make_float2(35.0f / 3.0f, 35.0f / 3.0f), c6 = make_float2(6.0f, 6.0f);
            const float2 u2a = mul2(ua, ua), u2b = mul2(ub, ub);
            va = mul2(mul2(mul2(u2a, u2a), u2a), fma2(fma2(c35, ra, c6), ra, one));
            vb = mul2(mul2(mul2(u2b, u2b), u2b), fma2(fma2(c35, rb, c6), rb, one));
        }
        out[k] = make_float4(tf32_part(d2a[k].x < th2[k].x ? va.x : 0.0f, lo), tf32_part(d2a[k].y < th2[k].y ? va.y : 0.0f, lo),
                             tf32_part(d2b[k].x < th2[k].z ? vb.x : 0.0f, lo), tf32_part(d2b[k].y < th2[k].w ? vb.y : 0.0f, lo));
    }
}
template <int FN, bool LO>
__device__ __forceinline__ float4 spatial_chunk_soa(const float4* g, float2 xx, float2 yy) {
    float4 o[1];
    spatial_chunks_soa<FN, LO, 1>(g, xx, yy, o);
    return o[0];
}
template <bool LO>
__device__ __forceinline__ float4 temporal_chunk_soa(const float4* g, float2 tt) {
    constexpr bool lo = LO;
    const float4 c = g[0], ib = g[1];
    const float2 kk = make_float2(-0.72134752044448170f, -0.72134752044448170f);
    const float2 sa = mul2(sub2(tt, make_float2(c.x, c.y)), make_float2(ib.x, ib.y));
    const float2 sb = mul2(sub2(tt, make_float2(c.z, c.w)), make_float2(ib.z, ib.w));
    const float2 ea = mul2(mul2(kk, sa), sa), eb = mul2(mul2(kk, sb), sb);
    return make_float4(tf32_part(ex2_approx(ea.x), lo), tf32_part(ex2_approx(ea.y), lo), tf32_part(ex2_approx(eb.x), lo),
                       tf32_part(ex2_approx(eb.y), lo));
}
// chunks [c_begin, c_end) of operand slab `slab` of row r, from the chunk tables (forward kernel)
template <int FN, bool LO, int NC>
__device__ __forceinline__ void gen_basis_slab_soa(const BasisP& B, const float4* tab, int slab, float x, float y, float t,
                                                   const float* xrow, uint32_t slab_saddr, uint32_t r, int c_begin, int c_end,
                                                   float* gslab) {
    constexpr bool lo = LO;
    const float2 xx = make_float2(x, x), yy = make_float2(y, y), tt = make_float2(t, t);
    const uint32_t rbase = slab_saddr + r * 128u, r7 = r & 7u;
    uint8_t* grow = gslab ? reinterpret_cast<uint8_t*>(gslab) + r * 128u : nullptr;
    auto chunk_value = [&](int kind, int f) -> float4 {
        if (kind == 0) return spatial_chunk_soa<FN, LO>(tab + f, xx, yy);
        if (kind == 1) return temporal_chunk_soa<LO>(tab + f, tt);
        if (kind == 3)
            return make_float4(tf32_part(feature_value(B, B.knots, B.tknots, f + 0, x, y, t, xrow), lo),
                               tf32_part(feature_value(B, B.knots, B.tknots, f + 1, x, y, t, xrow), lo),
                               tf32_part(feature_value(B, B.knots, B.tknots, f + 2, x, y, t, xrow), lo),
                               tf32_part(feature_value(B, B.knots, B.tknots, f + 3, x, y, t, xrow), lo));
        return make_float4(0.f, 0.f, 0.f, 0.f);
    };
    int c = c_begin;
#pragma unroll 1
    for (; c + NC <= c_end; c += NC) {     // groups of NC chunks: the common case is all spatial (or all temporal)
        const int f = slab * SLAB_K + 4 * c;
        bool all_spatial = true;
#pragma unroll
        for (int k = 0; k < NC; ++k) all_spatial &= chunk_kind(B, f + 4 * k) == 0;
        float4 v[NC];
        if (all_spatial) {
            spatial_chunks_soa<FN, LO, NC>(tab + f, xx, yy, v);
        } else {
#pragma unroll
            for (int k = 0; k < NC; ++k) v[k] = chunk_value(chunk_kind(B, f + 4 * k), f + 4 * k);
        }
#pragma unroll
        for (int k = 0; k < NC; ++k) {
            const uint32_t so = ((uint32_t)(c + k) ^ r7) << 4;
            st_shared_v4(rbase + so, v[k].x, v[k].y, v[k].z, v[k].w);
            if (grow) *reinterpret_cast<float4*>(grow + so) = v[k];
        }
    }
    for (; c < c_end; ++c) {
        const int f = slab * SLAB_K + 4 * c;
        const float4 v = chunk_value(chunk_kind(B, f), f);
        const uint32_t so = ((uint32_t)c ^ r7) << 4;
        st_shared_v4(rbase + so, v.x, v.y, v.z, v.w);
        if (grow) *reinterpret_cast<float4*>(grow + so) = v;
    }
}

// Generate chunks [c_begin, c_end) of one 128-row x 32-feature operand slab (this thread = row r) into swizzled SMEM.
__device__ __forceinline__ void gen_basis_slab(const BasisP& B, const float4* sk, const float2* st, int slab,
                                               float x, float y, float t, const float* xrow, uint32_t slab_saddr,
                                               uint32_t r, int c_begin = 0, int c_end = 8, float* gslab = nullptr,
                                               bool lo = false) {
#pragma unroll 1
    for (int c = c_begin; c < c_end; ++c) {
        float4 v = feature_chunk(B, sk, st, slab * SLAB_K + c * 4, x, y, t, xrow, lo);
        st_shared_v4(slab_saddr + swz_off(r, c), v.x, v.y, v.z, v.w);
        if (gslab)      // same slab, same swizzle, in the global operand image (read back by the backward / wgrad)
            *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(gslab) + swz_off(r, c)) = v;
    }
}

// Producer: B slab (n_pad rows of the weight image, split over its 128-row tiles) [+ A slab: a_bytes from a_tile_img,
// the whole 128-row slab or, for a 64-row tile, its half: 64 rows are 8 whole swizzle periods, so either half of an
// image slab is already in the MMA's layout].
// With `a_later`, the barrier is armed for both slabs but only the B slab is copied: the A slab comes from the
// predecessor kernel and is issued after pdl_wait() with issue_a_slab.
__device__ __forceinline__ void issue_a_slab(int slab, const float* a_tile_img, float* sA, uint64_t* bar,
                                             uint32_t a_bytes) {
    bulk_g2s(sA, a_tile_img + (size_t)slab * SLAB_FLOATS, a_bytes, bar);
}
__device__ __forceinline__ void issue_slab_copies(const float* w_img, int w_slabs, int slab, int n_pad,
                                                  const float* a_tile_img, float* sA, float* sB, uint64_t* bar,
                                                  uint32_t a_bytes = SLAB_BYTES, bool a_later = false) {
    uint32_t bytes = (uint32_t)n_pad * 128u + (a_tile_img ? a_bytes : 0u);
    mbar_arrive_expect_tx(bar, bytes);
    for (int r0 = 0; r0 < n_pad; r0 += TILE_M) {
        int rows = min(TILE_M, n_pad - r0);
        const float* src = w_img + ((size_t)(r0 / TILE_M) * w_slabs + slab) * SLAB_FLOATS;
        bulk_g2s(sB + (size_t)r0 * SLAB_K, src, (uint32_t)rows * 128u, bar);
    }
    if (a_tile_img && !a_later) issue_a_slab(slab, a_tile_img, sA, bar, a_bytes);
}

// Knot tables (knots4: cx, cy, theta'^2, 1/theta'; tknots2: c, 1/bw) -> shared memory with bulk async copies (TMA 1-D)
// completing on `bar` (initialised with count 1; consumers wait for phase 0).  Called by ONE thread after the barrier
// initialisation.  An odd last temporal knot (8 bytes, below the 16-byte granule) is copied by hand; it becomes
// visible with the __syncthreads() that follows in every caller.
__device__ __forceinline__ void stage_knots_async(const BasisP& B, float4* sk, float2* st, uint64_t* bar) {
    const uint32_t ks_bytes = (uint32_t)B.k_s * 16u, kt_bytes = ((uint32_t)B.k_t >> 1) * 16u;
    mbar_arrive_expect_tx(bar, ks_bytes + kt_bytes);
    if (ks_bytes) bulk_g2s(sk, B.knots, ks_bytes, bar);
    if (kt_bytes) bulk_g2s(st, B.tknots, kt_bytes, bar);
    if (B.k_t & 1) st[B.k_t - 1] = B.tknots[B.k_t - 1];
}

// MMA issuer: one 128-byte K slab = 4 MMAs of K=8 (TF32), advancing 32 bytes inside the swizzle atom.
__device__ __forceinline__ void issue_slab_mma(uint32_t tmem_acc, const float* sA, const float* sB, uint32_t idesc,
                                               bool first) {
    uint64_t ad = umma_desc_sw128(smem_u32(sA), 16, 1024);
    uint64_t bd = umma_desc_sw128(smem_u32(sB), 16, 1024);
#pragma unroll
    for (int k = 0; k < 4; ++k) umma_tf32(tmem_acc, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc,
                                          (first && k == 0) ? 0u : 1u);
}

// tf32x3 ("virtual slabs"): with passes = 3 every K slab is issued three times into the same accumulator, as
// (A_hi, B_hi), (A_hi, B_lo), (A_lo, B_hi); the stage ring, barriers and shared-memory footprint are those of the
// single-pass kernels, only the slab count and the image each copy reads from change.
__device__ __forceinline__ bool pass_a_lo(int p) { return p == 2; }
__device__ __forceinline__ bool pass_b_lo(int p) { return p == 1; }
// hi and residual image of one 32-column chunk of an output row (residual only in tf32x3 mode)
__device__ __forceinline__ void store_operand_chunk(float* img, float* img_lo, int tile, int slabs, int c0, uint32_t row,
                                                    const float (&v)[32]) {
    const size_t off = ((size_t)tile * slabs + (c0 / SLAB_K)) * SLAB_FLOATS;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float4 hi = make_float4(to_tf32(v[4 * c]), to_tf32(v[4 * c + 1]), to_tf32(v[4 * c + 2]), to_tf32(v[4 * c + 3]));
        *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(img + off) + swz_off(row, c)) = hi;
        if (img_lo)
            *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(img_lo + off) + swz_off(row, c)) =
                make_float4(to_tf32(v[4 * c] - hi.x), to_tf32(v[4 * c + 1] - hi.y), to_tf32(v[4 * c + 2] - hi.z),
                            to_tf32(v[4 * c + 3] - hi.w));
    }
}

// 1024-byte alignment of the dynamic shared-memory base, computed as an OFFSET from the extern array so the
// compiler keeps the pointer in the shared address space (LDS/STS instead of generic LD/ST).
__device__ __forceinline__ uint8_t* align_smem(uint8_t* p) {
    return p + ((1024u - (smem_u32(p) & 1023u)) & 1023u);
}

// v[i] += addend[row, c0 + i] for the valid columns of a 32-column chunk (rows of n_out floats, n_out % 4 == 0)
__device__ __forceinline__ void add_addend_chunk(float (&v)[32], const float* addend_row, int c0, int n_out) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        if (c0 + 4 * c < n_out) {
            float4 a = *reinterpret_cast<const float4*>(addend_row + c0 + 4 * c);
            v[4 * c] += a.x; v[4 * c + 1] += a.y; v[4 * c + 2] += a.z; v[4 * c + 3] += a.w;
        }
    }
}

// one thread's 32-column chunk of a row of an FP32 image (16-byte chunks, swizzled like every operand image)
__device__ __forceinline__ void image_store_chunk(float* img, int tile, int slabs, int c0, uint32_t row, const float (&v)[32]) {
    float* dst = img + ((size_t)tile * slabs + (c0 / SLAB_K)) * SLAB_FLOATS;
#pragma unroll
    for (int c = 0; c < 8; ++c)
        *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(dst) + swz_off(row, c)) =
            make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
}
__device__ __forceinline__ void image_load_chunk(const float* img, int tile, int slabs, int c0, uint32_t row, float (&v)[32]) {
    const float* src = img + ((size_t)tile * slabs + (c0 / SLAB_K)) * SLAB_FLOATS;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        float4 q = *reinterpret_cast<const float4*>(reinterpret_cast<const uint8_t*>(src) + swz_off(row, c));
        v[4 * c] = q.x; v[4 * c + 1] = q.y; v[4 * c + 2] = q.z; v[4 * c + 3] = q.w;
    }
}

// Pinball / MSE loss on one row: fills dy[q] (already scaled) and returns the row's loss contribution.
__device__ __forceinline__ float row_loss(const HeadP& H, const float* yh, float yt, float* dy) {
    float loss = 0.0f;
    const int q = H.q;
    if (H.loss_type == STDADK_LOSS_MSE) {
#pragma unroll
        for (int k = 0; k < STDADK_MAX_Q; ++k)
            if (k < q) {
                float e = yh[k] - yt;
                loss += e * e;
                dy[k] = 2.0f * e * H.inv_count;
            }
        loss *= H.inv_count;
    } else {
#pragma unroll
        for (int k = 0; k < STDADK_MAX_Q; ++k)
            if (k < q) {
                float tau = H.taus[k];
                float err = yt - yh[k];
                loss += fmaxf((tau - 1.0f) * err, tau * err);
                float g = err > 0.0f ? -tau : (err < 0.0f ? 1.0f - tau : 0.5f - tau);
                dy[k] = g * H.inv_count;
            }
        loss *= H.inv_count;
        if (H.nc_weight > 0.0f && q > 1) {  // sum_k relu(q_k - q_{k+1})^power, mean over rows
            float inv_rows = H.inv_count * (float)q;
            float pen = 0.0f;
#pragma unroll
            for (int k = 0; k < STDADK_MAX_Q - 1; ++k)
                if (k + 1 < q) {
                    float d = yh[k] - yh[k + 1];
                    if (d > 0.0f) {
                        float gd = (H.nc_power == 2 ? 2.0f * d : 1.0f) * H.nc_weight * inv_rows;
                        pen += (H.nc_power == 2 ? d * d : d);
                        dy[k] += gd;
                        dy[k + 1] -= gd;
                    }
                }
            loss += pen * H.nc_weight * inv_rows;
        }
    }
    return loss;
}

// ---------------------------------------------------------------- register-resident epilogue pieces (32-column chunks)
// bias add + shifted moments of one 32-column chunk held in registers (nv valid columns); packed FP32 throughout
__device__ __forceinline__ void pf_bias_stats(float (&v)[32], const float* sb, int nv, bool& have, float& K, float& S1,
                                              float& S2) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const float4 b = *reinterpret_cast<const float4*>(sb + 4 * c);
        const float2 lo = add2(make_float2(v[4 * c], v[4 * c + 1]), make_float2(b.x, b.y));
        const float2 hi = add2(make_float2(v[4 * c + 2], v[4 * c + 3]), make_float2(b.z, b.w));
        v[4 * c] = lo.x; v[4 * c + 1] = lo.y; v[4 * c + 2] = hi.x; v[4 * c + 3] = hi.y;
    }
    if (!have) {
        K = v[0];
        have = true;
    }
    if (nv >= 32) {
        // two independent packed accumulator pairs (= four scalar chains): with four warps per scheduler a single
        // 32-long FADD chain would stall
        const float2 nk = make_float2(-K, -K);
        float2 a1[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)}, a2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            const float2 d = add2(make_float2(v[i], v[i + 1]), nk);
            a1[(i >> 1) & 1] = add2(a1[(i >> 1) & 1], d);
            a2[(i >> 1) & 1] = fma2(d, d, a2[(i >> 1) & 1]);
        }
        S1 += (a1[0].x + a1[0].y) + (a1[1].x + a1[1].y);
        S2 += (a2[0].x + a2[0].y) + (a2[1].x + a2[1].y);
    } else {
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if (i < nv) {
                const float d = v[i] - K;
                S1 += d;
                S2 = fmaf(d, d, S2);
            }
    }
}

// v <- relu(LayerNorm(v)) (or relu(v)); columns >= nv forced to zero
__device__ __forceinline__ void pf_normalize(float (&v)[32], const float* sg, const float* sbt, bool has_ln, float rstd,
                                             float nmr, int nv) {
    if (has_ln) {
        const float2 r2 = make_float2(rstd, rstd), n2 = make_float2(nmr, nmr);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const float4 g = *reinterpret_cast<const float4*>(sg + 4 * c);
            const float4 b = *reinterpret_cast<const float4*>(sbt + 4 * c);
            const float2 y0 = fma2(fma2(make_float2(v[4 * c], v[4 * c + 1]), r2, n2), make_float2(g.x, g.y),
                                   make_float2(b.x, b.y));
            const float2 y1 = fma2(fma2(make_float2(v[4 * c + 2], v[4 * c + 3]), r2, n2), make_float2(g.z, g.w),
                                   make_float2(b.z, b.w));
            v[4 * c] = fmaxf(y0.x, 0.0f);
            v[4 * c + 1] = fmaxf(y0.y, 0.0f);
            v[4 * c + 2] = fmaxf(y1.x, 0.0f);
            v[4 * c + 3] = fmaxf(y1.y, 0.0f);
        }
    } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i], 0.0f);
    }
    if (nv < 32) {
#pragma unroll
        for (int i = 0; i < 32; ++i)
            if (i >= nv) v[i] = 0.0f;
    }
}

// keep bits of one 32-column chunk: four Philox calls (same keys as layer_fwd_kernel).  Computed BEFORE the accumulator
// is pulled into registers -- while the MMAs are still running -- so the calls neither sit on the critical path nor
// force the 64 accumulator registers to be saved around them.
__device__ __forceinline__ uint32_t pf_keep_mask(unsigned long long seed, uint32_t step, uint32_t layer,
                                                 unsigned long long key_row, int c0, uint32_t thresh16) {
    uint32_t keep = 0;
#pragma unroll 1
    for (int b = 0; b < 4; ++b) keep |= dropout_keep8(seed, step, layer, key_row, (uint32_t)(c0 / 8 + b), thresh16) << (8 * b);
    return keep;
}
// keep bits of each of the thread's 32-column chunks (the column loop of the epilogues), indexed by chunk; a chunk at
// n_pad (TM = 64) keeps everything, as its columns are dropped by col < n_out anyway
template <int TM, int CG, int MAXCH>
__device__ __forceinline__ void chunk_keep_masks(const LayerP& L, unsigned int thresh16, long long lrow, int cg, int lane,
                                                 int n_pad, uint32_t (&keeps)[MAXCH]) {
    using G = TileGeo<TM>;
    const bool drop = L.drop_p > 0.0f;
    const unsigned int step = drop ? dropout_step(L) : 0u;
    int ch = 0;
    for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += G::WARP_COLS * CG, ++ch) {
        const int c0 = wc + G::chunk_off(lane);
        const uint32_t kb = (drop && (TM == 128 || c0 < n_pad))
                                ? pf_keep_mask(L.seed, step, (uint32_t)L.layer_id, L.key_offset + (unsigned long long)lrow,
                                               c0, thresh16)
                                : 0xFFFFFFFFu;
#pragma unroll
        for (int k = 0; k < MAXCH; ++k)
            if (k == ch) keeps[k] = kb;
    }
}
__device__ __forceinline__ void pf_dropout(float (&v)[32], uint32_t keep, float scale) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = ((keep >> i) & 1u) ? v[i] * scale : 0.0f;
}
__device__ __forceinline__ void pf_head_partial(const float (&v)[32], const float* shw, int n_pad, int c0, int q,
                                                float (&yh)[STDADK_MAX_Q]) {
#pragma unroll 1
    for (int k = 0; k < q; ++k) {
        const float* wk = shw + k * n_pad + c0;
        float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const float4 w = *reinterpret_cast<const float4*>(wk + 4 * c);
            a0 = fmaf(v[4 * c], w.x, a0);
            a1 = fmaf(v[4 * c + 1], w.y, a1);
            a2 = fmaf(v[4 * c + 2], w.z, a2);
            a3 = fmaf(v[4 * c + 3], w.w, a3);
        }
        const float acc = (a0 + a1) + (a2 + a3);
#pragma unroll
        for (int kk = 0; kk < STDADK_MAX_Q; ++kk)
            if (kk == k) yh[kk] += acc;
    }
}

// =============================================================================================
// Forward
// =============================================================================================
// Epilogue of a forward block for one thread = (row, column group): two passes over the accumulator in tensor memory
// (a thread owns 256 / CG columns, more than the register file holds at two CTAs per SM), each on whole 32-column chunks
// in registers with packed FP32 math.
struct EpiCtx {
    const float* sbias;
    const float* sgam;
    const float* sbet;
    const float* shw;
    const float* shb;
    float* red;                    // (groups x TM) x RED_STRIDE floats of scratch
    uint32_t trow;                 // accumulator address of this warp's lane quarter
    int tile, row, irow, cg, lane; // tile / irow: image tile and row in it; row: row of the CTA's tile
    long long lrow, grow;
    bool rvalid, tile_valid;
};
// EARLY: the kernel form that may have formed the keep bits before the wait (P.keep_off).  They are found from the
// kernel parameter rather than a pointer, which would hold two registers across pass 1.
template <int CG, int TM, bool EARLY>
__device__ __forceinline__ void fwd_epilogue(const FwdK& P, const EpiCtx& E) {
    using G = TileGeo<TM>;
    constexpr int NW = n_work(CG), NG = G::groups(CG), WSTEP = G::WARP_COLS * CG;
    const float* sbias = E.sbias;
    const float* sgam = E.sgam;
    const float* sbet = E.sbet;
    const float* shw = E.shw;
    const float* shb = E.shb;
    float* red = E.red;
    const uint32_t trow = E.trow;
    const int tile = E.tile, row = E.row, irow = E.irow, cg = E.cg, lane = E.lane;
    const long long lrow = E.lrow, grow = E.grow;
    const bool rvalid = E.rvalid, tile_valid = E.tile_valid;
    const int n_pad = P.n_pad, n_out = P.L.n_out;
    const bool has_ln = P.L.gamma != nullptr;
    const int coff = G::chunk_off(lane), grp = G::group(cg, lane);
    float* myred = red + ((size_t)grp * TM + row) * RED_STRIDE;
    const float* arow = (P.addend && rvalid) ? P.addend + (size_t)lrow * n_out : nullptr;
    float v[32];
    float mean = 0.0f, rstd = 1.0f;
    if (has_ln) {
        // pass 1: shifted moments of x = A W^T + b (+ addend): per-thread shift K (the thread's first value) removes
        // the cancellation of the raw-moment formula; the NG column groups of a row publish (K, S1, S2, count) and
        // every thread combines them exactly:
        //   mean = sum_g (n_g K_g + S1_g) / n,   M2 = sum_g [S2_g - 2 (mean - K_g) S1_g + n_g (mean - K_g)^2]
        float K = 0.0f, S1 = 0.0f, S2 = 0.0f, cntv = 0.0f;
        bool have = false;
        for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += WSTEP) {
            const int c0 = wc + coff, nv = n_out - c0;
            if ((TM == 128 ? nv : n_out - wc) <= 0) break;      // warp-uniform: the half-warps' c0 differ at TM = 64
            acc_ld<TM>(trow + wc, v);
            if (TM == 128 || nv > 0) {
                if (arow) add_addend_chunk(v, arow, c0, n_out);
                pf_bias_stats(v, sbias + c0, min(nv, 32), have, K, S1, S2);
                cntv += (float)min(nv, 32);
            }
        }
        const float inv_n = 1.0f / (float)n_out;
        if (NG > 1) {
            *reinterpret_cast<float4*>(myred) = make_float4(K, S1, S2, cntv);
            worker_barrier(NW);
            float4 part[NG];
            float tot = 0.0f;
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                part[g] = *reinterpret_cast<const float4*>(red + ((size_t)g * TM + row) * RED_STRIDE);
                tot += fmaf(part[g].w, part[g].x, part[g].y);
            }
            mean = tot * inv_n;
            float m2 = 0.0f;
#pragma unroll
            for (int g = 0; g < NG; ++g) {
                float dk = mean - part[g].x;
                m2 += part[g].z - 2.0f * dk * part[g].y + part[g].w * dk * dk;
            }
            rstd = 1.0f / sqrtf(fmaxf(m2 * inv_n, 0.0f) + P.L.eps);
        } else {
            float m1 = S1 * inv_n;
            mean = K + m1;
            rstd = 1.0f / sqrtf(fmaxf(S2 * inv_n - m1 * m1, 0.0f) + P.L.eps);
        }
        if (P.stats && rvalid && grp == 0) {
            P.stats[2 * lrow] = mean;
            P.stats[2 * lrow + 1] = rstd;
        }
    }
    const float nmr = -mean * rstd;
    float yh[STDADK_MAX_Q];
#pragma unroll
    for (int k = 0; k < STDADK_MAX_Q; ++k) yh[k] = 0.0f;
    const bool drop = P.L.drop_p > 0.0f;
    const bool keep_early = EARLY && P.keep_off != 0;
    const unsigned int drop_step = (drop && !keep_early) ? dropout_step(P.L) : 0u;
    // pass 2: x -> LayerNorm -> ReLU -> dropout -> operand image (+ head partials, + x image for the backward)
    int ch = 0;
    for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += WSTEP, ++ch) {
        const int c0 = wc + coff;
        const bool cvalid = TM == 128 || c0 < n_pad;
        uint32_t keep = 0xFFFFFFFFu;
        if (drop && cvalid) {  // masks first: the Philox calls neither sit behind the TMEM load nor hold 32 live values
            if (keep_early) {
                extern __shared__ uint8_t smem_raw[];
                keep = reinterpret_cast<const uint32_t*>(align_smem(smem_raw) + P.keep_off)[ch * NW + (int)threadIdx.x];
            }
            else keep = pf_keep_mask(P.L.seed, drop_step, (uint32_t)P.L.layer_id, P.L.key_offset + (unsigned long long)lrow,
                                     c0, P.thresh16);
        }
        acc_ld<TM>(trow + wc, v);
        if (arow) add_addend_chunk(v, arow, c0, n_out);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const float4 b = *reinterpret_cast<const float4*>(sbias + c0 + 4 * c);
            const float2 lo = add2(make_float2(v[4 * c], v[4 * c + 1]), make_float2(b.x, b.y));
            const float2 hi = add2(make_float2(v[4 * c + 2], v[4 * c + 3]), make_float2(b.z, b.w));
            v[4 * c] = lo.x; v[4 * c + 1] = lo.y; v[4 * c + 2] = hi.x; v[4 * c + 3] = hi.y;
        }
        if (P.x_img && tile_valid && cvalid)  // training with a single wave of tiles: keep x for the backward
            image_store_chunk(P.x_img, tile, n_pad / SLAB_K, c0, (uint32_t)irow, v);
        const int nv = rvalid ? min(32, max(n_out - c0, 0)) : 0;      // padding rows / columns -> 0
        pf_normalize(v, sgam + c0, sbet + c0, has_ln, rstd, nmr, nv);
        if (drop) pf_dropout(v, keep, P.drop_scale);
        if (P.has_head && cvalid) pf_head_partial(v, shw, n_pad, c0, P.head.q, yh);
        if (P.out_img && tile_valid && cvalid)
            store_operand_chunk(P.out_img, P.out_img_lo, tile, n_pad / SLAB_K, c0, (uint32_t)irow, v);
    }
    if (P.has_head) {
        // head partials after the LayerNorm partials of the same scratch row, which slower threads may still be reading
        if (NG > 1) {
#pragma unroll
            for (int k = 0; k < STDADK_MAX_Q; ++k)
                if (k < P.head.q) myred[4 + k] = yh[k];
            worker_barrier(NW);
        }
        if (cg == 0) {
            float loss = 0.0f;
            if (rvalid && grp == 0) {
                float dy[STDADK_MAX_Q];
#pragma unroll
                for (int k = 0; k < STDADK_MAX_Q; ++k)
                    if (k < P.head.q) {
                        if (NG > 1) {
                            float acc = 0.0f;
#pragma unroll
                            for (int g = 0; g < NG; ++g) acc += red[((size_t)g * TM + row) * RED_STRIDE + 4 + k];
                            yh[k] = acc;
                        }
                        yh[k] += shb[k];
                        P.head.yhat[lrow * P.head.q + k] = yh[k];
                    }
                if (P.head.loss_type != STDADK_LOSS_NONE) {
                    loss = row_loss(P.head, yh, P.head.y[sample_of(P.pts, grow)], dy);
                    if (P.head.dyhat) {
#pragma unroll
                        for (int k = 0; k < STDADK_MAX_Q; ++k)
                            if (k < P.head.q) P.head.dyhat[lrow * P.head.q + k] = dy[k];
                    }
                }
            }
            if (P.head.loss_type != STDADK_LOSS_NONE) {
                loss = warp_sum(loss);
                if (lane == 0) atomicAdd(P.head.loss_acc, loss);
            }
        }
    }
}

// The wide form, CG = 4 with NS = 2 (MAX_N < n_pad <= MAX_W; 2 stages of up to 80 KB, one CTA per SM by its shared
// memory and by its tensor memory, all 512 columns at width 512): one UMMA takes N <= MAX_N, so every K slab is two
// MMAs, B rows [0, MAX_N) into accumulator columns [0, MAX_N) and the rest into [MAX_N, n_pad).  The accumulator is then
// the same n_pad contiguous columns the epilogue reads at any width.  The narrow forms are <CG = 4, NS = 4> and
// <CG = 2, NS = 2>.
template <bool BASIS, int TM, int CG, int NS>
__global__ void __launch_bounds__(n_threads(CG), CG <= 2 ? 2 : 1) layer_fwd_kernel(const __grid_constant__ FwdK P) {
    using G = TileGeo<TM>;
    constexpr bool WIDE = CG == 4 && NS == 2;
    constexpr int NW = n_work(CG), NT = n_threads(CG), NSTAGE = NS, NG = G::groups(CG);
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem(smem_raw);
    const SmemPlan sp = plan_smem(P.n_pad, P.has_head ? P.head.q : 0, BASIS ? P.basis.k_s : 0,
                                  BASIS ? P.basis.k_t : 0, false, CG, NS, BASIS ? P.k_slabs * 8 : 0);
    float* sA = reinterpret_cast<float*>(smem + sp.a_off);
    float* sB = reinterpret_cast<float*>(smem + sp.b_off);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + sp.bar_off);
    uint64_t* empty = full + NSTAGE;
    uint64_t* accf = full + 2 * NSTAGE;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + sp.tmem_off);
    float* sbias = reinterpret_cast<float*>(smem + sp.vec_off);    // per column bias | gamma | beta (one LDS.128 per 4 columns)
    float* sgam = sbias + P.n_pad;
    float* sbet = sgam + P.n_pad;
    float* shw = reinterpret_cast<float*>(smem + sp.headw_off);
    float* shb = shw + (P.has_head ? P.head.q * P.n_pad : 0);
    float4* ctab = reinterpret_cast<float4*>(smem + sp.knots_off);  // chunk tables of the generator (BASIS)
    float* red = reinterpret_cast<float*>(smem + sp.red_off);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef STDADK_PF_DEBUG
    unsigned long long t_prev_ = 0;
    if (P.dbg && tid == 0) {
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_prev_));
        atomicAdd(P.dbg + 8, 1ull);
    }
#endif
    // The grid has one CTA per tile, so tile_valid always holds.  It stays, with the tests it feeds, because ptxas
    // allocates registers better with it: without it the row index of layer_fwd_kernel<true, 2, 2> spills and a
    // 1M-row launch took 0.812 ms instead of 0.789 ms (B200, 1000 W power limit).
    const bool tile_valid = (int)blockIdx.x < P.n_tiles;
    const int tile = tile_valid ? (int)blockIdx.x : P.n_tiles - 1;
    const int itile = tile / (TILE_M / TM), irow0 = (tile % (TILE_M / TM)) * TM;   // image tile, first row in it
    const int n_pad = P.n_pad, n_out = P.L.n_out;
    const bool has_ln = P.L.gamma != nullptr;
    const size_t b_stage_floats = (size_t)n_pad * SLAB_K;

    if (tid == NW) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&full[s], BASIS ? 1 + NW / 32 : 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accf, 1);
        mbar_fence_init();
    }
    if (warp == 4 * CG) {
        __syncwarp();
        tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    }
    if (BASIS) build_chunk_tables(P.basis, ctab, P.k_slabs * 8, tid, NT);
    for (int i = tid; i < n_pad; i += NT) {
        bool ok = i < n_out;
        sbias[i] = ok ? P.L.bias[i] : 0.0f;
        sgam[i] = (ok && has_ln) ? P.L.gamma[i] : 1.0f;
        sbet[i] = (ok && has_ln) ? P.L.beta[i] : 0.0f;
    }
    if (P.has_head) {
        for (int i = tid; i < P.head.q * n_pad; i += NT) {
            int k = i / n_pad, c = i - k * n_pad;
            shw[i] = c < n_out ? P.head.w[(size_t)k * n_out + c] : 0.0f;
        }
        if (tid < P.head.q) shb[tid] = P.head.b[tid];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    FWD_T(0);       // prologue

    if (warp == 4 * CG) {
        // ---------------- producer
        if (lane == 0) {
            const size_t a_off = (size_t)itile * P.k_slabs * SLAB_FLOATS + (size_t)irow0 * SLAB_K;
            const int n_virt = P.k_slabs * P.passes;
            // blocks 2+: the weight slabs of the first stages (packed at least two launches back) go out before the
            // wait, the activation slabs (the previous block's output) after it.  Block 1's W1 is packed by the launch
            // just before this one.
            const int n_pre = BASIS ? 0 : min(n_virt, NSTAGE);
            for (int v = 0; v < n_pre; ++v) {
                const int s = v / P.passes, p = v - s * P.passes;
                issue_slab_copies(pass_b_lo(p) ? P.L.w_img_lo : P.L.w_img, P.k_slabs, s, n_pad,
                                  (pass_a_lo(p) ? P.a_img_lo : P.a_img) + a_off, sA + (size_t)v * SLAB_FLOATS,
                                  sB + v * b_stage_floats, &full[v], TM * 128u, true);
            }
            pdl_wait();
            pdl_launch_dependents();
            for (int v = 0; v < n_pre; ++v) {
                const int s = v / P.passes, p = v - s * P.passes;
                issue_a_slab(s, (pass_a_lo(p) ? P.a_img_lo : P.a_img) + a_off, sA + (size_t)v * SLAB_FLOATS, &full[v],
                             TM * 128u);
            }
            for (int v = n_pre; v < n_virt; ++v) {
                const int s = v / P.passes, p = v - s * P.passes;
                int stage = v % NSTAGE, it = v / NSTAGE;
                if (it > 0) FWD_WAIT(7, mbar_wait(&empty[stage], (it - 1) & 1));
                const float* w_src = pass_b_lo(p) ? P.L.w_img_lo : P.L.w_img;
                const float* a_tile = BASIS ? nullptr : (pass_a_lo(p) ? P.a_img_lo : P.a_img) + a_off;
                issue_slab_copies(w_src, P.k_slabs, s, n_pad, a_tile, sA + (size_t)stage * SLAB_FLOATS,
                                  sB + stage * b_stage_floats, &full[stage], TM * 128u);
            }
        }
        __syncwarp();
    } else if (warp == 4 * CG + 1) {
        // ---------------- MMA issuer
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_tf32((uint32_t)(WIDE ? MAX_N : n_pad), 0, 0, TM);
            const uint32_t idesc_hi = WIDE ? umma_idesc_tf32((uint32_t)(n_pad - MAX_N), 0, 0, TM) : 0u;
            const int n_virt = P.k_slabs * P.passes;
            for (int s = 0; s < n_virt; ++s) {
                int stage = s % NSTAGE, it = s / NSTAGE;
                FWD_WAIT(6, mbar_wait(&full[stage], it & 1));
                tc_fence_after();
                issue_slab_mma(tmem_base, sA + (size_t)stage * SLAB_FLOATS, sB + stage * b_stage_floats, idesc,
                               s == 0);
                if (WIDE)
                    issue_slab_mma(tmem_base + MAX_N, sA + (size_t)stage * SLAB_FLOATS,
                                   sB + stage * b_stage_floats + (size_t)MAX_N * SLAB_K, idesc_hi, s == 0);
                umma_commit(&empty[stage]);
            }
            umma_commit(accf);
        }
        __syncwarp();
    } else {
        // ---------------- workers: thread = (row, column group)
        const int q4 = warp & 3, cg = warp >> 2;
        const int row = G::row(q4, lane), grp = G::group(cg, lane);     // grp: the thread's 8 / NG chunks of each slab
        const long long lrow = (long long)tile * TM + row;
        const bool rvalid = tile_valid && lrow < P.pts.n_rows;
        const long long grow = P.pts.row_begin + lrow;
        // A one-wave training forward of block 2+ whose dropout step counter is settled (the previous step's tail
        // advanced it; ptx.cuh, rule 2) forms the keep bits of the thread's chunks here, while the previous launch still
        // runs, and parks them in shared memory for pass 2 of the epilogue: held in registers across the LayerNorm pass
        // they spill.  Block 1 (api.cu says why) and the 128-row forms keep the Philox calls in pass 2.
        if (!BASIS && TM == 64 && P.keep_off) {
            uint32_t* kw = reinterpret_cast<uint32_t*>(smem + P.keep_off) + tid;
            const unsigned int step = dropout_step(P.L);
            int ch = 0;
            for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += G::WARP_COLS * CG, ++ch) {
                const int c0 = wc + G::chunk_off(lane);
                if (c0 < n_pad)
                    kw[ch * NW] = pf_keep_mask(P.L.seed, step, (uint32_t)P.L.layer_id,
                                               P.L.key_offset + (unsigned long long)lrow, c0, P.thresh16);
            }
        }
        FWD_T(9);   // work before the wait
        // The points may have been written by the launch just before this one (a prediction call's inputs), the
        // addend by the support walk just before block 1, and the epilogue writes global memory: wait first.
        pdl_wait();
        FWD_T(10);  // wait for the previous launch
        if (BASIS) {
            float x = 0.f, y = 0.f, t = 0.f;
            const float* xrow = nullptr;
            if (rvalid) {
                load_point(P.pts, grow, x, y, t);
                if (P.basis.p_cov > 0 && P.pts.xcov) xrow = P.pts.xcov + sample_of(P.pts, grow) * P.basis.p_cov;
            }
            // one instantiation of the slab loop per basis function: the generator's inner code has no runtime switch
            auto gen_all = [&](auto fn_tag) {
                constexpr int FN = decltype(fn_tag)::value;
                int stage = 0, it = 0;
                for (int s = 0; s < P.k_slabs; ++s) {
                    float* gslab = (P.feat_img && tile_valid)
                                       ? P.feat_img + ((size_t)itile * P.k_slabs + s) * SLAB_FLOATS + (size_t)irow0 * SLAB_K
                                       : nullptr;
                    for (int p = 0; p < P.passes; ++p) {
                        if (it > 0) {
                            if (tid == 0) FWD_WAIT(5, mbar_wait(&empty[stage], (it - 1) & 1));
                            else mbar_wait(&empty[stage], (it - 1) & 1);
                        }
                        const uint32_t sa = smem_u32(sA + (size_t)stage * SLAB_FLOATS);
                        if (pass_a_lo(p))
                            gen_basis_slab_soa<FN, true, 2>(P.basis, ctab, s, x, y, t, xrow, sa, (uint32_t)row, grp * (8 / NG),
                                                         (grp + 1) * (8 / NG), nullptr);
                        else
                            gen_basis_slab_soa<FN, false, 2>(P.basis, ctab, s, x, y, t, xrow, sa, (uint32_t)row, grp * (8 / NG),
                                                          (grp + 1) * (8 / NG), p == 0 ? gslab : nullptr);
                        fence_proxy_async_smem();
                        mbar_arrive_warp(&full[stage]);
                        if (++stage == NSTAGE) { stage = 0; ++it; }
                    }
                }
            };
            if (P.basis.fn == STDADK_WENDLAND) gen_all(std::integral_constant<int, STDADK_WENDLAND>{});
            else if (P.basis.fn == STDADK_TRIANGULAR) gen_all(std::integral_constant<int, STDADK_TRIANGULAR>{});
            else gen_all(std::integral_constant<int, STDADK_GAUSSIAN>{});
        }
        FWD_T(1);   // operand generated (incl. waits for free stages)
        // ---------------- epilogue
        mbar_wait(accf, 0);
        tc_fence_after();
        FWD_T(2);   // wait for the accumulator
        EpiCtx E{sbias, sgam, sbet, shw, shb, red, tmem_base + ((uint32_t)(q4 * 32) << 16), itile, row, irow0 + row, cg, lane,
                 lrow, grow, rvalid, tile_valid};
        fwd_epilogue<CG, TM, !BASIS && TM == 64>(P, E);
        tc_fence_before();
        FWD_T(3);   // epilogue
    }
    __syncthreads();
    if (warp == 4 * CG) tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
    FWD_T(4);       // tail
}

// g[i] = sum_k dyh[k] * head_w[k, c0 + i]: the gradient entering the last hidden block, formed per row from the
// head (runtime loop over the Q outputs so the code stays small)
__device__ __forceinline__ void head_dh_chunk(float (&g)[32], const float (&dyh)[STDADK_MAX_Q], const float* shw, int n_pad,
                                              int c0, int q) {
#pragma unroll
    for (int i = 0; i < 32; ++i) g[i] = 0.0f;
#pragma unroll 1
    for (int k = 0; k < q; ++k) {
        float dk = 0.0f;
#pragma unroll
        for (int kk = 0; kk < STDADK_MAX_Q; ++kk)
            if (kk == k) dk = dyh[kk];
        const float* wk = shw + k * n_pad + c0;
#pragma unroll
        for (int i = 0; i < 32; ++i) g[i] = fmaf(dk, wk[i], g[i]);
    }
}

// =============================================================================================
// Backward
// =============================================================================================
// LN / HEAD are compile-time so that each instantiation carries only its own epilogue: the generic kernel was
// 150 KB of SASS and a one-wave launch (32 tiles) spent ~30% of its stall samples on instruction fetch.
// The wide form, NS = 2 (MAX_N < n_pad <= MAX_W; the narrow form has NS = 4): x comes from the forward's image only (no
// recompute GEMM, BASIS is false), so the dh accumulator starts at column 0 and spans up to MAX_W columns, two MMAs per
// K slab as in the wide forward.  There is no free half of tensor memory for x^: x_early stays off.
template <bool BASIS, int TM, int CG, int NS, bool LN, bool HEAD>
__global__ void __launch_bounds__(n_threads(CG), 1) layer_bwd_kernel(const __grid_constant__ BwdK P) {
    using G = TileGeo<TM>;
    constexpr bool WIDE = NS == 2;
    constexpr int NW = n_work(CG), NT = n_threads(CG), NSTAGE = NS, NG = G::groups(CG);
    constexpr int WSTEP = G::WARP_COLS * CG;
    constexpr int MAXCH = (WIDE ? MAX_W : MAX_N) / WSTEP;   // column chunks per thread
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem(smem_raw);
    const int q = HEAD ? P.head.q : 0;
    const SmemPlan sp = plan_smem(P.n_pad, q, BASIS ? P.basis.k_s : 0, BASIS ? P.basis.k_t : 0, true, CG, NS,
                                  BASIS ? P.k_slabs * 8 : 0);
    float* sA = reinterpret_cast<float*>(smem + sp.a_off);
    float* sB = reinterpret_cast<float*>(smem + sp.b_off);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + sp.bar_off);
    uint64_t* empty = full + NSTAGE;
    uint64_t* accf = full + 2 * NSTAGE;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + sp.tmem_off);
    float* sbias = reinterpret_cast<float*>(smem + sp.vec_off);
    float* sgam = sbias + P.n_pad;
    float* sbet = sgam + P.n_pad;
    float* shw = reinterpret_cast<float*>(smem + sp.headw_off);
    float4* ctab = reinterpret_cast<float4*>(smem + sp.knots_off);  // chunk tables of the generator (BASIS)
    float* cs_bias = reinterpret_cast<float*>(smem + sp.colsum_off);
    float* cs_gam = cs_bias + P.n_pad;
    float* cs_bet = cs_gam + P.n_pad;
    float* cs_hw = cs_bet + P.n_pad;
    float* cs_hb = cs_hw + q * P.n_pad;
    float* red = reinterpret_cast<float*>(smem + sp.red_off);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tile = blockIdx.x;
    STEP_T_BEGIN(P.dbg);
    const int itile = tile / (TILE_M / TM), irow0 = (tile % (TILE_M / TM)) * TM;   // image tile, first row in it
    const int n_pad = P.n_pad, n_out = P.L.n_out;
    constexpr bool has_ln = LN;
    const size_t b_stage_floats = (size_t)n_pad * SLAB_K;
    const int virt1 = P.k_slabs * P.passes;                 // GEMM 1 (recompute), then GEMM 2 (dgrad): virtual slabs
    const int total_slabs = virt1 + P.k_slabs2 * P.passes;
    const uint32_t acc1_off = WIDE ? 0u : (uint32_t)(P.tmem_cols / 2);

    if (tid == NW) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&full[s], BASIS ? 1 + NW / 32 : 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accf, 1);
        mbar_fence_init();
    }
    if (warp == 4 * CG) {
        __syncwarp();
        tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    }
    if (BASIS) build_chunk_tables(P.basis, ctab, P.k_slabs * 8, tid, NT);
    for (int i = tid; i < n_pad; i += NT) {
        bool ok = i < n_out;
        sbias[i] = ok ? P.L.bias[i] : 0.0f;
        sgam[i] = (ok && has_ln) ? P.L.gamma[i] : 1.0f;
        sbet[i] = (ok && has_ln) ? P.L.beta[i] : 0.0f;
    }
    for (int i = tid; i < (3 + q) * n_pad + STDADK_MAX_Q; i += NT) cs_bias[i] = 0.0f;
    if (HEAD) {
        for (int i = tid; i < q * n_pad; i += NT) {
            int k = i / n_pad, c = i - k * n_pad;
            shw[i] = c < n_out ? P.head.w[(size_t)k * n_out + c] : 0.0f;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    STEP_T(P.dbg, 0);   // prologue

    if (warp == 4 * CG) {
        if (lane == 0) {
            const size_t a_off = (size_t)itile * P.k_slabs * SLAB_FLOATS + (size_t)irow0 * SLAB_K;
            const size_t dzn_off = (size_t)itile * P.k_slabs2 * SLAB_FLOATS + (size_t)irow0 * SLAB_K;
            // Before the wait: the first stages' slabs that come from further back than the previous launch -- both
            // operands of the recompute GEMM (weights, earlier activations) and W_next^T of the dgrad GEMM.  dz_next
            // is the previous launch's output: its slabs of those stages are issued after the wait.
            const int n_pre = min(total_slabs, NSTAGE);
            auto wait_then_dz_next = [&]() {
                pdl_wait();
                pdl_launch_dependents();
                for (int v = virt1; v < n_pre; ++v) {
                    const int s = (v - virt1) / P.passes, p = (v - virt1) - s * P.passes;
                    issue_a_slab(s, (pass_a_lo(p) ? P.dz_next_img_lo : P.dz_next_img) + dzn_off,
                                 sA + (size_t)v * SLAB_FLOATS, &full[v], TM * 128u);
                }
            };
            for (int v = 0; v < total_slabs; ++v) {
                if (v == n_pre) wait_then_dz_next();
                int stage = v % NSTAGE, it = v / NSTAGE;
                if (it > 0) mbar_wait(&empty[stage], (it - 1) & 1);
                float* a_dst = sA + (size_t)stage * SLAB_FLOATS;
                float* b_dst = sB + stage * b_stage_floats;
                if (v < virt1) {
                    const int s = v / P.passes, p = v - s * P.passes;
                    const float* a_tile = BASIS ? nullptr : (pass_a_lo(p) ? P.a_img_lo : P.a_img) + a_off;
                    issue_slab_copies(pass_b_lo(p) ? P.L.w_img_lo : P.L.w_img, P.k_slabs, s, n_pad, a_tile, a_dst, b_dst,
                                      &full[stage], TM * 128u);
                } else {
                    const int s = (v - virt1) / P.passes, p = (v - virt1) - s * P.passes;
                    issue_slab_copies(pass_b_lo(p) ? P.wt_next_img_lo : P.wt_next_img, P.k_slabs2, s, n_pad,
                                      (pass_a_lo(p) ? P.dz_next_img_lo : P.dz_next_img) + dzn_off, a_dst, b_dst, &full[stage],
                                      TM * 128u, v < n_pre);
                }
            }
            if (total_slabs == n_pre) wait_then_dz_next();
        }
        __syncwarp();
    } else if (warp == 4 * CG + 1) {
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_tf32((uint32_t)(WIDE ? MAX_N : n_pad), 0, 0, TM);
            const uint32_t idesc_hi = WIDE ? umma_idesc_tf32((uint32_t)(n_pad - MAX_N), 0, 0, TM) : 0u;
            for (int s = 0; s < total_slabs; ++s) {
                int stage = s % NSTAGE, it = s / NSTAGE;
                mbar_wait(&full[stage], it & 1);
                tc_fence_after();
                bool second = s >= virt1;
                issue_slab_mma(tmem_base + (second ? acc1_off : 0u), sA + (size_t)stage * SLAB_FLOATS,
                               sB + stage * b_stage_floats, idesc, s == 0 || s == virt1);
                if (WIDE)
                    issue_slab_mma(tmem_base + MAX_N, sA + (size_t)stage * SLAB_FLOATS,
                                   sB + stage * b_stage_floats + (size_t)MAX_N * SLAB_K, idesc_hi, s == 0);
                umma_commit(&empty[stage]);
            }
            umma_commit(accf);
        }
        __syncwarp();
    } else {
        const int q4 = warp & 3, cg = warp >> 2;
        const int row = G::row(q4, lane), irow = irow0 + row, grp = G::group(cg, lane), coff = G::chunk_off(lane);
        const int c_begin = grp * (8 / NG), c_end = (grp + 1) * (8 / NG);     // chunks of each slab this thread generates
        const long long lrow = (long long)tile * TM + row;
        const bool rvalid = lrow < P.pts.n_rows;
        const long long grow = P.pts.row_begin + lrow;
        if (BASIS) {
            float x = 0.f, y = 0.f, t = 0.f;
            const float* xrow = nullptr;
            if (rvalid) {
                load_point(P.pts, grow, x, y, t);
                if (P.basis.p_cov > 0 && P.pts.xcov) xrow = P.pts.xcov + sample_of(P.pts, grow) * P.basis.p_cov;
            }
            // the forward's generator (chunk tables, packed FP32): the regenerated operand is the forward's bit for bit
            auto gen_all = [&](auto fn_tag) {
                constexpr int FN = decltype(fn_tag)::value;
                for (int v = 0; v < total_slabs; ++v) {
                    int stage = v % NSTAGE, it = v / NSTAGE;
                    if (it > 0) mbar_wait(&empty[stage], (it - 1) & 1);
                    if (v < virt1) {
                        const int s = v / P.passes, p = v - s * P.passes;
                        const uint32_t sa = smem_u32(sA + (size_t)stage * SLAB_FLOATS);
                        if (pass_a_lo(p))
                            gen_basis_slab_soa<FN, true, 2>(P.basis, ctab, s, x, y, t, xrow, sa, (uint32_t)row, c_begin,
                                                            c_end, nullptr);
                        else
                            gen_basis_slab_soa<FN, false, 2>(P.basis, ctab, s, x, y, t, xrow, sa, (uint32_t)row, c_begin,
                                                             c_end, nullptr);
                        fence_proxy_async_smem();
                    }
                    mbar_arrive_warp(&full[stage]);
                }
            };
            if (P.basis.fn == STDADK_WENDLAND) gen_all(std::integral_constant<int, STDADK_WENDLAND>{});
            else if (P.basis.fn == STDADK_TRIANGULAR) gen_all(std::integral_constant<int, STDADK_TRIANGULAR>{});
            else gen_all(std::integral_constant<int, STDADK_GAUSSIAN>{});
        }
        const uint32_t trow = tmem_base + ((uint32_t)(q4 * 32) << 16);
        const bool drop = P.L.drop_p > 0.0f;
        const float inv_n = 1.0f / (float)n_out;
        float mean = 0.0f, rstd = 1.0f;
        uint32_t actbits[MAXCH];     // before pass A of a chunk its keep bits (when formed before the wait), after it
                                     // its activation bits
        float z[32], g[32], tmp[32];
        auto load_stats = [&]() {
            if (has_ln && rvalid) {
                mean = P.stats[2 * lrow];
                rstd = P.stats[2 * lrow + 1];
            }
        };
        // Before the wait, when the caller says the inputs are settled (ptx.cuh, rule 2; the launcher passes the bits
        // to the one-wave x-image backward only, the recompute backward keeps its order): the keep bits and, for a
        // 64-row tile of a block below the head, whose x image and stats are at least two launches old, x^ and the
        // activation bits.  x^ goes to the half of tensor memory that the recompute GEMM would use (an x-image backward
        // has none): the warp's chunk at column wc sits in columns wc / 2 .. +31, one 32x32b lane per thread, so the
        // epilogue reads it back with one tcgen05.ld instead of two dependent trips to L2.
        constexpr bool X_EARLY_OK = TM == 64 && !HEAD && !WIDE;
        const bool keeps_early = P.step_settled != 0;
        const bool x_early = X_EARLY_OK && keeps_early && P.x_settled != 0;
        if (keeps_early) chunk_keep_masks<TM, CG, MAXCH>(P.L, P.thresh16, lrow, cg, lane, n_pad, actbits);
        if (x_early) {
            load_stats();
            int ch = 0;
            for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += WSTEP, ++ch) {
                const int c0 = wc + coff;
                const bool cvalid = c0 < n_pad;
                if (cvalid) image_load_chunk(P.x_img, itile, n_pad / SLAB_K, c0, (uint32_t)irow, z);
                else
#pragma unroll
                    for (int i = 0; i < 32; ++i) z[i] = 0.0f;
                uint32_t keep = 0, act = 0;
#pragma unroll
                for (int k = 0; k < MAXCH; ++k)
                    if (k == ch) keep = actbits[k];
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int col = c0 + i;
                    const float xh = has_ln ? (z[i] - mean) * rstd : z[i];
                    const float yv = has_ln ? fmaf(xh, sgam[col], sbet[col]) : z[i];
                    const bool on = (yv > 0.0f) && ((keep >> i) & 1u) && (col < n_out) && rvalid;
                    act |= (on ? 1u : 0u) << i;
                    z[i] = xh;
                }
#pragma unroll
                for (int k = 0; k < MAXCH; ++k)
                    if (k == ch) actbits[k] = act;
                tmem_st32(trow + (uint32_t)(wc / 2), z);
            }
            tmem_st_wait();
        }
        STEP_T(P.dbg, 1);   // work before the wait
        // the regenerated operand reads only points and knot tables, which the forward read before; the epilogue
        // reads the previous launch's output
        pdl_wait();
        STEP_T(P.dbg, 2);   // wait for the previous launch
        if (!x_early) load_stats();
        mbar_wait(accf, 0);
        tc_fence_after();
        STEP_T(P.dbg, 3);   // accumulator ready
        float* myred = red + ((size_t)grp * TM + row) * RED_STRIDE;
        const float* arow = (P.addend && rvalid) ? P.addend + (size_t)lrow * n_out : nullptr;
        float dyh[STDADK_MAX_Q];
#pragma unroll
        for (int k = 0; k < STDADK_MAX_Q; ++k)
            dyh[k] = (HEAD && rvalid && k < q) ? P.head.dyhat[lrow * q + k] : 0.0f;
        float Sa = 0.0f, Sb = 0.0f;

        // pass A: g = dL/dy (after dropout+ReLU backward); LN row sums; dgamma/dbeta/head column sums
        // a chunk at n_pad (TM = 64, odd number of 32-column chunks) reads zeros and writes nothing: its columns fail
        // col < n_out below, so it contributes nothing to the row and column sums
        int ch = 0;
        for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += WSTEP, ++ch) {
            const int c0 = wc + coff;
            const bool cvalid = TM == 128 || c0 < n_pad;
            if (x_early) {
                tmem_ld32(trow + (uint32_t)(wc / 2), z);       // x^
            } else if (WIDE || P.x_img) {
                if (cvalid) image_load_chunk(P.x_img, itile, n_pad / SLAB_K, c0, (uint32_t)irow, z);    // x saved by the forward
            } else {
                acc_ld<TM>(trow + wc, z);
                if (arow) add_addend_chunk(z, arow, c0, n_out);
#pragma unroll
                for (int i = 0; i < 32; ++i) z[i] += sbias[c0 + i];
            }
            if (!cvalid && !x_early)
#pragma unroll
                for (int i = 0; i < 32; ++i) z[i] = 0.0f;
            if (!HEAD) acc_ld<TM>(trow + acc1_off + wc, g);
            else head_dh_chunk(g, dyh, shw, n_pad, c0, cvalid ? q : 0);
            if (x_early) {
                uint32_t act = 0;
#pragma unroll
                for (int k = 0; k < MAXCH; ++k)
                    if (k == ch) act = actbits[k];
#pragma unroll
                for (int i = 0; i < 32; ++i) g[i] = ((act >> i) & 1u) ? g[i] * P.drop_scale : 0.0f;
            } else {
                uint32_t keep = 0xFFFFFFFFu, act = 0;
                if (keeps_early) {
#pragma unroll
                    for (int k = 0; k < MAXCH; ++k)
                        if (k == ch) keep = actbits[k];
                } else if (drop && cvalid) {
                    keep = pf_keep_mask(P.L.seed, dropout_step(P.L), (uint32_t)P.L.layer_id,
                                        P.L.key_offset + (unsigned long long)lrow, c0, P.thresh16);
                }
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int col = c0 + i;
                    float x = z[i];
                    float xh = has_ln ? (x - mean) * rstd : x;
                    float yv = has_ln ? fmaf(xh, sgam[col], sbet[col]) : x;
                    bool on = (yv > 0.0f) && ((keep >> i) & 1u) && (col < n_out) && rvalid;
                    act |= (on ? 1u : 0u) << i;
                    const float dh = g[i];
                    float h = on ? yv * P.drop_scale : 0.0f;  // forward activation (for the head gradient)
                    g[i] = on ? dh * P.drop_scale : 0.0f;
                    z[i] = xh;
                    tmp[i] = h;
                }
#pragma unroll
                for (int k = 0; k < MAXCH; ++k)
                    if (k == ch) actbits[k] = act;
            }
            if (HEAD) {
                for (int k = 0; k < q; ++k) {
                    float hv[32];
                    const float dk = dyh[k];
#pragma unroll
                    for (int i = 0; i < 32; ++i) hv[i] = dk * tmp[i];
                    colsum_chunk<TM>(cs_hw + k * n_pad, c0, cvalid, hv, lane);
                }
            }
            if (has_ln) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float gy = g[i] * sgam[c0 + i];
                    Sa += gy;
                    Sb = fmaf(gy, z[i], Sb);
                    tmp[i] = g[i] * z[i];
                }
                colsum_chunk<TM>(cs_gam, c0, cvalid, tmp, lane);
#pragma unroll
                for (int i = 0; i < 32; ++i) tmp[i] = g[i];
                colsum_chunk<TM>(cs_bet, c0, cvalid, tmp, lane);
            } else {
                if (cvalid) store_operand_chunk(P.dz_img, P.dz_img_lo, itile, n_pad / SLAB_K, c0, (uint32_t)irow, g);
                colsum_chunk<TM>(cs_bias, c0, cvalid, g, lane);
            }
        }
        STEP_T(P.dbg, 4);   // pass A
        if (HEAD && cg == 0) {
            for (int k = 0; k < q; ++k) {
                float s = warp_sum(TM == 128 || lane < 16 ? dyh[k] : 0.0f);    // a TM = 64 row sits in both half-warps
                if (lane == 0) atomicAdd(&cs_hb[k], s);
            }
        }
        // pass B (LayerNorm): dz = rstd * (gy - mean(gy) - xh * mean(gy * xh))
        if (has_ln) {
            if (NG > 1) {
                myred[0] = Sa;
                myred[1] = Sb;
                worker_barrier(NW);
                Sa = Sb = 0.0f;
#pragma unroll
                for (int gq = 0; gq < NG; ++gq) {
                    Sa += red[((size_t)gq * TM + row) * RED_STRIDE];
                    Sb += red[((size_t)gq * TM + row) * RED_STRIDE + 1];
                }
            }
            const float ma = Sa * inv_n, mb = Sb * inv_n;
            ch = 0;
            for (int wc = G::WARP_COLS * cg; wc < n_pad; wc += WSTEP, ++ch) {
                const int c0 = wc + coff;
                const bool cvalid = TM == 128 || c0 < n_pad;
                if (x_early) {
                    tmem_ld32(trow + (uint32_t)(wc / 2), z);   // x^
                } else if (WIDE || P.x_img) {
                    if (cvalid) image_load_chunk(P.x_img, itile, n_pad / SLAB_K, c0, (uint32_t)irow, z);
                } else {
                    acc_ld<TM>(trow + wc, z);
                    if (arow) add_addend_chunk(z, arow, c0, n_out);
#pragma unroll
                    for (int i = 0; i < 32; ++i) z[i] += sbias[c0 + i];
                }
                if (!cvalid && !x_early)
#pragma unroll
                    for (int i = 0; i < 32; ++i) z[i] = 0.0f;
                if (!HEAD) acc_ld<TM>(trow + acc1_off + wc, g);
                else head_dh_chunk(g, dyh, shw, n_pad, c0, cvalid ? q : 0);
                uint32_t act = 0;
#pragma unroll
                for (int k = 0; k < MAXCH; ++k)
                    if (k == ch) act = actbits[k];
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const int col = c0 + i;
                    float xh = x_early ? z[i] : (z[i] - mean) * rstd;
                    const float dh = g[i];
                    float gy = ((act >> i) & 1u) ? dh * P.drop_scale * sgam[col] : 0.0f;
                    float dz = rstd * (gy - ma - xh * mb);
                    g[i] = (col < n_out && rvalid) ? dz : 0.0f;
                }
                if (cvalid) store_operand_chunk(P.dz_img, P.dz_img_lo, itile, n_pad / SLAB_K, c0, (uint32_t)irow, g);
                colsum_chunk<TM>(cs_bias, c0, cvalid, g, lane);
            }
        }
        tc_fence_before();
        // flush the CTA's column sums
        worker_barrier(NW);
        for (int c = tid; c < n_out; c += NW) {
            atomicAdd(&P.d_bias[c], cs_bias[c]);
            if (has_ln) {
                atomicAdd(&P.d_gamma[c], cs_gam[c]);
                atomicAdd(&P.d_beta[c], cs_bet[c]);
            }
            for (int k = 0; k < q; ++k) atomicAdd(&P.d_head_w[(size_t)k * n_out + c], cs_hw[k * n_pad + c]);
        }
        if (tid < q) atomicAdd(&P.d_head_b[tid], cs_hb[tid]);
        STEP_T(P.dbg, 5);   // pass B, column-sum flush
    }
    __syncthreads();
    if (warp == 4 * CG) tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
}

// =============================================================================================
// Weight gradient: dW[o, i] += sum_rows dz[row, o] * A[row, i]
//
// The reduction runs over rows, so both operands are MN-major (the contiguous 128 bytes of an image
// row are 32 values of the M / N dimension).  For 32-bit (TF32) MN-major operands tcgen05 accepts a
// single shared-memory form, SWIZZLE_128B_BASE32B (32-byte units XOR-ed with row & 3, atoms of 4 rows
// x 128 B), which differs from the 16-byte-unit swizzle of the K-major images; the workers therefore
// restage each 64-row half tile HBM -> registers -> SMEM (coalesced 16-byte loads, conflict-free
// stores) and, for block 1, regenerate the basis straight into that form.
// =============================================================================================
struct WgradK {
    BasisP basis;
    PointsP pts;
    const float* a_img;
    const float* a_img_lo;      // tf32x3 residual images (NULL in TF32 mode)
    const float* dz_img;
    const float* dz_img_lo;
    float* dw;
    long long stride_o, stride_i;
    int n_in, n_out, a_slabs, dz_slabs, n_row_tiles, nt_slabs, tmem_cols, passes;
};
constexpr int WG_HALF_ROWS = 64;
constexpr int WG_CHUNK_BYTES = WG_HALF_ROWS * 128;           // 8 KB: 64 rows of one slab
constexpr int WG_A_BYTES = 4 * WG_CHUNK_BYTES;               // M = 128 = 4 chunks of 32
constexpr int WG_B_BYTES = 8 * WG_CHUNK_BYTES;               // N <= 256
constexpr int WG_STAGE_BYTES = WG_A_BYTES + WG_B_BYTES;

__host__ __device__ inline uint32_t wgrad_smem_bytes(int k_s, int k_t) {
    return WG_NSTAGE * WG_STAGE_BYTES + 64 + 16 + 16 + (uint32_t)k_s * 16u + (uint32_t)k_t * 8u + 16 + 1024;
}
// byte offset of logical 16-byte chunk `c16` of row `row` in the SWIZZLE_128B_BASE32B form
__device__ __forceinline__ uint32_t swz32_off(uint32_t row, uint32_t c16) {
    return row * 128u + ((((c16 >> 1) ^ (row & 3u)) << 5) | ((c16 & 1u) << 4));
}
__device__ __forceinline__ uint64_t umma_desc_sw128_32b(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (1ull << 61);
}
// Restage half-slabs (64 rows x 128 B each, image swizzle) of the dz tile and (optionally) of the A tile into the
// MN-major SMEM form.  ALL loads of the half tile are issued before the first store (8 + 16 16-byte loads per thread
// at 256 workers): the restage is bound by global-load latency, and with four loads in flight per thread it ran at
// ~16 GB/s per SM -- 26 us per row tile, which made wgrad the largest kernel of a large-batch step.
template <int NW>
__device__ __forceinline__ void restage_half_tiles(const float* dz_tile, int mslab0, int m_chunks, const float* a_tile,
                                                   int nslab0, int n_chunks, int half, uint32_t sa, uint32_t sb, int tid) {
    constexpr int BD = 2048 / NW, BA = 4096 / NW;      // dz: <= 4 chunks, A: <= 8 chunks of 512 units
    static_assert(NW * BD == 2048 && NW * BA == 4096, "worker count must divide the half-tile unit counts");
    const int units_d = m_chunks * 512, units_a = a_tile ? n_chunks * 512 : 0;
    const size_t hoff = (size_t)half * WG_HALF_ROWS * SLAB_K;
    float4 vd[BD], va[BA];
#pragma unroll
    for (int j = 0; j < BD; ++j) {
        const int u = tid + j * NW;
        if (u < units_d)
            vd[j] = __ldg(reinterpret_cast<const float4*>(dz_tile + (size_t)(mslab0 + (u >> 9)) * SLAB_FLOATS + hoff) + (u & 511));
    }
#pragma unroll
    for (int j = 0; j < BA; ++j) {
        const int u = tid + j * NW;
        if (u < units_a)
            va[j] = __ldg(reinterpret_cast<const float4*>(a_tile + (size_t)(nslab0 + (u >> 9)) * SLAB_FLOATS + hoff) + (u & 511));
    }
#pragma unroll
    for (int j = 0; j < BD; ++j) {
        const int u = tid + j * NW;
        if (u < units_d) {
            const int c = u >> 9, w = u & 511;
            const uint32_t r = (uint32_t)(w >> 3), lc = (uint32_t)(w & 7) ^ (r & 7u);
            st_shared_v4(sa + c * WG_CHUNK_BYTES + swz32_off(r, lc), vd[j].x, vd[j].y, vd[j].z, vd[j].w);
        }
    }
#pragma unroll
    for (int j = 0; j < BA; ++j) {
        const int u = tid + j * NW;
        if (u < units_a) {
            const int c = u >> 9, w = u & 511;
            const uint32_t r = (uint32_t)(w >> 3), lc = (uint32_t)(w & 7) ^ (r & 7u);
            st_shared_v4(sb + c * WG_CHUNK_BYTES + swz32_off(r, lc), va[j].x, va[j].y, va[j].z, va[j].w);
        }
    }
}

// Block 1's wgrad: the basis half (B operand, MN-major) of one stage for (row tile, half, tf32x3 pass), regenerated
// from the points and the knot tables.  Out of line: the kernel calls it before and after pdl_wait(), and two inlined
// copies cost the kernel six registers.
template <int NW>
__device__ __noinline__ void wgrad_gen_basis_half(const WgradK& P, const float4* sk, const float2* st, int rt, int half,
                                                  int pass, uint32_t sb, int row64, int par, int n_chunks) {
    float x = 0.f, y = 0.f, t = 0.f;
    const float* xrow = nullptr;
    long long lrow = (long long)rt * TILE_M + half * WG_HALF_ROWS + row64;
    if (lrow < P.pts.n_rows) {
        long long grow = P.pts.row_begin + lrow;
        load_point(P.pts, grow, x, y, t);
        if (P.basis.p_cov > 0 && P.pts.xcov) xrow = P.pts.xcov + sample_of(P.pts, grow) * P.basis.p_cov;
    }
    const int ni = blockIdx.z;
    for (int c = par; c < n_chunks; c += NW / 64) {
        const int slab = ni * P.nt_slabs + c;
#pragma unroll 1
        for (int c16 = 0; c16 < 8; ++c16) {
            float4 v = feature_chunk(P.basis, sk, st, slab * SLAB_K + c16 * 4, x, y, t, xrow, pass_b_lo(pass));
            st_shared_v4(sb + c * WG_CHUNK_BYTES + swz32_off((uint32_t)row64, (uint32_t)c16), v.x, v.y, v.z, v.w);
        }
    }
}

template <bool BASIS, int CG>
__global__ void __launch_bounds__(n_threads(CG), 1) wgrad_kernel(const __grid_constant__ WgradK P) {
    constexpr int NW = n_work(CG), NT = n_threads(CG);
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem(smem_raw);
    uint8_t* stage_base = smem;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + WG_NSTAGE * WG_STAGE_BYTES);
    uint64_t* empty = full + WG_NSTAGE;
    uint64_t* accf = full + 2 * WG_NSTAGE;
    uint64_t* kbar = accf + 1;                                       // knot tables have landed (BASIS)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + WG_NSTAGE * WG_STAGE_BYTES + 64);
    float4* sk = reinterpret_cast<float4*>(smem + WG_NSTAGE * WG_STAGE_BYTES + 96);
    float2* st = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(sk) + (size_t)(BASIS ? P.basis.k_s : 0) * 16);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int split = blockIdx.x, n_split = gridDim.x, mi = blockIdx.y, ni = blockIdx.z;
    const int m_chunks = min(4, P.dz_slabs - mi * 4);
    const int n_chunks = min(P.nt_slabs, P.a_slabs - ni * P.nt_slabs);
    const int n_mma = n_chunks * SLAB_K;
    int my_tiles = 0;
    for (int rt = split; rt < P.n_row_tiles; rt += n_split) ++my_tiles;
    const int n_iter = my_tiles * 2 * P.passes;     // (row tile, half, tf32x3 pass)

    if (tid == NW) {
        for (int s = 0; s < WG_NSTAGE; ++s) {
            mbar_init(&full[s], NW / 32);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accf, 1);
        mbar_init(kbar, 1);
        mbar_fence_init();
        if (BASIS) stage_knots_async(P.basis, sk, st, kbar);
    }
    if (warp == 4 * CG) {
        __syncwarp();
        tmem_alloc(tmem_slot, (uint32_t)P.tmem_cols);
    }
    // unused M chunks must read as zeros (they are never overwritten)
    if (m_chunks < 4) {
        for (int s = 0; s < WG_NSTAGE; ++s) {
            float4* zp = reinterpret_cast<float4*>(stage_base + s * WG_STAGE_BYTES + m_chunks * WG_CHUNK_BYTES);
            int n16 = (4 - m_chunks) * WG_CHUNK_BYTES / 16;
            for (int i = tid; i < n16; i += NT) zp[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (n_iter > 0) {
        if (warp == 4 * CG + 1) {
            if (lane == 0) {
                const uint32_t idesc = umma_idesc_tf32((uint32_t)n_mma, 1, 1);
                for (int itn = 0; itn < n_iter; ++itn) {
                    int stage = itn % WG_NSTAGE, it = itn / WG_NSTAGE;
                    mbar_wait(&full[stage], it & 1);
                    tc_fence_after();
                    uint32_t sa = smem_u32(stage_base + stage * WG_STAGE_BYTES);
                    uint32_t sb = sa + WG_A_BYTES;
#pragma unroll
                    for (int k8 = 0; k8 < WG_HALF_ROWS / 8; ++k8) {
                        uint64_t ad = umma_desc_sw128_32b(sa + k8 * 1024, WG_CHUNK_BYTES, 512);
                        uint64_t bd = umma_desc_sw128_32b(sb + k8 * 1024, WG_CHUNK_BYTES, 512);
                        umma_tf32(tmem_base, ad, bd, idesc, (itn == 0 && k8 == 0) ? 0u : 1u);
                    }
                    umma_commit(&empty[stage]);
                }
                umma_commit(accf);
            }
            __syncwarp();
        } else if (warp < 4 * CG) {
            const int row64 = tid & 63, par = tid >> 6;
            auto gen_basis = [&](int rt, int half, int pass, int stage) {
                wgrad_gen_basis_half<NW>(P, sk, st, rt, half, pass, smem_u32(stage_base + stage * WG_STAGE_BYTES) + WG_A_BYTES,
                                         row64, par, n_chunks);
            };
            // Before the wait: the basis halves of the first stages (points and knot tables, read by the forward
            // before).  After it: dz, the previous launch's output.
            const int n_pre = BASIS ? min(n_iter, WG_NSTAGE) : 0;
            int itn = 0;
            if (BASIS) {
                mbar_wait(kbar, 0);
                for (int rt = split; rt < P.n_row_tiles && itn < n_pre; rt += n_split)
                    for (int hp = 0; hp < 2 * P.passes && itn < n_pre; ++hp, ++itn)
                        gen_basis(rt, hp / P.passes, hp % P.passes, itn);
            }
            pdl_wait();
            pdl_launch_dependents();
            itn = 0;
            for (int rt = split; rt < P.n_row_tiles; rt += n_split)
                for (int hp = 0; hp < 2 * P.passes; ++hp, ++itn) {
                    const int half = hp / P.passes, pass = hp - half * P.passes;
                    int stage = itn % WG_NSTAGE, it = itn / WG_NSTAGE;
                    if (it > 0) mbar_wait(&empty[stage], (it - 1) & 1);
                    uint32_t sa = smem_u32(stage_base + stage * WG_STAGE_BYTES);
                    uint32_t sb = sa + WG_A_BYTES;
                    restage_half_tiles<NW>((pass_a_lo(pass) ? P.dz_img_lo : P.dz_img) + (size_t)rt * P.dz_slabs * SLAB_FLOATS,
                                           mi * 4, m_chunks,
                                           BASIS ? nullptr
                                                 : (pass_b_lo(pass) ? P.a_img_lo : P.a_img) + (size_t)rt * P.a_slabs * SLAB_FLOATS,
                                           ni * P.nt_slabs, n_chunks, half, sa, sb, tid);
                    if (BASIS && itn >= n_pre) gen_basis(rt, half, pass, stage);
                    fence_proxy_async_smem();
                    mbar_arrive_warp(&full[stage]);
                }
            mbar_wait(accf, 0);
            tc_fence_after();
            const int q4 = warp & 3, cg = warp >> 2;
            const uint32_t trow = tmem_base + ((uint32_t)(q4 * 32) << 16);
            const int o = mi * TILE_M + q4 * 32 + lane;
            float v[32];
            for (int c0 = 32 * cg; c0 < n_mma; c0 += 32 * CG) {
                tmem_ld32(trow + c0, v);
                if (o < P.n_out) {
                    float* dst = P.dw + (long long)o * P.stride_o;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        int col = ni * P.nt_slabs * SLAB_K + c0 + i;
                        if (col < P.n_in) atomicAdd(dst + (long long)col * P.stride_i, v[i]);
                    }
                }
            }
            tc_fence_before();
        }
    }
    __syncthreads();
    if (warp == 4 * CG) tmem_dealloc(tmem_base, (uint32_t)P.tmem_cols);
}

}  // namespace stdadk

// =============================================================================================
// Gradient of learnable knots (centres, log-bandwidths): G^T = W1s dz1^T on the tensor cores
// (M = 128 knots, N = 128 points, K = n_out), then the closed-form chain rule per (knot, point).
// =============================================================================================
namespace stdadk {

struct KnotGradK {
    BasisP basis;
    PointsP pts;
    const float* dz_img;
    const float* dz_img_lo;     // tf32x3 residual images (NULL in TF32 mode)
    const float* w1s_img;
    const float* w1s_img_lo;
    float* d_centers;
    float* d_log_bw;
    int n_out, k_slabs, passes, _p1;
};

template <int CG>
__global__ void __launch_bounds__(n_threads(CG)) knotgrad_kernel(const __grid_constant__ KnotGradK P) {
    constexpr int NW = n_work(CG), NSTAGE = 2;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem(smem_raw);
    const SmemPlan sp = plan_smem(TILE_M, 0, 0, 0, false);
    float* sA = reinterpret_cast<float*>(smem + sp.a_off);
    float* sB = reinterpret_cast<float*>(smem + sp.b_off);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + sp.bar_off);
    uint64_t* empty = full + NSTAGE;
    uint64_t* accf = full + 2 * NSTAGE;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + sp.tmem_off);
    float2* spt = reinterpret_cast<float2*>(smem + sp.vec_off);  // 128 points (x, y): 1 KB <= 3*128*4

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int ptile = blockIdx.x, ktile = blockIdx.y;
    if (tid == NW) {
        for (int s = 0; s < NSTAGE; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 1);
        }
        mbar_init(accf, 1);
        mbar_fence_init();
    }
    if (warp == 4 * CG) {
        __syncwarp();
        tmem_alloc(tmem_slot, TILE_M);
    }
    if (tid < TILE_M) {
        long long lrow = (long long)ptile * TILE_M + tid;
        float x = 0.f, y = 0.f, t = 0.f;
        if (lrow < P.pts.n_rows) load_point(P.pts, P.pts.row_begin + lrow, x, y, t);
        spt[tid] = make_float2(x, y);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4 * CG) {
        if (lane == 0) {
            const size_t a_off = (size_t)ktile * P.k_slabs * SLAB_FLOATS;
            for (int v = 0; v < P.k_slabs * P.passes; ++v) {
                const int s = v / P.passes, p = v - s * P.passes;
                int stage = v % NSTAGE, it = v / NSTAGE;
                if (it > 0) mbar_wait(&empty[stage], (it - 1) & 1);
                mbar_arrive_expect_tx(&full[stage], 2 * SLAB_BYTES);
                bulk_g2s(sA + (size_t)stage * SLAB_FLOATS,
                         (pass_a_lo(p) ? P.w1s_img_lo : P.w1s_img) + a_off + (size_t)s * SLAB_FLOATS, SLAB_BYTES, &full[stage]);
                bulk_g2s(sB + (size_t)stage * SLAB_FLOATS,
                         (pass_b_lo(p) ? P.dz_img_lo : P.dz_img) + ((size_t)ptile * P.k_slabs + s) * SLAB_FLOATS, SLAB_BYTES,
                         &full[stage]);
            }
        }
        __syncwarp();
    } else if (warp == 4 * CG + 1) {
        if (lane == 0) {
            const uint32_t idesc = umma_idesc_tf32(TILE_M, 0, 0);
            for (int s = 0; s < P.k_slabs * P.passes; ++s) {
                int stage = s % NSTAGE, it = s / NSTAGE;
                mbar_wait(&full[stage], it & 1);
                tc_fence_after();
                issue_slab_mma(tmem_base, sA + (size_t)stage * SLAB_FLOATS, sB + (size_t)stage * SLAB_FLOATS, idesc,
                               s == 0);
                umma_commit(&empty[stage]);
            }
            umma_commit(accf);
        }
        __syncwarp();
    } else {
        mbar_wait(accf, 0);
        tc_fence_after();
        const int q4 = warp & 3, cg = warp >> 2;
        const uint32_t trow = tmem_base + ((uint32_t)(q4 * 32) << 16);
        const int j = ktile * TILE_M + q4 * 32 + lane;
        const bool kvalid = j < P.basis.k_s;
        float4 kn = kvalid ? P.basis.knots[j] : make_float4(0.f, 0.f, 1.f, 1.f);
        const long long rows_left = P.pts.n_rows - (long long)ptile * TILE_M;
        float gcx = 0.f, gcy = 0.f, glb = 0.f;
        float v[32];
        for (int c0 = 32 * cg; c0 < TILE_M; c0 += 32 * CG) {
            tmem_ld32(trow + c0, v);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (c0 + i < rows_left) {
                    float2 pt = spt[c0 + i];
                    float dx = pt.x - kn.x, dy = pt.y - kn.y;
                    float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
                    bool in = (P.basis.fn == STDADK_GAUSSIAN) || (d2 < kn.z);
                    if (in && d2 > 0.0f) {
                        float d = sqrtf(d2);
                        float r = d * kn.w;
                        float coef = v[i] * phi_dr(P.basis.fn, r);
                        float s = coef * kn.w / d;  // coef / (d * theta')
                        gcx = fmaf(-dx, s, gcx);
                        gcy = fmaf(-dy, s, gcy);
                        glb = fmaf(-r, coef, glb);
                    }
                }
            }
        }
        if (kvalid) {
            atomicAdd(&P.d_centers[2 * j], gcx);
            atomicAdd(&P.d_centers[2 * j + 1], gcy);
            atomicAdd(&P.d_log_bw[j], glb);
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 4 * CG) tmem_dealloc(tmem_base, TILE_M);
}

}  // namespace stdadk
