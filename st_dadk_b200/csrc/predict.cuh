// Whole-network forward for prediction (evaluate_model / plot_spatial_mse / plot_temporal_series of upstream,
// scripts/train_st_interp.py:884-961, :1233-1248, :1380-1394): one persistent kernel per call, one CTA per SM.
//
// A CTA takes 128-row tiles in turn.  Per tile the activations never leave the SM:
//   block 1 : workers generate [X|phi|psi] slab by slab into a ring that lives in the (still unused) H buffer,
//             W1 slabs stream L2 -> SMEM through a bulk-copy ring, tcgen05.mma accumulates in TMEM;
//   epilogue: every worker thread pulls its 64 accumulator columns into registers ONCE, the LayerNorm statistics are
//             combined across the four column groups through a small scratch, and the normalised ReLU output is
//             written TF32-rounded into H (128 x 256 fp32 in the SWIZZLE_128B operand form) - slab by slab, each slab
//             with its own mbarrier, so the MMAs of the next block start while the rest is still being normalised;
//   block l : A = H, W_l slabs through the same ring, accumulator in the other half of TMEM;
//   last    : head dot products from registers (FP32), y_hat (rows x Q) is the only HBM write: 4Q bytes per point
//             against 12 (or 0 for a generated grid) in.
// HBM traffic per point is therefore ~16 bytes instead of the 4 KB of the layer-by-layer path; what remains is
// instruction issue in the worker warps and L2 -> SM weight streaming (720 KB per tile at 297-256-256-128).
#pragma once
#include "layer.cuh"

namespace stdadk {

constexpr int PF_MAX_LAYERS = 4;
constexpr int PF_CG = 4;
constexpr int PF_NW = 128 * PF_CG;          // 512 worker threads (16 warps)
constexpr int PF_NT = PF_NW + 64;           // + producer warp + MMA warp
constexpr int PF_WST = 2;                   // weight ring: 2 x (256 rows x 128 B)
constexpr int PF_AST = 6;                   // block-1 operand ring = H slabs 0..5; slabs 6,7 hold the head scratch
constexpr int PF_HSLABS = MAX_N / SLAB_K;   // 8

struct PredLayerP {
    const float* w_img;
    const float* bias;
    const float* gamma;
    const float* beta;
    int n_out, n_pad, k_slabs, has_ln;
    float eps;
    uint32_t prm_off;                       // byte offset of this layer's (bias | gamma | beta), n_pad floats each
};
struct PredSmem {
    uint32_t h_off, w_off, bar_off, tmem_off, headw_off, knots_off, tknots_off, red_off, total;
};
struct PredK {
    BasisP basis;
    PointsP pts;
    PredLayerP L[PF_MAX_LAYERS];
    PredSmem sm;
    const float* head_w;
    const float* head_b;
    float* yhat;
    int n_layers, q, n_tiles, _pad;
    unsigned long long* dbg;                // optional cycle counters (stdadk_debug_counters), NULL in production
};

// Development aid, compiled in with -DSTDADK_PF_DEBUG: cycles each role spends waiting / per phase, accumulated
// into P.dbg (stdadk_debug_counters, tools/prof_predict.py).  Production builds carry none of it.
#ifdef STDADK_PF_DEBUG
#define PF_DBG(...) __VA_ARGS__
#define PF_TIMED_WAIT(acc, ...)                   \
    do {                                          \
        if (P.dbg) {                              \
            long long t_ = clock64();             \
            __VA_ARGS__;                          \
            acc += (unsigned long long)(clock64() - t_); \
        } else {                                  \
            __VA_ARGS__;                          \
        }                                         \
    } while (0)
#else
#define PF_DBG(...)
#define PF_TIMED_WAIT(acc, ...) \
    do {                        \
        __VA_ARGS__;            \
    } while (0)
#endif

// Fills the per-layer offsets and the carve-up; returns the dynamic shared-memory bytes needed.
__host__ inline uint32_t plan_predict(PredK& K) {
    uint32_t o = 0;
    K.sm.h_off = o; o += PF_HSLABS * SLAB_BYTES;                       // 128 KB
    K.sm.w_off = o; o += PF_WST * MAX_N * 128u;                        // 64 KB
    K.sm.bar_off = o; o += 320;
    K.sm.tmem_off = o; o += 16;
    for (int l = 0; l < K.n_layers; ++l) {
        K.L[l].prm_off = o;
        o += 3u * (uint32_t)K.L[l].n_pad * 4u;
    }
    K.sm.headw_off = o; o += (uint32_t)(K.q * K.L[K.n_layers - 1].n_pad + STDADK_MAX_Q) * 4u;
    o = (o + 15u) & ~15u;
    K.sm.knots_off = o; o += (uint32_t)K.basis.k_s * 16u;
    K.sm.tknots_off = o; o += (uint32_t)K.basis.k_t * 8u;
    o = (o + 15u) & ~15u;
    K.sm.red_off = o; o += 2u * PF_CG * TILE_M * 16u;                  // LayerNorm partials, double-buffered
    K.sm.total = o + 1024;
    return K.sm.total;
}

// One thread generates its row of a whole 32-feature slab (eight 16-byte chunks): column group cg owns slabs
// cg, cg + 4, ... so a slab costs one barrier arrival per thread of that group and 32 independent evaluations.
__device__ __forceinline__ void pf_gen_slab(const BasisP& B, const float4* sk, const float2* st, int slab, float x, float y,
                                         float t, const float* xrow, uint32_t row_saddr, uint32_t rx) {
#pragma unroll 1
    for (int c2 = 0; c2 < 8; c2 += 2) {        // two chunks (8 evaluations) in flight
        const float4 v0 = feature_chunk(B, sk, st, slab * SLAB_K + c2 * 4, x, y, t, xrow);
        const float4 v1 = feature_chunk(B, sk, st, slab * SLAB_K + c2 * 4 + 4, x, y, t, xrow);
        st_shared_v4(row_saddr + (((uint32_t)c2 ^ rx) << 4), v0.x, v0.y, v0.z, v0.w);
        st_shared_v4(row_saddr + (((uint32_t)(c2 + 1) ^ rx) << 4), v1.x, v1.y, v1.z, v1.w);
    }
}

__device__ __forceinline__ void pf_store_slab(const float (&v)[32], uint32_t slab_saddr, uint32_t rowoff, uint32_t rx) {
#pragma unroll
    for (int c = 0; c < 8; ++c)
        st_shared_v4(slab_saddr + rowoff + (((uint32_t)c ^ rx) << 4), to_tf32(v[4 * c]), to_tf32(v[4 * c + 1]),
                     to_tf32(v[4 * c + 2]), to_tf32(v[4 * c + 3]));
}

// Eval mode: no dropout, and nothing but y_hat leaves the SM.
__global__ void __launch_bounds__(PF_NT, 1) predict_fused_kernel(const __grid_constant__ PredK P) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = align_smem(smem_raw);
    float* sH = reinterpret_cast<float*>(smem + P.sm.h_off);
    float* sW = reinterpret_cast<float*>(smem + P.sm.w_off);
    uint64_t* wfull = reinterpret_cast<uint64_t*>(smem + P.sm.bar_off);
    uint64_t* wempty = wfull + PF_WST;
    uint64_t* afull = wempty + PF_WST;
    uint64_t* aempty = afull + PF_AST;
    uint64_t* hfull = aempty + PF_AST;
    uint64_t* hfree = hfull + PF_HSLABS;   // H slab j (j < PF_AST) no longer read by the last block of the current tile
    uint64_t* accf = hfree + PF_AST;       // [2]: accumulator-ready of even / odd tiles
    uint64_t* kbar = accf + 2;             // knot tables have landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + P.sm.tmem_off);
    float* shw = reinterpret_cast<float*>(smem + P.sm.headw_off);
    float4* sk = reinterpret_cast<float4*>(smem + P.sm.knots_off);
    float2* st = reinterpret_cast<float2*>(smem + P.sm.tknots_off);
    float4* red = reinterpret_cast<float4*>(smem + P.sm.red_off);
    float* hscr = sH + (size_t)PF_AST * SLAB_FLOATS;          // head partials [cg][row][MAX_Q] in H slabs 6,7

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nl = P.n_layers;
    const int last_pad = P.L[nl - 1].n_pad, last_out = P.L[nl - 1].n_out;
    float* shb = shw + P.q * last_pad;

    if (tid == PF_NW) {
        for (int s = 0; s < PF_WST; ++s) {
            mbar_init(&wfull[s], 1);
            mbar_init(&wempty[s], 1);
        }
        for (int s = 0; s < PF_AST; ++s) {
            mbar_init(&afull[s], TILE_M / 32);
            mbar_init(&aempty[s], 1);
        }
        for (int s = 0; s < PF_HSLABS; ++s) mbar_init(&hfull[s], TILE_M / 32);
        for (int s = 0; s < PF_AST; ++s) mbar_init(&hfree[s], 1);
        mbar_init(&accf[0], 1);
        mbar_init(&accf[1], 1);
        mbar_init(kbar, 1);
        mbar_fence_init();
        stage_knots_async(P.basis, sk, st, kbar);
    }
    if (warp == 4 * PF_CG) {
        __syncwarp();
        tmem_alloc(tmem_slot, 512u);
    }
    for (int l = 0; l < nl; ++l) {
        const PredLayerP& Ly = P.L[l];
        float* prm = reinterpret_cast<float*>(smem + Ly.prm_off);
        for (int i = tid; i < Ly.n_pad; i += PF_NT) {
            const bool ok = i < Ly.n_out;
            prm[i] = ok ? Ly.bias[i] : 0.0f;
            prm[Ly.n_pad + i] = (ok && Ly.has_ln) ? Ly.gamma[i] : 1.0f;
            prm[2 * Ly.n_pad + i] = (ok && Ly.has_ln) ? Ly.beta[i] : 0.0f;
        }
    }
    for (int i = tid; i < P.q * last_pad; i += PF_NT) {
        const int k = i / last_pad, c = i - k * last_pad;
        shw[i] = c < last_out ? P.head_w[(size_t)k * last_out + c] : 0.0f;
    }
    if (tid < P.q) shb[tid] = P.head_b[tid];
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 4 * PF_CG) {
        // ---------------- producer: weight slabs of every block of every tile, in consumption order
        if (lane == 0) {
            uint32_t stage = 0, phase = 0;
            PF_DBG(unsigned long long w_empty = 0;)
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
                for (int l = 0; l < nl; ++l) {
                    const PredLayerP& Ly = P.L[l];
                    for (int s = 0; s < Ly.k_slabs; ++s) {
                        PF_TIMED_WAIT(w_empty, mbar_wait(&wempty[stage], phase ^ 1u));
                        issue_slab_copies(Ly.w_img, Ly.k_slabs, s, Ly.n_pad, nullptr, nullptr,
                                          sW + (size_t)stage * MAX_N * SLAB_K, &wfull[stage]);
                        if (++stage == PF_WST) {
                            stage = 0;
                            phase ^= 1u;
                        }
                    }
                }
            }
            PF_DBG(if (P.dbg) atomicAdd(&P.dbg[7], w_empty);)
        }
        __syncwarp();
    } else if (warp == 4 * PF_CG + 1) {
        // ---------------- MMA issuer
        if (lane == 0) {
            uint32_t wstage = 0, wphase = 0, astage = 0, aphase = 0, hph = 0, it = 0;
            PF_DBG(unsigned long long w_a = 0, w_w = 0; const long long t_begin = clock64();)
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
                // every block of a tile accumulates into the same half of TMEM (the epilogue has drained it into
                // registers before it releases the next block's first operand slab); tiles alternate halves so that
                // block 1 of the next tile runs under the last epilogue of this one
                const uint32_t acc = tmem_base + (it & 1u) * MAX_N;
                for (int l = 0; l < nl; ++l) {
                    const PredLayerP& Ly = P.L[l];
                    const uint32_t idesc = umma_idesc_tf32((uint32_t)Ly.n_pad, 0, 0);
                    const bool last = l == nl - 1;
                    for (int s = 0; s < Ly.k_slabs; ++s) {
                        const float* a;
                        if (l == 0) {
                            PF_TIMED_WAIT(w_a, mbar_wait(&afull[astage], aphase));
                            a = sH + (size_t)astage * SLAB_FLOATS;
                        } else {
                            PF_TIMED_WAIT(w_a, mbar_wait(&hfull[s], (hph >> s) & 1u));
                            hph ^= 1u << s;
                            a = sH + (size_t)s * SLAB_FLOATS;
                        }
                        PF_TIMED_WAIT(w_w, mbar_wait(&wfull[wstage], wphase));
                        tc_fence_after();
                        issue_slab_mma(acc, a, sW + (size_t)wstage * MAX_N * SLAB_K, idesc, s == 0);
                        umma_commit(&wempty[wstage]);
                        if (l == 0) {
                            umma_commit(&aempty[astage]);
                            if (++astage == PF_AST) {
                                astage = 0;
                                aphase ^= 1u;
                            }
                        } else if (last && s < PF_AST) {
                            umma_commit(&hfree[s]);      // the next tile's block-1 operand may overwrite this H slab
                        }
                        if (++wstage == PF_WST) {
                            wstage = 0;
                            wphase ^= 1u;
                        }
                    }
                    umma_commit(&accf[it & 1u]);
                }
            }
            PF_DBG(if (P.dbg) {
                atomicAdd(&P.dbg[0], w_a);
                atomicAdd(&P.dbg[1], w_w);
                atomicAdd(&P.dbg[2], (unsigned long long)(clock64() - t_begin));
            })
        }
        __syncwarp();
    } else {
        // ---------------- workers: thread = (row, column group)
        const int q4 = warp & 3, cg = warp >> 2;
        const int row = q4 * 32 + lane;
        const uint32_t rowoff = (uint32_t)row * 128u, rx = (uint32_t)row & 7u;
        const uint32_t trow = tmem_base + ((uint32_t)(q4 * 32) << 16);
        const uint32_t sH_addr = smem_u32(sH);
        uint32_t astage = 0, aphase = 0, accn = 0;
#ifdef STDADK_PF_DEBUG
        unsigned long long w_acc = 0, w_ae = 0, w_bar = 0, ph_gen = 0, ph_ld = 0, ph_norm = 0, ph_head = 0;
        const long long t_begin = clock64();
        long long t_last = t_begin;
#define PF_PHASE(var)                                    \
    do {                                                 \
        if (P.dbg) {                                     \
            const long long n_ = clock64();              \
            var += (unsigned long long)(n_ - t_last);    \
            t_last = n_;                                 \
        }                                                \
    } while (0)
#else
#define PF_PHASE(var)
#endif
        // generated grid: this thread's row index decomposed once ((k*nx + i)*ny + j, 64-bit), then advanced by the
        // tile stride with 32-bit divisions (the 64-bit div/mod triple costs ~500 instructions per row otherwise)
        const bool is_grid = P.pts.nx > 0;
        uint32_t gk = 0, gi = 0, gj = 0;
        const uint32_t gstep = (uint32_t)TILE_M * gridDim.x;
        if (is_grid) {
            const long long g0 = P.pts.row_begin + (long long)blockIdx.x * TILE_M + row;
            const long long r0 = g0 / P.pts.ny;
            gj = (uint32_t)(g0 - r0 * P.pts.ny);
            gk = (uint32_t)(r0 / P.pts.nx);
            gi = (uint32_t)(r0 - (long long)gk * P.pts.nx);
        }
        // Software pipeline over this CTA's tiles: the operand of block 1 of the NEXT tile is generated just before the
        // last epilogue of the current one (into H slabs the last block has already consumed), so those MMAs run
        // under the epilogue + head instead of leaving the workers waiting for them.
        const int k_last = nl >= 2 ? P.L[nl - 1].k_slabs : 0;
        mbar_wait(kbar, 0);
        long long lrow = 0, nxt_lrow = 0;
        bool rvalid = false, nxt_valid = false, have_cur = false;
        uint32_t it = 0;                                   // iteration index of the current tile
        for (int next = blockIdx.x; have_cur || next < P.n_tiles; next += gridDim.x) {
            const bool have_next = next < P.n_tiles;
            for (int l = have_cur ? 0 : nl - 1; l < nl; ++l) {
                if (l == nl - 1) {
                    if (have_next) {
                        nxt_lrow = (long long)next * TILE_M + row;
                        nxt_valid = nxt_lrow < P.pts.n_rows;
                        const long long grow = P.pts.row_begin + nxt_lrow;
                        float x = 0.f, y = 0.f, t = 0.f;
                        const float* xrow = nullptr;
                        if (is_grid) {
                            x = P.pts.nx > 1 ? __fdiv_rn((float)gi, (float)(P.pts.nx - 1)) : 0.0f;     // as load_point()
                            y = P.pts.ny > 1 ? __fdiv_rn((float)gj, (float)(P.pts.ny - 1)) : 0.0f;
                            t = P.pts.nt > 1 ? __fdiv_rn((float)gk, (float)(P.pts.nt - 1)) : 0.0f;
                            const uint32_t jj = gj + gstep, qj = jj / (uint32_t)P.pts.ny;
                            gj = jj - qj * (uint32_t)P.pts.ny;
                            const uint32_t ii = gi + qj, qi = ii / (uint32_t)P.pts.nx;
                            gi = ii - qi * (uint32_t)P.pts.nx;
                            gk += qi;
                        } else if (nxt_valid) {
                            load_point(P.pts, grow, x, y, t);
                        }
                        if (nxt_valid && P.basis.p_cov > 0 && P.pts.xcov)
                            xrow = P.pts.xcov + sample_of(P.pts, grow) * P.basis.p_cov;
                        for (int s = 0; s < P.L[0].k_slabs; ++s) {
                            if ((s & (PF_CG - 1)) == cg) {
                                PF_TIMED_WAIT(w_ae, mbar_wait(&aempty[astage], aphase ^ 1u));
                                if (have_cur && s < PF_AST && (int)astage < k_last)   // H slab still feeds the last block?
                                    PF_TIMED_WAIT(w_ae, mbar_wait(&hfree[astage], it & 1u));
                                pf_gen_slab(P.basis, sk, st, s, x, y, t, xrow,
                                            sH_addr + astage * (uint32_t)SLAB_BYTES + rowoff, rx);
                                fence_proxy_async_smem();
                                mbar_arrive_warp(&afull[astage]);
                            }
                            if (++astage == PF_AST) {
                                astage = 0;
                                aphase ^= 1u;
                            }
                        }
                    }
                    PF_PHASE(ph_gen);
                    if (!have_cur) break;
                }
                const PredLayerP& Ly = P.L[l];
                const float* sb = reinterpret_cast<const float*>(smem + Ly.prm_off);
                const float* sg = sb + Ly.n_pad;
                const float* sbt = sg + Ly.n_pad;
                const int c0a = 32 * cg, c0b = 32 * cg + 128;
                const bool ha = c0a < Ly.n_pad, hb = c0b < Ly.n_pad;
                const int nva = min(32, Ly.n_out - c0a), nvb = min(32, Ly.n_out - c0b);
                float4* redl = red + (size_t)(accn & 1u) * (PF_CG * TILE_M);
                PF_TIMED_WAIT(w_acc, mbar_wait(&accf[it & 1u], ((it >> 1) * (uint32_t)nl + (uint32_t)l) & 1u));
                PF_DBG(if (P.dbg) t_last = clock64();)
                ++accn;
                tc_fence_after();
                const uint32_t acc = trow + (it & 1u) * MAX_N;
                // both arrays are DEFINED on every path right here: a register written only under `if (ha)` and read
                // under a later `if (ha)` looks live from the top of the tile loop to the register allocator, which then
                // keeps 64 registers away from the basis generation
                float va[32], vb[32];
                if (ha) {
                    tmem_ld32_issue(acc + (uint32_t)c0a, va);
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) va[i] = 0.0f;
                }
                if (hb) {
                    tmem_ld32_issue(acc + (uint32_t)c0b, vb);
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) vb[i] = 0.0f;
                }
                tmem_ld_wait(va);
                tmem_ld_wait(vb);
                bool have = false;
                float K = 0.0f, S1 = 0.0f, S2 = 0.0f;
                if (ha) pf_bias_stats(va, sb + c0a, nva, have, K, S1, S2);
                if (hb) pf_bias_stats(vb, sb + c0b, nvb, have, K, S1, S2);
                float rstd = 1.0f, nmr = 0.0f;
                if (Ly.has_ln) {
                    const float cntv = (float)((ha ? max(nva, 0) : 0) + (hb ? max(nvb, 0) : 0));
                    redl[cg * TILE_M + row] = make_float4(K, S1, S2, cntv);
                    PF_PHASE(ph_ld);
                    PF_TIMED_WAIT(w_bar, worker_barrier(PF_NW));
                    PF_DBG(if (P.dbg) t_last = clock64();)
                    if (ha) {
                        const float inv_n = 1.0f / (float)Ly.n_out;
                        float4 part[PF_CG];
                        float tot = 0.0f;
#pragma unroll
                        for (int g = 0; g < PF_CG; ++g) {
                            part[g] = redl[g * TILE_M + row];
                            tot += fmaf(part[g].w, part[g].x, part[g].y);
                        }
                        const float mean = tot * inv_n;
                        float m2 = 0.0f;
#pragma unroll
                        for (int g = 0; g < PF_CG; ++g) {
                            const float dk = mean - part[g].x;
                            m2 += part[g].z - 2.0f * dk * part[g].y + part[g].w * dk * dk;
                        }
                        rstd = 1.0f / sqrtf(fmaxf(m2 * inv_n, 0.0f) + Ly.eps);
                        nmr = -mean * rstd;
                    }
                } else {
                    worker_barrier(PF_NW);   // every thread has seen this accumulator phase before the next can complete
                }
                if (l + 1 < nl) {
                    if (ha) {
                        pf_normalize(va, sg + c0a, sbt + c0a, Ly.has_ln != 0, rstd, nmr, nva);
                        pf_store_slab(va, sH_addr + (uint32_t)cg * SLAB_BYTES, rowoff, rx);
                        fence_proxy_async_smem();
                        tc_fence_before();
                        mbar_arrive_warp(&hfull[cg]);
                    }
                    if (hb) {
                        pf_normalize(vb, sg + c0b, sbt + c0b, Ly.has_ln != 0, rstd, nmr, nvb);
                        pf_store_slab(vb, sH_addr + (uint32_t)(cg + 4) * SLAB_BYTES, rowoff, rx);
                        fence_proxy_async_smem();
                        tc_fence_before();
                        mbar_arrive_warp(&hfull[cg + 4]);
                    }
                    PF_PHASE(ph_norm);
                } else {
                    float yh[STDADK_MAX_Q];
#pragma unroll
                    for (int k = 0; k < STDADK_MAX_Q; ++k) yh[k] = 0.0f;
                    if (ha) {
                        pf_normalize(va, sg + c0a, sbt + c0a, Ly.has_ln != 0, rstd, nmr, nva);
                        pf_head_partial(va, shw, Ly.n_pad, c0a, P.q, yh);
                    }
                    if (hb) {
                        pf_normalize(vb, sg + c0b, sbt + c0b, Ly.has_ln != 0, rstd, nmr, nvb);
                        pf_head_partial(vb, shw, Ly.n_pad, c0b, P.q, yh);
                    }
                    float* mine = hscr + ((size_t)cg * TILE_M + row) * STDADK_MAX_Q;
                    *reinterpret_cast<float4*>(mine) = make_float4(yh[0], yh[1], yh[2], yh[3]);
                    *reinterpret_cast<float4*>(mine + 4) = make_float4(yh[4], yh[5], yh[6], yh[7]);
                    worker_barrier(PF_NW);
                    if (cg == 0 && rvalid) {
#pragma unroll
                        for (int k = 0; k < STDADK_MAX_Q; ++k) {
                            if (k < P.q) {
                                float acc_k = shb[k];
#pragma unroll
                                for (int g = 0; g < PF_CG; ++g)
                                    acc_k += hscr[((size_t)g * TILE_M + row) * STDADK_MAX_Q + k];
                                P.yhat[lrow * P.q + k] = acc_k;
                            }
                        }
                    }
                    PF_PHASE(ph_head);
                }
            }
            if (have_cur) ++it;
            have_cur = have_next;
            lrow = nxt_lrow;
            rvalid = nxt_valid;
        }
        PF_DBG(if (P.dbg && tid == 0) {
            atomicAdd(&P.dbg[3], w_acc);
            atomicAdd(&P.dbg[4], w_ae);
            atomicAdd(&P.dbg[5], (unsigned long long)(clock64() - t_begin));
            atomicAdd(&P.dbg[6], w_bar);
            atomicAdd(&P.dbg[8], ph_gen);
            atomicAdd(&P.dbg[9], ph_ld);
            atomicAdd(&P.dbg[10], ph_norm);
            atomicAdd(&P.dbg[11], ph_head);
        })
        tc_fence_before();
    }
    __syncthreads();
    if (warp == 4 * PF_CG) tmem_dealloc(tmem_base, 512u);
}

}  // namespace stdadk
