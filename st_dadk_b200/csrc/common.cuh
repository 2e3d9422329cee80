// Shared device-side definitions: flat kernel parameter blocks, basis evaluation, dropout RNG.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

#include "../../include/stdadk.h"
#include "ptx.cuh"

namespace stdadk {

// Development aid of the training step's kernels (-DSTDADK_PF_DEBUG builds, stdadk_debug_step_counters): thread 0 of
// each CTA adds the globaltimer nanoseconds since its previous stamp to dbg[slot] (slots 0-6) and counts the CTA in
// dbg[7].  Production builds carry none of it.
#ifdef STDADK_PF_DEBUG
#define STEP_T_BEGIN(dbg)                                                  \
    unsigned long long t_prev_ = 0;                                        \
    if ((dbg) && threadIdx.x == 0) {                                       \
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_prev_));        \
        atomicAdd((dbg) + 7, 1ull);                                        \
    }
#define STEP_T(dbg, slot)                                                  \
    do {                                                                   \
        if ((dbg) && threadIdx.x == 0) {                                   \
            unsigned long long now_;                                       \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now_));       \
            atomicAdd((dbg) + (slot), now_ - t_prev_);                     \
            t_prev_ = now_;                                                \
        }                                                                  \
    } while (0)
#else
#define STEP_T_BEGIN(dbg)
#define STEP_T(dbg, slot)
#endif

constexpr int TILE_M = 128;                  // rows (points) per tile = TMEM lanes
constexpr int SLAB_K = 32;                   // fp32/tf32 elements per 128-byte operand row
constexpr int SLAB_FLOATS = TILE_M * SLAB_K; // 4096 floats = 16 KB
constexpr int SLAB_BYTES = SLAB_FLOATS * 4;
constexpr int MAX_N = 256;                   // widest block of the whole-network and field kernels (one UMMA N); layout
                                             // constant of their weight ring and tensor-memory halves
constexpr int MAX_W = STDADK_MAX_WIDTH;      // widest block of the per-block kernels: one FP32 accumulator column per
                                             // output unit in the 512 tensor-memory columns of an SM
static_assert(MAX_W == 2 * MAX_N, "a wide block is two MMAs of N <= MAX_N per K slab");

__host__ __device__ inline int pad32(int x) { return (x + 31) & ~31; }
__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

struct BasisP {
    const float4* knots;
    const float2* tknots;
    int k_s, k_t, p_cov, fn;
};
struct PointsP {
    const float* coords;
    const float* t;
    const float* xcov;
    const long long* index;
    int nx, ny, nt, _pad;
    long long row_begin;
    long long n_rows;
};
struct HeadP {
    const float* w;
    const float* b;
    const float* y;
    float* yhat;
    float* dyhat;
    float* loss_acc;
    int q, loss_type, nc_power, _pad;
    float inv_count, nc_weight;
    float taus[STDADK_MAX_Q];
};
struct LayerP {
    const float* w_img;
    const float* w_img_lo;      // tf32x3: image of W - tf32(W); NULL = single-pass TF32
    const float* bias;
    const float* gamma;
    const float* beta;
    int n_in, n_out, layer_id, _pad;
    float eps, drop_p;
    unsigned int step, _pad2;
    unsigned long long seed;
    const int* step_ptr;
    unsigned long long key_offset;
};
__device__ __forceinline__ unsigned int dropout_step(const LayerP& L) {
    return L.step_ptr ? (unsigned int)(*L.step_ptr) : L.step;
}
// sample index of global row g (identity unless a gather index is given)
__device__ __forceinline__ long long sample_of(const PointsP& P, long long g) { return P.index ? P.index[g] : g; }

// ---------------------------------------------------------------- basis evaluation
// Spatial basis value from the coordinate difference; the support predicate d2 < th2 is evaluated
// with explicitly rounded products (no FMA contraction) so that index sets match oracle/basis_ref.c
// bit for bit.  Reference: stnf/models/st_interp.py:462-491.
// MUFU-only helpers (no denormal / special-case wrappers): rsqrt and exp2 to ~2^-22 relative error.
__device__ __forceinline__ float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float ex2_approx(float x) {
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// phi from the squared distance.  The support test d2 < th2 is exact; inside the support the value uses
// sqrt(d2) = d2 * rsqrt(d2) (two instructions instead of the IEEE square root's ten: relative error ~2e-7 in r,
// far inside the 1e-5 parity tolerance) and the polynomial with 1/3 folded into its coefficients.
template <int FN>
__device__ __forceinline__ float phi_from_d2(float d2, float th2, float inv_th) {
    if (FN == STDADK_GAUSSIAN) return ex2_approx(-0.72134752044448170f * (d2 * inv_th * inv_th));  // exp(-r^2/2)
    const float r = d2 * rsqrt_approx(fmaxf(d2, 1e-30f)) * inv_th;
    const float u = fmaxf(1.0f - r, 0.0f);
    float v;
    if (FN == STDADK_TRIANGULAR) {
        v = u;
    } else {
        const float u2 = u * u;
        v = (u2 * u2) * u2 * fmaf(fmaf(35.0f / 3.0f, r, 6.0f), r, 1.0f);
    }
    return d2 < th2 ? v : 0.0f;
}
__device__ __forceinline__ float phi_eval(int fn, float dx, float dy, float th2, float inv_th) {
    const float d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    if (fn == STDADK_GAUSSIAN) return phi_from_d2<STDADK_GAUSSIAN>(d2, th2, inv_th);
    if (!(d2 < th2)) return 0.0f;
    if (fn == STDADK_TRIANGULAR) return phi_from_d2<STDADK_TRIANGULAR>(d2, th2, inv_th);
    return phi_from_d2<STDADK_WENDLAND>(d2, th2, inv_th);
}
// d phi / d r (SURVEY.md 9.1): wendland -(56/3) r (5r+1) (1-r)^5; gaussian -r exp(-r^2/2); triangular -1.
__device__ __forceinline__ float phi_dr(int fn, float r) {
    if (fn == STDADK_GAUSSIAN) return -r * exp2f(-0.72134752044448170f * r * r);
    if (!(r < 1.0f)) return 0.0f;
    if (fn == STDADK_TRIANGULAR) return -1.0f;
    float u = 1.0f - r;
    float u2 = u * u;
    return -(56.0f / 3.0f) * r * fmaf(5.0f, r, 1.0f) * u2 * u2 * u;
}
// Temporal Gaussian basis (st_interp.py:583-596).
__device__ __forceinline__ float psi_eval(float t, float c, float inv_bw) {
    float s = (t - c) * inv_bw;
    return ex2_approx(-0.72134752044448170f * s * s);
}

// Coordinates of global row g: from the arrays, or from the dense grid n = (k*nx + i)*ny + j.
__device__ __forceinline__ void load_point(const PointsP& P, long long g, float& x, float& y, float& t) {
    if (P.nx > 0) {
        long long j = g % P.ny;
        long long i = (g / P.ny) % P.nx;
        long long k = g / ((long long)P.ny * P.nx);
        x = P.nx > 1 ? __fdiv_rn((float)i, (float)(P.nx - 1)) : 0.0f;
        y = P.ny > 1 ? __fdiv_rn((float)j, (float)(P.ny - 1)) : 0.0f;
        t = P.nt > 1 ? __fdiv_rn((float)k, (float)(P.nt - 1)) : 0.0f;
    } else {
        long long sidx = sample_of(P, g);
        float2 c = *reinterpret_cast<const float2*>(P.coords + 2 * sidx);
        x = c.x;
        y = c.y;
        t = P.t[sidx];
    }
}

// Feature f of the first Linear layer's input row: [X | phi | psi | 0-padding] (st_interp.py:843-846).
__device__ __forceinline__ float feature_value(const BasisP& B, const float4* sk, const float2* st, int f, float x,
                                               float y, float t, const float* xrow) {
    if (f < B.p_cov) return xrow ? xrow[f] : 0.0f;
    f -= B.p_cov;
    if (f < B.k_s) {
        float4 kn = sk[f];
        return phi_eval(B.fn, x - kn.x, y - kn.y, kn.z, kn.w);
    }
    f -= B.k_s;
    if (f < B.k_t) {
        float2 tk = st[f];
        return psi_eval(t, tk.x, tk.y);
    }
    return 0.0f;
}

// ---------------------------------------------------------------- dropout RNG
// Philox4x32-10, counter = (row_lo, col_block, layer | row_hi<<8, step), key = seed.  One call yields
// eight 16-bit uniforms = 8 consecutive columns; keep iff u16 >= floor(p * 65536).  Keyed on the GLOBAL
// row so the mask is invariant to sharding.  Mirrored by oracle.dropout_keep_mask.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// bit e of the result = keep flag of column (block*8 + e)
// not inlined: one copy of the 10 Philox rounds per kernel keeps the instruction footprint (and the cold I-cache
// misses of one-wave launches) down
__device__ __noinline__ uint32_t dropout_keep8(unsigned long long seed, uint32_t step, uint32_t layer,
                                                  unsigned long long row, uint32_t block, uint32_t thresh16) {
    uint32_t o[4];
    philox4x32_10((uint32_t)row, block, layer | ((uint32_t)(row >> 32) << 8), step, (uint32_t)seed,
                  (uint32_t)(seed >> 32), o);
    uint32_t bits = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        uint32_t u = (o[e >> 1] >> ((e & 1) * 16)) & 0xFFFFu;
        bits |= (u >= thresh16 ? 1u : 0u) << e;
    }
    return bits;
}
__host__ __device__ inline uint32_t dropout_thresh16(float p) {
    int t = (int)(p * 65536.0f);
    return (uint32_t)(t < 0 ? 0 : (t > 65535 ? 65535 : t));
}

// Sum of v[c] over the 32 lanes of a warp for all 32 indices c at once: on return lane c holds the
// column sum of index c (31 shuffles instead of 32 x 5).
__device__ __forceinline__ float warp_transpose_sum(float (&v)[32], int lane) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            float send = upper ? v[i] : v[i + off];
            float keep = upper ? v[i + off] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
    }
    return v[0];
}
__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) x += __shfl_xor_sync(0xffffffffu, x, off);
    return x;
}

}  // namespace stdadk
