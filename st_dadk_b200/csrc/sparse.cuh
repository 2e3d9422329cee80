// Large-knot-count regime (K_s ~ 1e5, BASELINE config 4; also any knot set too large for the dense operand): the spatial
// part of block 1 walks only the knots inside each point's compact support instead of generating K_s dense columns.
//
//   sparse_spatial_fwd_kernel  : zs[n, :] = sum_{j in supp(s_n)} phi_j(s_n) * W1t[p + j, :]      (N x n_out, FP32)
//   sparse_spatial_wgrad_kernel: dW1t[p + j, :] += phi_j(s_n) * dz1[n, :] for j in supp(s_n)       (vector atomics)
//                                and, for learnable knots, the closed-form chain rule of SURVEY.md 9.1 into
//                                d_centers / d_log_bw with G_nj = dz1[n, :] . W1t[p + j, :]
//
// W1t is the knot-major storage of the first Linear layer ((n_in, n_out)-contiguous: one knot = one contiguous row,
// 1 KB at n_out = 256), so a gather is a coalesced row read.  The dense temporal / covariate columns still run on
// the tensor cores (layer_fwd/bwd with a k_s = 0 basis); zs enters their epilogue as an addend before LayerNorm.
//
// Candidate knots of a point, per resolution level, come from one of two sources:
//   * fixed uniform lattice (knot j of a level at node (j / side, j % side), st_interp.py:152-185): the closed-form
//     window [ceil((x - th) g) - 1, floor((x + th) g) + 1] x the same in y, g = side - 1;
//   * any other knot set (gmm / random_site / kmeans_balanced placement, learnable knots that move every step,
//     st_interp.py:94-108, :187-431): a per-level CELL LIST built on the device by celllist_build_kernel -- cells of
//     edge h_l >= max theta' of the level, knots counting-sorted by cell, a point visits the 3 x 3 cells around it.
// Either way the exact FP32 support predicate of phi_eval decides membership, so index sets equal the dense path's.
//
// One warp per point.  Lanes evaluate 32 candidates at a time; the active ones are consumed immediately (ballot, then
// one broadcast per set bit), so there is no per-point list and no limit on the number of knots in a support.
#pragma once
#include "common.cuh"

namespace stdadk {

constexpr int SP_MAX_LEVELS = 8;
constexpr int SP_WARPS = 8;
constexpr int CL_GMAX = 128;                 // cells per axis and level, at most (cell edge >= 1/128 and >= theta'_max)
constexpr int CL_THREADS = 1024;

struct Lattice {
    int n_levels;
    int side[SP_MAX_LEVELS];
    int offset[SP_MAX_LEVELS];
    float thetap[SP_MAX_LEVELS];
};

// Device-resident cell list (built per step when the knots are learnable).  Layout of the int32 workspace:
//   [0, 8 * SP_MAX_LEVELS)            level descriptors: {G, cell_base, knot_begin, knot_end, -, -, -, -}
//   starts[ n_levels * (GMAX^2 + 1) ] first sorted position of every cell (exclusive scan, + level base)
//   cursor[ n_levels * GMAX^2 ]       scatter cursors
//   order[ K ]                        knot index at every sorted position
// followed (16-byte aligned) by sorted_knots4[K]: the knot table in sorted order (coalesced candidate loads).
struct CellList {
    const int* desc;
    const int* starts;
    const int* order;
    const float4* sorted;
    int n_levels, _pad;
};
__host__ __device__ inline size_t celllist_ints(int k_s, int n_levels) {
    return (size_t)8 * SP_MAX_LEVELS + (size_t)n_levels * (CL_GMAX * CL_GMAX + 1) + (size_t)n_levels * CL_GMAX * CL_GMAX +
           (size_t)k_s;
}
__host__ __device__ inline size_t celllist_bytes(int k_s, int n_levels) {
    size_t b = celllist_ints(k_s, n_levels) * 4;
    b = (b + 15) & ~(size_t)15;
    return b + (size_t)k_s * 16;
}
__device__ __forceinline__ int cell_of(float v, int G) {
    int c = (int)floorf(v * (float)G);
    return min(max(c, 0), G - 1);      // knots / points outside [0,1] fall into the border cells (clamping is monotone
}                                      // and 1-Lipschitz, so |cell(point) - cell(knot)| <= 1 still holds inside a support)

struct CellBuildK {
    const float4* knots;               // (cx, cy, theta'^2, 1/theta')
    int k_s, n_levels;
    int level_begin[SP_MAX_LEVELS + 1];
    int* ws;
    float4* sorted;
};
// One CTA: per level max theta' -> G, histogram of knots per cell, exclusive scan, scatter.  ~1e5 knots: tens of us.
__global__ void __launch_bounds__(CL_THREADS) celllist_build_kernel(const __grid_constant__ CellBuildK P) {
    __shared__ float s_red[CL_THREADS / 32];
    __shared__ int s_scan[CL_THREADS / 32];
    __shared__ int s_G, s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int* desc = P.ws;
    int* starts = P.ws + 8 * SP_MAX_LEVELS;
    int* cursor = starts + (size_t)P.n_levels * (CL_GMAX * CL_GMAX + 1);
    int* order = cursor + (size_t)P.n_levels * CL_GMAX * CL_GMAX;
    for (int l = 0; l < P.n_levels; ++l) {
        const int kb = P.level_begin[l], ke = P.level_begin[l + 1];
        // ---- largest support radius of the level
        float th = 0.0f;
        for (int j = kb + tid; j < ke; j += CL_THREADS) th = fmaxf(th, sqrtf(P.knots[j].z));
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) th = fmaxf(th, __shfl_xor_sync(0xffffffffu, th, o));
        if (lane == 0) s_red[warp] = th;
        __syncthreads();
        if (tid == 0) {
            float m = 0.0f;
            for (int w = 0; w < CL_THREADS / 32; ++w) m = fmaxf(m, s_red[w]);
            int G = m > 0.0f ? (int)floorf(1.0f / m) : CL_GMAX;      // cell edge 1/G >= theta'_max
            s_G = min(max(G, 1), CL_GMAX);
        }
        __syncthreads();
        const int G = s_G, ncell = G * G;
        int* st_l = starts + (size_t)l * (CL_GMAX * CL_GMAX + 1);
        int* cu_l = cursor + (size_t)l * CL_GMAX * CL_GMAX;
        for (int c = tid; c <= ncell; c += CL_THREADS) st_l[c] = 0;
        __syncthreads();
        for (int j = kb + tid; j < ke; j += CL_THREADS) {
            const float4 kn = P.knots[j];
            atomicAdd(&st_l[cell_of(kn.x, G) * G + cell_of(kn.y, G)], 1);
        }
        __syncthreads();
        // ---- exclusive scan of the counts (chunks of CL_THREADS cells, carry between chunks)
        if (tid == 0) s_carry = kb;
        __syncthreads();
        for (int c0 = 0; c0 < ncell; c0 += CL_THREADS) {
            const int c = c0 + tid;
            const int v = c < ncell ? st_l[c] : 0;
            int inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int n = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += n;
            }
            if (lane == 31) s_scan[warp] = inc;
            __syncthreads();
            if (warp == 0) {
                int w = s_scan[lane];
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    int n = __shfl_up_sync(0xffffffffu, w, o);
                    if (lane >= o) w += n;
                }
                s_scan[lane] = w;
            }
            __syncthreads();
            const int before = s_carry + (warp > 0 ? s_scan[warp - 1] : 0) + inc - v;
            if (c < ncell) {
                st_l[c] = before;
                cu_l[c] = before;
            }
            __syncthreads();
            if (tid == 0) s_carry += s_scan[CL_THREADS / 32 - 1];
            __syncthreads();
        }
        if (tid == 0) {
            st_l[ncell] = ke;
            desc[8 * l + 0] = G;
            desc[8 * l + 1] = l * (CL_GMAX * CL_GMAX + 1);
            desc[8 * l + 2] = kb;
            desc[8 * l + 3] = ke;
        }
        __syncthreads();
        for (int j = kb + tid; j < ke; j += CL_THREADS) {
            const float4 kn = P.knots[j];
            const int pos = atomicAdd(&cu_l[cell_of(kn.x, G) * G + cell_of(kn.y, G)], 1);
            order[pos] = j;
            P.sorted[pos] = kn;
        }
        __syncthreads();
    }
}

struct SparseK {
    PointsP pts;
    Lattice lat;
    CellList cl;             // cl.desc != NULL: candidates from the cell list; else the lattice's closed-form window
    const float4* knots;
    const float* w1t;        // (n_in, n_out) contiguous; spatial rows start at row p_cov
    float* zs;               // fwd: out (n_rows x n_out)
    const float* dz_img;     // wgrad: image (n_rows x n_out)
    float* dw1t;             // wgrad: += into the same geometry as w1t
    float* d_centers;        // wgrad, learnable knots: (k_s x 2) +=, or NULL
    float* d_log_bw;         // (k_s) +=
    int n_out, p_cov, fn, _pad;
};

// Calls f(j, phi, dx, dy, d2, inv_theta) for every knot j of the point's support, warp-uniformly (all lanes take part in
// every call; the arguments are broadcast from the lane that evaluated the candidate).
template <typename F>
__device__ __forceinline__ void sparse_for_each_active(const SparseK& P, float x, float y, int lane, F&& f) {
    auto consume = [&](bool valid, int j, float4 kn) {
        float dx = 0.f, dy = 0.f, d2 = 0.f, val = 0.f;
        if (valid) {
            dx = x - kn.x;
            dy = y - kn.y;
            d2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
            val = phi_eval(P.fn, dx, dy, kn.z, kn.w);
        }
        unsigned m = __ballot_sync(0xffffffffu, val > 0.0f);
        while (m) {
            const int b = __ffs(m) - 1;
            m &= m - 1;
            f(__shfl_sync(0xffffffffu, j, b), __shfl_sync(0xffffffffu, val, b), __shfl_sync(0xffffffffu, dx, b),
              __shfl_sync(0xffffffffu, dy, b), __shfl_sync(0xffffffffu, d2, b), __shfl_sync(0xffffffffu, kn.w, b));
        }
    };
    if (P.cl.desc) {
        for (int l = 0; l < P.cl.n_levels; ++l) {
            const int G = P.cl.desc[8 * l], base = P.cl.desc[8 * l + 1];
            const int* st = P.cl.starts + base;
            const int cx = cell_of(x, G), cy = cell_of(y, G);
            const int y0 = max(cy - 1, 0), y1 = min(cy + 1, G - 1);
            for (int ix = max(cx - 1, 0); ix <= min(cx + 1, G - 1); ++ix) {
                const int p0 = st[ix * G + y0], p1 = st[ix * G + y1 + 1];       // cells (ix, y0..y1) are contiguous
                for (int pbase = p0; pbase < p1; pbase += 32) {
                    const int p = pbase + lane;
                    const bool valid = p < p1;
                    consume(valid, valid ? P.cl.order[p] : 0, valid ? __ldg(&P.cl.sorted[p]) : make_float4(0.f, 0.f, 0.f, 0.f));
                }
            }
        }
    } else {
        const Lattice& Lt = P.lat;
        for (int l = 0; l < Lt.n_levels; ++l) {
            const int side = Lt.side[l];
            const float g = (float)(side - 1), th = Lt.thetap[l];
            int ix0 = max(0, (int)ceilf((x - th) * g) - 1), ix1 = min(side - 1, (int)floorf((x + th) * g) + 1);
            int iy0 = max(0, (int)ceilf((y - th) * g) - 1), iy1 = min(side - 1, (int)floorf((y + th) * g) + 1);
            if (side == 1) { ix0 = ix1 = iy0 = iy1 = 0; }
            const int ny = iy1 - iy0 + 1, ncand = (ix1 - ix0 + 1) * ny;
            for (int cb = 0; cb < ncand; cb += 32) {
                const int c = cb + lane;
                const bool valid = c < ncand;
                const int j = valid ? Lt.offset[l] + (ix0 + c / ny) * side + (iy0 + c % ny) : 0;
                consume(valid, j, valid ? __ldg(&P.knots[j]) : make_float4(0.f, 0.f, 0.f, 0.f));
            }
        }
    }
}

__global__ void __launch_bounds__(SP_WARPS * 32) sparse_spatial_fwd_kernel(const __grid_constant__ SparseK P) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_warps = (long long)gridDim.x * SP_WARPS;
    const int ngroups = P.n_out >> 2;
    for (long long r = (long long)blockIdx.x * SP_WARPS + warp; r < P.pts.n_rows; r += n_warps) {
        float x, y, t;
        load_point(P.pts, P.pts.row_begin + r, x, y, t);
        float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
        sparse_for_each_active(P, x, y, lane, [&](int j, float f, float, float, float, float) {
            const float4* row = reinterpret_cast<const float4*>(P.w1t + (size_t)(P.p_cov + j) * P.n_out);
            if (lane < ngroups) {
                float4 w = __ldg(row + lane);
                acc0.x = fmaf(f, w.x, acc0.x); acc0.y = fmaf(f, w.y, acc0.y);
                acc0.z = fmaf(f, w.z, acc0.z); acc0.w = fmaf(f, w.w, acc0.w);
            }
            if (lane + 32 < ngroups) {
                float4 w = __ldg(row + lane + 32);
                acc1.x = fmaf(f, w.x, acc1.x); acc1.y = fmaf(f, w.y, acc1.y);
                acc1.z = fmaf(f, w.z, acc1.z); acc1.w = fmaf(f, w.w, acc1.w);
            }
        });
        float4* out = reinterpret_cast<float4*>(P.zs + (size_t)r * P.n_out);
        if (lane < ngroups) out[lane] = acc0;
        if (lane + 32 < ngroups) out[lane + 32] = acc1;
    }
}

// element group (row r, columns 4*g4 .. 4*g4+3) of an operand image
__device__ __forceinline__ float4 image_load4(const float* img, int slabs, long long r, int g4) {
    const long long tile = r / TILE_M;
    const uint32_t row = (uint32_t)(r - tile * TILE_M);
    const int slab = g4 >> 3, chunk = g4 & 7;
    const uint8_t* base = reinterpret_cast<const uint8_t*>(img + ((size_t)tile * slabs + slab) * SLAB_FLOATS);
    return *reinterpret_cast<const float4*>(base + swz_off(row, (uint32_t)chunk));
}

__global__ void __launch_bounds__(SP_WARPS * 32) sparse_spatial_wgrad_kernel(const __grid_constant__ SparseK P) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_warps = (long long)gridDim.x * SP_WARPS;
    const int ngroups = P.n_out >> 2;
    const int slabs = pad32(P.n_out) / SLAB_K;
    const bool knot_grads = P.d_centers != nullptr;
    for (long long r = (long long)blockIdx.x * SP_WARPS + warp; r < P.pts.n_rows; r += n_warps) {
        float x, y, t;
        load_point(P.pts, P.pts.row_begin + r, x, y, t);
        float4 d0 = make_float4(0.f, 0.f, 0.f, 0.f), d1 = d0;
        if (lane < ngroups) d0 = image_load4(P.dz_img, slabs, r, lane);
        if (lane + 32 < ngroups) d1 = image_load4(P.dz_img, slabs, r, lane + 32);
        sparse_for_each_active(P, x, y, lane, [&](int j, float f, float dx, float dy, float d2, float inv_th) {
            float4* row = reinterpret_cast<float4*>(P.dw1t + (size_t)(P.p_cov + j) * P.n_out);
            if (lane < ngroups) atomicAdd(row + lane, make_float4(f * d0.x, f * d0.y, f * d0.z, f * d0.w));
            if (lane + 32 < ngroups) atomicAdd(row + lane + 32, make_float4(f * d1.x, f * d1.y, f * d1.z, f * d1.w));
            if (knot_grads) {
                // G = dz1[n, :] . W1t[p + j, :]; then dL/dc_j += G phi'(r) (-(s - c)/(d theta')), dL/dlog theta_j += G phi'(r) (-r)
                const float4* wr = reinterpret_cast<const float4*>(P.w1t + (size_t)(P.p_cov + j) * P.n_out);
                float g = 0.0f;
                if (lane < ngroups) {
                    const float4 w = __ldg(wr + lane);
                    g = fmaf(d0.x, w.x, fmaf(d0.y, w.y, fmaf(d0.z, w.z, d0.w * w.w)));
                }
                if (lane + 32 < ngroups) {
                    const float4 w = __ldg(wr + lane + 32);
                    g += fmaf(d1.x, w.x, fmaf(d1.y, w.y, fmaf(d1.z, w.z, d1.w * w.w)));
                }
                g = warp_sum(g);
                if (lane == 0 && d2 > 0.0f) {
                    const float d = sqrtf(d2), rr = d * inv_th;
                    const float coef = g * phi_dr(P.fn, rr);
                    const float s = coef * inv_th / d;
                    atomicAdd(&P.d_centers[2 * j], -dx * s);
                    atomicAdd(&P.d_centers[2 * j + 1], -dy * s);
                    atomicAdd(&P.d_log_bw[j], -rr * coef);
                }
            }
        });
    }
}

// Blocks 1 wider than MAX_N (up to MAX_W outputs): the columns of a row are LANE_SETS = 4 float4 groups per lane,
// lane + 32 k, where the kernels above take two.  Kept apart from them so that their code stays as it is.
template <int LANE_SETS>
__device__ __forceinline__ void sparse_fwd_rows(const SparseK& P) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_warps = (long long)gridDim.x * SP_WARPS;
    const int ngroups = P.n_out >> 2;
    for (long long r = (long long)blockIdx.x * SP_WARPS + warp; r < P.pts.n_rows; r += n_warps) {
        float x, y, t;
        load_point(P.pts, P.pts.row_begin + r, x, y, t);
        float4 acc[LANE_SETS];
#pragma unroll
        for (int k = 0; k < LANE_SETS; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        sparse_for_each_active(P, x, y, lane, [&](int j, float f, float, float, float, float) {
            const float4* row = reinterpret_cast<const float4*>(P.w1t + (size_t)(P.p_cov + j) * P.n_out);
#pragma unroll
            for (int k = 0; k < LANE_SETS; ++k)
                if (lane + 32 * k < ngroups) {
                    float4 w = __ldg(row + lane + 32 * k);
                    acc[k].x = fmaf(f, w.x, acc[k].x); acc[k].y = fmaf(f, w.y, acc[k].y);
                    acc[k].z = fmaf(f, w.z, acc[k].z); acc[k].w = fmaf(f, w.w, acc[k].w);
                }
        });
        float4* out = reinterpret_cast<float4*>(P.zs + (size_t)r * P.n_out);
#pragma unroll
        for (int k = 0; k < LANE_SETS; ++k)
            if (lane + 32 * k < ngroups) out[lane + 32 * k] = acc[k];
    }
}
__global__ void __launch_bounds__(SP_WARPS * 32) sparse_spatial_fwd_wide_kernel(const __grid_constant__ SparseK P) {
    sparse_fwd_rows<4>(P);
}

template <int LANE_SETS>
__device__ __forceinline__ void sparse_wgrad_rows(const SparseK& P) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_warps = (long long)gridDim.x * SP_WARPS;
    const int ngroups = P.n_out >> 2;
    const int slabs = pad32(P.n_out) / SLAB_K;
    const bool knot_grads = P.d_centers != nullptr;
    for (long long r = (long long)blockIdx.x * SP_WARPS + warp; r < P.pts.n_rows; r += n_warps) {
        float x, y, t;
        load_point(P.pts, P.pts.row_begin + r, x, y, t);
        float4 d[LANE_SETS];
#pragma unroll
        for (int k = 0; k < LANE_SETS; ++k)
            d[k] = lane + 32 * k < ngroups ? image_load4(P.dz_img, slabs, r, lane + 32 * k) : make_float4(0.f, 0.f, 0.f, 0.f);
        sparse_for_each_active(P, x, y, lane, [&](int j, float f, float dx, float dy, float d2, float inv_th) {
            float4* row = reinterpret_cast<float4*>(P.dw1t + (size_t)(P.p_cov + j) * P.n_out);
#pragma unroll
            for (int k = 0; k < LANE_SETS; ++k)
                if (lane + 32 * k < ngroups)
                    atomicAdd(row + lane + 32 * k, make_float4(f * d[k].x, f * d[k].y, f * d[k].z, f * d[k].w));
            if (knot_grads) {
                // G = dz1[n, :] . W1t[p + j, :]; then dL/dc_j += G phi'(r) (-(s - c)/(d theta')), dL/dlog theta_j += G phi'(r) (-r)
                const float4* wr = reinterpret_cast<const float4*>(P.w1t + (size_t)(P.p_cov + j) * P.n_out);
                float g = 0.0f;
#pragma unroll
                for (int k = 0; k < LANE_SETS; ++k)
                    if (lane + 32 * k < ngroups) {
                        const float4 w = __ldg(wr + lane + 32 * k);
                        const float gk = fmaf(d[k].x, w.x, fmaf(d[k].y, w.y, fmaf(d[k].z, w.z, d[k].w * w.w)));
                        g = k == 0 ? gk : g + gk;
                    }
                g = warp_sum(g);
                if (lane == 0 && d2 > 0.0f) {
                    const float d = sqrtf(d2), rr = d * inv_th;
                    const float coef = g * phi_dr(P.fn, rr);
                    const float s = coef * inv_th / d;
                    atomicAdd(&P.d_centers[2 * j], -dx * s);
                    atomicAdd(&P.d_centers[2 * j + 1], -dy * s);
                    atomicAdd(&P.d_log_bw[j], -rr * coef);
                }
            }
        });
    }
}
// at least two CTAs per SM, i.e. up to 128 registers: with the default bound ptxas held the kernel to 64 and spilled
__global__ void __launch_bounds__(SP_WARPS * 32, 2) sparse_spatial_wgrad_wide_kernel(const __grid_constant__ SparseK P) {
    sparse_wgrad_rows<4>(P);
}

}  // namespace stdadk
