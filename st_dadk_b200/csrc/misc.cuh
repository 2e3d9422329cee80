// Elementwise / streaming kernels: operand-image packing, knot tables, unfused basis (parity checks),
// gradient norm and the fused clip + AdamW + EMA update.  All are HBM-bound; grids are sized in
// multiples of the SM count and accesses are 16-byte vectors where the layout allows.
#pragma once
#include "common.cuh"

namespace stdadk {

// ---------------------------------------------------------------- images
// One thread per 16-byte chunk of the image.
__global__ void pack_image_kernel(const float* __restrict__ src, long long row_stride, long long col_stride,
                                  long long rows, long long cols, float* __restrict__ img, long long n_chunks,
                                  int slabs) {
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n_chunks;
         idx += (long long)gridDim.x * blockDim.x) {
        int chunk = (int)(idx & 7);
        int row = (int)((idx >> 3) & 127);
        long long ts = idx >> 10;  // tile * slabs + slab
        int slab = (int)(ts % slabs);
        long long tile = ts / slabs;
        long long r = tile * TILE_M + row;
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            long long c = (long long)slab * SLAB_K + chunk * 4 + e;
            v[e] = (r < rows && c < cols) ? to_tf32(src[r * row_stride + c * col_stride]) : 0.0f;
        }
        float* dst = img + ts * SLAB_FLOATS;
        *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(dst) + swz_off((uint32_t)row, (uint32_t)chunk)) =
            make_float4(v[0], v[1], v[2], v[3]);
    }
}

struct PackBatch {
    stdadk_pack_desc d[STDADK_MAX_PACK];
    int n;
};
// blockIdx.y selects the matrix; same per-chunk work as pack_image_kernel
__global__ void pack_images_kernel(PackBatch B) {
    pdl_wait();                 // the sources are parameters the previous kernel may have written
    pdl_launch_dependents();
    const stdadk_pack_desc D = B.d[blockIdx.y];
    const int slabs = (int)((D.cols + SLAB_K - 1) / SLAB_K);
    const long long n_chunks = ((D.rows + TILE_M - 1) / TILE_M) * slabs * (long long)(SLAB_FLOATS / 4);
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n_chunks;
         idx += (long long)gridDim.x * blockDim.x) {
        int chunk = (int)(idx & 7);
        int row = (int)((idx >> 3) & 127);
        long long ts = idx >> 10;
        int slab = (int)(ts % slabs);
        long long tile = ts / slabs;
        long long r = tile * TILE_M + row;
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            long long c = (long long)slab * SLAB_K + chunk * 4 + e;
            v[e] = (r < D.rows && c < D.cols) ? tf32_part(D.src[r * D.row_stride + c * D.col_stride], D.part != 0) : 0.0f;
        }
        float* dst = D.img + ts * SLAB_FLOATS;
        *reinterpret_cast<float4*>(reinterpret_cast<uint8_t*>(dst) + swz_off((uint32_t)row, (uint32_t)chunk)) =
            make_float4(v[0], v[1], v[2], v[3]);
    }
}

__global__ void unpack_image_kernel(const float* __restrict__ img, long long rows, long long cols,
                                    float* __restrict__ dst, int slabs) {
    long long n = rows * cols;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < n;
         idx += (long long)gridDim.x * blockDim.x) {
        long long r = idx / cols, c = idx - r * cols;
        long long tile = r / TILE_M;
        uint32_t row = (uint32_t)(r - tile * TILE_M);
        int slab = (int)(c / SLAB_K);
        int cc = (int)(c - (long long)slab * SLAB_K);
        const uint8_t* base = reinterpret_cast<const uint8_t*>(img + (tile * slabs + slab) * SLAB_FLOATS);
        dst[idx] = *reinterpret_cast<const float*>(base + swz_off(row, (uint32_t)(cc >> 2)) + (cc & 3) * 4);
    }
}

// ---------------------------------------------------------------- knot tables
__global__ void knots_prepare_kernel(const float* __restrict__ centers, const float* __restrict__ bw,
                                     const float* __restrict__ log_bw, float calib, int k,
                                     float4* __restrict__ out) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    float b = log_bw ? expf(log_bw[j]) : bw[j];
    float th = __fmul_rn(b, calib);
    out[j] = make_float4(centers[2 * j], centers[2 * j + 1], __fmul_rn(th, th), 1.0f / th);
}
__global__ void tknots_prepare_kernel(const float* __restrict__ centers, const float* __restrict__ bw, int k,
                                      float2* __restrict__ out) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    out[j] = make_float2(centers[j], 1.0f / bw[j]);
}

// ---------------------------------------------------------------- unfused basis (debug / parity)
// phi (N x k_s) and psi (N x k_t) dense FP32; thread = (row, feature), consecutive threads = features.
__global__ void basis_fwd_kernel(BasisP B, PointsP P, float* __restrict__ phi, float* __restrict__ psi) {
    const int kf = B.k_s + B.k_t;
    const long long total = P.n_rows * (long long)kf;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        long long r = idx / kf;
        int f = (int)(idx - r * kf);
        float x, y, t;
        load_point(P, P.row_begin + r, x, y, t);
        if (f < B.k_s) {
            if (phi) {
                float4 kn = B.knots[f];
                phi[r * B.k_s + f] = phi_eval(B.fn, x - kn.x, y - kn.y, kn.z, kn.w);
            }
        } else if (psi) {
            float2 tk = B.tknots[f - B.k_s];
            psi[r * B.k_t + (f - B.k_s)] = psi_eval(t, tk.x, tk.y);
        }
    }
}

// ---------------------------------------------------------------- gradient norm + AdamW + EMA
struct GroupsP {
    long long end[8];
    int n;
};
__device__ __forceinline__ int group_of(const GroupsP& G, long long i) {
    int g = 0;
#pragma unroll
    for (int k = 0; k < 7; ++k)
        if (k + 1 < G.n && i >= G.end[k]) g = k + 1;
    return g;
}

// Deterministic (bitwise run-to-run and rank-to-rank: data-parallel replicas must derive the same clip coefficient):
// fixed grid, fixed per-thread stride, ordered in-block reduction, per-block partials written to `ws`, and the last
// block to finish (atomic ticket) adds the partials in block order.  ws: gridDim.x * 8 floats + 1 counter.
constexpr int SQNORM_BLOCKS = 592;      // 4 x 148 SMs
constexpr int SQNORM_THREADS = 256;
__global__ void sqnorm_kernel(const float* __restrict__ g, long long n, GroupsP G, float* __restrict__ out,
                              float* __restrict__ ws) {
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.0f;
    // 16-byte loads, four independent chains per thread; the element -> thread map is fixed, so the result is too
    const long long n4 = n >> 2;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4;
         i += (long long)gridDim.x * blockDim.x) {
        float4 v = __ldg(g4 + i);
        const long long e = i << 2;
        const int g0 = group_of(G, e), g3 = group_of(G, e + 3);
        if (g0 == g3) {
            float q = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, v.w * v.w)));
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (k == g0) acc[k] += q;
        } else {
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                int gi = group_of(G, e + j);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (k == gi) acc[k] = fmaf(vv[j], vv[j], acc[k]);
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {          // tail (n not a multiple of 4)
        long long i = (n4 << 2) + threadIdx.x;
        float v = g[i];
        int gi = group_of(G, i);
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k == gi) acc[k] = fmaf(v, v, acc[k]);
    }
    __shared__ float wsum[SQNORM_THREADS / 32][8];
    __shared__ bool last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float s = warp_sum(acc[k]);          // xor-butterfly: same order every run
        if (lane == 0) wsum[warp][k] = s;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float s = 0.0f;
        for (int w = 0; w < SQNORM_THREADS / 32; ++w) s += wsum[w][threadIdx.x];
        ws[blockIdx.x * 8 + threadIdx.x] = s;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int* ticket = reinterpret_cast<unsigned int*>(ws + gridDim.x * 8);
        unsigned int t = atomicAdd(ticket, 1u);
        last = (t == gridDim.x - 1);
        if (last) *ticket = 0u;              // ready for the next call
    }
    __syncthreads();
    if (last && threadIdx.x < G.n) {
        __threadfence();
        float s = 0.0f;
        for (unsigned int b = 0; b < gridDim.x; ++b) s += ws[b * 8 + threadIdx.x];
        out[threadIdx.x] = s;
    }
}

// ---------------------------------------------------------------- data-parallel gradient exchange over peer memory
// One-shot all-reduce of the flat gradient between the GPUs of one box (NVLink 5 / NVSwitch), fused with the gradient
// norm that follows it in a step, replacing {graph boundary, ncclAllReduce, graph boundary, sqnorm launch}.
//
// Low-latency protocol (flag travels WITH the data, as in NCCL's LL): every rank pushes its gradient to every peer's
// receive area with 16-byte remote stores {v0, epoch, v1, epoch} -- two self-validating 8-byte packets -- and then
// reduces: for each element it reads the W - 1 packets that the peers pushed into ITS receive area (local memory),
// spinning on the epoch, and adds them to its own value in RANK ORDER, so every rank forms bit-identical sums.  No
// separate barrier, no second pass, the result is written in place.  Receive areas are double-buffered by epoch
// parity: a rank can only be one exchange ahead of its slowest peer (it cannot finish exchange e+1 before every peer
// has pushed e+1, which a peer does after it finished reading e), so parity e+2 never overwrites unread data.
// epoch = *step_count + 1 (device-side, equal on all ranks, grows by one per step: graph-replay safe, never 0).
// Traffic per rank: 8 B x n x (W - 1) pushed (0.7 MB gradient, 8 ranks: 10 MB, ~13 us at NVLink rate); waits are
// bounded (trap after ~2 s instead of hanging the GPU).
constexpr int PEER_MAX = 8;
struct PeerK {
    float* g;                         // this rank's gradient, reduced in place
    long long n2;                     // float pairs
    uint4* recv[PEER_MAX];            // rank p's receive area as mapped here: [2 parities][W sources][n2] packets
    const int* step_count;
    int rank, world;
    int two_phase;                    // 0: every rank pushes everything to everyone; 1: reduce-scatter + all-gather
    GroupsP G;                        // fused squared norm of g[0 : n_norm) per group (G.n == 0: no norm)
    long long n_norm;
    float* sq_out;
    float* ws;                        // gridDim.x * 8 partials + ticket
};
__device__ __forceinline__ void st_sys_v4(uint4* p, uint4 v) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_sys_v4(const uint4* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
// spin until the packet at `src` carries this exchange's epoch in both halves (bounded: trap after ~2 s)
__device__ __forceinline__ float2 peer_wait_packet(const uint4* src, unsigned int epoch) {
    uint4 q = ld_sys_v4(src);
    if (q.y != epoch || q.w != epoch) {
        unsigned long long t0 = 0, now;
        do {
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 2000000000ull) __trap();
            q = ld_sys_v4(src);
        } while (q.y != epoch || q.w != epoch);
    }
    return make_float2(__uint_as_float(q.x), __uint_as_float(q.z));
}
constexpr int PEER_THREADS = 256;
// Two-phase form (P.two_phase, worlds of 4 and more): the pairs are cut into W contiguous chunks, chunk c is OWNED by
// rank c.  (1) every rank pushes its values of chunk c to rank c only; (2) the owner adds the W contributions in rank
// order -- the same order as the one-shot form, so both give the same bits -- and pushes the sum to every peer;
// (3) every rank picks up the W - 1 foreign chunks.  Pushed per rank: ~(1 + 6/8) n packets at W = 8 instead of 7 n
// (measured at 8 GPUs, 176k floats: 35.7 us one-shot), at the price of a second NVLink traversal.  Slots never collide:
// in rank r's area, source s writes chunk r in phase 1 and its own chunk s in phase 2.  The thread -> element mapping
// is the same grid-stride mapping in every phase, so a thread only ever re-reads what it wrote itself, and the norm
// is accumulated in a last pass in a rank-independent order (replicas must compute the same clip coefficient).
__device__ __forceinline__ void peer_two_phase(const PeerK& P, unsigned int epoch, long long par_off, long long i0,
                                               long long stride) {
    float2* g2 = reinterpret_cast<float2*>(P.g);
    const long long m = (P.n2 + P.world - 1) / P.world;
    const long long own_lo = (long long)P.rank * m, own_hi = min(P.n2, own_lo + m);
    const uint4* mine = P.recv[P.rank];
    for (long long i = i0; i < P.n2; i += stride) {
        if (i >= own_lo && i < own_hi) continue;
        const int owner = (int)(i / m);
        const float2 v = g2[i];
        uint4* dst = nullptr;
#pragma unroll
        for (int p = 0; p < PEER_MAX; ++p)
            if (p == owner) dst = P.recv[p];
        st_sys_v4(dst + (par_off + P.rank) * P.n2 + i, make_uint4(__float_as_uint(v.x), epoch, __float_as_uint(v.y), epoch));
    }
    for (long long i = i0; i < P.n2; i += stride) {
        if (i < own_lo || i >= own_hi) continue;
        const float2 own = g2[i];
        float2 sum = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int s = 0; s < PEER_MAX; ++s)
            if (s < P.world) {
                const float2 v = s == P.rank ? own : peer_wait_packet(mine + (par_off + s) * P.n2 + i, epoch);
                sum.x += v.x;
                sum.y += v.y;
            }
        g2[i] = sum;
        const uint4 pkt = make_uint4(__float_as_uint(sum.x), epoch, __float_as_uint(sum.y), epoch);
#pragma unroll
        for (int p = 0; p < PEER_MAX; ++p)
            if (p < P.world && p != P.rank) st_sys_v4(P.recv[p] + (par_off + P.rank) * P.n2 + i, pkt);
    }
    for (long long i = i0; i < P.n2; i += stride) {
        if (i >= own_lo && i < own_hi) continue;
        const int owner = (int)(i / m);
        g2[i] = peer_wait_packet(mine + (par_off + owner) * P.n2 + i, epoch);
    }
}
__global__ void __launch_bounds__(PEER_THREADS) peer_allreduce_kernel(const __grid_constant__ PeerK P) {
    const unsigned int epoch = (unsigned int)(*P.step_count) + 1u;
    const long long par_off = (long long)(epoch & 1u) * P.world;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    float2* g2 = reinterpret_cast<float2*>(P.g);
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.0f;
    if (P.two_phase) {
        peer_two_phase(P, epoch, par_off, i0, stride);
        if (P.G.n == 0) return;
        for (long long i = i0; i < P.n2; i += stride) {
            const float2 sum = g2[i];
            const long long e = i << 1;
            const float vv[2] = {sum.x, sum.y};
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (e + j < P.n_norm) {
                    const int gi = group_of(P.G, e + j);
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (k == gi) acc[k] = fmaf(vv[j], vv[j], acc[k]);
                }
        }
    } else {
    // ---- push my gradient into every peer's receive area
    for (long long i = i0; i < P.n2; i += stride) {
        const float2 v = g2[i];
        const uint4 pkt = make_uint4(__float_as_uint(v.x), epoch, __float_as_uint(v.y), epoch);
#pragma unroll
        for (int p = 0; p < PEER_MAX; ++p)
            if (p < P.world && p != P.rank) st_sys_v4(P.recv[p] + (par_off + P.rank) * P.n2 + i, pkt);
    }
    // ---- reduce in rank order what the peers pushed into mine
    const uint4* mine = P.recv[P.rank];
    for (long long i = i0; i < P.n2; i += stride) {
        const float2 own = g2[i];
        float2 sum = make_float2(0.0f, 0.0f);
#pragma unroll
        for (int s = 0; s < PEER_MAX; ++s)
            if (s < P.world) {
                float2 v = own;
                if (s != P.rank) v = peer_wait_packet(mine + (par_off + s) * P.n2 + i, epoch);
                sum.x += v.x;
                sum.y += v.y;
            }
        g2[i] = sum;
        if (P.G.n > 0) {
            const long long e = i << 1;
            const float vv[2] = {sum.x, sum.y};
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (e + j < P.n_norm) {
                    const int gi = group_of(P.G, e + j);
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (k == gi) acc[k] = fmaf(vv[j], vv[j], acc[k]);
                }
        }
    }
    }
    if (P.G.n == 0) return;
    // ---- deterministic finish of the norm: ordered in-block reduction, last block adds the partials in block order
    __shared__ float wsum[PEER_THREADS / 32][8];
    __shared__ bool last;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float s = warp_sum(acc[k]);
        if (lane == 0) wsum[warp][k] = s;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float s = 0.0f;
        for (int w = 0; w < PEER_THREADS / 32; ++w) s += wsum[w][threadIdx.x];
        P.ws[blockIdx.x * 8 + threadIdx.x] = s;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int* ticket = reinterpret_cast<unsigned int*>(P.ws + gridDim.x * 8);
        unsigned int t = atomicAdd(ticket, 1u);
        last = (t == gridDim.x - 1);
        if (last) *ticket = 0u;
    }
    __syncthreads();
    if (last && threadIdx.x < P.G.n) {
        __threadfence();
        float s = 0.0f;
        for (unsigned int b = 0; b < gridDim.x; ++b) s += P.ws[b * 8 + threadIdx.x];
        P.sq_out[threadIdx.x] = s;
    }
}

struct AdamK {
    float* p;
    const float* g;
    float* m;
    float* v;
    float* shadow;
    long long n;
    GroupsP G;
    const float* hyper;    // (n_groups x 4): lr, weight_decay, max_norm (<=0: no clipping), unused
    const float* sqnorms;  // (n_groups) or null
    const int* step_count; // device; holds the 1-based step index of THIS update
    float beta1, beta2, eps, ema_decay;
    float* g_zero;         // == g when the kernel should leave the gradient buffer zeroed for the next step, else null
    float* loss_acc;       // optional: *loss_sum += *loss_acc; *loss_acc = 0 (one thread), saves two tiny launches
    float* loss_sum;
    float* loss_last;      // optional: the step's loss before the accumulator is cleared
    // fused step tail (adamw_fused_kernel): the kernel itself forms the squared gradient norms (written to sq_out),
    // and advances the step counter -- one launch instead of {sqnorm, step counter, adamw}
    float* sq_out;
    float* norm_ws;        // gridDim.x * 8 partials, then two uint32: arrival counter, generation
    int* step_rw;
    int state_early;       // stdadk_adamw_args.state_early (fused tail only)
    unsigned long long* dbg;   // phase stamps of -DSTDADK_PF_DEBUG builds (STEP_T), else NULL
};
// torch.optim.AdamW (decoupled decay, bias correction) + clip_grad_norm_ coefficient + ModelEMA.update
// in one pass: 20 B read + 16 B written per parameter (28 B without EMA).
// Fused tail: a thread's float4 of p / m / v / shadow (at most TAIL_RES of them) and of g stay in registers from
// before the wait and the grid barrier to the update, so the update pass takes no memory round trip after the
// barrier.  A larger model takes the streaming loop.  Either way element i4 belongs to thread i4 mod (grid x 256) and
// both norm reductions keep their order, so the results are the same bits.
constexpr int TAIL_RES = 2;
template <bool FUSED>
__global__ void __launch_bounds__(256) adamw_ema_kernel(AdamK A) {
    __shared__ float s_sq[8];
    const long long n4 = A.n >> 2;
    const long long i0 = blockIdx.x * (long long)blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    const float4* g4 = reinterpret_cast<const float4*>(A.g);
    float4* p4 = reinterpret_cast<float4*>(A.p);
    float4* m4 = reinterpret_cast<float4*>(A.m);
    float4* v4 = reinterpret_cast<float4*>(A.v);
    float4* s4 = reinterpret_cast<float4*>(A.shadow);
    const bool early = FUSED && A.state_early;
    const bool resident = early && n4 <= TAIL_RES * stride;
    float4 rg[TAIL_RES], rp[TAIL_RES], rm[TAIL_RES], rv[TAIL_RES], rs[TAIL_RES];
    float hy[8][3];
    int step;
    auto load_state = [&]() {
        step = FUSED ? *A.step_count + 1 : *A.step_count;  // fused: read BEFORE the grid barrier, block 0 publishes it
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < A.G.n) {
                hy[k][0] = A.hyper[4 * k];
                hy[k][1] = A.hyper[4 * k + 1];
                hy[k][2] = A.hyper[4 * k + 2];
            }
        if (resident) {
#pragma unroll
            for (int r = 0; r < TAIL_RES; ++r) {
                const long long i = i0 + r * stride;
                if (i < n4) {
                    rp[r] = p4[i];
                    rm[r] = m4[i];
                    rv[r] = v4[i];
                    rs[r] = s4 ? s4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        }
    };
    STEP_T_BEGIN(A.dbg);
    // with state_early, hyper-parameters, the step counter and the optimizer state were written by the previous step's
    // tail or by copies before this step's first kernel: they are loaded before the wait (ptx.cuh, rule 2)
    if (early) load_state();
    STEP_T(A.dbg, 0);   // early loads
    if (FUSED) {
        pdl_wait();             // g comes from the backward; the grid barrier below needs its CTAs gone
        STEP_T(A.dbg, 1);   // wait for the backward
        if (!early) load_state();
        if (resident) {
#pragma unroll
            for (int r = 0; r < TAIL_RES; ++r)
                if (i0 + r * stride < n4) rg[r] = __ldg(g4 + i0 + r * stride);
        }
        // ---- phase 1: squared norm per group.  Deterministic: the element -> thread map is a function of the grid
        // (itself a function of n), in-block reduction and the sum over blocks are ordered.
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.0f;
        if (A.sqnorms) {                                // (sqnorms != NULL <=> clipping is on)
            auto add_sq = [&](const float4 v, long long i) {
                const long long e = i << 2;
                const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int gi = group_of(A.G, e + j);
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (k == gi) acc[k] = fmaf(vv[j], vv[j], acc[k]);
                }
            };
            if (resident) {
#pragma unroll
                for (int r = 0; r < TAIL_RES; ++r)
                    if (i0 + r * stride < n4) add_sq(rg[r], i0 + r * stride);
            } else {
                for (long long i = i0; i < n4; i += stride) add_sq(__ldg(g4 + i), i);
            }
            if (blockIdx.x == 0 && threadIdx.x < (A.n & 3)) {
                const long long i = (n4 << 2) + threadIdx.x;
                const float v = A.g[i];
                const int gi = group_of(A.G, i);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    if (k == gi) acc[k] = fmaf(v, v, acc[k]);
            }
        }
        __shared__ float wsum[8][8];
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float sk = warp_sum(acc[k]);
            if (lane == 0) wsum[warp][k] = sk;
        }
        __syncthreads();
        if (threadIdx.x < 8) {
            float sk = 0.0f;
            for (int w = 0; w < 8; ++w) sk += wsum[w][threadIdx.x];
            A.norm_ws[blockIdx.x * 8 + threadIdx.x] = sk;
        }
        STEP_T(A.dbg, 2);   // g, norm partials
        // ---- grid barrier (the grid is at most one block per SM and every block is resident): arrival counter +
        // generation word; bounded wait
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned int* cnt = reinterpret_cast<unsigned int*>(A.norm_ws + gridDim.x * 8);
            volatile unsigned int* gen = cnt + 1;
            const unsigned int my_gen = *gen;
            if (atomicAdd(cnt, 1u) == gridDim.x - 1) {
                *cnt = 0u;
                __threadfence();
                atomicAdd(const_cast<unsigned int*>(gen), 1u);
            } else {
                long long t0 = clock64();
                while (*gen == my_gen) {
                    if (clock64() - t0 > 4000000000LL) __trap();
                }
            }
            __threadfence();
        }
        __syncthreads();
        if (threadIdx.x < 8) {
            float sk = 0.0f;
            for (unsigned int b = 0; b < gridDim.x; ++b) sk += __ldcg(&A.norm_ws[b * 8 + threadIdx.x]);
            s_sq[threadIdx.x] = sk;
            if (blockIdx.x == 0 && A.sq_out && threadIdx.x < A.G.n) A.sq_out[threadIdx.x] = sk;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) *A.step_rw = step;
        __syncthreads();
        STEP_T(A.dbg, 3);   // grid barrier, norms
    } else {
        load_state();
    }
    const float bc1 = 1.0f - powf(A.beta1, (float)step);
    const float bc2 = 1.0f - powf(A.beta2, (float)step);
    const float inv_sqrt_bc2 = 1.0f / sqrtf(bc2);
    float lr[8], wd[8], clip[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        lr[k] = wd[k] = 0.0f;
        clip[k] = 1.0f;
        if (k < A.G.n) {
            lr[k] = hy[k][0];
            wd[k] = hy[k][1];
            float mx = hy[k][2];
            if (A.sqnorms && mx > 0.0f) clip[k] = fminf(1.0f, mx / (sqrtf(FUSED ? s_sq[k] : A.sqnorms[k]) + 1e-6f));
        }
    }
    auto update = [&](long long i, float g, float& p, float& m, float& v, float& sh) {
        int gi = group_of(A.G, i);
        float l = lr[0], w = wd[0], c = clip[0];
#pragma unroll
        for (int k = 1; k < 8; ++k)
            if (k == gi) { l = lr[k]; w = wd[k]; c = clip[k]; }
        g *= c;
        p *= (1.0f - l * w);
        m = A.beta1 * m + (1.0f - A.beta1) * g;
        v = A.beta2 * v + (1.0f - A.beta2) * g * g;
        float denom = sqrtf(v) * inv_sqrt_bc2 + A.eps;
        p -= (l / bc1) * (m / denom);
        sh = A.ema_decay * sh + (1.0f - A.ema_decay) * p;
    };
    auto update4 = [&](long long i, float4 g, float4 p, float4 m, float4 v, float4 sh) {
        const long long e = i << 2;
        update(e, g.x, p.x, m.x, v.x, sh.x);
        update(e + 1, g.y, p.y, m.y, v.y, sh.y);
        update(e + 2, g.z, p.z, m.z, v.z, sh.z);
        update(e + 3, g.w, p.w, m.w, v.w, sh.w);
        p4[i] = p;
        m4[i] = m;
        v4[i] = v;
        if (s4) s4[i] = sh;
        if (A.g_zero) reinterpret_cast<float4*>(A.g_zero)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    };
    if (resident) {
#pragma unroll
        for (int r = 0; r < TAIL_RES; ++r)
            if (i0 + r * stride < n4) update4(i0 + r * stride, rg[r], rp[r], rm[r], rv[r], rs[r]);
    } else {
        for (long long i = i0; i < n4; i += stride)
            update4(i, __ldg(g4 + i), p4[i], m4[i], v4[i], s4 ? s4[i] : make_float4(0.f, 0.f, 0.f, 0.f));
    }
    STEP_T(A.dbg, 4);       // update pass
    if (blockIdx.x == 0 && threadIdx.x == 0 && A.loss_acc && A.loss_sum) {
        const float step_loss = *A.loss_acc;
        *A.loss_sum += step_loss;
        if (A.loss_last) *A.loss_last = step_loss;
        *A.loss_acc = 0.0f;
    }
    if (blockIdx.x == 0 && threadIdx.x < (A.n & 3)) {
        long long i = (n4 << 2) + threadIdx.x;
        float p = A.p[i], m = A.m[i], v = A.v[i], sh = A.shadow ? A.shadow[i] : 0.0f;
        update(i, A.g[i], p, m, v, sh);
        A.p[i] = p;
        A.m[i] = m;
        A.v[i] = v;
        if (A.shadow) A.shadow[i] = sh;
        if (A.g_zero) A.g_zero[i] = 0.0f;
    }
}

}  // namespace stdadk
