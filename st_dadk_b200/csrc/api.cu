// C ABI of libstdadk.so (see include/stdadk.h): argument validation on the host, kernel launches on the
// caller's stream.  No device allocation, no CPU fallback.
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "layer.cuh"
#include "misc.cuh"
#include "sparse.cuh"
#include "predict.cuh"
#include "field.cuh"

using namespace stdadk;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
static int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
    return 0;
}
#define REQUIRE(cond, ...) \
    do {                   \
        if (!(cond)) return fail(-1, __VA_ARGS__); \
    } while (0)

static int g_sm_count = 0;
static int check_device() {
    static thread_local int ok_dev = -1;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail((int)e, "cudaGetDevice: %s (libstdadk has no CPU fallback)", cudaGetErrorString(e));
    if (dev == ok_dev) return 0;
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, dev);
    if (e != cudaSuccess) return fail((int)e, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (p.major != 10) return fail(-2, "libstdadk requires an sm_100 (B200) device, found sm_%d%d", p.major, p.minor);
    g_sm_count = p.multiProcessorCount;
    ok_dev = dev;
    return 0;
}
static int grid_for(long long work_items, int threads, int per_sm = 8) {
    long long blocks = (work_items + threads - 1) / threads;
    long long cap = (long long)(g_sm_count > 0 ? g_sm_count : 148) * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}
static int pow2_cols(int n) {
    int c = 32;
    while (c < n) c <<= 1;
    return c;
}
// A 64-row tile's warps read the accumulator 64 columns at a time (two 32-column chunks, one per half-warp), so the
// allocation covers n_pad rounded up to 64.
static int tmem_cols_m64(int n_pad) { return pow2_cols((n_pad + 63) & ~63); }
template <typename K>
static int set_smem(K kernel, uint32_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return fail((int)e, "cudaFuncSetAttribute(%u B smem): %s", bytes, cudaGetErrorString(e));
    return 0;
}

// Launch of a kernel of the training step's chain (pack, layer_fwd, layer_bwd, wgrad, the fused tail) with
// programmatic stream serialisation: it may start while the previous kernel on the stream runs and waits for it in
// pdl_wait() (ptx.cuh states the rules the kernels keep).  Only a grid of at most one CTA per SM starts early: the
// CTAs of a larger one would sit waiting on every SM its predecessor frees and keep the concurrent kernels of the
// other stream off them (batch 65,536 on B200: 0.791 -> 0.817 ms per step with every grid starting early).  Errors
// surface through check_launch.
template <typename... KArgs, typename... Args>
static void launch_chained(void (*kernel)(KArgs...), dim3 grid, int threads, uint32_t smem, void* stream,
                           Args&&... args) {
    const long long ctas = (long long)grid.x * grid.y * grid.z;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = ctas <= (g_sm_count > 0 ? g_sm_count : 148) ? 1 : 0;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = (cudaStream_t)stream;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    (void)cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

static BasisP to_basis(const stdadk_basis* b) {
    BasisP B{};
    if (b) {
        B.knots = reinterpret_cast<const float4*>(b->knots4);
        B.tknots = reinterpret_cast<const float2*>(b->tknots2);
        B.k_s = b->k_s;
        B.k_t = b->k_t;
        B.p_cov = b->p_cov;
        B.fn = b->basis_fn;
    }
    return B;
}
static PointsP to_points(const stdadk_points& p) {
    PointsP P{};
    P.coords = p.coords;
    P.t = p.t;
    P.xcov = p.xcov;
    P.index = reinterpret_cast<const long long*>(p.index);
    P.nx = p.grid_nx;
    P.ny = p.grid_ny;
    P.nt = p.grid_nt;
    P.row_begin = p.row_begin;
    P.n_rows = p.n_rows;
    return P;
}
static LayerP to_layer(const stdadk_layer& l, const stdadk_dropout& d) {
    LayerP L{};
    L.w_img = l.w_img;
    L.w_img_lo = l.w_img_lo;
    L.bias = l.bias;
    L.gamma = l.gamma;
    L.beta = l.beta;
    L.n_in = l.n_in;
    L.n_out = l.n_out;
    L.layer_id = l.layer_id;
    L.eps = l.ln_eps;
    L.drop_p = d.p;
    L.step = d.step;
    L.seed = d.seed;
    L.step_ptr = d.step_ptr;
    L.key_offset = d.key_offset;
    return L;
}
static HeadP to_head(const stdadk_head* h) {
    HeadP H{};
    if (h) {
        H.w = h->w;
        H.b = h->b;
        H.y = h->y;
        H.yhat = h->yhat;
        H.dyhat = h->dyhat;
        H.loss_acc = h->loss_acc;
        H.q = h->q;
        H.loss_type = h->loss_type;
        H.nc_power = h->nc_power;
        H.inv_count = h->inv_count;
        H.nc_weight = h->nc_weight;
        memcpy(H.taus, h->taus, sizeof(H.taus));
    }
    return H;
}
static int check_basis_points(const stdadk_basis* b, const stdadk_points& p, int n_in) {
    REQUIRE(b->knots4 || b->k_s == 0, "basis: knots4 is NULL");
    REQUIRE(b->tknots2 || b->k_t == 0, "basis: tknots2 is NULL");
    REQUIRE(((reinterpret_cast<uintptr_t>(b->knots4) | reinterpret_cast<uintptr_t>(b->tknots2)) & 15) == 0,
            "basis: knots4 / tknots2 must be 16-byte aligned (staged into shared memory with bulk async copies)");
    REQUIRE(b->k_s >= 0 && b->k_t >= 0 && b->p_cov >= 0, "basis: negative sizes");
    REQUIRE(b->basis_fn >= 0 && b->basis_fn <= 2, "basis: unknown basis_fn %d", b->basis_fn);
    REQUIRE(n_in < 0 || b->p_cov + b->k_s + b->k_t == n_in, "basis: p+k_s+k_t=%d != layer n_in=%d",
            b->p_cov + b->k_s + b->k_t, n_in);
    if (p.grid_nx > 0) {
        REQUIRE(p.grid_ny > 0 && p.grid_nt > 0, "points: grid sizes must all be positive");
    } else if (p.n_rows > 0) {       // an empty batch (X of shape (0, p), st_interp.py:836-846) has no storage to point at
        REQUIRE(p.coords && p.t, "points: coords/t are NULL and no grid was given");
        REQUIRE((reinterpret_cast<uintptr_t>(p.coords) & 7) == 0, "points: coords must be 8-byte aligned");
    }
    REQUIRE(b->p_cov == 0 || p.xcov || p.grid_nx > 0 || p.n_rows <= 0, "points: xcov is NULL but p_cov > 0");
    return 0;
}

extern "C" {

int stdadk_version(void) { return STDADK_VERSION; }
const char* stdadk_last_error(void) { return g_err; }

size_t stdadk_sizeof(int which) {
    switch (which) {
        case 0: return sizeof(stdadk_basis);
        case 1: return sizeof(stdadk_points);
        case 2: return sizeof(stdadk_layer);
        case 3: return sizeof(stdadk_dropout);
        case 4: return sizeof(stdadk_head);
        case 5: return sizeof(stdadk_fwd_args);
        case 6: return sizeof(stdadk_bwd_args);
        case 7: return sizeof(stdadk_wgrad_args);
        case 8: return sizeof(stdadk_knotgrad_args);
        case 9: return sizeof(stdadk_adamw_args);
        case 10: return sizeof(stdadk_pack_desc);
        case 11: return sizeof(stdadk_sparse_args);
        case 12: return sizeof(stdadk_predict_args);
        case 14: return sizeof(stdadk_peer_allreduce_args);
        case 15: return sizeof(stdadk_field_args);
        default: return 0;
    }
}

size_t stdadk_image_floats(int64_t rows, int64_t cols) {
    return (size_t)(ceil_div64(rows, TILE_M) * ceil_div64(cols, SLAB_K)) * SLAB_FLOATS;
}

int stdadk_knots_prepare(const float* centers, const float* bw, const float* log_bw, float calib, int k,
                         float* knots4, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(k >= 0 && centers && (bw || log_bw) && knots4, "knots_prepare: bad arguments");
    REQUIRE((reinterpret_cast<uintptr_t>(knots4) & 15) == 0, "knots_prepare: knots4 must be 16-byte aligned");
    if (k == 0) return 0;
    knots_prepare_kernel<<<(k + 127) / 128, 128, 0, (cudaStream_t)stream>>>(centers, bw, log_bw, calib, k,
                                                                             reinterpret_cast<float4*>(knots4));
    return check_launch("knots_prepare");
}

int stdadk_tknots_prepare(const float* centers, const float* bw, int k, float* tknots2, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(k >= 0 && centers && bw && tknots2, "tknots_prepare: bad arguments");
    if (k == 0) return 0;
    tknots_prepare_kernel<<<(k + 127) / 128, 128, 0, (cudaStream_t)stream>>>(centers, bw, k,
                                                                              reinterpret_cast<float2*>(tknots2));
    return check_launch("tknots_prepare");
}

int stdadk_basis_fwd(const stdadk_basis* basis, const stdadk_points* pts, float* phi, float* psi, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(basis && pts, "basis_fwd: NULL descriptor");
    if (int r = check_basis_points(basis, *pts, -1)) return r;
    if (pts->n_rows <= 0) return 0;
    long long total = pts->n_rows * (long long)(basis->k_s + basis->k_t);
    if (total == 0) return 0;
    basis_fwd_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(to_basis(basis), to_points(*pts), phi,
                                                                              psi);
    return check_launch("basis_fwd");
}

int stdadk_pack_image(const float* src, int64_t row_stride, int64_t col_stride, int64_t rows, int64_t cols,
                      float* img, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(src && img && rows > 0 && cols > 0, "pack_image: bad arguments");
    REQUIRE((reinterpret_cast<uintptr_t>(img) & 127) == 0, "pack_image: image must be 128-byte aligned");
    int slabs = (int)ceil_div64(cols, SLAB_K);
    long long chunks = (long long)ceil_div64(rows, TILE_M) * slabs * (SLAB_FLOATS / 4);
    pack_image_kernel<<<grid_for(chunks, 256), 256, 0, (cudaStream_t)stream>>>(src, row_stride, col_stride, rows, cols,
                                                                                img, chunks, slabs);
    return check_launch("pack_image");
}

int stdadk_pack_images(const stdadk_pack_desc* descs, int n, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(descs && n >= 1 && n <= STDADK_MAX_PACK, "pack_images: 1..%d descriptors, got %d", STDADK_MAX_PACK, n);
    PackBatch B{};
    B.n = n;
    long long max_chunks = 0;
    for (int i = 0; i < n; ++i) {
        REQUIRE(descs[i].src && descs[i].img && descs[i].rows > 0 && descs[i].cols > 0, "pack_images: bad descriptor %d", i);
        REQUIRE((reinterpret_cast<uintptr_t>(descs[i].img) & 127) == 0, "pack_images: image %d must be 128-byte aligned", i);
        B.d[i] = descs[i];
        long long chunks = ceil_div64(descs[i].rows, TILE_M) * ceil_div64(descs[i].cols, SLAB_K) * (SLAB_FLOATS / 4);
        if (chunks > max_chunks) max_chunks = chunks;
    }
    dim3 grid(grid_for(max_chunks, 256, 2), n);
    launch_chained(pack_images_kernel, grid, 256, 0, stream, B);
    return check_launch("pack_images");
}

int stdadk_unpack_image(const float* img, int64_t rows, int64_t cols, float* dst, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(dst && img && rows > 0 && cols > 0, "unpack_image: bad arguments");
    int slabs = (int)ceil_div64(cols, SLAB_K);
    unpack_image_kernel<<<grid_for(rows * cols, 256), 256, 0, (cudaStream_t)stream>>>(img, rows, cols, dst, slabs);
    return check_launch("unpack_image");
}

static int check_layer(const stdadk_layer& l, const char* who) {
    REQUIRE(l.w_img && l.bias, "%s: weight image / bias is NULL", who);
    REQUIRE(l.n_out >= 1 && l.n_out <= MAX_N, "%s: n_out=%d outside [1,%d] (one UMMA N / LayerNorm row per thread)", who,
            l.n_out, MAX_N);
    REQUIRE(l.n_in >= 1, "%s: n_in=%d", who, l.n_in);
    REQUIRE((l.gamma == nullptr) == (l.beta == nullptr), "%s: gamma and beta must both be given or both NULL", who);
    REQUIRE(((reinterpret_cast<uintptr_t>(l.w_img) | reinterpret_cast<uintptr_t>(l.w_img_lo)) & 127) == 0,
            "%s: weight images must be 128-byte aligned", who);
    return 0;
}

// Shared memory of the layer_fwd / layer_bwd launches.  stdadk_dense_basis_supported checks block 1's launches with
// these same functions (and wgrad_smem_bytes), so the executor's regime choice and the launch checks cannot disagree.
constexpr uint32_t SMEM_LIMIT = 227 * 1024;
constexpr int BWD_CG = 2, BWD_NS = 4;
// cg = 4 (latency configuration, 4 stages) or 2 (two CTAs per SM, 2 stages); tab_chunks = k_slabs * 8 with a basis
static uint32_t fwd_smem(int n_pad, int q, int k_s, int k_t, int tab_chunks, int cg) {
    return plan_smem(n_pad, q, k_s, k_t, false, cg, cg == 2 ? 2 : 4, tab_chunks).total;
}
static uint32_t bwd_smem(int n_pad, int q, int k_s, int k_t, int tab_chunks) {
    return plan_smem(n_pad, q, k_s, k_t, true, BWD_CG, BWD_NS, tab_chunks).total;
}

static unsigned long long* g_predict_dbg = nullptr;   // stdadk_debug_counters (profiling builds)
int stdadk_layer_fwd(const stdadk_fwd_args* a, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(a, "layer_fwd: NULL args");
    if (int r = check_layer(a->layer, "layer_fwd")) return r;
    REQUIRE((a->basis != nullptr) != (a->a_img != nullptr), "layer_fwd: give exactly one of basis / a_img");
    if (a->basis)
        if (int r = check_basis_points(a->basis, a->pts, a->layer.n_in)) return r;
    REQUIRE(a->drop.p >= 0.0f && a->drop.p < 1.0f, "layer_fwd: dropout p=%f", a->drop.p);
    REQUIRE(!a->addend || (a->layer.n_out % 4 == 0 && (reinterpret_cast<uintptr_t>(a->addend) & 15) == 0),
            "layer_fwd: addend needs n_out %% 4 == 0 and 16-byte alignment");
    if (a->head) {
        REQUIRE(a->head->q >= 1 && a->head->q <= STDADK_MAX_Q, "layer_fwd: head q=%d outside [1,%d]", a->head->q,
                STDADK_MAX_Q);
        REQUIRE(a->head->w && a->head->b && a->head->yhat, "layer_fwd: head w/b/yhat NULL");
        REQUIRE(a->head->loss_type == STDADK_LOSS_NONE || (a->head->y && a->head->loss_acc),
                "layer_fwd: loss requested without y / loss_acc");
    } else {
        REQUIRE(a->out_img, "layer_fwd: out_img is NULL and there is no head");
    }
    const bool x3 = a->layer.w_img_lo != nullptr;
    if (x3) {
        REQUIRE(!a->a_img || a->a_img_lo, "layer_fwd: tf32x3 needs a_img_lo next to a_img");
        REQUIRE(!a->out_img || a->out_img_lo, "layer_fwd: tf32x3 needs out_img_lo next to out_img");
        REQUIRE(!a->feat_img, "layer_fwd: feat_img is not available in tf32x3 mode");
    }
    if (a->pts.n_rows <= 0) return 0;
    FwdK K{};
    K.basis = to_basis(a->basis);
    K.pts = to_points(a->pts);
    K.L = to_layer(a->layer, a->drop);
    K.head = to_head(a->head);
    K.a_img = a->a_img;
    K.a_img_lo = a->a_img_lo;
    K.out_img_lo = x3 ? a->out_img_lo : nullptr;
    K.passes = x3 ? 3 : 1;
    K.addend = a->addend;
    K.x_img = a->x_img;
    K.feat_img = a->basis ? a->feat_img : nullptr;
    K.dbg = g_predict_dbg;
    K.out_img = a->out_img;
    K.stats = a->stats;
    K.has_head = a->head ? 1 : 0;
    K.k_slabs = pad32(a->layer.n_in) / SLAB_K;
    K.n_pad = pad32(a->layer.n_out);
    K.thresh16 = dropout_thresh16(a->drop.p);
    K.drop_scale = a->drop.p > 0.0f ? 1.0f / (1.0f - a->drop.p) : 1.0f;
    const bool basis = a->basis != nullptr;
    int tiles = (int)ceil_div64(a->pts.n_rows, TILE_M);
    // few tiles (a training batch): 16 worker warps per CTA hide the latency of the serial phases; many tiles
    // (dense prediction): 8 worker warps and two CTAs per SM so one tile's epilogue overlaps the other's MMAs
    const int sms = g_sm_count > 0 ? g_sm_count : 148;
    const int cg = tiles >= 2 * sms ? 2 : 4;
    // a batch that fits in one wave of 64-row tiles runs on twice the SMs, each walking half the rows.  Both halves of
    // every 128-row image tile get a CTA, so the padding rows of the last tile are written (zeros) as on the 128-row
    // path: wgrad and the knot gradient read whole 128-row tiles.
    const bool half_tiles = 2 * tiles <= sms;
    if (half_tiles) tiles *= 2;
    K.tmem_cols = half_tiles ? tmem_cols_m64(K.n_pad) : pow2_cols(K.n_pad);
    // 1 CTA/SM in the latency configuration: spend the shared memory on pipeline depth (4 stages, else 2)
    const uint32_t smem = fwd_smem(K.n_pad, K.has_head ? K.head.q : 0, basis ? K.basis.k_s : 0, basis ? K.basis.k_t : 0,
                                   basis ? K.k_slabs * 8 : 0, cg);
    REQUIRE(smem <= SMEM_LIMIT, "layer_fwd: needs %u B of shared memory (> 227 KB): too many knots for the dense path",
            smem);
    K.n_tiles = tiles;
#define LAUNCH_FWD(B, TM, C)                                                                                 \
    do {                                                                                                     \
        if (int r = set_smem(layer_fwd_kernel<B, TM, C, (C == 2 ? 2 : 4)>, smem)) return r;                  \
        launch_chained(layer_fwd_kernel<B, TM, C, (C == 2 ? 2 : 4)>, dim3(tiles), n_threads(C), smem, stream, K); \
    } while (0)
    if (basis) {
        if (half_tiles) LAUNCH_FWD(true, 64, 4);
        else if (cg == 2) LAUNCH_FWD(true, 128, 2);
        else LAUNCH_FWD(true, 128, 4);
    } else {
        if (half_tiles) LAUNCH_FWD(false, 64, 4);
        else if (cg == 2) LAUNCH_FWD(false, 128, 2);
        else LAUNCH_FWD(false, 128, 4);
    }
#undef LAUNCH_FWD
    return check_launch("layer_fwd");
}

// Development aid (not part of include/stdadk.h): 16 device counters of cycles the fused prediction kernel's roles spend
// waiting; see tools/prof_predict.py.
extern "C" void stdadk_debug_counters(void* dev_u64x16) { g_predict_dbg = static_cast<unsigned long long*>(dev_u64x16); }
// Phase stamps of the training step (STEP_T, profiling builds): 8 counters per kernel, layer_bwd of layer l at 8 l
// (l < 7), the fused tail at 56.  Launches read the pointer when they are made, so a graph keeps the one it was
// captured with.
static unsigned long long* g_step_dbg = nullptr;
extern "C" void stdadk_debug_step_counters(void* dev_u64x64) { g_step_dbg = static_cast<unsigned long long*>(dev_u64x64); }

// The hidden blocks of the whole-network kernels: each block's n_in must be the previous block's n_out.
static int fill_pred_layers(const stdadk_layer* layers, int n_layers, PredLayerP* out, const char* who) {
    for (int l = 0; l < n_layers; ++l) {
        const stdadk_layer& y = layers[l];
        if (int r = check_layer(y, who)) return r;
        REQUIRE(l == 0 || y.n_in == layers[l - 1].n_out, "%s: block %d n_in=%d != previous n_out=%d", who, l, y.n_in,
                layers[l - 1].n_out);
        PredLayerP& L = out[l];
        L.w_img = y.w_img;
        L.bias = y.bias;
        L.gamma = y.gamma;
        L.beta = y.beta;
        L.n_out = y.n_out;
        L.n_pad = pad32(y.n_out);
        L.k_slabs = pad32(y.n_in) / SLAB_K;
        L.has_ln = y.gamma != nullptr;
        L.eps = y.ln_eps;
    }
    return 0;
}

static int predict_fill(const stdadk_predict_args* a, PredK* K) {
    REQUIRE(a && a->basis && a->head, "predict: NULL args / basis / head");
    REQUIRE(a->n_layers >= 1 && a->n_layers <= PF_MAX_LAYERS, "predict: %d hidden blocks outside [1,%d]", a->n_layers,
            PF_MAX_LAYERS);
    if (int r = check_basis_points(a->basis, a->pts, a->layers[0].n_in)) return r;
    REQUIRE(a->head->q >= 1 && a->head->q <= STDADK_MAX_Q, "predict: head q=%d outside [1,%d]", a->head->q, STDADK_MAX_Q);
    REQUIRE(a->head->w && a->head->b && a->head->yhat, "predict: head w/b/yhat NULL");
    *K = PredK{};
    K->basis = to_basis(a->basis);
    K->pts = to_points(a->pts);
    K->n_layers = a->n_layers;
    K->q = a->head->q;
    K->head_w = a->head->w;
    K->head_b = a->head->b;
    K->yhat = a->head->yhat;
    if (int r = fill_pred_layers(a->layers, a->n_layers, K->L, "predict")) return r;
    uint32_t bytes = plan_predict(*K);
    REQUIRE(bytes <= 227 * 1024, "predict: the fused kernel needs %u B of shared memory (> 227 KB) for this shape", bytes);
    K->n_tiles = (int)ceil_div64(a->pts.n_rows, TILE_M);
    K->dbg = g_predict_dbg;
    return 0;
}

int stdadk_predict_supported(const stdadk_predict_args* a) {
    PredK K;
    return predict_fill(a, &K) == 0 ? 1 : 0;
}

int stdadk_predict(const stdadk_predict_args* a, void* stream) {
    if (int r = check_device()) return r;
    PredK Kl;
    if (int r = predict_fill(a, &Kl)) return r;
    if (a->pts.n_rows <= 0) return 0;
    if (int r = set_smem(predict_fused_kernel, Kl.sm.total)) return r;
    const int sms = g_sm_count > 0 ? g_sm_count : 148;
    const int grid = Kl.n_tiles < sms ? Kl.n_tiles : sms;
    predict_fused_kernel<<<grid, PF_NT, Kl.sm.total, (cudaStream_t)stream>>>(Kl);
    return check_launch("predict");
}

static int field_fill(const stdadk_field_args* a, FieldK* K) {
    REQUIRE(a && a->basis && a->head, "predict_field: NULL args / basis / head");
    REQUIRE(a->n_layers >= 1 && a->n_layers <= PF_MAX_LAYERS, "predict_field: %d hidden blocks outside [1,%d]", a->n_layers,
            PF_MAX_LAYERS);
    const stdadk_basis* b = a->basis;
    REQUIRE(b->p_cov == 0, "predict_field: covariates (p_cov=%d) are per (site, time): use stdadk_predict", b->p_cov);
    REQUIRE(b->k_s >= 1 && b->knots4 && (b->k_t == 0 || b->tknots2), "predict_field: basis tables missing");
    REQUIRE(((reinterpret_cast<uintptr_t>(b->knots4)) & 15) == 0, "predict_field: knots4 must be 16-byte aligned");
    REQUIRE(b->basis_fn >= 0 && b->basis_fn <= 2, "predict_field: unknown basis_fn %d", b->basis_fn);
    REQUIRE(a->layers[0].n_in == b->k_s, "predict_field: layers[0] is the spatial part: n_in=%d != k_s=%d", a->layers[0].n_in,
            b->k_s);
    REQUIRE(a->n_sites >= 1 && a->n_times >= 1, "predict_field: n_sites / n_times");
    REQUIRE(a->sites || (a->grid_nx > 0 && a->grid_ny > 0 && (int64_t)a->grid_nx * a->grid_ny == a->n_sites),
            "predict_field: give sites or a lattice with nx*ny == n_sites");
    REQUIRE(!a->sites || (reinterpret_cast<uintptr_t>(a->sites) & 7) == 0, "predict_field: sites must be 8-byte aligned");
    REQUIRE(0 <= a->k_begin && a->k_begin <= a->k_end && a->k_end <= a->n_times, "predict_field: time range");
    REQUIRE(0 <= a->site_begin && a->site_begin <= a->site_end && a->site_end <= a->n_sites, "predict_field: site range");
    REQUIRE(a->out_k_stride >= 0, "predict_field: out_k_stride");
    REQUIRE(a->head->q >= 1 && a->head->q <= STDADK_MAX_Q && a->head->w && a->head->b && a->head->yhat,
            "predict_field: head q / w / b / yhat");
    REQUIRE(a->w1 && a->zt_ws && (reinterpret_cast<uintptr_t>(a->zt_ws) & 15) == 0, "predict_field: w1 / zt_ws");
    *K = FieldK{};
    K->basis = to_basis(b);
    K->basis.k_t = 0;
    K->basis.tknots = nullptr;
    K->sites = a->sites;
    K->nx = a->grid_nx;
    K->ny = a->grid_ny;
    K->n_sites = a->n_sites;
    K->site_begin = a->site_begin;
    K->site_end = a->site_end;
    K->k_begin = a->k_begin;
    K->k_end = a->k_end;
    K->n_layers = a->n_layers;
    K->q = a->head->q;
    K->head_w = a->head->w;
    K->head_b = a->head->b;
    K->yhat = a->head->yhat;
    K->row_base = a->row_base;
    K->out_k_stride = a->out_k_stride > 0 ? a->out_k_stride : a->n_sites;
    K->zt = a->zt_ws;
    K->dbg = g_predict_dbg;
    if (int r = fill_pred_layers(a->layers, a->n_layers, K->L, "predict_field")) return r;
    REQUIRE(K->L[0].k_slabs <= PF_HSLABS, "predict_field: %d spatial knots exceed the resident operand (%d)", b->k_s,
            PF_HSLABS * SLAB_K);
    uint32_t bytes = plan_field(*K);
    REQUIRE(bytes <= 227 * 1024, "predict_field: the kernel needs %u B of shared memory (> 227 KB) for this shape", bytes);
    // work units: (tile of 128 sites) x (chunk of time steps).  Every unit pays the basis + block-1 GEMM of its tile
    // (about one time step of work), so chunks are as long as the SM count allows: minimise waves * (chunk + 1).
    const int sms = g_sm_count > 0 ? g_sm_count : 148;
    const long long n_s = a->site_end - a->site_begin;
    const int tk = a->k_end - a->k_begin;
    K->n_site_tiles = (int)ceil_div64(n_s, TILE_M);
    int best_chunk = tk > 0 ? tk : 1;
    double best_cost = 1e30;
    for (int chunk = 1; chunk <= tk; ++chunk) {
        const long long units = (long long)K->n_site_tiles * ((tk + chunk - 1) / chunk);
        const double cost = (double)ceil_div64(units, sms) * (chunk + 1.0);
        if (cost < best_cost - 1e-9 || (cost < best_cost + 1e-9 && chunk > best_chunk)) {
            best_cost = cost;
            best_chunk = chunk;
        }
    }
    K->k_chunk = best_chunk;
    K->n_kchunks = tk > 0 ? (tk + best_chunk - 1) / best_chunk : 0;
    const long long units = (long long)K->n_site_tiles * K->n_kchunks;
    REQUIRE(units < (1ll << 31), "predict_field: too many work units");
    K->n_units = (int)units;
    return 0;
}

int stdadk_predict_field_supported(const stdadk_field_args* a) {
    FieldK K;
    return field_fill(a, &K) == 0 ? 1 : 0;
}

int stdadk_predict_field(const stdadk_field_args* a, void* stream) {
    if (int r = check_device()) return r;
    FieldK K;
    if (int r = field_fill(a, &K)) return r;
    if (K.n_units <= 0) return 0;
    const int pad0 = K.L[0].n_pad, total = a->n_times * pad0;
    field_zt_kernel<<<(total + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        a->w1, a->w1_row_stride, a->w1_col_stride, a->basis->k_s, a->layers[0].bias,
        reinterpret_cast<const float2*>(a->basis->tknots2), a->basis->k_t, K.L[0].n_out, pad0, a->n_times, a->zt_ws);
    if (int r = check_launch("predict_field (zt)")) return r;
    if (int r = set_smem(predict_field_kernel, K.sm.total)) return r;
    const int sms = g_sm_count > 0 ? g_sm_count : 148;
    const int grid = K.n_units < sms ? K.n_units : sms;
    predict_field_kernel<<<grid, PF_NT, K.sm.total, (cudaStream_t)stream>>>(K);
    return check_launch("predict_field");
}

int stdadk_layer_bwd(const stdadk_bwd_args* a, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(a, "layer_bwd: NULL args");
    if (int r = check_layer(a->layer, "layer_bwd")) return r;
    REQUIRE(a->x_img || ((a->basis != nullptr) != (a->a_img != nullptr)), "layer_bwd: give exactly one of basis / a_img");
    if (a->basis && !a->x_img)
        if (int r = check_basis_points(a->basis, a->pts, a->layer.n_in)) return r;
    REQUIRE((a->head != nullptr) != (a->dz_next_img != nullptr), "layer_bwd: give exactly one of head / dz_next_img");
    REQUIRE(a->dz_img && a->d_bias, "layer_bwd: dz_img / d_bias NULL");
    REQUIRE(!a->layer.gamma || (a->d_gamma && a->d_beta && a->stats), "layer_bwd: LayerNorm needs d_gamma/d_beta/stats");
    if (a->head) {
        REQUIRE(a->head->q >= 1 && a->head->q <= STDADK_MAX_Q && a->head->w && a->head->dyhat && a->d_head_w &&
                    a->d_head_b,
                "layer_bwd: head arguments incomplete");
    } else {
        REQUIRE(a->wt_next_img && a->n_next >= 1 && a->n_next <= MAX_N, "layer_bwd: wt_next_img / n_next invalid");
    }
    const bool x3 = a->layer.w_img_lo != nullptr;
    if (x3) {
        REQUIRE(a->x_img || !a->a_img || a->a_img_lo, "layer_bwd: tf32x3 needs a_img_lo next to a_img");
        REQUIRE(a->head || (a->dz_next_img_lo && a->wt_next_img_lo), "layer_bwd: tf32x3 needs dz_next_img_lo / wt_next_img_lo");
        REQUIRE(a->dz_img_lo, "layer_bwd: tf32x3 needs dz_img_lo");
    }
    if (a->pts.n_rows <= 0) return 0;
    BwdK K{};
    K.basis = to_basis(a->basis);
    K.pts = to_points(a->pts);
    K.L = to_layer(a->layer, a->drop);
    K.head = to_head(a->head);
    K.a_img = a->a_img;
    K.a_img_lo = a->a_img_lo;
    K.dz_next_img_lo = a->dz_next_img_lo;
    K.wt_next_img_lo = a->wt_next_img_lo;
    K.dz_img_lo = x3 ? a->dz_img_lo : nullptr;
    K.passes = x3 ? 3 : 1;
    K.addend = a->addend;
    K.x_img = a->x_img;
    K.step_settled = a->x_img && (a->settled & STDADK_SETTLED_STEP) ? 1 : 0;   // only the x-image backward reads
    K.x_settled = a->x_img && (a->settled & STDADK_SETTLED_X) ? 1 : 0;         // inputs early
#ifdef STDADK_PF_DEBUG
    K.dbg = g_step_dbg && a->layer.layer_id < 7 ? g_step_dbg + 8 * a->layer.layer_id : nullptr;
#endif
    K.stats = a->stats;
    K.dz_next_img = a->dz_next_img;
    K.wt_next_img = a->wt_next_img;
    K.dz_img = a->dz_img;
    K.d_bias = a->d_bias;
    K.d_gamma = a->d_gamma;
    K.d_beta = a->d_beta;
    K.d_head_w = a->d_head_w;
    K.d_head_b = a->d_head_b;
    K.has_head = a->head ? 1 : 0;
    K.k_slabs = a->x_img ? 0 : pad32(a->layer.n_in) / SLAB_K;      // x saved by the forward: no recomputation GEMM
    K.k_slabs2 = a->head ? 0 : pad32(a->n_next) / SLAB_K;
    K.n_pad = pad32(a->layer.n_out);
    K.thresh16 = dropout_thresh16(a->drop.p);
    K.drop_scale = a->drop.p > 0.0f ? 1.0f / (1.0f - a->drop.p) : 1.0f;
    const bool basis = a->basis != nullptr && a->x_img == nullptr;
    constexpr int BCG = BWD_CG, BNS = BWD_NS;
    const uint32_t smem = bwd_smem(K.n_pad, K.has_head ? K.head.q : 0, basis ? K.basis.k_s : 0, basis ? K.basis.k_t : 0,
                                   basis ? K.k_slabs * 8 : 0);
    REQUIRE(smem <= SMEM_LIMIT, "layer_bwd: needs %u B of shared memory (> 227 KB)", smem);
    int tiles = (int)ceil_div64(a->pts.n_rows, TILE_M);
    // one wave of 64-row tiles (as in layer_fwd), only with x saved by the forward: there is no recompute GEMM then
    const int sms = g_sm_count > 0 ? g_sm_count : 148;
    const bool half_tiles = a->x_img && 2 * tiles <= sms;
    if (half_tiles) tiles *= 2;
    K.tmem_cols = 2 * (half_tiles ? tmem_cols_m64(K.n_pad) : pow2_cols(K.n_pad));
    const bool ln = a->layer.gamma != nullptr, hd = a->head != nullptr;
#define LAUNCH_BWD(B, TM, LNV, HD)                                                                          \
    do {                                                                                                    \
        if (int r = set_smem(layer_bwd_kernel<B, TM, BCG, BNS, LNV, HD>, smem)) return r;                   \
        launch_chained(layer_bwd_kernel<B, TM, BCG, BNS, LNV, HD>, dim3(tiles), n_threads(BCG), smem, stream, K); \
    } while (0)
    if (half_tiles) {
        if (ln && hd) LAUNCH_BWD(false, 64, true, true);
        else if (ln) LAUNCH_BWD(false, 64, true, false);
        else if (hd) LAUNCH_BWD(false, 64, false, true);
        else LAUNCH_BWD(false, 64, false, false);
    } else if (basis) {
        if (ln && hd) LAUNCH_BWD(true, 128, true, true);
        else if (ln) LAUNCH_BWD(true, 128, true, false);
        else if (hd) LAUNCH_BWD(true, 128, false, true);
        else LAUNCH_BWD(true, 128, false, false);
    } else {
        if (ln && hd) LAUNCH_BWD(false, 128, true, true);
        else if (ln) LAUNCH_BWD(false, 128, true, false);
        else if (hd) LAUNCH_BWD(false, 128, false, true);
        else LAUNCH_BWD(false, 128, false, false);
    }
#undef LAUNCH_BWD
    return check_launch("layer_bwd");
}

int stdadk_wgrad(const stdadk_wgrad_args* a, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(a, "wgrad: NULL args");
    REQUIRE((a->basis != nullptr) != (a->a_img != nullptr), "wgrad: give exactly one of basis / a_img");
    REQUIRE(a->dz_img && a->dw, "wgrad: dz_img / dw NULL");
    REQUIRE(a->n_out >= 1 && a->n_out <= MAX_N && a->n_in >= 1, "wgrad: bad sizes n_in=%d n_out=%d", a->n_in, a->n_out);
    if (a->basis)
        if (int r = check_basis_points(a->basis, a->pts, a->n_in)) return r;
    if (a->pts.n_rows <= 0) return 0;
    const bool x3 = a->dz_img_lo != nullptr;
    REQUIRE(!x3 || !a->a_img || a->a_img_lo, "wgrad: tf32x3 needs a_img_lo next to a_img");
    WgradK K{};
    K.basis = to_basis(a->basis);
    K.pts = to_points(a->pts);
    K.a_img = a->a_img;
    K.a_img_lo = a->a_img_lo;
    K.dz_img_lo = a->dz_img_lo;
    K.passes = x3 ? 3 : 1;
    K.dz_img = a->dz_img;
    K.dw = a->dw;
    K.stride_o = a->stride_o;
    K.stride_i = a->stride_i;
    K.n_in = a->n_in;
    K.n_out = a->n_out;
    K.a_slabs = pad32(a->n_in) / SLAB_K;
    K.dz_slabs = pad32(a->n_out) / SLAB_K;
    K.n_row_tiles = (int)ceil_div64(a->pts.n_rows, TILE_M);
    int n_tiles_n = (K.a_slabs + 7) / 8;
    K.nt_slabs = (K.a_slabs + n_tiles_n - 1) / n_tiles_n;
    K.tmem_cols = pow2_cols(K.nt_slabs * SLAB_K);
    int m_tiles = (K.dz_slabs + 3) / 4;
    int per = m_tiles * n_tiles_n;
    int sms = g_sm_count > 0 ? g_sm_count : 148;
    int splits = sms / per;
    if (splits < 1) splits = 1;
    if (splits > K.n_row_tiles) splits = K.n_row_tiles;
    const bool basis = a->basis != nullptr;
    uint32_t smem = wgrad_smem_bytes(basis ? K.basis.k_s : 0, basis ? K.basis.k_t : 0);
    REQUIRE(smem <= SMEM_LIMIT, "wgrad: needs %u B of shared memory (> 227 KB)", smem);
    dim3 grid(splits, m_tiles, n_tiles_n);
    constexpr int WCG = 2;
    if (basis) {
        if (int r = set_smem(wgrad_kernel<true, WCG>, smem)) return r;
        launch_chained(wgrad_kernel<true, WCG>, grid, n_threads(WCG), smem, stream, K);
    } else {
        if (int r = set_smem(wgrad_kernel<false, WCG>, smem)) return r;
        launch_chained(wgrad_kernel<false, WCG>, grid, n_threads(WCG), smem, stream, K);
    }
    return check_launch("wgrad");
}

// The block-1 launches of the dense path: layer_fwd in both CTA configurations (every forward), and with `training`
// also layer_bwd regenerating the basis (batches the forward saves no x for) and the basis-form wgrad.
static int dense_basis_check(int n_in, int n_out, int k_s, int k_t, int q_head, int training) {
    REQUIRE(n_out >= 1 && n_out <= MAX_N && k_s >= 0 && k_t >= 0 && n_in >= k_s + k_t && q_head >= 0 &&
                q_head <= STDADK_MAX_Q,
            "dense_basis_supported: bad sizes n_in=%d n_out=%d k_s=%d k_t=%d q_head=%d", n_in, n_out, k_s, k_t, q_head);
    const int n_pad = pad32(n_out), tab_chunks = pad32(n_in) / SLAB_K * 8;
    for (int cg : {4, 2}) {
        const uint32_t b = fwd_smem(n_pad, q_head, k_s, k_t, tab_chunks, cg);
        REQUIRE(b <= SMEM_LIMIT, "layer_fwd: needs %u B of shared memory (> 227 KB): too many knots for the dense path", b);
    }
    if (!training) return 0;
    const uint32_t bb = bwd_smem(n_pad, q_head, k_s, k_t, tab_chunks);
    REQUIRE(bb <= SMEM_LIMIT, "layer_bwd: needs %u B of shared memory (> 227 KB)", bb);
    const uint32_t wb = wgrad_smem_bytes(k_s, k_t);
    REQUIRE(wb <= SMEM_LIMIT, "wgrad: needs %u B of shared memory (> 227 KB)", wb);
    return 0;
}

int stdadk_dense_basis_supported(int32_t n_in, int32_t n_out, int32_t k_s, int32_t k_t, int32_t q_head, int32_t training) {
    return dense_basis_check(n_in, n_out, k_s, k_t, q_head, training) == 0 ? 1 : 0;
}

int32_t stdadk_dense_max_knots(int32_t p_cov, int32_t k_t, int32_t n_out, int32_t q_head, int32_t training) {
    if (p_cov < 0 || dense_basis_check(p_cov + k_t, n_out, 0, k_t, q_head, training)) return -1;
    // shared memory grows with k_s in every launch: bisect for the last k_s that fits.  Each layer_fwd chunk of 4
    // features takes 64 B of table, so 1 << 14 knots exceed 227 KB in every configuration.
    int lo = 0, hi = 1 << 14;
    while (hi - lo > 1) {
        const int mid = (lo + hi) / 2;
        if (dense_basis_check(p_cov + mid + k_t, n_out, mid, k_t, q_head, training) == 0) lo = mid;
        else hi = mid;
    }
    return lo;
}

int stdadk_knot_grad(const stdadk_knotgrad_args* a, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(a && a->basis && a->dz_img && a->w1s_img && a->d_centers && a->d_log_bw, "knot_grad: NULL argument");
    if (int r = check_basis_points(a->basis, a->pts, -1)) return r;
    REQUIRE(a->n_out >= 1 && a->n_out <= MAX_N, "knot_grad: n_out=%d", a->n_out);
    if (a->pts.n_rows <= 0 || a->basis->k_s == 0) return 0;
    KnotGradK K{};
    K.basis = to_basis(a->basis);
    K.pts = to_points(a->pts);
    REQUIRE((a->dz_img_lo != nullptr) == (a->w1s_img_lo != nullptr), "knot_grad: give both residual images or neither");
    K.dz_img = a->dz_img;
    K.w1s_img = a->w1s_img;
    K.dz_img_lo = a->dz_img_lo;
    K.w1s_img_lo = a->w1s_img_lo;
    K.passes = a->dz_img_lo ? 3 : 1;
    K.d_centers = a->d_centers;
    K.d_log_bw = a->d_log_bw;
    K.n_out = a->n_out;
    K.k_slabs = pad32(a->n_out) / SLAB_K;
    SmemPlan sp = plan_smem(TILE_M, 0, 0, 0, false);
    if (int r = set_smem(knotgrad_kernel<2>, sp.total)) return r;
    dim3 grid((unsigned)ceil_div64(a->pts.n_rows, TILE_M), (unsigned)((a->basis->k_s + TILE_M - 1) / TILE_M));
    knotgrad_kernel<2><<<grid, n_threads(2), sp.total, (cudaStream_t)stream>>>(K);
    return check_launch("knot_grad");
}

static int sparse_fill(const stdadk_sparse_args* a, SparseK* K, bool wgrad) {
    REQUIRE(a, "sparse_l1: NULL args");
    REQUIRE(a->n_levels >= 1 && a->n_levels <= SP_MAX_LEVELS, "sparse_l1: 1..%d lattice levels, got %d", SP_MAX_LEVELS,
            a->n_levels);
    REQUIRE(a->basis_fn == STDADK_WENDLAND || a->basis_fn == STDADK_TRIANGULAR,
            "sparse_l1: only compactly supported bases can be walked (the gaussian basis is dense)");
    REQUIRE(a->n_out >= 4 && a->n_out <= MAX_N && a->n_out % 4 == 0, "sparse_l1: n_out=%d must be a multiple of 4 <= %d",
            a->n_out, MAX_N);
    REQUIRE(a->knots4, "sparse_l1: knots4 is NULL");
    REQUIRE(a->pts.grid_nx > 0 || a->pts.coords != nullptr, "sparse_l1: no point source");
    REQUIRE(a->pts.grid_nx > 0 || (reinterpret_cast<uintptr_t>(a->pts.coords) & 7) == 0, "sparse_l1: coords alignment");
    if (wgrad) {
        REQUIRE(a->dz_img && a->dw1t && (reinterpret_cast<uintptr_t>(a->dw1t) & 15) == 0, "sparse_l1_wgrad: dz_img / dw1t");
    } else {
        REQUIRE(a->w1t && a->zs && (reinterpret_cast<uintptr_t>(a->w1t) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(a->zs) & 15) == 0, "sparse_l1_fwd: w1t / zs NULL or misaligned");
    }
    K->pts = to_points(a->pts);
    K->lat.n_levels = a->n_levels;
    if (a->celllist) {
        REQUIRE((reinterpret_cast<uintptr_t>(a->celllist) & 15) == 0 && a->celllist_k_s >= 1, "sparse_l1: cell list workspace");
        const int* wsi = static_cast<const int*>(a->celllist);
        K->cl.desc = wsi;
        K->cl.starts = wsi + 8 * SP_MAX_LEVELS;
        K->cl.order = K->cl.starts + (size_t)a->n_levels * (CL_GMAX * CL_GMAX + 1) + (size_t)a->n_levels * CL_GMAX * CL_GMAX;
        size_t ib = (celllist_ints(a->celllist_k_s, a->n_levels) * 4 + 15) & ~(size_t)15;
        K->cl.sorted = reinterpret_cast<const float4*>(static_cast<const uint8_t*>(a->celllist) + ib);
        K->cl.n_levels = a->n_levels;
    } else {
        for (int l = 0; l < a->n_levels; ++l) {
            REQUIRE(a->side[l] >= 1 && a->thetap[l] > 0.0f, "sparse_l1: level %d side=%d theta'=%f", l, a->side[l], a->thetap[l]);
            K->lat.side[l] = a->side[l];
            K->lat.offset[l] = a->offset[l];
            K->lat.thetap[l] = a->thetap[l];
        }
    }
    REQUIRE((a->d_centers == nullptr) == (a->d_log_bw == nullptr), "sparse_l1: give d_centers and d_log_bw together");
    REQUIRE(!(wgrad && a->d_centers) || (a->w1t && (reinterpret_cast<uintptr_t>(a->w1t) & 15) == 0),
            "sparse_l1_wgrad: knot gradients need w1t (G = dz1 . W1t row)");
    K->d_centers = wgrad ? a->d_centers : nullptr;
    K->d_log_bw = wgrad ? a->d_log_bw : nullptr;
    K->knots = reinterpret_cast<const float4*>(a->knots4);
    K->w1t = a->w1t;
    K->zs = a->zs;
    K->dz_img = a->dz_img;
    K->dw1t = a->dw1t;
    K->n_out = a->n_out;
    K->p_cov = a->p_cov;
    K->fn = a->basis_fn;
    return 0;
}

static int make_groups(int n_groups, const int64_t* group_end, int64_t n, GroupsP* G) {
    REQUIRE(n_groups >= 1 && n_groups <= 8 && group_end, "optimizer: 1..8 parameter groups supported, got %d", n_groups);
    int64_t prev = 0;
    for (int i = 0; i < n_groups; ++i) {
        REQUIRE(group_end[i] >= prev, "optimizer: group_end must be non-decreasing");
        G->end[i] = prev = group_end[i];
    }
    REQUIRE(prev == n, "optimizer: last group_end (%lld) != n (%lld)", (long long)prev, (long long)n);
    G->n = n_groups;
    return 0;
}

size_t stdadk_celllist_ws_bytes(int32_t k_s, int32_t n_levels) {
    if (k_s < 0 || n_levels < 1 || n_levels > SP_MAX_LEVELS) return 0;
    return celllist_bytes(k_s, n_levels);
}

int stdadk_celllist_build(const float* knots4, int32_t k_s, const int32_t* level_begin, int32_t n_levels, void* ws,
                          size_t ws_bytes, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(knots4 && level_begin && ws && k_s >= 1, "celllist_build: NULL argument / no knots");
    REQUIRE(n_levels >= 1 && n_levels <= SP_MAX_LEVELS, "celllist_build: 1..%d levels, got %d", SP_MAX_LEVELS, n_levels);
    REQUIRE(((reinterpret_cast<uintptr_t>(ws) | reinterpret_cast<uintptr_t>(knots4)) & 15) == 0,
            "celllist_build: knots4 / workspace must be 16-byte aligned");
    REQUIRE(ws_bytes >= celllist_bytes(k_s, n_levels), "celllist_build: workspace of %zu B, need %zu B", ws_bytes,
            celllist_bytes(k_s, n_levels));
    CellBuildK K{};
    K.knots = reinterpret_cast<const float4*>(knots4);
    K.k_s = k_s;
    K.n_levels = n_levels;
    for (int l = 0; l <= n_levels; ++l) {
        REQUIRE(level_begin[l] >= (l ? level_begin[l - 1] : 0) && level_begin[l] <= k_s, "celllist_build: level_begin not monotone");
        K.level_begin[l] = level_begin[l];
    }
    REQUIRE(level_begin[0] == 0 && level_begin[n_levels] == k_s, "celllist_build: levels must cover [0, k_s)");
    K.ws = static_cast<int*>(ws);
    size_t ib = (celllist_ints(k_s, n_levels) * 4 + 15) & ~(size_t)15;
    K.sorted = reinterpret_cast<float4*>(static_cast<uint8_t*>(ws) + ib);
    celllist_build_kernel<<<1, CL_THREADS, 0, (cudaStream_t)stream>>>(K);
    return check_launch("celllist_build");
}

size_t stdadk_sqnorm_ws_floats(void) { return (size_t)SQNORM_BLOCKS * 8 + 8; }

int stdadk_grad_sqnorm(const float* g, int64_t n, int n_groups, const int64_t* group_end, float* sqnorms,
                       float* workspace, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(g && sqnorms && workspace && n > 0, "grad_sqnorm: bad arguments (workspace of stdadk_sqnorm_ws_floats() "
            "zero-initialised floats is required)");
    REQUIRE((reinterpret_cast<uintptr_t>(g) & 15) == 0, "grad_sqnorm: g must be 16-byte aligned");
    GroupsP G{};
    if (int r = make_groups(n_groups, group_end, n, &G)) return r;
    // grid sized by n alone (four 16-byte loads per thread), so the summation order is a function of n: the result is
    // the same on every run and on every data-parallel rank; a 177k-float gradient takes 44 blocks, not 592
    long long blocks = ((n >> 2) + SQNORM_THREADS * 4 - 1) / (SQNORM_THREADS * 4);
    if (blocks < 1) blocks = 1;
    if (blocks > SQNORM_BLOCKS) blocks = SQNORM_BLOCKS;
    sqnorm_kernel<<<(int)blocks, SQNORM_THREADS, 0, (cudaStream_t)stream>>>(g, n, G, sqnorms, workspace);
    return check_launch("grad_sqnorm");
}

int stdadk_sparse_l1_fwd(const stdadk_sparse_args* a, void* stream) {
    if (int r = check_device()) return r;
    SparseK K{};
    if (int r = sparse_fill(a, &K, false)) return r;
    if (a->pts.n_rows <= 0) return 0;
    int blocks = grid_for(a->pts.n_rows, SP_WARPS, 8);
    sparse_spatial_fwd_kernel<<<blocks, SP_WARPS * 32, 0, (cudaStream_t)stream>>>(K);
    return check_launch("sparse_l1_fwd");
}

int stdadk_sparse_l1_wgrad(const stdadk_sparse_args* a, void* stream) {
    if (int r = check_device()) return r;
    SparseK K{};
    if (int r = sparse_fill(a, &K, true)) return r;
    if (a->pts.n_rows <= 0) return 0;
    int blocks = grid_for(a->pts.n_rows, SP_WARPS, 8);
    sparse_spatial_wgrad_kernel<<<blocks, SP_WARPS * 32, 0, (cudaStream_t)stream>>>(K);
    return check_launch("sparse_l1_wgrad");
}

__global__ void step_inc_kernel(int* c) { *c += 1; }

int stdadk_peer_allreduce(const stdadk_peer_allreduce_args* a, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(a && a->g && a->step_count, "peer_allreduce: NULL argument");
    REQUIRE(a->world >= 2 && a->world <= PEER_MAX && a->rank >= 0 && a->rank < a->world,
            "peer_allreduce: world=%d rank=%d outside [2,%d]", a->world, a->rank, PEER_MAX);
    REQUIRE(a->n > 0 && a->n % 4 == 0, "peer_allreduce: n=%lld must be a positive multiple of 4", (long long)a->n);
    static_assert(PEER_MAX == STDADK_MAX_PEERS, "peer limits differ");
    REQUIRE((reinterpret_cast<uintptr_t>(a->g) & 15) == 0, "peer_allreduce: g must be 16-byte aligned");
    PeerK K{};
    for (int r = 0; r < a->world; ++r) {
        REQUIRE(a->recv[r] && (reinterpret_cast<uintptr_t>(a->recv[r]) & 15) == 0,
                "peer_allreduce: rank %d receive area not mapped / not 16-byte aligned", r);
        K.recv[r] = static_cast<uint4*>(a->recv[r]);
    }
    K.g = a->g;
    K.n2 = a->n / 2;
    K.step_count = a->step_count;
    K.rank = a->rank;
    K.world = a->world;
    REQUIRE(a->mode >= 0 && a->mode <= 2, "peer_allreduce: mode=%d (0 automatic, 1 one-shot, 2 two-phase)", a->mode);
    K.two_phase = a->mode == 2 || (a->mode == 0 && a->world >= 4);
    if (a->n_groups > 0) {
        REQUIRE(a->group_end && a->sqnorms && a->workspace, "peer_allreduce: fused norm needs group_end / sqnorms / workspace");
        K.n_norm = a->group_end[a->n_groups - 1];
        REQUIRE(K.n_norm <= a->n, "peer_allreduce: norm range exceeds n");
        if (int r = make_groups(a->n_groups, a->group_end, K.n_norm, &K.G)) return r;
        K.sq_out = a->sqnorms;
        K.ws = a->workspace;
    }
    // grid: a function of n alone (the norm's summation order must not depend on the device), at most one block per SM
    long long blocks = (K.n2 + PEER_THREADS * 2 - 1) / (PEER_THREADS * 2);
    if (blocks > 148) blocks = 148;
    if (blocks < 1) blocks = 1;
    peer_allreduce_kernel<<<(int)blocks, PEER_THREADS, 0, (cudaStream_t)stream>>>(K);
    return check_launch("peer_allreduce");
}

int stdadk_adamw_ema_step(const stdadk_adamw_args* a, void* stream) {
    if (int r = check_device()) return r;
    REQUIRE(a && a->p && a->g && a->m && a->v && a->hyper && a->step_count && a->n > 0, "adamw: bad arguments");
    AdamK K{};
    if (int r = make_groups(a->n_groups, a->group_end, a->n, &K.G)) return r;
    K.p = a->p;
    K.g = a->g;
    K.m = a->m;
    K.v = a->v;
    K.shadow = a->shadow;
    K.n = a->n;
    K.hyper = a->hyper;
    K.sqnorms = a->sqnorms;
    K.step_count = a->step_count;
    K.beta1 = a->beta1;
    K.beta2 = a->beta2;
    K.eps = a->eps;
    K.ema_decay = a->ema_decay;
    K.g_zero = a->zero_grad ? const_cast<float*>(a->g) : nullptr;
    K.state_early = a->fuse_norm && a->state_early ? 1 : 0;
    K.dbg = g_step_dbg ? g_step_dbg + 56 : nullptr;
    K.loss_acc = a->loss_acc;
    K.loss_sum = a->loss_sum;
    K.loss_last = a->loss_last;
    REQUIRE(((reinterpret_cast<uintptr_t>(a->p) | reinterpret_cast<uintptr_t>(a->g) | reinterpret_cast<uintptr_t>(a->m) |
              reinterpret_cast<uintptr_t>(a->v) | reinterpret_cast<uintptr_t>(a->shadow)) & 15) == 0,
            "adamw: buffers must be 16-byte aligned");
    if (a->fuse_norm) {
        REQUIRE(a->norm_ws, "adamw: fuse_norm needs norm_ws");
        K.sq_out = const_cast<float*>(a->sqnorms);
        K.norm_ws = a->norm_ws;
        K.step_rw = a->step_count;
        // every block must be resident for the grid barrier: at most one block per SM; the grid is a function of n only
        long long blocks = ((a->n + 3) / 4 + 255) / 256;
        if (blocks > 148) blocks = 148;
        const int sms = g_sm_count > 0 ? g_sm_count : 148;
        if (blocks > sms) blocks = sms;
        if (blocks < 1) blocks = 1;
        launch_chained(adamw_ema_kernel<true>, dim3((unsigned)blocks), 256, 0, stream, K);
        return check_launch("adamw_ema_step (fused tail)");
    }
    step_inc_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(a->step_count);     // only once every argument check has passed
    adamw_ema_kernel<false><<<grid_for((a->n + 3) / 4, 256, 8), 256, 0, (cudaStream_t)stream>>>(K);
    return check_launch("adamw_ema_step");
}

}  // extern "C"
