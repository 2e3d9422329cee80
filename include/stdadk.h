/* libstdadk.so -- C ABI of the B200-native ST-DADK hot path.
 *
 * The reference (STLABTW/ST-DADK) is pure Python/PyTorch and has no FFI of its own; the boundary it
 * exposes for this path is the nn.Module API.  These entry points are what a binding underneath that
 * API calls; each cites the reference code it replaces (path:line under the upstream repo root).
 * INTEGRATION.md shows the ctypes stub a maintainer would add to stnf/models/st_interp.py.
 *
 * Conventions
 *  - every pointer is a raw DEVICE address owned by the caller (PyTorch); the library allocates no
 *    device memory; work is enqueued on `stream` (a cudaStream_t passed as void*) and returns at once;
 *  - return value: 0 ok, <0 argument error found on the host before launch, >0 cudaError_t of the
 *    launch; the message is available from stdadk_last_error() (thread local);
 *  - no CPU fallback and no other backend: a device that is not sm_100 is an error.
 *
 * Operand images.  Activations and weights that feed the tensor cores live in HBM as "images":
 * tiles of 128 rows x 32 fp32 columns (a 16 KB slab), rows 128 bytes long with their eight 16-byte
 * chunks XOR-swizzled by (row & 7) -- byte for byte the SWIZZLE_128B shared-memory form tcgen05
 * reads, so a slab moves HBM -> SMEM with one bulk copy and the same slab serves as a K-major
 * operand (forward, dgrad) and as an MN-major operand (wgrad).  Matrix (rows x cols) image:
 * [ceil(rows/128)][ceil(cols/32)][128][32] floats; stdadk_image_floats() gives the size.
 */
#ifndef STDADK_H
#define STDADK_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STDADK_VERSION 100
#define STDADK_MAX_Q 8

enum { STDADK_WENDLAND = 0, STDADK_GAUSSIAN = 1, STDADK_TRIANGULAR = 2 };
enum { STDADK_LOSS_NONE = 0, STDADK_LOSS_MSE = 1, STDADK_LOSS_PINBALL = 2 };

/* Basis description.  knots4[j] = (cx, cy, theta'^2, 1/theta'), theta' = bandwidth * calibration
 * (st_interp.py:447-448, CALIBRATION_FACTORS :56-60); tknots2[k] = (c, 1/bw) (st_interp.py:583-596).
 * Feature order of the first Linear layer: [X (p_cov) | phi (k_s) | psi (k_t)] (st_interp.py:843-846).
 * Both tables must be 16-byte aligned (they are staged into shared memory with bulk async copies). */
typedef struct {
    const float* knots4;
    const float* tknots2;
    int32_t k_s, k_t, p_cov, basis_fn;
} stdadk_basis;

/* Point source: arrays (coords (N,2), t (N,1), xcov (N,p) row-major FP32) or, when grid_nx > 0,
 * the dense space-time grid n = (k*nx + i)*ny + j, x=i/(nx-1), y=j/(ny-1), t=k/(nt-1) generated on
 * the device (train_st_interp.py:1233-1248, :1380-1394).  row_begin = first GLOBAL row of this call
 * (index into the arrays / grid, and the dropout key), n_rows = rows processed. */
typedef struct {
    const float* coords;
    const float* t;
    const float* xcov;
    const int64_t* index;   /* optional gather: row r reads sample index[row_begin + r] of the arrays (and of y):
                               a mini-batch is a slice of a device-resident permutation, no collate copy
                               (replaces train_st_interp.py:453-460) */
    int32_t grid_nx, grid_ny, grid_nt, _pad;
    int64_t row_begin;
    int64_t n_rows;
} stdadk_points;

/* One hidden block Linear -> LayerNorm -> ReLU -> Dropout (st_interp.py:659-666). */
typedef struct {
    const float* w_img;  /* image of W (n_out x n_in), K-major forward operand */
    const float* bias;   /* (n_out) */
    const float* gamma;  /* (n_out) LayerNorm weight or NULL when layernorm=False */
    const float* beta;   /* (n_out) */
    int32_t n_in, n_out;
    float ln_eps;
    int32_t layer_id;    /* dropout stream id */
    const float* w_img_lo; /* precision "tf32x3": image of W - tf32(W) (stdadk_pack_desc.part = 1); NULL = plain TF32.
                              With it every GEMM of the call runs three tensor-core passes hi*hi + hi*lo + lo*hi into the
                              same FP32 accumulator (FP32-faithful products; the reference is FP32 throughout,
                              st_interp.py:656-692), and every operand image of the call needs its *_lo twin. */
} stdadk_layer;

typedef struct {
    float p;                  /* 0 => off (eval mode) */
    uint32_t step;            /* stream position; masks are keyed by (seed, step, layer, key_offset + r, column) */
    uint64_t seed;
    const int32_t* step_ptr;  /* if non-NULL the step is read from this DEVICE counter (graph replay) */
    uint64_t key_offset;      /* position of this call's row 0 in the GLOBAL batch: a data-parallel rank passes the
                                 offset of its shard, so masks do not depend on how the batch is split */
} stdadk_dropout;

/* Output head + loss (st_interp.py:689 / :849-877 through an effective (Q x d) matrix;
 * train_st_interp.py:37-50, :620-631).  loss = mean over rows and quantiles; inv_count = 1/(B*Q)
 * with B the GLOBAL batch so that data-parallel ranks sum to the global mean. */
typedef struct {
    const float* w;      /* (q x d) row-major */
    const float* b;      /* (q) */
    int32_t q;
    int32_t loss_type;
    const float* y;      /* (N) targets, NULL for prediction */
    float taus[STDADK_MAX_Q];
    float inv_count;
    float nc_weight;     /* prediction-level non-crossing penalty weight (train_st_interp.py:53-85) */
    int32_t nc_power;
    int32_t _pad;
    float* yhat;         /* (N x q) out */
    float* dyhat;        /* (N x q) out, dLoss/dyhat, NULL for prediction */
    float* loss_acc;     /* (1) += loss contribution of these rows */
} stdadk_head;

/* Forward of one hidden block.  A operand = basis generated in-kernel (basis != NULL; the N x K
 * basis matrix is never written to HBM) or the previous block's activation image (a_img). */
typedef struct {
    const stdadk_basis* basis;
    stdadk_points pts;       /* rows; for a_img mode only row_begin/n_rows are used */
    const float* a_img;
    stdadk_layer layer;
    stdadk_dropout drop;
    float* out_img;          /* image (rows x n_out) of the block output, or NULL */
    float* stats;            /* (rows x 2) LayerNorm mean, rstd for backward, or NULL */
    const stdadk_head* head; /* non-NULL on the last hidden block: fuses head (+ loss) */
    const float* addend;     /* optional (rows x n_out) FP32 row-major term added to A W^T + b before LayerNorm: the
                                support-walked spatial part of block 1 in the large-knot regime (stdadk_sparse_l1_fwd) */
    float* feat_img;         /* optional out, block 1 only: image (rows x n_in) of the generated operand [X|phi|psi] (TF32).
                                Large batches pay the basis evaluation three times per step (forward, the backward's
                                recompute GEMM, wgrad); with this image the other two read it back instead -- pass it as
                                a_img (and basis = NULL) to stdadk_layer_bwd / stdadk_wgrad of block 1. */
    float* x_img;            /* optional out: image (rows x n_out) of the pre-LayerNorm value x = A W^T + b (+ addend),
                                FP32.  A backward that receives it skips the recomputation GEMM -- worth its 1 KB/row
                                when the batch is a single wave of tiles and latency, not bandwidth, is the limit. */
    const float* a_img_lo;   /* tf32x3 (layer.w_img_lo != NULL): residual image of a_img */
    float* out_img_lo;       /* tf32x3: residual image of out_img (written together with it) */
} stdadk_fwd_args;

/* stdadk_bwd_args.settled: the dropout step counter (drop.step_ptr) / the saved x image and its stats */
#define STDADK_SETTLED_STEP 1
#define STDADK_SETTLED_X 2

/* Backward of one hidden block: recomputes z = A W^T (for block 1 this recomputes the basis),
 * forms dh (from the head, or dz_next * W_next on the tensor cores), and writes dz image + bias /
 * LayerNorm / head gradients (accumulated with atomics into zero-initialised buffers). */
typedef struct {
    const stdadk_basis* basis;
    stdadk_points pts;
    const float* a_img;
    stdadk_layer layer;
    stdadk_dropout drop;
    const float* stats;        /* from forward */
    /* upstream gradient: exactly one of (head) or (dz_next_img, wt_next_img) */
    const stdadk_head* head;   /* uses head->dyhat, head->w */
    float* d_head_w;           /* (q x d) += */
    float* d_head_b;           /* (q) += */
    const float* dz_next_img;  /* image (rows x n_next) */
    const float* wt_next_img;  /* image of W_next^T (n_out x n_next): dgrad operand */
    int32_t n_next;
    int32_t settled;           /* STDADK_SETTLED_* bits: inputs that the kernel launched just before this one does not
                                  write, so a one-wave x-image backward may read them while that kernel still runs */
    float* dz_img;             /* out: image (rows x n_out) */
    float* d_bias;             /* (n_out) += */
    float* d_gamma;            /* (n_out) += or NULL */
    float* d_beta;             /* (n_out) += or NULL */
    const float* addend;       /* as in stdadk_fwd_args (the recomputed z needs the same term) */
    const float* x_img;        /* optional: x saved by the forward; then a_img / basis / addend are not read */
    /* tf32x3 (layer.w_img_lo != NULL): residual images of a_img, dz_next_img, wt_next_img and (out) dz_img */
    const float* a_img_lo;
    const float* dz_next_img_lo;
    const float* wt_next_img_lo;
    float* dz_img_lo;
} stdadk_bwd_args;

/* Weight gradient dW (n_out x n_in) += dz^T A, reduction over rows on the tensor cores (both
 * operands MN-major from the same images the forward wrote).  A = a_img or the recomputed basis.
 * dW element (o, i) is accumulated at dw[o*stride_o + i*stride_i]. */
typedef struct {
    const stdadk_basis* basis;
    stdadk_points pts;
    const float* a_img;
    const float* dz_img;
    int32_t n_in, n_out;
    float* dw;
    int64_t stride_o, stride_i;
    const float* a_img_lo;     /* tf32x3: residual images; dz_img_lo != NULL selects the three-pass product */
    const float* dz_img_lo;
} stdadk_wgrad_args;

/* Gradient of the learnable knots (st_interp.py:94-108, closed form of SURVEY.md 9.1):
 * G = dz1 * W1[:, p:p+k_s] on the tensor cores, then d_centers (k_s x 2) and d_log_bw (k_s) +=. */
typedef struct {
    const stdadk_basis* basis;
    stdadk_points pts;
    const float* dz_img;      /* image (rows x n_out) of block-1 dz */
    const float* w1s_img;     /* image of W1[:, p:p+k_s]^T (k_s x n_out) */
    int32_t n_out, _pad;
    float* d_centers;
    float* d_log_bw;
    const float* dz_img_lo;   /* tf32x3: residual images (both or neither) */
    const float* w1s_img_lo;
} stdadk_knotgrad_args;

/* Fused clip + AdamW + EMA over one flat buffer (train_st_interp.py:696-718, torch.optim.AdamW,
 * ema.py:52-66).  Groups are contiguous ranges; hyper[g] = (lr, weight_decay, max_norm, unused) is
 * read from DEVICE memory so a captured graph picks up schedule changes; norms[g] holds the squared
 * L2 norm written by stdadk_grad_sqnorm; step_count (device int) is incremented by the kernel. */
typedef struct {
    float* p;
    const float* g;
    float* m;
    float* v;
    float* shadow;            /* EMA or NULL */
    int64_t n;
    int32_t n_groups;
    int32_t zero_grad;        /* != 0: g is overwritten with zeros once consumed (optimizer.zero_grad() of the next step,
                                 train_st_interp.py:612, without a separate fill launch) */
    const int64_t* group_end; /* host array (n_groups): exclusive end offset of each group */
    const float* hyper;       /* device (n_groups x 4) */
    const float* sqnorms;     /* device (n_groups) or NULL (no clipping) */
    int32_t* step_count;      /* device */
    float beta1, beta2, eps, ema_decay;
    float* loss_acc;          /* optional pair (device scalars): *loss_sum += *loss_acc; *loss_acc = 0 -- the running */
    float* loss_sum;          /* epoch loss of train_st_interp.py:721 kept on the device                              */
    float* loss_last;         /* optional: receives this step's loss (what loss.item() returns upstream, :721)        */
    int32_t fuse_norm;        /* != 0: ONE launch for the whole step tail -- the kernel forms the squared gradient norms
                                 itself (two phases around a grid barrier; bitwise deterministic), writes them to sqnorms
                                 (which then only needs to be non-NULL when clipping is on), and advances step_count */
    int32_t state_early;      /* fuse_norm only, != 0: the kernel launched just before this one writes none of hyper,
                                 step_count, p, m, v, shadow (it may write g), so they are loaded while it still runs
                                 and kept in registers across the grid barrier (n <= 8 x 256 x blocks) */
    float* norm_ws;           /* fuse_norm: (148 * 8 + 8) floats, zero-initialised once */
} stdadk_adamw_args;

int stdadk_version(void);
const char* stdadk_last_error(void);
/* sizeof() of the argument structs, for bindings to verify their layout:
 * 0 basis, 1 points, 2 layer, 3 dropout, 4 head, 5 fwd_args, 6 bwd_args, 7 wgrad_args, 8 knotgrad_args, 9 adamw_args,
 * 10 pack_desc, 11 sparse_args, 12 predict_args, 13 unused (returns 0), 14 peer_allreduce_args, 15 field_args */
size_t stdadk_sizeof(int which);

size_t stdadk_image_floats(int64_t rows, int64_t cols);

/* theta' = bw*calib (or exp(log_bw)*calib when log_bw != NULL) -> knots4 (st_interp.py:144-150, :447-448) */
int stdadk_knots_prepare(const float* centers, const float* bw, const float* log_bw, float calib, int k,
                         float* knots4, void* stream);
int stdadk_tknots_prepare(const float* centers, const float* bw, int k, float* tknots2, void* stream);

/* Unfused basis for parity checks: phi (N x k_s), psi (N x k_t) dense FP32 (st_interp.py:433-491, :583-596) */
int stdadk_basis_fwd(const stdadk_basis* basis, const stdadk_points* pts, float* phi, float* psi, void* stream);

/* Row-major (strided) matrix -> image with TF32 rounding, and back (testing) */
int stdadk_pack_image(const float* src, int64_t row_stride, int64_t col_stride, int64_t rows, int64_t cols,
                      float* img, void* stream);
int stdadk_unpack_image(const float* img, int64_t rows, int64_t cols, float* dst, void* stream);
/* Several matrices -> images in ONE launch (a training step repacks every weight matrix and its transpose) */
#define STDADK_MAX_PACK 8
typedef struct {
    const float* src;
    int64_t row_stride, col_stride, rows, cols;
    float* img;
    int32_t part;             /* 0: tf32(src) (the operand image); 1: tf32(src - tf32(src)), the tf32x3 residual image */
    int32_t _pad;
} stdadk_pack_desc;
int stdadk_pack_images(const stdadk_pack_desc* descs, int n, void* stream);

/* Large-knot regime of block 1 (K_s up to ~1e5+; BASELINE config 4): walk only the knots in each point's compact
 * support.
 *   fwd  : zs[n,:]  = sum_{j in supp(s_n)} phi_j(s_n) * w1t[p_cov + j, :]
 *   wgrad: dw1t[p_cov + j, :] += phi_j(s_n) * dz1[n,:]; with d_centers / d_log_bw also the knot gradients
 *          (st_interp.py:94-108, closed form of SURVEY.md 9.1)
 * w1t / dw1t: first Linear layer stored knot-major, (n_in x n_out) contiguous.
 * Candidate knots per level: the fixed uniform lattice (knot j of level l at node (j / side, j % side),
 * st_interp.py:152-185) is walked in closed form; ANY other knot set (gmm / random_site / kmeans_balanced placement,
 * learnable knots: st_interp.py:187-431) goes through a cell list built on the device by stdadk_celllist_build
 * (per level: cells of edge >= the level's largest theta', knots counting-sorted by cell; rebuilt every step when the
 * knots move).  No limit on the number of knots inside a support. */
size_t stdadk_celllist_ws_bytes(int32_t k_s, int32_t n_levels);
/* level_begin: HOST array of n_levels + 1 knot offsets (levels are contiguous knot ranges); ws: device workspace of
 * stdadk_celllist_ws_bytes() bytes, 16-byte aligned */
int stdadk_celllist_build(const float* knots4, int32_t k_s, const int32_t* level_begin, int32_t n_levels, void* ws,
                          size_t ws_bytes, void* stream);
#define STDADK_MAX_LEVELS 8
typedef struct {
    stdadk_points pts;
    const float* knots4;      /* as in stdadk_basis */
    int32_t n_levels, basis_fn, n_out, p_cov;
    int32_t side[STDADK_MAX_LEVELS];
    int32_t offset[STDADK_MAX_LEVELS];   /* index of the level's first knot */
    float thetap[STDADK_MAX_LEVELS];     /* bandwidth * calibration of the level */
    const float* w1t;
    float* zs;                /* fwd out (rows x n_out) */
    const float* dz_img;      /* wgrad in: image (rows x n_out) */
    float* dw1t;              /* wgrad out, += */
    const void* celllist;     /* workspace filled by stdadk_celllist_build for these knots (then side/offset/thetap are
                                 not read; n_levels and celllist_k_s must be the values it was built with), or NULL */
    int32_t celllist_k_s, _pad;
    float* d_centers;         /* wgrad, learnable knots: (k_s x 2) +=, or NULL */
    float* d_log_bw;          /* (k_s) += */
} stdadk_sparse_args;
int stdadk_sparse_l1_fwd(const stdadk_sparse_args* a, void* stream);
int stdadk_sparse_l1_wgrad(const stdadk_sparse_args* a, void* stream);

/* Whole-network forward for prediction (evaluate_model / plot_spatial_mse / plot_temporal_series,
 * train_st_interp.py:884-961, :1233-1248, :1380-1394; STInterpMLP.forward in eval mode, st_interp.py:827-882):
 * basis -> hidden blocks -> head in ONE persistent kernel; activations stay in shared / tensor memory, the only
 * per-point HBM traffic is the point (12 B, or 0 for a generated grid) and y_hat (4Q B).  Dropout is the identity.
 * Limits: 1..STDADK_MAX_HIDDEN hidden blocks of width <= 256, dense basis (all knots resident in shared memory);
 * stdadk_predict_supported() tells whether a shape fits, otherwise chain stdadk_layer_fwd calls. */
#define STDADK_MAX_HIDDEN 4
typedef struct {
    const stdadk_basis* basis;
    stdadk_points pts;
    int32_t n_layers, _pad;
    stdadk_layer layers[STDADK_MAX_HIDDEN];   /* layers[l].w_img = image of W_l; layers[0].n_in = p + k_s + k_t */
    const stdadk_head* head;                  /* w, b, q, yhat are used */
} stdadk_predict_args;
int stdadk_predict_supported(const stdadk_predict_args* a);   /* 1 yes, 0 no (reason in stdadk_last_error) */
int stdadk_predict(const stdadk_predict_args* a, void* stream);

/* Space-time FIELD prediction: every site of a set (explicit sites, or the lattice grid_nx x grid_ny with site = i*ny + j)
 * at the time steps k_begin .. k_end-1 of an n_times-step axis, t_k = k/(n_times-1) -- the T x S field of upstream's
 * plot_spatial_mse loop (train_st_interp.py:1233-1248), plot_temporal_series (:1380-1394) and the dense grid of
 * stdadk_points.  Same function as stdadk_predict on those points; the kernel exploits that the first Linear layer
 * separates, W1 [phi(s) | psi(t)] + b1 = zs(s) + zt(t): a CTA evaluates the basis and block 1 once per tile of 128
 * sites and loops over the time steps.  Needs p_cov == 0 and the limits of stdadk_predict.
 *   layers[0].w_img : image of W1[:, 0:k_s] (n_1 x k_s), the spatial columns only; layers[0].n_in = k_s
 *   w1 / strides    : W1 itself (n_1 x (k_s + k_t)), read for the temporal columns
 *   yhat row of point (k, s) = k * n_sites + s - row_base     (the caller's shard of the (t, s) row-major field)
 *   zt_ws           : workspace of n_times * pad32(n_1) floats */
typedef struct {
    const stdadk_basis* basis;
    const float* sites;
    int32_t grid_nx, grid_ny;
    int64_t n_sites;
    int32_t n_times, k_begin, k_end, n_layers;
    int64_t site_begin, site_end;
    stdadk_layer layers[STDADK_MAX_HIDDEN];
    const float* w1;
    int64_t w1_row_stride, w1_col_stride;
    const stdadk_head* head;
    int64_t row_base;
    float* zt_ws;
    int64_t out_k_stride;     /* rows of yhat between consecutive time steps: point (k, site) is written to row
                                 k * out_k_stride + site - row_base.  0 = n_sites (the (t, s) row-major field).  A site-sharded
                                 rank passes its own site count and row_base = site_begin: a dense (n_times, sites) block */
} stdadk_field_args;
int stdadk_predict_field_supported(const stdadk_field_args* a);   /* 1 yes, 0 no (reason in stdadk_last_error) */
int stdadk_predict_field(const stdadk_field_args* a, void* stream);

int stdadk_layer_fwd(const stdadk_fwd_args* a, void* stream);
int stdadk_layer_bwd(const stdadk_bwd_args* a, void* stream);
int stdadk_wgrad(const stdadk_wgrad_args* a, void* stream);

/* Whether block 1 can generate its basis densely in shared memory: the block-1 launches fit in 227 KB, by the same
 * shared-memory plans the launchers check.  training = 0: the forward only (stdadk_layer_fwd in both CTA
 * configurations), what a prediction runs; training = 1: also stdadk_layer_bwd regenerating the basis and stdadk_wgrad
 * in basis form, every launch a training step can make.  n_in = p_cov + k_s + k_t inputs, n_out outputs; q_head = Q
 * when block 1 is also the last hidden block (it carries the head), else 0.  Host-only: no device is needed.  1 yes,
 * 0 no (the launch that does not fit in stdadk_last_error). */
int stdadk_dense_basis_supported(int32_t n_in, int32_t n_out, int32_t k_s, int32_t k_t, int32_t q_head, int32_t training);
/* Largest k_s for which stdadk_dense_basis_supported(p_cov + k_s + k_t, n_out, k_s, k_t, q_head, training) holds, -1 if
 * none. */
int32_t stdadk_dense_max_knots(int32_t p_cov, int32_t k_t, int32_t n_out, int32_t q_head, int32_t training);
int stdadk_knot_grad(const stdadk_knotgrad_args* a, void* stream);

/* sqnorms[g] = sum of squares of g over each group.  Bitwise deterministic (replicas of a data-parallel run must
 * compute the same clip coefficient).  workspace: stdadk_sqnorm_ws_floats() floats, zeroed once by the caller. */
size_t stdadk_sqnorm_ws_floats(void);
int stdadk_grad_sqnorm(const float* g, int64_t n, int n_groups, const int64_t* group_end, float* sqnorms,
                       float* workspace, void* stream);
int stdadk_adamw_ema_step(const stdadk_adamw_args* a, void* stream);

/* Data-parallel training (SURVEY.md section 8e: one sum of the flat gradient per step; upstream itself is single
 * device): one-shot all-reduce over NVLink peer memory, low-latency protocol (every 8-byte packet carries its own epoch
 * flag), result IN PLACE in g, optionally fused with the gradient norm of stdadk_grad_sqnorm.
 *   recv[p]  rank p's receive area as mapped into THIS process (CUDA VMM / symmetric memory, own rank included):
 *            2 * world * (n / 2) packets of 16 bytes, zero-initialised once before the first call
 *   n        floats, a multiple of 4; g 16-byte aligned
 *   step_count  device counter, equal on all ranks, must grow by exactly one between calls (the AdamW step counter)
 *   n_groups > 0: sqnorms[k] = sum of squares of the REDUCED g[0 : n_norm) over group k (bitwise deterministic);
 *            workspace = (148 * 8 + 8) zero-initialised floats */
#define STDADK_MAX_PEERS 8
typedef struct {
    int32_t world, rank;
    float* g;
    int64_t n;
    void* recv[STDADK_MAX_PEERS];
    const int32_t* step_count;
    int32_t n_groups;
    int32_t mode;               /* 0 = automatic, 1 = one-shot (every rank pushes everything to every peer, one NVLink
                                   traversal), 2 = two-phase (chunk owners reduce and publish: ~4x fewer bytes at 8 ranks,
                                   two traversals; automatic choice from 4 ranks on).  Same bits either way. */
    const int64_t* group_end;   /* host array (n_groups), last entry = n_norm */
    float* sqnorms;
    float* workspace;
} stdadk_peer_allreduce_args;
int stdadk_peer_allreduce(const stdadk_peer_allreduce_args* a, void* stream);

#ifdef __cplusplus
}
#endif
#endif
