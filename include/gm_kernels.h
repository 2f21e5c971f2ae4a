/*
 * gm_kernels.h -- C-ABI of libgm_b200.so: the B200 (sm_100a) kernels behind the
 * graphembed training hot path (pair distance + gradient, distortion loss,
 * Riemannian optimizer step, BFS graph-distance targets).
 *
 * The reference (dalab/matrix-manifolds, `graphembed`) has no FFI: its "plugin
 * API" for this path is the Python Manifold / optimizer interface.  Every entry
 * point below therefore cites the reference *Python* function(s) it replaces
 * (paths relative to /root/reference/graphembed/).  The Python drop-in package
 * (matrix-manifolds_b200/graphembed) binds these with ctypes; INTEGRATION.md
 * shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers unless
 *     the name ends in `_host`; `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, a negative GM_E* code for bad
 *     arguments (nothing launched) or a positive cudaError_t from the launch.
 *   - kernels never allocate; outputs/workspaces are caller-owned.
 *   - dtype selects the arithmetic AND storage type of all `void*` real arrays.
 *   - re-entrant: no global mutable state; uses the caller's current device.
 */
#ifndef GM_KERNELS_H
#define GM_KERNELS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gm_stream_t; /* cudaStream_t */

/* ---- error codes -------------------------------------------------------- */
#define GM_OK 0
#define GM_EINVAL (-1)       /* bad argument combination            */
#define GM_EUNSUPPORTED (-2) /* (kind, n, p, dtype) not instantiated */
#define GM_ENULL (-3)        /* required pointer is NULL            */

/* ---- enums -------------------------------------------------------------- */
enum gm_dtype { GM_F32 = 0, GM_F64 = 1 };

enum gm_manifold_kind {
  GM_SPD_AI = 0,    /* manifolds/spd.py:171-181  affine-invariant squared distance        */
  GM_SPD_STEIN = 1, /* manifolds/spd.py:183-194,246-295  symmetric Stein divergence         */
  GM_LORENTZ = 2,   /* manifolds/lorentz.py:72-77                                          */
  GM_SPHERE = 3,    /* manifolds/sphere.py:68-74                                           */
  GM_GRASSMANN = 4, /* manifolds/grassmann.py:91-96                                        */
  GM_EUCLIDEAN = 5, /* manifolds/euclidean.py:46-50 via base.py:56-57                      */
  GM_UNIVERSAL = 6  /* manifolds/universal.py:76-81 + manifolds/impl/math.py:567-572: kappa-stereographic model
                       (c > 0: Poincare ball of curvature -c, c < 0: stereographic sphere), learnable c       */
};

/* gm_manifold_t.flags */
#define GM_FAST_EIG 1u  /* SPD n=2,3: closed-form eigenvalues with the reference's eps terms (linalg/fast.py:53-91)   */
#define GM_FAST_CHOL 2u /* SPD n=2: closed-form (inverse) Cholesky with eps terms (linalg/fast.py:94-134)             */
#define GM_FAST_SVD 4u  /* Grassmann p=2: closed-form singular values (linalg/fast.py:138-159)                         */

typedef struct gm_manifold {
  int32_t kind;  /* gm_manifold_kind */
  int32_t dtype; /* gm_dtype */
  int32_t n;     /* SPD: matrix size; Lorentz: ambient dim; Sphere/Euclidean: #elements per point; Grassmann: rows */
  int32_t p;     /* Grassmann: columns; otherwise 0 */
  uint32_t flags;
  int32_t reserved;
  double wmin; /* SPD eigenvalue / distance clamp (spd.py:28-29), default 1e-8 */
  double wmax; /* default 1e8 */
  /* GM_UNIVERSAL only (ignored otherwise; zero-initialise).  The curvature parameter is read ON THE DEVICE so that a
   * curvature optimizer can update it between steps without a host round trip (universal.py:28-32 get_c()). */
  const void* c_dev; /* DEVICE pointer to one scalar of `dtype`: c = Universal.get_c(), must be non-zero          */
  double* c_grad;    /* optional DEVICE double: gm_pairs_grad / gm_pairs_loss_fused add sum_k w_k d(d2_k)/dc to it
                        (w_k = the per-pair weight the point gradients are scaled with); NULL: not wanted        */
} gm_manifold_t;

/* How the P pairs of one launch are enumerated. */
enum gm_pairs_mode {
  GM_PAIRS_ELEMENTWISE = 0, /* pair k = (xa[k], xb[k])                       -- Manifold.dist(x, y)  (base.py:56-57)        */
  GM_PAIRS_LIST = 1,        /* pair k = (xa[idx_i[k]], xb[idx_j[k]])         -- dist(x[I], x[J]) incl. the gather           */
  GM_PAIRS_TRIU = 2,        /* pair k = (k0+k)-th (a<b) of triu_indices(B,B,1), rows
                               xa[nodes[a]], xb[nodes[b]] (nodes NULL: a, b) -- Manifold.pdist (base.py:59-63) fused with
                                                                                x[indices] (modules.py:84-88)              */
  GM_PAIRS_SAMPLED = 3      /* pairs DRAWN ON THE DEVICE (new capability: BASELINE config 5 "sampled pairs"; the reference
                               only enumerates all pairs of a node batch, train.py:206-213).  Pair k belongs to source
                               group g = k / per_src:  i = idx_i[g] (int32 node id of the BFS source),
                               j = the gm_sample_j(seed, k, i, n_nodes)-th node != i (counter-based: the same (seed, k)
                               always gives the same j, on any grid -- oracle/sampler_oracle.py is the host statement),
                               hop = levels[slot_g * n_nodes + j] with slot_g = slots ? slots[g] : g.
                               The kernels see the pair as the packed word (hop << 24) | j, i.e. exactly a LIST pair with
                               GM_TGT_HOPS_PACKED targets, but nothing per pair is uploaded or read from memory: a step
                               uploads the G source ids.  Needs n_nodes < 2^24, hop counts < 255 (uint8 levels).      */
};

typedef struct gm_pairs {
  int32_t mode;      /* gm_pairs_mode */
  int32_t idx64;     /* 1: idx_i/idx_j/nodes are int64, 0: int32 */
  int64_t P;         /* number of pairs (TRIU: k0 + P <= B(B-1)/2) */
  const void* idx_i; /* LIST */
  const void* idx_j; /* LIST */
  int64_t B;         /* TRIU */
  const void* nodes; /* TRIU, optional */
  int64_t k0;        /* TRIU: first pair of the triangle covered by this launch (0 for the whole triangle); per-pair
                        vectors (out_d2, gout, VECTOR / HOPS targets) are indexed by the LOCAL pair number 0..P-1.
                        A rank of a pair-sharded job passes its slice [k0, k0+P) (SURVEY 8e) */
  /* GM_PAIRS_SAMPLED only (zero otherwise) */
  const void* levels; /* uint8 (S, n_nodes) hop counts from gm_bfs_multi_source, resident on the device */
  const void* slots;  /* int32 (G): row of `levels` that belongs to group g; NULL: row g                */
  int64_t n_nodes;    /* rows of the point table == columns of `levels`                                 */
  int64_t per_src;    /* targets drawn per source; G = ceil(P / per_src)                                */
  uint64_t seed;      /* stream id of this step's draws (the caller mixes its seed with the step number) */
  /* GM_PAIRS_LIST, optional locality hint (0 or 1: none).  The list is `segments` consecutive parts of
   * ceil(P / segments) pairs (the last may be shorter) and the training kernels walk the parts one after another with
   * the whole grid instead of giving every warp one contiguous range of the list.  A sampler that orders a batch by
   * (window of the target row, source) -- segment s holding the pairs whose target lies in rows
   * [s N / segments, (s+1) N / segments) -- thereby keeps the gradient rows and point rows the grid is scattering into
   * and gathering from inside a window that fits the L2 cache; the result is the same sum over the same pairs (only the
   * order of the floating-point reductions changes, as it does from launch to launch anyway). */
  int32_t segments;
  int32_t reserved;
} gm_pairs_t;

/* The draw of GM_PAIRS_SAMPLED, stated once so that host code can reproduce a step's pairs bit for bit:
 *   z = seed + (k + 1) * 0x9E3779B97F4A7C15;  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9;
 *   z = (z ^ (z >> 27)) * 0x94D049BB133111EB;  z ^= z >> 31;          (the splitmix64 output function, mod 2^64)
 *   r = z >> 32;  j = (r * (n_nodes - 1)) >> 32;  if (j >= i) j += 1;  (uniform over the n_nodes - 1 nodes != i)      */

/* Loss on (graph target g, manifold squared distance m) -- objectives.py:16-45. */
enum gm_loss_kind { GM_LOSS_QUOTIENT = 0, GM_LOSS_STRESS = 1 };
typedef struct gm_loss {
  int32_t kind;
  int32_t inc_l1; /* QuotientLoss(inc_l1) : sum |m/(alpha g) - 1|            */
  int32_t inc_l2; /* QuotientLoss(inc_l2) : sum |alpha g/(m+eps) - 1|        */
  int32_t reserved;
  double alpha; /* objectives.py:25 (Stress ignores it)                    */
  double eps;   /* 1/(epoch+1), objectives.py:30                           */
} gm_loss_t;

/* Where the per-pair target g comes from. */
enum gm_target_mode {
  GM_TGT_VECTOR = 0, /* data[k], same dtype as the manifold -- GraphDataset.__getitem__ result (data/dataset.py:19-27) */
  GM_TGT_DENSE = 1,  /* data[u*ld + v], u,v = node ids of the pair -- GraphDataset.pdists, fuses the double gather +
                        masked_select of data/dataset.py:23-27 (LIST/TRIU modes only)                               */
  GM_TGT_HOPS_U8 = 2, /* uint8 BFS hop count h per pair; g = (h*h)/max_sq computed in the manifold dtype exactly as
                        data/dataset.py:11-12 does (pow(2) then div_(max))                                           */
  GM_TGT_HOPS_U16 = 3,
  GM_TGT_HOPS_PACKED = 4 /* LIST pairs with int32 indices only: the hop count rides in the top 8 bits of idx_j[k]
                            (row = idx_j[k] & 0xFFFFFF, h = idx_j[k] >> 24; needs < 2^24 rows); `data` is ignored.
                            One 4-byte word per pair instead of 5 bytes to upload and read (gm_pairs_loss_fused only).
                            Also the target mode of GM_PAIRS_SAMPLED pairs, whose packed word is computed on the fly */
};
typedef struct gm_targets {
  int32_t mode;
  int32_t reserved;
  const void* data;
  int64_t ld;    /* DENSE: row stride in elements */
  double max_sq; /* HOPS: max over the graph of h*h */
} gm_targets_t;

/* ---- pair kernels -------------------------------------------------------- */

/* out_d2[k] = squared manifold distance (Stein: divergence) of pair k, with the reference's value-only clamps.
 * Replaces Manifold.dist/pdist(..., squared=True): spd.py:171-194, lorentz.py:72-77, sphere.py:68-74,
 * grassmann.py:91-96, base.py:56-63 and the linalg they call (linalg/torch_batch.py, linalg/fast.py). */
int gm_pairs_dist2(const gm_manifold_t* man, const void* xa, const void* xb, const gm_pairs_t* pairs,
                   void* out_d2, gm_stream_t stream);

/* Backward of gm_pairs_dist2: for every pair k adds coef*gout[k]*d(d2_k)/d(x) to the rows of ga / gb the pair
 * touches (ELEMENTWISE: plain stores to row k; LIST/TRIU: atomic accumulation into row idx -- the fused
 * index_put_(accumulate=True) of autograd, SURVEY 8a A11).  ga/gb may alias.  SPD gradients are symmetric
 * (what egrad2rgrad's sym() keeps, spd.py:134-135).  Straight-through clamps as in the reference. */
int gm_pairs_grad(const gm_manifold_t* man, const void* xa, const void* xb, const gm_pairs_t* pairs,
                  const void* gout, double coef, void* ga, void* gb, gm_stream_t stream);

/* Single-factor fused hot path: distance, loss term and gradient in one pass.
 *   m_k = scale_sp * d2_k;  loss += l(g_k, m_k);  grad[rows] += l'(g_k, m_k) * scale_sp * d(d2_k)/dx
 *   acc[0] += sum_k l(g_k, m_k)          (double)
 *   acc[1] += sum_k l'(g_k, m_k) * d2_k  (double; times sigmoid(scale) it is d loss / d scale, modules.py:84-88)
 * out_d2 (optional, may be NULL) receives d2_k.  x is the (N, ...) parameter, grad the (N, ...) gradient to accumulate
 * into (caller zeroes it).  Replaces BatchedObjective.forward + loss.backward() for one factor
 * (modules.py:84-105, objectives.py:16-45, train.py:213-216). */
int gm_pairs_loss_fused(const gm_manifold_t* man, const void* x, const gm_pairs_t* pairs,
                        const gm_targets_t* targets, const gm_loss_t* loss, double scale_sp, void* out_d2,
                        double* acc, void* grad, gm_stream_t stream);

/* Product-manifold loss over F factor distance vectors (modules.py:84-88 + objectives.py):
 *   m_k = sum_f sp[f]*d2[f][k];  acc[0] += sum_k l(g_k, m_k);  acc[1+f] += sum_k l'_k * d2[f][k];  out_g[k] = l'_k.
 * d2_ptrs_host / sp_host are HOST arrays of length F (F <= 8).  `pairs` (LIST / TRIU, pairs->P == P) is needed only
 * for DENSE targets, whose matrix is indexed by the pair's node ids -- the fused form of
 * GraphDataset.__getitem__ (data/dataset.py:19-27); pass NULL otherwise. */
int gm_product_loss(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                    const gm_pairs_t* pairs, const gm_targets_t* targets, const gm_loss_t* loss, int64_t P, double* acc,
                    void* out_g, gm_stream_t stream);

/* Fused pair kernel of a PRODUCT manifold (modules.py:84-105 with F factors + objectives.py:16-45 + loss.backward()):
 * ONE launch evaluates every factor's d2 of a pair, m_k = sum_f sp[f] * d2_f[k] (left to right, as Python's sum() over the
 * factor list), the loss of m_k against the pair's target, and adds every factor's gradient into grad[f]:
 *   acc[0] += sum_k l(g_k, m_k);   acc[1+f] += sum_k l'_k * d2_f[k];   grad[f][i_k], grad[f][j_k] += l'_k sp[f] d(d2_f)/d(x, y).
 * Host arrays of length F: mans, x, grad, sp.  Pairs / targets as gm_pairs_loss_fused (LIST / TRIU / SAMPLED; every
 * target mode).  Supported products: at most one SPD factor (either divergence) and up to three of Lorentz / Sphere /
 * Euclidean, 2 <= F <= 4, one dtype; anything else returns GM_EUNSUPPORTED and the caller keeps the unfused sequence
 * gm_pairs_dist2 x F -> gm_product_loss -> gm_pairs_grad x F.  gm_train_epoch_product uses it when it can. */
int gm_pairs_product_fused(int32_t F, const gm_manifold_t* mans, void* const* x, const gm_pairs_t* pairs,
                           const gm_targets_t* targets, const gm_loss_t* loss, const double* sp, double* acc,
                           void* const* grad, gm_stream_t stream);

/* Validation metrics over a pair set, streamed (TrainingEngine._validate, train.py:230-265; metrics.average_distortion
 * and metrics.pearsonr, metrics.py:13-17,46-56) without materialising the N(N-1)/2 distance vectors:
 *   squared_inputs != 0:  m_k = sqrt(sum_f sp[f]*d2[f][k]),  g_k = sqrt(target_k)   (train.py:231-232)
 *   squared_inputs == 0:  m_k = d2[0][k] (F must be 1),      g_k = target_k         (plain metrics.py call)
 *   acc[0] += #pairs           acc[1] += sum |m-g|/g     acc[2] += sum m     acc[3] += sum g
 *   acc[4] += sum m*m          acc[5] += sum g*g         acc[6] += sum m*g   (all double; acc has 8 slots)
 * d2[f] are per-pair vectors of this launch (local index); targets may be VECTOR / DENSE / HOPS_*; `pairs` gives the
 * node ids for DENSE targets (may be NULL otherwise; pairs->P is the number of pairs). */
int gm_pairs_metrics(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                     const gm_pairs_t* pairs, const gm_targets_t* targets, int32_t squared_inputs, double* acc,
                     gm_stream_t stream);

/* KL-divergence objective with the stochastic-neighbour inference model (objectives.py:48-76,
 * inference/stochastic_neighbors.py:8-24) over ALL pairs of a batch of B nodes, condensed triu order.
 *   m_k = sum_f sp[f]*d2[f][k];  inclusive: theta_x = -alpha*g, theta_z = -m;  else theta_x = -m, theta_z = -alpha*g
 *   KL = A_z - A_x - margs_x . (theta_z - theta_x),  A = sum_rows logsumexp_{j != i} theta_ij
 * gm_sne_row_stats: one pass per row i over its B-1 entries (online softmax):
 *   row_stats[0*B+i] = logsumexp theta_x row i;  row_stats[1*B+i] = logsumexp theta_z row i;
 *   row_stats[2*B+i] = E_{p_x(i,.)}[theta_z - theta_x]
 * gm_sne_pair_terms: acc[0] += KL, out_g[k] = dKL/dm_k, acc[1+f] += sum_k out_g[k]*d2[f][k] (scale gradients).
 * g is a VECTOR target (condensed, dtype of the manifold).  row_stats: 3*B elements of `dtype`. */
int gm_sne_row_stats(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                     const void* g, int64_t B, double alpha, int32_t inclusive, void* row_stats, gm_stream_t stream);
int gm_sne_pair_terms(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                      const void* g, int64_t B, double alpha, int32_t inclusive, const void* row_stats, double* acc,
                      void* out_g, gm_stream_t stream);

/* ---- optimizer ---------------------------------------------------------- */
enum gm_optim_kind { GM_OPT_RSGD = 0, GM_OPT_RADAM = 1 };
typedef struct gm_optim {
  int32_t kind;
  int32_t exact;      /* 1: manifold.exp, 0: manifold.retr (radam.py:66, rsgd.py:60)              */
  int32_t has_clip;   /* max_grad_norm is not None                                                 */
  int32_t step;       /* RAdam: state['step'] BEFORE the update (starts at 1, radam.py:56)          */
  int32_t has_momentum; /* RSGD: momentum > 0                                                      */
  int32_t first_step; /* RSGD+momentum: buffer is initialised to the Euclidean grad (rsgd.py:53-54) */
  int32_t grassmann_retr_qr; /* Grassmann(retr='qr')                                               */
  int32_t zero_grad;  /* gm_optim_step only: 1 = overwrite every gradient row with zeros once it has been read, i.e.
                         fold the next step's `zero_grad()` (train.py:214) into this kernel -- saves one full pass
                         over the gradient table per step; `grad` must then be writable.  0: grad is left untouched */
  double lr, beta1, beta2, momentum, dampening, max_grad_norm, eps;
} gm_optim_t;

/* One fused in-place optimizer update over all N points (optim/radam.py:43-98, optim/rsgd.py:40-82 and the
 * manifold callees egrad2rgrad / norm / exp|retr / transp of SURVEY 8a A14-A16).
 *   RAdam: buf1 = exp_avg, buf2 = exp_avg_sq (both full parameter shape).  RSGD: buf1 = momentum buffer or NULL. */
int gm_optim_step(const gm_manifold_t* man, const gm_optim_t* opt, void* x, void* grad, void* buf1, void* buf2,
                  int64_t N, gm_stream_t stream);

/* One whole training epoch over node mini-batches in ONE call (TrainingEngine._train, train.py:198-228, for a single
 * manifold): for every slice `perm[i : i + batch_nodes]` of the node permutation (slices shorter than drop_last_n end
 * the epoch, train.py:209-211) launch  zero(grad) -> gm_pairs_loss_fused over all pairs of the slice (TRIU order,
 * DENSE targets indexed by node id) -> gm_optim_step  back to back on `stream`, with no host work in between.  A
 * 512-node batch is 130 816 pairs: its kernels take ~50 us, a Python-driven step ~200 us -- this entry point is what
 * makes BASELINE configs 2-3 kernel-bound.
 *   opt   : optimizer settings; opt->step is RAdam's state['step'] BEFORE the first update (it is advanced by one per
 *           slice), opt->first_step applies to the first slice only
 *   acc   : [max_steps][2] doubles, zeroed by the caller; slice k accumulates into acc[2k] (loss) and acc[2k+1]
 *           (sum l' d2, for the scale gradient)
 *   returns the number of slices processed in *n_steps (host), or a negative / CUDA error code */
int gm_train_epoch(const gm_manifold_t* man, const gm_optim_t* opt, void* x, void* grad, void* buf1, void* buf2,
                   int64_t N, const void* perm, int32_t perm_is_int64, int64_t n_perm, int64_t batch_nodes,
                   int64_t drop_last_n, const gm_targets_t* targets, const gm_loss_t* loss, double scale_sp, double* acc,
                   int64_t max_steps, int64_t* n_steps, gm_stream_t stream);

/* gm_train_epoch for a PRODUCT of F manifolds (modules.py:84-88: m = sum_f sp[f] * d2_f): per slice
 * zero(grad_f) x F -> gm_pairs_dist2 x F -> gm_product_loss -> gm_pairs_grad x F -> gm_optim_step x F (or, for the
 * products gm_pairs_product_fused takes: zero x F -> gm_pairs_product_fused -> gm_optim_step x F), all enqueued from
 * this one call.  Host arrays of length F: mans, opts (opts[f].step / first_step as in gm_train_epoch), x, grad, buf1,
 * buf2, sp, d2_ws (device workspaces of >= batch_nodes*(batch_nodes-1)/2 elements of the dtype each); g_ws is one more
 * such workspace.  acc: [max_steps][1 + F] doubles, zeroed by the caller (slice k: loss, then sum l' d2_f per factor).
 * All factors share dtype and N.  Universal factors are not supported here (see gm_train_epoch). */
int gm_train_epoch_product(int32_t F, const gm_manifold_t* mans, const gm_optim_t* opts, void* const* x,
                           void* const* grad, void* const* buf1, void* const* buf2, int64_t N, const void* perm,
                           int32_t perm_is_int64, int64_t n_perm, int64_t batch_nodes, int64_t drop_last_n,
                           const gm_targets_t* targets, const gm_loss_t* loss, const double* sp, void* const* d2_ws,
                           void* g_ws, double* acc, int64_t max_steps, int64_t* n_steps, gm_stream_t stream);

/* ---- multi-GPU: fused reduce-scatter + optimizer update + all-gather over NVLink peer memory ---------------------
 * New capability (the reference's only multi-GPU mechanism is nn.DataParallel, train.py:107-109,203-204).  Pairs are
 * sharded over ranks; every rank accumulates a full (N, ...) table of partial gradients.  Rank r owns rows
 * [row_lo, row_lo + N_owned): gm_optim_step_peer sums those rows over ALL ranks' gradient tables through peer loads,
 * applies the optimizer update of gm_optim_step to them (buf1/buf2 hold the owned rows only) and stores the new rows
 * into EVERY rank's point table through peer stores -- one kernel instead of ncclReduceScatter + update +
 * ncclAllGather.  The kernel carries its own cross-GPU barriers (flag words in the arenas): on entry it waits until
 * every rank has launched it (=> all partial gradients are final), and it only completes once every rank has finished
 * reading this rank's gradients and writing this rank's points.  All ranks must call it in lock step with the same
 * `epoch`, which must increase by one from call to call starting at 1.
 * The tables must live in memory obtained from gm_peer_alloc and mapped into the peers with gm_peer_export /
 * gm_peer_open (CUDA IPC, one process per GPU on one NVLink domain).  Each rank's flag block is
 * GM_PEER_FLAG_BYTES of zero-initialised arena memory. */
#define GM_MAX_PEERS 8
#define GM_PEER_FLAG_BYTES ((2 * GM_MAX_PEERS + 2) * 8)
#define GM_PEER_HANDLE_BYTES 64
typedef struct gm_peers {
  int32_t world, rank;
  int64_t row_lo;
  uint64_t epoch;
  void* x[GM_MAX_PEERS];          /* rank r's full point table (as mapped in THIS process)                  */
  const void* grad[GM_MAX_PEERS]; /* rank r's full partial-gradient table                                   */
  void* flags[GM_MAX_PEERS];      /* rank r's flag block                                                    */
  const void* acc[GM_MAX_PEERS];  /* rank r's double[n_acc] step accumulator (loss, scale grads) or NULL    */
  void* acc_out;                  /* local double[n_acc]: sum over ranks of acc                             */
  int32_t n_acc, reserved;
  void* gsum;                     /* optional LOCAL workspace of N_owned rows (dtype of the points).  Non-NULL selects the
                                     pipelined exchange: the owned rows are cut into chunks; a light kernel pulls and
                                     sums chunk c+1 of every rank's gradient table into gsum over NVLink while a second
                                     kernel, on a second stream, updates chunk c from gsum and pushes the new rows to
                                     every rank -- inbound and outbound NVLink traffic overlap instead of alternating
                                     inside one kernel.  NULL: the single fused kernel                         */
} gm_peers_t;
int gm_peer_alloc(size_t bytes, void** ptr);            /* zero-filled device memory on the current device  */
int gm_peer_free(void* ptr);
int gm_peer_export(const void* ptr, void* handle);      /* writes GM_PEER_HANDLE_BYTES                      */
int gm_peer_open(const void* handle, void** ptr);       /* maps a peer's arena; enables peer access         */
int gm_peer_close(void* ptr);
int gm_optim_step_peer(const gm_manifold_t* man, const gm_optim_t* opt, const gm_peers_t* peers, void* buf1,
                       void* buf2, int64_t N_owned, gm_stream_t stream);

/* ---- row-sharded embeddings (SURVEY 8(e) second scheme; BASELINE config 5 "embeddings row-sharded over NVLink") ----
 * The (N, ...) point table and its gradient table are cut over `world` GPUs of one NVLink domain, CYCLICALLY: global
 * row v is row v / world of the shard of rank v % world (world a power of two, <= GM_MAX_PEERS; a cyclic cut needs no
 * division in the kernel and spreads correlated node ids -- the hubs of a preferential-attachment graph are its first
 * ids -- evenly).  x[r] / grad[r] are rank r's shards as mapped into THIS process (CUDA IPC, gm_peer_open; the local
 * shard for r == rank).  The training kernel gathers a pair's rows from whichever shard holds them (16-byte cp.async
 * over NVLink for remote rows) and adds its gradient rows into the owning shard with red.global.add (NVLink atomics),
 * so after a step every rank holds the COMPLETE gradient of the rows it owns, and the optimizer update is local:
 *     gm_pairs_loss_fused_sharded (every rank, its slice of the pair batch)
 *     gm_peer_barrier(phase 0)    -- all ranks' reductions into my shard are final; acc_out = sum of the ranks' acc
 *     gm_optim_step               (local shard, zero_grad folded)
 *     gm_peer_barrier(phase 1)    -- all shards updated and all gradient shards zero: the next step may start
 * No point row is ever replicated; no collective library call is on the step path.  The reference has no counterpart
 * (its only multi-GPU mechanism is nn.DataParallel over node chunks, train.py:107-109,203-204).
 * SPD manifolds (the streaming pair kernels), GM_PAIRS_LIST / GM_PAIRS_SAMPLED; GM_EUNSUPPORTED otherwise. */
typedef struct gm_row_shards {
  int32_t world, reserved;
  const void* x[GM_MAX_PEERS];
  void* grad[GM_MAX_PEERS];
} gm_row_shards_t;
int gm_pairs_loss_fused_sharded(const gm_manifold_t* man, const gm_row_shards_t* shards, const gm_pairs_t* pairs,
                                const gm_targets_t* targets, const gm_loss_t* loss, double scale_sp, void* out_d2,
                                double* acc, gm_stream_t stream);
/* Lock-step barrier over the flag blocks of gm_peers_t (only world, rank, epoch, flags[], acc[], acc_out, n_acc are
 * read).  `epoch` must increase by one per step and be the same on every rank; phase 0 and 1 use separate flag words.
 * Phase 0 additionally sums acc[r][0..n_acc) over the ranks into acc_out. */
int gm_peer_barrier(const gm_peers_t* peers, int32_t phase, gm_stream_t stream);

/* ---- deterministic gradient accumulation (SURVEY 8a A11) ------------------------------------------------------- */
/* out[dst[c]] (row of E elements; dst == NULL: row c) = sum, left to right, of src[order[k]] (order == NULL: row k) for
 * chunk_start[c] <= k < chunk_end[c].  Plain stores, no atomics: bit-reproducible.  The autograd scatter it can stand
 * in for is index_put_(accumulate=True) behind x[m[0]], x[m[1]] (manifolds/base.py:62-63), which adds in whatever
 * order the device schedules.  graphembed.engine.PairTrainer(deterministic=True) builds a step from per-pair gradient
 * rows (gm_pairs_grad, GM_PAIRS_ELEMENTWISE) and two calls of this (fixed-size chunks of each row's sorted incidence
 * list, then the chunk sums of each row). */
int gm_segment_sum(int32_t dtype, int32_t E, const void* src, const int64_t* order, const int64_t* chunk_start,
                   const int64_t* chunk_end, const int64_t* dst, int64_t n_chunks, void* out, gm_stream_t stream);

/* ---- per-point manifold operations (Manifold API, manifolds/base.py:7-81) ----------------------------------- */
enum gm_point_op {
  GM_OP_EXP = 0,         /* out = exp_x(u)                      */
  GM_OP_RETR = 1,        /* out = retr_x(u)                     */
  GM_OP_LOG = 2,         /* out = log_x(u) with u := y          */
  GM_OP_PROJU = 3,       /* out = proju(x, u)                   */
  GM_OP_PROJX = 4,       /* out = projx(x)                      */
  GM_OP_EGRAD2RGRAD = 5, /* out = egrad2rgrad(x, u)             */
  GM_OP_INNER = 6,       /* out[k] = <u, v>_x (one scalar)      */
  GM_OP_NORM2 = 7,       /* out[k] = manifold.norm(x,u)^2 with the reference's clamp (one scalar) */
  GM_OP_TRANSP = 8,      /* out = transp(x, y := u, v)          */
  GM_OP_RETR_QR = 9,     /* Grassmann qr retraction             */
  GM_OP_SPD_SQRTM = 10   /* SPD only: out = x^{1/2} via eigendecomposition, eigenvalues clamped to [wmin, wmax]
                            (tb.spdsqrtm, linalg/torch_batch.py:169-171; used by SPD.randvec, spd.py:210-221) */
};
int gm_point_op(const gm_manifold_t* man, int32_t op, const void* x, const void* u, const void* v, void* out,
                int64_t N, gm_stream_t stream);

/* ---- graph-distance targets ---------------------------------------------------------------------------------- */

/* Unweighted multi-source BFS on a CSR graph (both directions of every undirected edge present).
 * levels[s*N + v] = hop count from sources[s] to v, GM_BFS_UNREACHED if not reachable.
 * Replaces networkit APSP at data/graph.py:66-87; in-tree spec pyx/impl/precision.cpp:44-63.  Bit-exact.
 * level_bytes: 1 (uint8, unreached = 255), 2 (uint16, 65535) or 4 (int32, -1).
 * workspace: at least gm_bfs_workspace_bytes(N, S) bytes of device memory. */
size_t gm_bfs_workspace_bytes(int32_t N, int32_t S);
int gm_bfs_multi_source(const int32_t* rowptr, const int32_t* colidx, int32_t N, const int32_t* sources, int32_t S,
                        int32_t level_bytes, void* levels, void* workspace, size_t workspace_bytes,
                        gm_stream_t stream);

/* Condensed (scipy.squareform order) float targets from a full S==N level matrix:
 * out[k] = (float|double) levels[a*N+b] for the k-th a<b (data/graph.py:78-82). */
int gm_levels_to_condensed(int32_t level_bytes, const void* levels, int32_t N, int32_t dtype, void* out,
                           gm_stream_t stream);

/* GraphDataset.__init__ (data/dataset.py:9-13): dense[u*N+v] = (h(u,v)^2)/max_sq in `dtype`, from a full level matrix. */
int gm_levels_to_dense_targets(int32_t level_bytes, const void* levels, int32_t N, double max_sq, int32_t dtype,
                               void* dense, gm_stream_t stream);

/* Gather per-pair hop counts: out[k] = levels[row_of[k]*N + col[k]] (row_of indexes the S sources). */
int gm_gather_levels(int32_t level_bytes, const void* levels, int32_t N, const int32_t* src_slot, const int32_t* col,
                     int64_t P, void* out, gm_stream_t stream);

/* Source-grouped (CSR-like) pair lists -> explicit first-endpoint index vector for gm_pairs_t LIST mode:
 * out_i[k] = group_row[g] for offsets[g] <= k < offsets[g+1], g < G; offsets[G] == P.  The grouped form is what a
 * per-source sampler produces (BASELINE config 5: S BFS sources x targets) and is 4 bytes/pair cheaper to upload
 * than the (i, j) lists base.py:62-63 builds with triu_indices. */
int gm_expand_groups(const int32_t* group_row, const int64_t* offsets, int32_t G, int32_t* out_i, int64_t P,
                     gm_stream_t stream);

/* Upload format of sampled pair batches, 3 bytes per pair: little-endian 24-bit words, bits 0-20 = second-endpoint row
 * (N <= 2^21), bits 21-23 = hop count - 1 (1 <= hops <= 8).  Expands them on the device to the 4-byte words of
 * GM_TGT_HOPS_PACKED, out[k] = (hops << 24) | j -- the end-to-end step is PCIe bound at 4 bytes per pair on one GPU
 * (67 MB per 2^24-pair step), this is 25 % less over the bus for a 20 us kernel.  src3: 4-byte aligned, 3*P bytes
 * (readable up to the next multiple of 4); out: 16-byte aligned, P words. */
int gm_unpack_pairs3(const void* src3, int64_t P, int32_t* out, gm_stream_t stream);

/* Upload format of source-grouped sampled pair batches, 2 bytes per pair.  A sampler that draws its targets per BFS
 * source can hand every source's targets over SORTED by row; consecutive targets of a group are then close (2^24 pairs
 * over 1024 sources and 2 M rows: mean gap 122 rows), and a pair fits a 16-bit word: bits 0-12 = j_k - j_{k-1}
 * (0 .. 8191; j_{-1} := base[g], so the first word of a group is usually 0), bits 13-15 = hop count - 1
 * (1 <= hops <= 8).  A batch with a larger gap or hop count is not representable -- the host packer
 * (graphembed.engine.pack_hops2) then declines and the caller uploads the 4-byte words.  offsets (G + 1 entries) are the
 * same group offsets gm_expand_groups takes.  Expands to the 4-byte words of GM_TGT_HOPS_PACKED,
 * out[k] = (hops << 24) | j_k, with a segmented prefix sum per group (one block per group).  Half the bytes of the
 * 4-byte form over PCIe: 33.5 MB instead of 67 MB per 2^24-pair step.  group_row / out_i (both or neither): also write
 * the first-endpoint vector out_i[k] = group_row[g] in the same pass (gm_expand_groups folded in). */
int gm_unpack_pairs2(const void* words, const int32_t* base, const int64_t* offsets, int32_t G, int32_t* out,
                     const int32_t* group_row, int32_t* out_i, gm_stream_t stream);

/* ---- ranking metrics (evaluation) ------------------------------------------------------------------------------
 * FastPrecision on the GPU (graphembed/pyx/impl/precision.cpp:249-291 mean average precision, :321-446 per-layer F1
 * scores; bound to Python in graphembed/pyx/precision.pyx:48-127).  For every shortest-path-tree root u in
 * [root_lo, root_hi): sort the other nodes by manifold distance from u (row u of the condensed `mpdists`, N(N-1)/2
 * values of `dtype`, squareform order) and compare that order with the BFS layering `levels_u8` (full N x N uint8 hop
 * matrix from gm_bfs_multi_source, connected graph with < 255 layers).  Everything is ACCUMULATED into caller-zeroed
 * device arrays of length n_layers - 1 (n_layers = max hop count + 1, precision.cpp:191-199):
 *   f1_m1 / f1_m2 / f1_cnt : sum f1, sum f1^2, count per layer over all (root, node) with
 *                            min_degree <= degree(root) <= max_degree          -- LayerMeanF1Scores (:397-420)
 *   af_m1 / af_m2 / af_cnt : the same after averaging within each root first   -- LayerMeanAverageF1Scores (:422-446)
 *   ap_sum[0]              : sum over roots of the average precision            -- MeanAveragePrecision (:268-303)
 * means = m1 / cnt, "stds" = m2 / cnt - means^2 as the reference reports them.  A rank of a multi-GPU job passes its
 * slice of roots and the accumulators are summed across ranks.  N <= 32768 (fp32) / 16384 (fp64): one root's sort
 * lives in one SM's shared memory. */
int gm_rank_metrics(int32_t dtype, const void* mpdists, const void* levels_u8, int32_t N, int32_t root_lo,
                    int32_t root_hi, int32_t min_degree, int32_t max_degree, int32_t n_layers, double* f1_m1,
                    double* f1_m2, int64_t* f1_cnt, double* af_m1, double* af_m2, int64_t* af_cnt, double* ap_sum,
                    gm_stream_t stream);

/* ---- introspection ------------------------------------------------------------------------------------------- */
const char* gm_version(void);
/* 1 if (kind, n, p, dtype, flags) has a compiled kernel */
int gm_supported(const gm_manifold_t* man);
/* number of kernel launches issued by this library in this process (for bench.py's gpu_launches) */
int64_t gm_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GM_KERNELS_H */
