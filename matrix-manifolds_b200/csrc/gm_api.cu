// C-ABI entry points of libgm_b200.so (declared in include/gm_kernels.h):
// argument validation and dispatch to the templated kernel launchers.
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <cuda_runtime.h>
#include "gm_point_kernels.cuh"

namespace gm {

static std::atomic<long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int check_launch() { return (int)cudaGetLastError(); }

// one side stream + event set per device for the pipelined exchange (created on first use, kept for the process)
PeerPipe& peer_pipe() {
  static std::mutex mu;
  static PeerPipe pipes[64];
  int dev = 0;
  cudaGetDevice(&dev);
  std::lock_guard<std::mutex> lock(mu);
  PeerPipe& p = pipes[dev & 63];
  if (!p.side) {
    if (cudaStreamCreateWithFlags(&p.side, cudaStreamNonBlocking) != cudaSuccess) { p.side = nullptr; return p; }
    for (auto& e : p.pulled) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&p.joined, cudaEventDisableTiming);
  }
  return p;
}


int validate_pairs(const gm_pairs_t* p) {
  if (!p) return GM_ENULL;
  if (p->P < 0) return GM_EINVAL;
  switch (p->mode) {
    case GM_PAIRS_ELEMENTWISE:
      return GM_OK;
    case GM_PAIRS_LIST:
      if (p->P > 0 && (!p->idx_i || !p->idx_j)) return GM_ENULL;
      if (p->segments < 0 || p->segments > 64) return GM_EINVAL;
      return GM_OK;
    case GM_PAIRS_TRIU:
      if (p->B < 0 || p->k0 < 0) return GM_EINVAL;
      if (p->k0 + p->P > p->B * (p->B - 1) / 2) return GM_EINVAL;
      return GM_OK;
    case GM_PAIRS_SAMPLED:
      if (p->idx64 || p->per_src < 1 || p->n_nodes < 2 || p->n_nodes >= (1LL << 24)) return GM_EINVAL;
      if (p->P > 0 && (!p->idx_i || !p->levels)) return GM_ENULL;
      return GM_OK;
    default:
      return GM_EINVAL;
  }
}

// the set of compiled SPD sizes comes from the Makefile (-DGM_SPD_LIST="X(1) X(2) ...")
#ifndef GM_SPD_LIST
#define GM_SPD_LIST X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10)
#endif
#define X(n) int spd_launch_##n(const PairArgs& a); int spd_point_##n(const PointArgs& a);
GM_SPD_LIST
#undef X
int vec_launch(const PairArgs& a);
int vec_point_0(const PointArgs& a);
int vec_point_1(const PointArgs& a);
int vec_point_2(const PointArgs& a);
int vec_point_3(const PointArgs& a);
int vec_point_4(const PointArgs& a);
static int vec_point(const PointArgs& a) {
  switch (a.kind) {
    case GM_LORENTZ: return vec_point_0(a);
    case GM_SPHERE: return vec_point_1(a);
    case GM_EUCLIDEAN: return vec_point_2(a);
    case GM_GRASSMANN: return vec_point_3(a);
    case GM_UNIVERSAL: return vec_point_4(a);
    default: return GM_EINVAL;
  }
}

// Cross-GPU barrier of the row-sharded step (gm_peer_barrier): tell every peer "I have passed point `phase` of step
// pt.epoch" and wait until every peer has said the same.  It runs in stream order after the kernel whose effects it
// publishes (the pair kernel's reductions into the peers' gradient shards for phase 0, the optimizer's writes of the
// local point shard for phase 1); kernel completion makes those visible at system scope before the release stores
// here.  Phase 0 also sums the ranks' per-step scalars (loss, sum l' d2) into the local acc_out.
__global__ void __launch_bounds__(64)
peer_barrier_kernel(PeerTable pt, int phase) {
  const int tid = threadIdx.x;
  unsigned long long* mine = pt.flags[pt.rank] + (phase ? kMaxPeers : 0);
  __threadfence_system();
  if (tid < pt.world) {
    flag_store_release(pt.flags[tid] + (phase ? kMaxPeers : 0) + pt.rank, pt.epoch);
    flag_wait(mine + tid, pt.epoch, pt.timeout_ns);
  }
  __syncthreads();
  if (tid < pt.n_acc) {
    double s = 0.0;
    for (int r = 0; r < pt.world; ++r) s += pt.acc[r][tid];
    pt.acc_out[tid] = s;
  }
}
static int launch_peer_barrier(const PeerTable& pt, int phase, cudaStream_t stream) {
  peer_barrier_kernel<<<1, 64, 0, stream>>>(pt, phase);
  note_launch();
  return check_launch();
}

static int point_dispatch(const PointArgs& a) {
  if (a.kind == GM_SPD_AI || a.kind == GM_SPD_STEIN) {
    switch (a.n) {
#define X(n) case n: return spd_point_##n(a);
      GM_SPD_LIST
#undef X
      default: return GM_EUNSUPPORTED;
    }
  }
  return vec_point(a);
}

static int spd_dispatch(const PairArgs& a) {
  switch (a.n) {
#define X(n) case n: return spd_launch_##n(a);
    GM_SPD_LIST
#undef X
    default: return GM_EUNSUPPORTED;
  }
}

static bool spd_size_compiled(int n) {
  switch (n) {
#define X(n) case n: return true;
    GM_SPD_LIST
#undef X
    default: return false;
  }
}

static int manifold_ok(const gm_manifold_t* m) {
  if (!m) return GM_ENULL;
  if (m->dtype != GM_F32 && m->dtype != GM_F64) return GM_EINVAL;
  switch (m->kind) {
    case GM_SPD_AI:
    case GM_SPD_STEIN:
      if (!spd_size_compiled(m->n)) return GM_EUNSUPPORTED;
      if ((m->flags & GM_FAST_CHOL) && m->n != 2) return GM_EINVAL;
      if ((m->flags & GM_FAST_EIG) && m->n != 2 && m->n != 3) return GM_EINVAL;
      return GM_OK;
    case GM_LORENTZ:
      return m->n >= 2 ? GM_OK : GM_EINVAL;
    case GM_SPHERE:
    case GM_EUCLIDEAN:
      return m->n >= 1 ? GM_OK : GM_EINVAL;
    case GM_UNIVERSAL:
      if (m->n < 1) return GM_EINVAL;
      return m->c_dev ? GM_OK : GM_ENULL;
    case GM_GRASSMANN:
      if (m->n < 1 || m->p < 1 || m->p > m->n) return GM_EINVAL;
      if (m->p > 5) return GM_EUNSUPPORTED;
      if ((m->flags & GM_FAST_SVD) && m->p != 2) return GM_EINVAL;
      return GM_OK;
    default:
      return GM_EINVAL;
  }
}

static void fill_manifold(PairArgs& a, const gm_manifold_t* m) {
  a.kind = m->kind; a.dtype = m->dtype; a.n = m->n; a.p = m->p; a.flags = m->flags;
  a.wmin = m->wmin; a.wmax = m->wmax;
  a.c_dev = m->c_dev; a.c_grad = m->c_grad;
  a.sh = no_shards();
}

static int pair_dispatch(const PairArgs& a) {
  if (a.kind == GM_SPD_AI || a.kind == GM_SPD_STEIN) return spd_dispatch(a);
  return vec_launch(a);
}

// the loss request: QuotientLoss needs at least one of its two terms
int check_loss(const gm_loss_t* loss) {
  if (loss->kind != GM_LOSS_QUOTIENT && loss->kind != GM_LOSS_STRESS) return GM_EINVAL;
  if (loss->kind == GM_LOSS_QUOTIENT && !loss->inc_l1 && !loss->inc_l2) return GM_EINVAL;
  return GM_OK;
}

// targets of a K_FUSED request: hop counts packed into the top byte of idx_j need int32 LIST or SAMPLED pairs, drawn
// pairs bring their hop count with them, and every other target mode reads targets->data
static int check_fused_targets(const gm_pairs_t* pairs, const gm_targets_t* targets) {
  if (pairs->mode == GM_PAIRS_ELEMENTWISE) return GM_EINVAL;
  if (targets->mode < GM_TGT_VECTOR || targets->mode > GM_TGT_HOPS_PACKED) return GM_EINVAL;
  const bool packed = targets->mode == GM_TGT_HOPS_PACKED;
  if (packed && ((pairs->mode != GM_PAIRS_LIST && pairs->mode != GM_PAIRS_SAMPLED) || pairs->idx64)) return GM_EINVAL;
  if (pairs->mode == GM_PAIRS_SAMPLED && !packed) return GM_EINVAL;
  if (pairs->P > 0 && !packed && !targets->data) return GM_ENULL;
  return GM_OK;
}

static bool optim_kind_ok(const gm_optim_t* opt) { return opt->kind == GM_OPT_RSGD || opt->kind == GM_OPT_RADAM; }

// the optimizer request: RAdam needs both moment buffers and step >= 1, RSGD with momentum its momentum buffer
static int check_optim(const gm_optim_t* opt, const void* buf1, const void* buf2) {
  if (!optim_kind_ok(opt)) return GM_EINVAL;
  if (opt->kind == GM_OPT_RADAM && (!buf1 || !buf2 || opt->step < 1)) return GM_EINVAL;
  if (opt->kind == GM_OPT_RSGD && opt->has_momentum && !buf1) return GM_ENULL;
  return GM_OK;
}

// PointArgs of `man`; with an optimizer, its step (op -1) and the state buffers that step uses
static PointArgs point_args(const gm_manifold_t* man, const gm_optim_t* opt, void* buf1, void* buf2) {
  PointArgs a{};
  a.kind = man->kind; a.dtype = man->dtype; a.n = man->n; a.p = man->p; a.flags = man->flags;
  a.wmin = man->wmin; a.wmax = man->wmax; a.c_dev = man->c_dev;
  a.op = -1;
  if (opt) {
    a.oc = make_optim_cfg(opt);
    a.grassmann_retr_qr = opt->grassmann_retr_qr;
    a.buf1 = (opt->kind == GM_OPT_RSGD && !opt->has_momentum) ? nullptr : buf1;
    a.buf2 = (opt->kind == GM_OPT_RADAM) ? buf2 : nullptr;
  }
  return a;
}

// One rank's PeerTable.  phase < 0: the owner update of gm_optim_step_peer, which also reads every rank's point and
// gradient shard; phase 0 / 1: gm_peer_barrier (phase 1 sums no per-step scalars).
static int peer_table(const gm_peers_t* peers, int phase, PeerTable& pt) {
  static const long long timeout_s = [] { const char* e = getenv("GM_PEER_TIMEOUT_S"); return e ? atoll(e) : 300LL; }();
  static const int chunks = [] { const char* e = getenv("GM_PEER_CHUNKS"); return e ? atoi(e) : 4; }();
  pt = PeerTable{};
  pt.world = peers->world; pt.rank = peers->rank; pt.row_lo = peers->row_lo; pt.epoch = peers->epoch;
  pt.n_acc = phase == 1 ? 0 : peers->n_acc;
  for (int r = 0; r < peers->world; ++r) {
    if (!peers->flags[r] || (phase < 0 && (!peers->x[r] || !peers->grad[r]))) return GM_ENULL;
    if (pt.n_acc > 0 && !peers->acc[r]) return GM_ENULL;
    pt.x[r] = peers->x[r]; pt.g[r] = peers->grad[r];
    pt.flags[r] = (unsigned long long*)peers->flags[r];
    pt.acc[r] = (const double*)peers->acc[r];
  }
  if (pt.n_acc > 0 && !peers->acc_out) return GM_ENULL;
  pt.acc_out = (double*)peers->acc_out;
  pt.gsum = peers->gsum;
  pt.timeout_ns = timeout_s > 0 ? (unsigned long long)timeout_s * 1000000000ull : 0ull;
  pt.chunks = chunks;
  return GM_OK;
}

// The K_FUSED launch request shared by the fused entry points; the caller adds the point / gradient tables.
static PairArgs fused_args(const gm_manifold_t* man, const gm_pairs_t* pairs, const gm_targets_t* targets,
                           const gm_loss_t* loss, double scale_sp, double* acc, gm_stream_t stream) {
  PairArgs a{};
  fill_manifold(a, man);
  a.kmode = K_FUSED;
  a.ps = make_pairs(pairs);
  a.tg = make_targets(targets);
  if (targets->mode == GM_TGT_HOPS_PACKED) { a.tg.data = pairs->idx_j; a.ps.jmask = 0x00ffffffu; }
  a.lc = make_loss(loss);
  a.scale_sp = scale_sp;
  a.acc = acc;
  a.stream = (cudaStream_t)stream;
  return a;
}

// The TRIU node batches of one epoch: batch k is the upper triangle of perm[i, i + b), b = batch_nodes except for the
// last.  The walk stops at the first batch shorter than drop_last_n (or than 2 nodes); a walk longer than max_steps is
// an error.  body(k, pairs) returns a code; *n_steps is the number of batches walked.
template <class Body>
static int for_each_node_batch(const void* perm, int32_t perm_is_int64, int64_t n_perm, int64_t batch_nodes,
                               int64_t drop_last_n, int64_t max_steps, int64_t* n_steps, Body&& body) {
  const size_t idx_bytes = perm_is_int64 ? 8 : 4;
  int64_t k = 0;
  for (int64_t i = 0; i < n_perm; i += batch_nodes, ++k) {
    const int64_t b = (n_perm - i < batch_nodes) ? (n_perm - i) : batch_nodes;
    if (b < drop_last_n || b < 2) break;
    if (k >= max_steps) return GM_EINVAL;
    gm_pairs_t pr{};
    pr.mode = GM_PAIRS_TRIU; pr.idx64 = perm_is_int64; pr.P = b * (b - 1) / 2; pr.B = b;
    pr.nodes = (const char*)perm + (size_t)i * idx_bytes; pr.k0 = 0;
    int rc = body(k, pr);
    if (rc) return rc;
  }
  *n_steps = k;
  return GM_OK;
}

}  // namespace gm

using namespace gm;

static int64_t point_elems(const gm_manifold_t* man) {
  switch (man->kind) {
    case GM_SPD_AI: case GM_SPD_STEIN: return (int64_t)man->n * man->n;
    case GM_GRASSMANN: return (int64_t)man->n * man->p;
    default: return man->n;
  }
}

extern "C" {
#pragma GCC visibility push(default)

const char* gm_version(void) { return "gm_b200 0.1 (sm_100a)"; }
int64_t gm_launch_count(void) { return (int64_t)g_launches.load(); }
int gm_supported(const gm_manifold_t* man) { return manifold_ok(man) == GM_OK; }

int gm_pairs_dist2(const gm_manifold_t* man, const void* xa, const void* xb, const gm_pairs_t* pairs,
                   void* out_d2, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  rc = validate_pairs(pairs);
  if (rc) return rc;
  if (pairs->P == 0) return GM_OK;
  if (!xa || !xb || !out_d2) return GM_ENULL;
  PairArgs a{};
  fill_manifold(a, man);
  a.kmode = K_FWD;
  a.ps = make_pairs(pairs);
  a.xa = xa; a.xb = xb; a.out_d2 = out_d2;
  a.stream = (cudaStream_t)stream;
  return pair_dispatch(a);
}

int gm_pairs_grad(const gm_manifold_t* man, const void* xa, const void* xb, const gm_pairs_t* pairs,
                  const void* gout, double coef, void* ga, void* gb, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  rc = validate_pairs(pairs);
  if (rc) return rc;
  if (pairs->P == 0) return GM_OK;
  if (!xa || !xb || !gout || !ga || !gb) return GM_ENULL;
  if (pairs->mode == GM_PAIRS_ELEMENTWISE && ga == gb) return GM_EINVAL;
  PairArgs a{};
  fill_manifold(a, man);
  a.kmode = K_BWD;
  a.ps = make_pairs(pairs);
  a.xa = xa; a.xb = xb; a.gout = gout; a.coef = coef; a.ga = ga; a.gb = gb;
  a.stream = (cudaStream_t)stream;
  return pair_dispatch(a);
}

int gm_pairs_loss_fused(const gm_manifold_t* man, const void* x, const gm_pairs_t* pairs,
                        const gm_targets_t* targets, const gm_loss_t* loss, double scale_sp, void* out_d2,
                        double* acc, void* grad, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  rc = validate_pairs(pairs);
  if (rc) return rc;
  if (!targets || !loss) return GM_ENULL;
  if ((rc = check_loss(loss)) || (rc = check_fused_targets(pairs, targets))) return rc;
  if (pairs->P == 0) return GM_OK;
  if (!x || !acc || !grad) return GM_ENULL;
  PairArgs a = fused_args(man, pairs, targets, loss, scale_sp, acc, stream);
  a.xa = x; a.xb = x; a.ga = grad; a.gb = grad; a.out_d2 = out_d2;
  return pair_dispatch(a);
}

int gm_pairs_loss_fused_sharded(const gm_manifold_t* man, const gm_row_shards_t* shards, const gm_pairs_t* pairs,
                                const gm_targets_t* targets, const gm_loss_t* loss, double scale_sp, void* out_d2,
                                double* acc, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  if (!shards) return GM_ENULL;
  const int W = shards->world;
  if (W < 1 || W > GM_MAX_PEERS || (W & (W - 1)) != 0) return GM_EINVAL;  // cyclic ownership by the low bits of the row id
  if (man->kind != GM_SPD_AI && man->kind != GM_SPD_STEIN) return GM_EUNSUPPORTED;
  rc = validate_pairs(pairs);
  if (rc) return rc;
  if (!targets || !loss) return GM_ENULL;
  if (pairs->mode != GM_PAIRS_LIST && pairs->mode != GM_PAIRS_SAMPLED) return GM_EINVAL;
  if ((rc = check_loss(loss)) || (rc = check_fused_targets(pairs, targets))) return rc;
  if (pairs->P == 0) return GM_OK;
  if (!acc) return GM_ENULL;
  PairArgs a = fused_args(man, pairs, targets, loss, scale_sp, acc, stream);
  a.sh.log2w = 0;
  while ((1 << a.sh.log2w) < W) ++a.sh.log2w;
  a.sh.mask = (unsigned)W - 1u;
  for (int r = 0; r < W; ++r) {
    if (!shards->x[r] || !shards->grad[r]) return GM_ENULL;
    a.sh.x[r] = shards->x[r]; a.sh.g[r] = shards->grad[r];
  }
  a.xa = shards->x[0]; a.xb = shards->x[0]; a.ga = shards->grad[0]; a.gb = shards->grad[0]; a.out_d2 = out_d2;
  return pair_dispatch(a);
}

int gm_optim_step(const gm_manifold_t* man, const gm_optim_t* opt, void* x, void* grad, void* buf1, void* buf2,
                  int64_t N, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  if (!opt) return GM_ENULL;
  if (N < 0) return GM_EINVAL;
  if (!optim_kind_ok(opt)) return GM_EINVAL;
  if (N == 0) return GM_OK;
  if (!x || !grad) return GM_ENULL;
  rc = check_optim(opt, buf1, buf2);
  if (rc) return rc;
  PointArgs a = point_args(man, opt, buf1, buf2);
  a.x = x; a.u = grad;
  a.N = N;
  a.stream = (cudaStream_t)stream;
  return point_dispatch(a);
}

int gm_train_epoch(const gm_manifold_t* man, const gm_optim_t* opt, void* x, void* grad, void* buf1, void* buf2,
                   int64_t N, const void* perm, int32_t perm_is_int64, int64_t n_perm, int64_t batch_nodes,
                   int64_t drop_last_n, const gm_targets_t* targets, const gm_loss_t* loss, double scale_sp, double* acc,
                   int64_t max_steps, int64_t* n_steps, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  if (!opt || !targets || !loss || !n_steps) return GM_ENULL;
  *n_steps = 0;
  if (man->kind == GM_UNIVERSAL) return GM_EUNSUPPORTED;  // the curvature gradient needs the autograd-side chain rule
  if (N <= 0 || n_perm < 0 || batch_nodes < 2 || max_steps < 0) return GM_EINVAL;
  if (targets->mode != GM_TGT_DENSE || !targets->data) return GM_EINVAL;
  if (!optim_kind_ok(opt)) return GM_EINVAL;
  rc = check_loss(loss);
  if (rc) return rc;
  if (!x || !grad || !perm || !acc) return GM_ENULL;
  rc = check_optim(opt, buf1, buf2);
  if (rc) return rc;
  const size_t grad_bytes = (size_t)N * point_elems(man) * (man->dtype == GM_F32 ? 4 : 8);
  cudaStream_t st = (cudaStream_t)stream;
  gm_optim_t o = *opt;
  return for_each_node_batch(perm, perm_is_int64, n_perm, batch_nodes, drop_last_n, max_steps, n_steps,
                             [&](int64_t k, const gm_pairs_t& pr) -> int {
    cudaError_t e = cudaMemsetAsync(grad, 0, grad_bytes, st);
    if (e != cudaSuccess) return (int)e;
    int rc = gm_pairs_loss_fused(man, x, &pr, targets, loss, scale_sp, nullptr, acc + 2 * k, grad, stream);
    if (rc) return rc;
    rc = gm_optim_step(man, &o, x, grad, buf1, buf2, N, stream);
    if (rc) return rc;
    o.step += 1;       // RAdam: state['step'] += 1 (radam.py:98)
    o.first_step = 0;  // RSGD momentum buffer exists from now on
    return GM_OK;
  });
}

// Can the fused product kernel (gm_product.cuh) take this factor list?  At most one SPD factor, the rest Lorentz /
// Sphere / Euclidean, one dtype.
static bool product_fusable(int F, const gm_manifold_t* mans) {
  if (F < 2 || F > 1 + kMaxVecExtra) return false;
  int n_spd = 0, n_vec = 0;
  for (int f = 0; f < F; ++f) {
    const int k = mans[f].kind;
    if (mans[f].dtype != mans[0].dtype) return false;
    if (k == GM_SPD_AI || k == GM_SPD_STEIN) ++n_spd;
    else if (k == GM_LORENTZ || k == GM_SPHERE || k == GM_EUCLIDEAN) ++n_vec;
    else return false;
  }
  return n_spd <= 1 && n_vec <= kMaxVecExtra;
}

int gm_pairs_product_fused(int32_t F, const gm_manifold_t* mans, void* const* x, const gm_pairs_t* pairs,
                           const gm_targets_t* targets, const gm_loss_t* loss, const double* sp, double* acc,
                           void* const* grad, gm_stream_t stream) {
  if (!mans || !x || !grad || !sp || !targets || !loss) return GM_ENULL;
  if (F < 1 || F > 8) return GM_EINVAL;
  for (int f = 0; f < F; ++f) {
    int rc = manifold_ok(&mans[f]);
    if (rc) return rc;
  }
  if (!product_fusable(F, mans)) return GM_EUNSUPPORTED;
  int rc = validate_pairs(pairs);
  if (rc) return rc;
  if ((rc = check_loss(loss)) || (rc = check_fused_targets(pairs, targets))) return rc;
  if (pairs->P == 0) return GM_OK;
  if (!acc) return GM_ENULL;
  ProductExtra px{};
  px.F = F; px.lead_slot = -1; px.nvec = 0;
  for (int f = 0; f < F; ++f) {
    if (!x[f] || !grad[f]) return GM_ENULL;
    if (mans[f].kind == GM_SPD_AI || mans[f].kind == GM_SPD_STEIN) { px.lead_slot = f; continue; }
    VecExtra& v = px.v[px.nvec++];
    v.kind = mans[f].kind; v.n = mans[f].n; v.slot = f; v.x = x[f]; v.g = grad[f]; v.sp = sp[f];
  }
  const int lead = px.lead_slot;
  // without an SPD factor, mans[0] gives the dtype and the factors themselves travel in px
  PairArgs a = fused_args(&mans[lead >= 0 ? lead : 0], pairs, targets, loss, lead >= 0 ? sp[lead] : 0.0, acc, stream);
  if (lead >= 0) {
    a.xa = a.xb = x[lead];
    a.ga = a.gb = grad[lead];
  }
  a.px = &px;
  return pair_dispatch(a);
}

int gm_train_epoch_product(int32_t F, const gm_manifold_t* mans, const gm_optim_t* opts, void* const* x,
                           void* const* grad, void* const* buf1, void* const* buf2, int64_t N, const void* perm,
                           int32_t perm_is_int64, int64_t n_perm, int64_t batch_nodes, int64_t drop_last_n,
                           const gm_targets_t* targets, const gm_loss_t* loss, const double* sp, void* const* d2_ws,
                           void* g_ws, double* acc, int64_t max_steps, int64_t* n_steps, gm_stream_t stream) {
  if (!mans || !opts || !x || !grad || !buf1 || !buf2 || !targets || !loss || !sp || !d2_ws || !n_steps) return GM_ENULL;
  *n_steps = 0;
  if (F < 1 || F > 8 || N <= 0 || n_perm < 0 || batch_nodes < 2 || max_steps < 0) return GM_EINVAL;
  if (targets->mode != GM_TGT_DENSE || !targets->data || !perm || !acc || !g_ws) return GM_EINVAL;
  for (int f = 0; f < F; ++f) {
    int rc = manifold_ok(&mans[f]);
    if (rc) return rc;
    if (mans[f].kind == GM_UNIVERSAL) return GM_EUNSUPPORTED;
    if (mans[f].dtype != mans[0].dtype) return GM_EINVAL;
    if (!x[f] || !grad[f] || !d2_ws[f]) return GM_ENULL;
    rc = check_optim(&opts[f], buf1[f], buf2[f]);
    if (rc) return rc;
  }
  const size_t s_bytes = mans[0].dtype == GM_F32 ? 4 : 8;
  cudaStream_t st = (cudaStream_t)stream;
  gm_optim_t o[8];
  for (int f = 0; f < F; ++f) o[f] = opts[f];
  const bool fused = product_fusable(F, mans);
  return for_each_node_batch(perm, perm_is_int64, n_perm, batch_nodes, drop_last_n, max_steps, n_steps,
                             [&](int64_t k, const gm_pairs_t& pr) -> int {
    for (int f = 0; f < F; ++f) {
      cudaError_t e = cudaMemsetAsync(grad[f], 0, (size_t)N * point_elems(&mans[f]) * s_bytes, st);
      if (e != cudaSuccess) return (int)e;
      if (fused) continue;
      int rc = gm_pairs_dist2(&mans[f], x[f], x[f], &pr, d2_ws[f], stream);
      if (rc) return rc;
    }
    int rc = fused ? gm_pairs_product_fused(F, mans, x, &pr, targets, loss, sp, acc + (1 + F) * k, grad, stream)
                   : gm_product_loss(mans[0].dtype, F, (const void* const*)d2_ws, sp, &pr, targets, loss, pr.P,
                                     acc + (1 + F) * k, g_ws, stream);
    if (rc) return rc;
    for (int f = 0; f < F; ++f) {
      if (!fused) {
        rc = gm_pairs_grad(&mans[f], x[f], x[f], &pr, g_ws, sp[f], grad[f], grad[f], stream);
        if (rc) return rc;
      }
      rc = gm_optim_step(&mans[f], &o[f], x[f], grad[f], buf1[f], buf2[f], N, stream);
      if (rc) return rc;
      o[f].step += 1;
      o[f].first_step = 0;
    }
    return GM_OK;
  });
}

int gm_peer_alloc(size_t bytes, void** ptr) {
  if (!ptr) return GM_ENULL;
  if (bytes == 0) return GM_EINVAL;
  cudaError_t e = cudaMalloc(ptr, bytes);
  if (e != cudaSuccess) return (int)e;
  return (int)cudaMemset(*ptr, 0, bytes);
}
int gm_peer_free(void* ptr) { return ptr ? (int)cudaFree(ptr) : GM_OK; }
int gm_peer_export(const void* ptr, void* handle) {
  if (!ptr || !handle) return GM_ENULL;
  static_assert(sizeof(cudaIpcMemHandle_t) == GM_PEER_HANDLE_BYTES, "IPC handle size");
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, const_cast<void*>(ptr));
  if (e != cudaSuccess) return (int)e;
  memcpy(handle, &h, sizeof(h));
  return GM_OK;
}
int gm_peer_open(const void* handle, void** ptr) {
  if (!handle || !ptr) return GM_ENULL;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  return (int)cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess);
}
int gm_peer_close(void* ptr) { return ptr ? (int)cudaIpcCloseMemHandle(ptr) : GM_OK; }

int gm_optim_step_peer(const gm_manifold_t* man, const gm_optim_t* opt, const gm_peers_t* peers, void* buf1,
                       void* buf2, int64_t N_owned, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  if (!opt || !peers) return GM_ENULL;
  if (N_owned <= 0 || peers->row_lo < 0 || peers->epoch == 0) return GM_EINVAL;  // every rank must launch: no empty shards
  if (peers->world < 1 || peers->world > GM_MAX_PEERS || peers->rank < 0 || peers->rank >= peers->world) return GM_EINVAL;
  if (peers->n_acc < 0 || peers->n_acc > 64) return GM_EINVAL;
  rc = check_optim(opt, buf1, buf2);
  if (rc) return rc;
  PeerTable pt;
  rc = peer_table(peers, -1, pt);
  if (rc) return rc;
  PointArgs a = point_args(man, opt, buf1, buf2);
  a.N = N_owned;
  a.stream = (cudaStream_t)stream;
  a.peer = &pt;
  return point_dispatch(a);
}

int gm_peer_barrier(const gm_peers_t* peers, int32_t phase, gm_stream_t stream) {
  if (!peers) return GM_ENULL;
  if (peers->world < 1 || peers->world > GM_MAX_PEERS || peers->rank < 0 || peers->rank >= peers->world) return GM_EINVAL;
  if (phase < 0 || phase > 1 || peers->epoch == 0 || peers->n_acc < 0 || peers->n_acc > 64) return GM_EINVAL;
  PeerTable pt;
  int rc = peer_table(peers, phase, pt);
  if (rc) return rc;
  return launch_peer_barrier(pt, phase, (cudaStream_t)stream);
}

int gm_point_op(const gm_manifold_t* man, int32_t op, const void* x, const void* u, const void* v, void* out,
                int64_t N, gm_stream_t stream) {
  int rc = manifold_ok(man);
  if (rc) return rc;
  if (N < 0 || op < GM_OP_EXP || op > GM_OP_SPD_SQRTM) return GM_EINVAL;
  if (op == GM_OP_SPD_SQRTM && man->kind != GM_SPD_AI && man->kind != GM_SPD_STEIN) return GM_EINVAL;
  if (N == 0) return GM_OK;
  if (!x || !out) return GM_ENULL;
  const bool needs_u = op != GM_OP_PROJX && op != GM_OP_SPD_SQRTM;
  const bool needs_v = op == GM_OP_INNER || op == GM_OP_TRANSP;
  if ((needs_u && !u) || (needs_v && !v)) return GM_ENULL;
  PointArgs a = point_args(man, nullptr, nullptr, nullptr);
  a.op = op;
  if (op == GM_OP_RETR_QR) { a.op = GM_OP_RETR; a.grassmann_retr_qr = 1; }
  a.x = const_cast<void*>(x); a.u = u; a.v = v; a.out = out;
  a.N = N;
  a.stream = (cudaStream_t)stream;
  return point_dispatch(a);
}

#pragma GCC visibility pop
}  // extern "C"
