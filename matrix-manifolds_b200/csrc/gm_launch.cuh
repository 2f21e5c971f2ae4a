// Kernel-side plumbing shared by all pair kernels: pair enumeration, target
// fetch, vectorised row I/O, warp-aggregated gradient accumulation.
#pragma once
#include <stdint.h>
#include "../../include/gm_kernels.h"
#include "gm_manifolds.cuh"

namespace gm {

// ---- launch accounting (gm_launch_count) -----------------------------------
void note_launch();
int check_launch();  // returns cudaGetLastError() as int

// ---- POD copies of the C-ABI structs, passed to kernels by value -------------
struct PairSpec {
  int mode, idx64;
  long long P, B;
  const void* idx_i;
  const void* idx_j;
  const void* nodes;
  long long k0;    // TRIU: triangle index of local pair 0
  unsigned jmask;  // LIST + int32: row = idx_j[k] & jmask (0xFFFFFF when hop counts ride in the top byte)
  // SAMPLED
  const unsigned char* levels;
  const int* slots;
  long long n_nodes, per_src;
  unsigned long long seed;
  int per_shift;  // log2(per_src) if it is a power of two, else -1
  // LIST: the list is nseg consecutive segments of seg_len pairs (the last one may be shorter); the streaming kernels
  // walk them one after another with the whole grid (seg_len is filled in by the launcher)
  int nseg;
  long long seg_len;
};
// Row-sharded point / gradient tables (gm_row_shards_t): global row v is row (v >> log2w) of shard (v & mask).
// log2w < 0: not sharded (the kernels use their plain base pointers).
struct ShardTab {
  int log2w;
  unsigned mask;
  const void* x[8];
  void* g[8];
};
inline ShardTab no_shards() {
  ShardTab t{};
  t.log2w = -1;
  return t;
}
struct TargetSpec {
  int mode;
  const void* data;
  long long ld;
  double max_sq;
};

inline PairSpec make_pairs(const gm_pairs_t* p) {
  PairSpec s;
  s.mode = p->mode; s.idx64 = p->idx64; s.P = p->P; s.B = p->B;
  s.idx_i = p->idx_i; s.idx_j = p->idx_j; s.nodes = p->nodes;
  s.k0 = (p->mode == GM_PAIRS_TRIU) ? p->k0 : 0;
  s.jmask = 0xffffffffu;
  s.levels = nullptr; s.slots = nullptr; s.n_nodes = 0; s.per_src = 1; s.seed = 0; s.per_shift = 0;
  s.nseg = (p->mode == GM_PAIRS_LIST && p->segments > 1) ? p->segments : 1;
  s.seg_len = (p->P + s.nseg - 1) / s.nseg;
  if (p->mode == GM_PAIRS_SAMPLED) {
    s.levels = (const unsigned char*)p->levels; s.slots = (const int*)p->slots;
    s.n_nodes = p->n_nodes; s.per_src = p->per_src; s.seed = p->seed;
    s.jmask = 0x00ffffffu;
    s.per_shift = -1;
    for (int b = 0; b < 62; ++b)
      if (p->per_src == (1LL << b)) s.per_shift = b;
  }
  return s;
}
inline TargetSpec make_targets(const gm_targets_t* t) {
  TargetSpec s;
  s.mode = t->mode; s.data = t->data; s.ld = t->ld; s.max_sq = t->max_sq;
  return s;
}
inline LossCfg make_loss(const gm_loss_t* l) {
  LossCfg c;
  c.kind = l->kind; c.inc_l1 = l->inc_l1; c.inc_l2 = l->inc_l2; c.alpha = l->alpha; c.eps = l->eps;
  return c;
}
int validate_pairs(const gm_pairs_t* p);
int check_loss(const gm_loss_t* loss);

// factor distance vectors of a product manifold and their softplus(scale) weights (modules.py:84-88)
struct FactorPtrs {
  const void* d2[8];
  double sp[8];
};

// ---- fused product-manifold launch: the vector factors evaluated next to the lead factor (gm_product.cuh) ----
constexpr int kMaxVecExtra = 3;
struct VecExtra {
  int kind, n, slot;  // slot: position of the factor in the product's factor list
  const void* x;
  void* g;
  double sp;          // softplus(scale) of the factor
};
struct ProductExtra {
  int F, lead_slot, nvec;  // lead_slot: slot of the SPD factor, -1 when the product has none
  VecExtra v[kMaxVecExtra];
};

// ---- one pair-kernel launch request (filled by gm_api.cu) --------------------
enum { K_FWD = 0, K_BWD = 1, K_FUSED = 2 };
struct PairArgs {
  int kind, dtype, n, p;
  unsigned flags;
  double wmin, wmax;
  const void* c_dev;  // GM_UNIVERSAL: device scalar c
  double* c_grad;     // GM_UNIVERSAL: optional device accumulator of d(loss)/dc
  int kmode;
  PairSpec ps;
  const void* xa;
  const void* xb;
  const void* gout;
  double coef;
  void* ga;
  void* gb;
  void* out_d2;
  TargetSpec tg;
  LossCfg lc;
  double scale_sp;
  double* acc;
  cudaStream_t stream;
  const ProductExtra* px;  // K_FUSED only: non-null = product-manifold launch (acc has 1 + F slots)
  ShardTab sh;             // row-sharded tables (xa / xb / ga / gb ignored) when sh.log2w >= 0
};

// The per-mode kernel arguments of a pair launch: the buffers a mode does not use are passed as NULL / 0.
template <typename T, int KMODE>
struct ModeArgs {
  static constexpr int kmode = KMODE;
  const T* gout;
  T coef;
  T* ga;
  T* gb;
  T* out_d2;
  T scale_sp;
  double* acc;
  double* c_grad;
  explicit ModeArgs(const PairArgs& a)
      : gout(KMODE == K_BWD ? (const T*)a.gout : nullptr), coef(KMODE == K_BWD ? (T)a.coef : (T)0),
        ga(KMODE == K_FWD ? nullptr : (T*)a.ga), gb(KMODE == K_FWD ? nullptr : (T*)a.gb),
        out_d2(KMODE == K_BWD ? nullptr : (T*)a.out_d2), scale_sp(KMODE == K_FUSED ? (T)a.scale_sp : (T)0),
        acc(KMODE == K_FUSED ? a.acc : nullptr), c_grad(KMODE == K_FWD ? nullptr : a.c_grad) {}
};

// launch(ModeArgs<T, a.kmode>) for a one-pair-per-thread kernel, counted
template <typename T, class Launch>
int launch_by_mode(const PairArgs& a, Launch&& launch) {
  switch (a.kmode) {
    case K_FWD: launch(ModeArgs<T, K_FWD>(a)); break;
    case K_BWD: launch(ModeArgs<T, K_BWD>(a)); break;
    default: launch(ModeArgs<T, K_FUSED>(a));
  }
  note_launch();
  return check_launch();
}

// ---- pair enumeration --------------------------------------------------------
__device__ __forceinline__ long long load_index(const void* p, long long k, int idx64) {
  return idx64 ? ((const long long*)p)[k] : (long long)((const int*)p)[k];
}

// first pair index of row a in torch.triu_indices(B, B, 1) order (base.py:62)
__device__ __forceinline__ long long triu_row_start(long long a, long long B) {
  return a * (2 * B - a - 1) / 2;
}

// k -> (a, b), a < b, row-major upper triangle; exact for B up to 2^31
__device__ __forceinline__ void triu_decode(long long k, long long B, long long& a, long long& b) {
  double tb = (double)(2 * B - 1);
  long long r = (long long)floor((tb - sqrt(tb * tb - 8.0 * (double)k)) * 0.5);
  if (r < 0) r = 0;
  if (r > B - 2) r = B - 2;
  while (r + 1 <= B - 2 && triu_row_start(r + 1, B) <= k) ++r;
  while (r > 0 && triu_row_start(r, B) > k) --r;
  a = r;
  b = k - triu_row_start(r, B) + r + 1;
}

// GM_PAIRS_SAMPLED: source row of pair k and the packed word (hop << 24) | j of its drawn target
// (include/gm_kernels.h states the draw; oracle/sampler_oracle.py restates it on the host).
__host__ __device__ __forceinline__ unsigned sample_hash32(unsigned long long seed, unsigned long long k) {
  unsigned long long z = seed + (k + 1ull) * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (unsigned)(z >> 32);
}
// the drawn target j of pair k, its source row `ra`, and WHERE its hop count lives (so that a pipelined caller can
// issue that load long before it needs the value)
__device__ __forceinline__ unsigned sampled_j(const PairSpec& ps, long long k, long long& ra,
                                              const unsigned char*& hop_ptr) {
  const long long g = ps.per_shift >= 0 ? (k >> ps.per_shift) : (k / ps.per_src);
  const unsigned i = (unsigned)((const int*)ps.idx_i)[g];
  const long long slot = ps.slots ? (long long)ps.slots[g] : g;
  unsigned j = __umulhi(sample_hash32(ps.seed, (unsigned long long)k), (unsigned)(ps.n_nodes - 1));
  j += (j >= i) ? 1u : 0u;
  hop_ptr = ps.levels + slot * ps.n_nodes + j;
  ra = (long long)i;
  return j;
}
// One random byte out of a multi-GB table per pair: streaming (evict-first) so that it does not push the gradient and
// point tables out of L2.
__device__ __forceinline__ unsigned load_hop(const unsigned char* p) { return (unsigned)__ldcs(p); }
__device__ __forceinline__ unsigned sampled_word(const PairSpec& ps, long long k, long long& ra) {
  const unsigned char* hp;
  const unsigned j = sampled_j(ps, k, ra, hp);
  return (load_hop(hp) << 24) | j;
}

// rows of xa / xb touched by pair k (also the rows gradients go to)
__device__ __forceinline__ void decode_pair(const PairSpec& ps, long long k, long long& ra, long long& rb) {
  if (ps.mode == GM_PAIRS_ELEMENTWISE) {
    ra = k; rb = k;
  } else if (ps.mode == GM_PAIRS_SAMPLED) {
    rb = (long long)(sampled_word(ps, k, ra) & 0x00ffffffu);
  } else if (ps.mode == GM_PAIRS_LIST) {
    ra = load_index(ps.idx_i, k, ps.idx64);
    rb = ps.idx64 ? ((const long long*)ps.idx_j)[k] : (long long)(((const unsigned*)ps.idx_j)[k] & ps.jmask);
  } else {
    long long a, b;
    triu_decode(k + ps.k0, ps.B, a, b);
    if (ps.nodes) { ra = load_index(ps.nodes, a, ps.idx64); rb = load_index(ps.nodes, b, ps.idx64); }
    else { ra = a; rb = b; }
  }
}

// graph target of pair k (data/dataset.py:9-27)
template <typename T>
__device__ __forceinline__ T fetch_target(const TargetSpec& tg, long long k, long long ra, long long rb) {
  if (tg.mode == GM_TGT_VECTOR) return ((const T*)tg.data)[k];
  if (tg.mode == GM_TGT_DENSE) return ((const T*)tg.data)[ra * tg.ld + rb];
  T h = (tg.mode == GM_TGT_HOPS_U8) ? (T)((const unsigned char*)tg.data)[k]
        : (tg.mode == GM_TGT_HOPS_U16) ? (T)((const unsigned short*)tg.data)[k]
                                       : (T)(((const unsigned*)tg.data)[k] >> 24);  // HOPS_PACKED: data == idx_j
  return (h * h) / (T)tg.max_sq;  // pow(2) then div_(max): dataset.py:11-12
}

// fetch_target for kernels that enumerate pairs themselves: SAMPLED pairs carry their hop count in the drawn word
template <typename T>
__device__ __forceinline__ T fetch_target_ps(const PairSpec& ps, const TargetSpec& tg, long long k, long long ra,
                                             long long rb) {
  if (ps.mode == GM_PAIRS_SAMPLED && tg.mode == GM_TGT_HOPS_PACKED) {
    long long dummy;
    T h = (T)(sampled_word(ps, k, dummy) >> 24);
    return (h * h) / (T)tg.max_sq;
  }
  return fetch_target<T>(tg, k, ra, rb);
}

// m_k = sum_f sp_f * d2_f[k]: sum() of a Python list starts from int 0 and adds left to right (modules.py:84-88)
template <typename T>
__device__ __forceinline__ T product_dist2(int F, const FactorPtrs& fp, long long k) {
  T m = (T)0;
  for (int f = 0; f < F; ++f) {
    T term = (T)fp.sp[f] * ((const T*)fp.d2[f])[k];
    m = (f == 0) ? term : m + term;
  }
  return m;
}

// ---- row I/O ---------------------------------------------------------------
template <typename T, int E>
__device__ __forceinline__ void load_row(const T* __restrict__ base, long long row, T (&r)[E]) {
  const T* p = base + row * E;
  if constexpr ((E * sizeof(T)) % 16 == 0) {
    constexpr int V = 16 / sizeof(T);
    const float4* q = reinterpret_cast<const float4*>(p);
    GM_UNROLL for (int k = 0; k < E / V; ++k) {
      float4 t = __ldg(q + k);
      const T* tt = reinterpret_cast<const T*>(&t);
      GM_UNROLL for (int j = 0; j < V; ++j) r[k * V + j] = tt[j];
    }
  } else if constexpr ((E * sizeof(T)) % 8 == 0) {
    constexpr int V = 8 / sizeof(T);
    const float2* q = reinterpret_cast<const float2*>(p);
    GM_UNROLL for (int k = 0; k < E / V; ++k) {
      float2 t = __ldg(q + k);
      const T* tt = reinterpret_cast<const T*>(&t);
      GM_UNROLL for (int j = 0; j < V; ++j) r[k * V + j] = tt[j];
    }
  } else {
    GM_UNROLL for (int k = 0; k < E; ++k) r[k] = __ldg(p + k);
  }
}

template <typename T, int E>
__device__ __forceinline__ void store_row(T* __restrict__ base, long long row, const T (&r)[E]) {
  T* p = base + row * E;
  if constexpr ((E * sizeof(T)) % 16 == 0) {
    constexpr int V = 16 / sizeof(T);
    float4* q = reinterpret_cast<float4*>(p);
    GM_UNROLL for (int k = 0; k < E / V; ++k) {
      float4 t;
      T* tt = reinterpret_cast<T*>(&t);
      GM_UNROLL for (int j = 0; j < V; ++j) tt[j] = r[k * V + j];
      q[k] = t;
    }
  } else {
    GM_UNROLL for (int k = 0; k < E; ++k) p[k] = r[k];
  }
}

// red.global.add of one row; fp32 rows whose byte size is a multiple of 16 use the
// sm_90+ 128-bit vector reduction (REDG.E.ADD.F32x4), fp64 uses scalar REDG.64.
template <typename T, int E>
__device__ __forceinline__ void atomic_add_row(T* __restrict__ base, long long row, const T (&r)[E]) {
  T* p = base + row * E;
  if constexpr (sizeof(T) == 4 && E % 4 == 0) {
    GM_UNROLL for (int k = 0; k < E / 4; ++k)
      atomicAdd(reinterpret_cast<float4*>(p) + k, make_float4(r[4 * k], r[4 * k + 1], r[4 * k + 2], r[4 * k + 3]));
  } else if constexpr (sizeof(T) == 4 && E % 2 == 0) {
    GM_UNROLL for (int k = 0; k < E / 2; ++k)
      atomicAdd(reinterpret_cast<float2*>(p) + k, make_float2(r[2 * k], r[2 * k + 1]));
  } else {
    GM_UNROLL for (int k = 0; k < E; ++k) atomicAdd(p + k, r[k]);
  }
}

// Accumulate one gradient row per lane.  Lanes of a warp that target the same
// row (the common case for the `a` side of TRIU / source-major pair lists) are
// first summed with shuffles so that one lane issues the reduction.
// Must be called by all 32 lanes; `row < 0` marks an idle lane.
template <typename T, int E>
__device__ __forceinline__ void warp_accumulate_row(T* __restrict__ base, long long row, T (&r)[E]) {
  const unsigned full = 0xffffffffu;
  long long row0 = __shfl_sync(full, row, 0);
  bool uniform = __all_sync(full, row == row0);
  if (uniform) {
    if (row0 < 0) return;
    GM_UNROLL for (int k = 0; k < E; ++k) r[k] = warp_sum(r[k]);
    if ((threadIdx.x & 31) == 0) atomic_add_row<T, E>(base, row0, r);
  } else if (row >= 0) {
    atomic_add_row<T, E>(base, row, r);
  }
}

}  // namespace gm
