// SPD pair kernels (affine-invariant distance and Stein divergence), one pair
// per thread, the n x n math register resident.  Compiled once per matrix size:
//   nvcc -DGM_N=<n> ... gm_pairs_spd.cu -o gm_pairs_spd_<n>.o
// and exposes gm::spd_launch_<n>(...) to the dispatcher in gm_api.cu.
//
// Replaces SymmetricPositiveDefinite.dist / pdist / stein_div / stein_pdiv and
// their autograd backward (manifolds/spd.py:171-194,246-295), fused with the
// gather x[m[0]], x[m[1]] (base.py:62-63), the loss (objectives.py:16-45) and
// the index_put_ scatter-add of the gradients (SURVEY 8a A3-A5, A10, A11).
#include "gm_product.cuh"

#ifndef GM_N
#error "compile with -DGM_N=<matrix size>"
#endif

namespace gm {

template <class Op, typename T, int KMODE>
__global__ void __launch_bounds__(128)
spd_pair_kernel(Op op, PairSpec ps, const T* __restrict__ xa, const T* __restrict__ xb,
                const T* __restrict__ gout, T coef, T* __restrict__ ga, T* __restrict__ gb,
                T* __restrict__ out_d2, TargetSpec tg, LossCfg lc, T scale_sp, double* __restrict__ acc) {
  constexpr int E = Op::E;
  __shared__ double red[2][4];
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = k < ps.P;
  long long ra = -1, rb = -1;
  double loss_v = 0.0, gd2_v = 0.0;
  T gx[E], gy[E];
  if (active) {
    decode_pair(ps, k, ra, rb);
    T x[E], y[E];
    load_row<T, E>(xa, ra, x);
    load_row<T, E>(xb, rb, y);
    if constexpr (KMODE == K_FWD) {
      out_d2[k] = op.dist2(x, y);
    } else {
      T d2 = op.dist2_grad(x, y, gx, gy);
      T w;
      if constexpr (KMODE == K_BWD) {
        w = coef * gout[k];
      } else {
        T g = fetch_target_ps<T>(ps, tg, k, ra, rb);
        T m = scale_sp * d2;
        T dm;
        T lv = loss_term<T>(lc, g, m, dm);
        loss_v = (double)lv;
        gd2_v = (double)dm * (double)d2;
        w = dm * scale_sp;
        if (out_d2) out_d2[k] = d2;
      }
      GM_UNROLL for (int e = 0; e < E; ++e) { gx[e] *= w; gy[e] *= w; }
    }
  }
  if constexpr (KMODE != K_FWD) {
    if (ps.mode == GM_PAIRS_ELEMENTWISE) {
      if (active) {
        store_row<T, E>(ga, ra, gx);
        store_row<T, E>(gb, rb, gy);
      }
    } else {
      warp_accumulate_row<T, E>(ga, ra, gx);
      warp_accumulate_row<T, E>(gb, rb, gy);
    }
  }
  if constexpr (KMODE == K_FUSED) {
    block_accumulate(loss_v, acc, red[0]);
    block_accumulate(gd2_v, acc + 1, red[1]);
  }
}

// ---------------------------------------------------------------------------
// Streaming variant for LIST / TRIU pair sets (the training hot path).
//
// Persistent grid; every warp owns a contiguous range of pairs and walks it 32
// pairs at a time.  Per lane, a 3-deep software pipeline hides the gather:
//   iteration it   : compute pair k(it) from rows staged in shared memory
//   issued in `it` : cp.async (LDGSTS) of both endpoint rows + target of pair k(it+1)
//                    index loads of pair k(it+2)
// Each thread stages into its own slots (layout [stage][row][16B-chunk][thread],
// bank-conflict free), so no block barrier is needed inside the loop.
// Consecutive pairs of a warp usually share the first endpoint (TRIU order,
// source-major pair lists): its inverse Cholesky factor is cached in registers
// and its gradient is accumulated in registers across iterations, reduced over
// the warp with shuffles and flushed with ONE vector reduction when the row
// changes.  The loss is accumulated per thread and block-reduced once.
// ---------------------------------------------------------------------------
template <int BYTES>
__device__ __forceinline__ void cp_async(void* smem, const void* gmem) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  if constexpr (BYTES == 16)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem) : "memory");
  else if constexpr (BYTES == 8)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(s), "l"(gmem) : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(s), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }
template <int PENDING>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;\n" ::"n"(PENDING) : "memory"); }

template <typename T, int E, int STAGES = 2>
struct RowStage {
  static constexpr int ROWB = E * (int)sizeof(T);
  static constexpr int CPB = (ROWB % 16 == 0) ? 16 : ((ROWB % 8 == 0) ? 8 : 4);
  static constexpr int NCH = ROWB / CPB;
  static constexpr int THREADS = 128;
  static constexpr int BYTES = STAGES * 2 /*rows*/ * ROWB * THREADS;
  // slot of chunk c of row r (0: a side, 1: b side) of stage s for thread t
  __device__ __forceinline__ static char* slot(char* base, int s, int r, int c, int t) {
    return base + ((((s * 2 + r) * NCH + c) * THREADS + t) * CPB);
  }
  __device__ __forceinline__ static void issue(char* base, int s, int r, int t, const T* row) {
    const char* g = reinterpret_cast<const char*>(row);
    GM_UNROLL for (int c = 0; c < NCH; ++c) cp_async<CPB>(slot(base, s, r, c, t), g + c * CPB);
  }
  __device__ __forceinline__ static void read(char* base, int s, int r, int t, T (&out)[E]) {
    GM_UNROLL for (int c = 0; c < NCH; ++c) {
      if constexpr (CPB == 16) {
        float4 v = *reinterpret_cast<const float4*>(slot(base, s, r, c, t));
        const T* tv = reinterpret_cast<const T*>(&v);
        GM_UNROLL for (int j = 0; j < 16 / (int)sizeof(T); ++j) out[c * (16 / (int)sizeof(T)) + j] = tv[j];
      } else if constexpr (CPB == 8) {
        float2 v = *reinterpret_cast<const float2*>(slot(base, s, r, c, t));
        const T* tv = reinterpret_cast<const T*>(&v);
        GM_UNROLL for (int j = 0; j < 8 / (int)sizeof(T); ++j) out[c * (8 / (int)sizeof(T)) + j] = tv[j];
      } else {
        out[c] = *reinterpret_cast<const T*>(slot(base, s, r, c, t));
      }
    }
  }
};

// TRIU position of one lane's look-ahead pair: walks k, k+32, k+64, ... (LIST pairs need no state beyond k)
struct PairCursor {
  long long a, pos;  // TRIU: row a, position inside the row
  int slot;          // SAMPLED: level row of the cached group
  __device__ __forceinline__ void init(const PairSpec& ps, long long k0) {
    if (ps.mode == GM_PAIRS_TRIU && k0 < ps.P) {
      long long b;
      triu_decode(k0 + ps.k0, ps.B, a, b);
      pos = b - a - 1;
    } else {
      a = -1; pos = 0; slot = 0;  // SAMPLED: no group cached yet
    }
  }
  __device__ __forceinline__ void rows(const PairSpec& ps, long long k, long long& ra, long long& rb) const {
    if (ps.mode == GM_PAIRS_LIST) {
      ra = load_index(ps.idx_i, k, ps.idx64);
      rb = load_index(ps.idx_j, k, ps.idx64);  // raw word: HOPS_PACKED callers split off the top byte
    } else if (ps.mode == GM_PAIRS_SAMPLED) {
      const unsigned char* hp;  // callers that want the hop count use rows_sampled()
      rb = (long long)sampled_j(ps, k, ra, hp);
    } else {
      long long b = a + 1 + pos;
      if (ps.nodes) { ra = load_index(ps.nodes, a, ps.idx64); rb = load_index(ps.nodes, b, ps.idx64); }
      else { ra = a; rb = b; }
    }
  }
  // SAMPLED: the drawn pair, plus its hop count as a load issued NOW and (by a pipelined caller) consumed an
  // iteration later -- nothing is read per pair except that one byte
  // The source id and level row of the lane's current group are cached (a group is thousands of consecutive pairs):
  // the draw itself then depends on no load at all, and the hop load can be issued straight away.
  __device__ __forceinline__ void rows_sampled(const PairSpec& ps, long long k, long long& ra, long long& rb,
                                               unsigned& hop) {
    const int g = (int)(ps.per_shift >= 0 ? (k >> ps.per_shift) : (k / ps.per_src));
    if (g != a) {  // (a, pos) are free in SAMPLED mode: a = cached group, pos = its source id; row in `slot`
      a = g;
      pos = ((const int*)ps.idx_i)[g];
      slot = ps.slots ? ps.slots[g] : g;
    }
    const unsigned i = (unsigned)pos;
    unsigned j = __umulhi(sample_hash32(ps.seed, (unsigned long long)k), (unsigned)(ps.n_nodes - 1));
    j += (j >= i) ? 1u : 0u;
    hop = load_hop(ps.levels + (long long)slot * ps.n_nodes + j);
    ra = (long long)i;
    rb = (long long)j;
  }
  __device__ __forceinline__ void advance(const PairSpec& ps) {
    if (ps.mode == GM_PAIRS_TRIU) {
      pos += 32;
      while (a < ps.B - 1 && pos >= ps.B - a - 1) { pos -= ps.B - a - 1; ++a; }
    }
  }
};

// Row ids are carried as 32-bit values when a table of 2^32 such rows cannot exist (>= 64-byte rows: 274 GB).
template <int ROWBYTES, bool SMALL = (ROWBYTES >= 64)> struct RowId { using type = long long; };
template <int ROWBYTES> struct RowId<ROWBYTES, true> { using type = unsigned; };

// Raw per-pair scalar carried through the pipeline: the bits of a T (explicit target / upstream gradient) or, for
// hop-count targets, the integer hop count.  Hop counts are mapped to (h^2)/max -- dataset.py:11-12, IEEE division so
// that the value is bit-identical to the reference's -- through a 256-entry table built once per block (HOPS_U8) or
// on the fly (HOPS_U16).
template <typename T> struct RawScalar;
template <> struct RawScalar<float> {
  using type = unsigned;
  __device__ __forceinline__ static unsigned pack(float v) { return __float_as_uint(v); }
  __device__ __forceinline__ static float unpack(unsigned r) { return __uint_as_float(r); }
};
template <> struct RawScalar<double> {
  using type = unsigned long long;
  __device__ __forceinline__ static unsigned long long pack(double v) { return (unsigned long long)__double_as_longlong(v); }
  __device__ __forceinline__ static double unpack(unsigned long long r) { return __longlong_as_double((long long)r); }
};

// SPEC = 1: the launch is known to be explicit int32 lists in window order (gm_pairs_t.segments > 1) with the hop count
// packed into the top byte of idx_j and plain (not row-sharded) tables -- the BASELINE config 5 training step as
// bench.py runs it.  Every mode test folds away at compile time and the walk position is carried as (segment, offset)
// instead of being divided out: measured 0.957 vs 1.040 ms for the general instantiation on the same window-ordered
// batch (profiles/r02_pair_kernel_ab.txt run 10); with resident rows the kernel is issue bound and these count.
template <class Op, typename T, int KMODE, int MINB, int DEPTH, int SPEC = 0>
__global__ void __launch_bounds__(128, MINB)
spd_pair_stream_kernel(Op op, PairSpec ps, const T* __restrict__ xa, const T* __restrict__ xb,
                       const T* __restrict__ gout, T coef, T* __restrict__ ga, T* __restrict__ gb,
                       T* __restrict__ out_d2, TargetSpec tg, LossCfg lc, T scale_sp, double* __restrict__ acc,
                       long long chunk, const ShardTab sh) {
  constexpr int E = Op::E;
  constexpr int N = GM_N;
  constexpr int EU = N * (N + 1) / 2;  // gradients are symmetric: the run-length accumulator keeps the upper triangle
  constexpr int D = DEPTH;  // a pair's rows are in flight for D iterations of the loop (D + 1 staging slots per thread)
  using Stage = RowStage<T, E, D + 1>;
  using Raw = RawScalar<T>;
  using raw_t = typename Raw::type;
  extern __shared__ __align__(16) char stage_mem[];
  __shared__ double red[2][4];
  __shared__ T hop_lut[256];
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned full = 0xffffffffu;
  const long long warp_id = (long long)blockIdx.x * 4 + (tid >> 5);
  // A warp owns `chunk` consecutive pairs of every segment of the list (one segment unless the caller cut a LIST into
  // ps.nseg parts that the whole grid should walk one after another -- see gm_pairs_t.segments): position t of its
  // walk, t = 0, 32, 64, ..., is pair (t / chunk) * seg_len + warp_id * chunk + t % chunk + lane.
  const long long wbase = warp_id * chunk + lane;
  const int nseg = ps.nseg;
  auto locate = [&](int t, long long& k) -> bool {
    int s = 0, o = t;
    if (nseg > 1) {
      s = t / (int)chunk;
      o = t - s * (int)chunk;
      if (s >= nseg) return false;
    } else if (t >= chunk) {
      return false;
    }
    const long long in_seg = wbase + o;
    k = (long long)s * ps.seg_len + in_seg;
    return in_seg < ps.seg_len && k < ps.P;
  };
  [[maybe_unused]] auto locate_so = [&](int s, int o, long long& k) -> bool {  // SPEC: position given as (segment, offset)
    if (s >= nseg) return false;
    const long long in_seg = wbase + o;
    k = (long long)s * ps.seg_len + in_seg;
    return in_seg < ps.seg_len && k < ps.P;
  };
  const bool hopsP = SPEC ? true : (KMODE == K_FUSED) && tg.mode == GM_TGT_HOPS_PACKED;  // hop count in the top byte of idx_j
  const bool hops8 = SPEC ? true : (KMODE == K_FUSED) && (tg.mode == GM_TGT_HOPS_U8 || hopsP);
  const bool hops16 = SPEC ? false : (KMODE == K_FUSED) && tg.mode == GM_TGT_HOPS_U16;
  const bool rawj = SPEC ? true : hopsP || ps.mode == GM_PAIRS_SAMPLED;  // j arrives with a hop count in its top byte
  if (hops8) {
    for (int h = tid; h < 256; h += 128) hop_lut[h] = ((T)h * (T)h) / (T)tg.max_sq;
    __syncthreads();
  }

  // ---- pipeline registers -------------------------------------------------------------------------------------
  using row_t = typename RowId<E * (int)sizeof(T)>::type;
  const row_t kNoRow = (row_t)-1;
  // Row-sharded tables (gm_row_shards_t, sh.log2w >= 0): global row v is row v >> log2w of rank (v & mask)'s shard --
  // local memory or a peer's, mapped over NVLink -- for the point gathers and the gradient reductions alike.
  const bool sharded = SPEC ? false : sh.log2w >= 0;
  auto xrow = [&](const T* base, row_t r) -> const T* {
    if (sharded) return (const T*)sh.x[(unsigned)r & sh.mask] + (size_t)((unsigned long long)r >> sh.log2w) * E;
    return base + (size_t)r * E;
  };
  auto grow = [&](T* base, row_t r, long long& lr) -> T* {
    lr = (long long)r;
    if (sharded) { base = (T*)sh.g[(unsigned)r & sh.mask]; lr = (long long)((unsigned long long)r >> sh.log2w); }
    return base;
  };
  int tc = 0;         // position (in the warp's walk) of the pair computed in this iteration (rows staged in `stage`)
  PairCursor ahead;   // TRIU position of the furthest pair whose indices have been loaded
  // queue of the pairs at positions tc + 32 q: q = 0 is computed now, q = 1..D-1 have their rows in flight, q = D has its indices (rows
  // are issued this iteration), q = D + 1 is the pair whose indices are being loaded
  row_t ra[D + 2], rb[D + 2];
  raw_t tgq[D + 1];    // target (K_FUSED) or upstream gradient (K_BWD) of the pair, raw
  bool v[D + 2];
  unsigned hopn = 0;   // SAMPLED: hop count of pair q = D (load in flight since the previous iteration)
  GM_UNROLL for (int q = 0; q < D + 2; ++q) { ra[q] = kNoRow; rb[q] = kNoRow; v[q] = false; }
  GM_UNROLL for (int q = 0; q < D + 1; ++q) tgq[q] = 0;
  const bool sampled = SPEC ? false : ps.mode == GM_PAIRS_SAMPLED;
  int stage = 0;

  auto fetch_scalar = [&](long long k, row_t ra, row_t rb) -> raw_t {
    if constexpr (KMODE == K_BWD) {
      return Raw::pack(gout[k]);
    } else {
      if (hopsP) return (raw_t)(((unsigned)rb) >> 24);  // (SAMPLED pairs: see the callers)
      if (hops8) return (raw_t)((const unsigned char*)tg.data)[k];
      if (hops16) return (raw_t)((const unsigned short*)tg.data)[k];
      return Raw::pack(fetch_target<T>(tg, k, (long long)ra, (long long)rb));
    }
  };
  auto scalar_value = [&](raw_t r) -> T {
    if constexpr (KMODE == K_BWD) {
      return Raw::unpack(r);
    } else {
      if (hops8) return hop_lut[r];
      if (hops16) { T h = (T)r; return (h * h) / (T)tg.max_sq; }
      return Raw::unpack(r);
    }
  };
  auto load_rows = [&](long long k, row_t& ra, row_t& rb, unsigned& hop) {
    if constexpr (SPEC != 0) {
      ra = (row_t)((const int*)ps.idx_i)[k];
      rb = (row_t)(unsigned)((const int*)ps.idx_j)[k];
      return;
    }
    long long a, b;
    if (sampled) ahead.rows_sampled(ps, k, a, b, hop);
    else ahead.rows(ps, k, a, b);
    ra = (row_t)a; rb = (row_t)b;
  };

  ahead.init(ps, wbase);
  GM_UNROLL for (int q = 0; q < D; ++q) {
    long long kq = 0;
    v[q] = locate(32 * q, kq);
    if (v[q]) {
      unsigned hop = 0;
      load_rows(kq, ra[q], rb[q], hop);
      tgq[q] = (sampled && hopsP) ? (raw_t)hop : fetch_scalar(kq, ra[q], rb[q]);
      if (rawj) rb[q] &= (row_t)0x00ffffffu;
      Stage::issue(stage_mem, q, 0, tid, xrow(xa, ra[q]));
      Stage::issue(stage_mem, q, 1, tid, xrow(xb, rb[q]));
    }
    cp_async_commit();
    ahead.advance(ps);
  }
  {
    long long kq = 0;
    v[D] = locate(32 * D, kq);
    if (v[D]) load_rows(kq, ra[D], rb[D], hopn);
  }
  // SPEC: (segment, offset) of the walk position whose indices are loaded next, tc + 32 (D + 1)
  [[maybe_unused]] int hs = SPEC ? (32 * (D + 1)) / (int)chunk : 0;
  [[maybe_unused]] int ho = SPEC ? 32 * (D + 1) - hs * (int)chunk : 0;

  // ---- per-lane running state -------------------------------------------------------------------------------------
  double loss_v = 0.0, gd2_v = 0.0;
  row_t acc_row = kNoRow;  // warp-uniform row whose gradient is being accumulated in gacc
  T gacc[EU];
  GM_UNROLL for (int e = 0; e < EU; ++e) gacc[e] = (T)0;
  row_t prep_row = kNoRow;
  T ap[Op::kPrepSize];

  auto flush = [&]() {
    if (acc_row != kNoRow) {
      GM_UNROLL for (int e = 0; e < EU; ++e) gacc[e] = warp_sum(gacc[e]);
      if (lane == 0) {
        T gfull[E];
        GM_UNROLL for (int i = 0; i < N; ++i)
          GM_UNROLL for (int j = i; j < N; ++j) {
            gfull[i * N + j] = gacc[i * N - i * (i - 1) / 2 + (j - i)];
            gfull[j * N + i] = gfull[i * N + j];
          }
        long long lr;
        T* gbase = grow(ga, acc_row, lr);
        atomic_add_row<T, E>(gbase, lr, gfull);
      }
      GM_UNROLL for (int e = 0; e < EU; ++e) gacc[e] = (T)0;
      acc_row = kNoRow;
    }
  };

  // one segment: the walk ends at the first position nobody holds a pair at.  Several: the warp that straddles the end
  // of a segment idles through the rest of its chunk and resumes in the next segment, so the walk runs to its end.
  const int t_end = (nseg > 1 && wbase - lane < ps.seg_len) ? nseg * (int)chunk : 0;
  while (nseg > 1 ? tc < t_end : __any_sync(full, v[0])) {
    // (1) rows of the current pair have landed in my slots (the D - 1 younger groups may still be in flight)
    cp_async_wait_group<D - 1>();
    const bool v0 = v[0];
    const row_t ra0 = ra[0], rb0 = rb[0];
    const raw_t tg0 = tgq[0];
    T x[E], y[E];
    if (v0) {
      Stage::read(stage_mem, stage, 1, tid, y);
      if (!Op::kCanPrep || ra0 != prep_row) Stage::read(stage_mem, stage, 0, tid, x);
    }
    // (2) issue the rows of pair q = D: rows via LDGSTS, scalar via LDG; (3) indices of the pair after it
    tgq[D] = 0;
    if (v[D]) {
      long long kq = 0;
      if (KMODE == K_BWD || !hopsP) locate(tc + 32 * D, kq);  // (a packed hop count needs no pair index)
      tgq[D] = (sampled && hopsP) ? (raw_t)hopn : fetch_scalar(kq, ra[D], rb[D]);
      if (rawj) rb[D] &= (row_t)0x00ffffffu;
      int sn = stage + D;
      if (sn > D) sn -= D + 1;
      Stage::issue(stage_mem, sn, 0, tid, xrow(xa, ra[D]));
      Stage::issue(stage_mem, sn, 1, tid, xrow(xb, rb[D]));
    }
    cp_async_commit();
    ahead.advance(ps);
    long long kh = 0;
    if constexpr (SPEC != 0) {
      v[D + 1] = locate_so(hs, ho, kh);
      ho += 32;
      if (ho >= (int)chunk) { ho -= (int)chunk; ++hs; }
    } else {
      v[D + 1] = locate(tc + 32 * (D + 1), kh);
    }
    ra[D + 1] = kNoRow; rb[D + 1] = kNoRow;
    unsigned hop_next = 0;
    if (v[D + 1]) load_rows(kh, ra[D + 1], rb[D + 1], hop_next);

    // (4) the math
    T gx[E], gy[E];
    if (v0) {
      T d2, w;
      [[maybe_unused]] typename Op::EigState st;
      if constexpr (Op::kCanPrep) {
        if (ra0 != prep_row) { op.prep(x, ap); prep_row = ra0; }
        d2 = op.eig_forward_prepped(ap, y, st);
      } else {
        d2 = op.dist2_grad(x, y, gx, gy);
      }
      if constexpr (KMODE == K_BWD) {
        w = coef * scalar_value(tg0);
      } else {
        T m = scale_sp * d2;
        T dm;
        T lv = loss_term<T, true>(lc, scalar_value(tg0), m, dm);
        loss_v += (double)lv;
        gd2_v += (double)dm * (double)d2;
        w = dm * scale_sp;
        if (out_d2) {
          long long k0 = 0;
          locate(tc, k0);
          out_d2[k0] = d2;
        }
      }
      if constexpr (Op::kCanPrep) {
        op.eig_backward(st, w, gx, gy);  // loss weight folded into the N eigen-coefficients
      } else {
        GM_UNROLL for (int e = 0; e < E; ++e) { gx[e] *= w; gy[e] *= w; }
      }
      long long lrb;
      T* gbb = grow(gb, rb0, lrb);
      atomic_add_row<T, E>(gbb, lrb, gy);
    }
    // (5) first-endpoint gradient: run-length accumulation in registers
    {
      row_t r0 = __shfl_sync(full, ra0, 0);
      bool uniform = __all_sync(full, v0 && ra0 == r0);
      if (uniform && r0 == acc_row) {
        GM_UNROLL for (int i = 0; i < N; ++i)
          GM_UNROLL for (int j = i; j < N; ++j) gacc[i * N - i * (i - 1) / 2 + (j - i)] += gx[i * N + j];
      } else {
        flush();
        if (uniform) {
          acc_row = r0;
          GM_UNROLL for (int i = 0; i < N; ++i)
            GM_UNROLL for (int j = i; j < N; ++j) gacc[i * N - i * (i - 1) / 2 + (j - i)] = gx[i * N + j];
        } else if (v0) {
          long long lra;
          T* gba = grow(ga, ra0, lra);
          atomic_add_row<T, E>(gba, lra, gx);
        }
      }
    }
    // (6) rotate the pipeline
    tc += 32;
    GM_UNROLL for (int q = 0; q < D + 1; ++q) { ra[q] = ra[q + 1]; rb[q] = rb[q + 1]; v[q] = v[q + 1]; }
    GM_UNROLL for (int q = 0; q < D; ++q) tgq[q] = tgq[q + 1];
    hopn = hop_next;
    stage = (stage == D) ? 0 : stage + 1;
  }
  flush();
  if constexpr (KMODE == K_FUSED) {
    block_accumulate(loss_v, acc, red[0]);
    block_accumulate(gd2_v, acc + 1, red[1]);
  }
}

template <class Op, typename T>
static int launch_op(const Op& op, const PairArgs& a) {
  if (a.ps.P <= 0) return 0;
  if (a.px) return a.sh.log2w >= 0 ? GM_EUNSUPPORTED : launch_product<SpdLead<Op>, T>(SpdLead<Op>{op}, a);
  const int threads = 128;
  long long blocks = (a.ps.P + threads - 1) / threads;
  if (blocks > 0x7fffffffLL) return GM_EINVAL;
  dim3 grid((unsigned)blocks), block(threads);
  const T* xa = (const T*)a.xa;
  const T* xb = (const T*)a.xb;
  constexpr int MINB = sizeof(T) == 4 ? 4 : 2;  // resident CTAs per SM the streaming kernel is built for
  constexpr int DEPTH = 1;                      // a pair's rows are in flight for one iteration of its loop
  using Stage = RowStage<T, Op::E, DEPTH + 1>;
  if (a.kmode != K_FWD && a.ps.mode != GM_PAIRS_ELEMENTWISE && RowStage<T, Op::E, 2>::BYTES <= 64 * 1024) {
    int dev = 0, sms = 0, occ = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    auto launch_stream = [&](auto m) -> int {
      constexpr int KMODE = decltype(m)::kmode;
      auto kern = spd_pair_stream_kernel<Op, T, KMODE, MINB, DEPTH>;
      cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Stage::BYTES);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, Stage::BYTES);
      if (occ < 1) occ = 1;
      long long max_blocks = (long long)sms * occ;
      long long want = (a.ps.P + threads - 1) / threads;
      long long nb = want < max_blocks ? want : max_blocks;
      long long warps = nb * (threads / 32);
      PairSpec ps = a.ps;
      if (ps.mode != GM_PAIRS_LIST || ps.nseg < 2 || ps.P < ps.nseg * 32LL * warps) ps.nseg = 1;  // (tiny lists: one walk)
      ps.seg_len = (ps.P + ps.nseg - 1) / ps.nseg;
      long long chunk = ((ps.seg_len + warps - 1) / warps + 31) / 32 * 32;
      if (chunk * ps.nseg > 0x7fffffffLL) return GM_EINVAL;
      if constexpr (KMODE == K_FUSED && GM_N == 4 && sizeof(T) == 4 && Op::kCanPrep) {  // the window-ordered config 5 step: see SPEC
        if (ps.nseg > 1 && !ps.idx64 && a.tg.mode == GM_TGT_HOPS_PACKED && a.sh.log2w < 0) {
          auto spec = spd_pair_stream_kernel<Op, T, K_FUSED, MINB, DEPTH, 1>;
          cudaFuncSetAttribute(spec, cudaFuncAttributeMaxDynamicSharedMemorySize, Stage::BYTES);
          spec<<<(unsigned)nb, threads, Stage::BYTES, a.stream>>>(op, ps, xa, xb, m.gout, m.coef, m.ga, m.gb, m.out_d2,
                                                                   a.tg, a.lc, m.scale_sp, m.acc, chunk, a.sh);
          note_launch();
          return check_launch();
        }
      }
      kern<<<(unsigned)nb, threads, Stage::BYTES, a.stream>>>(op, ps, xa, xb, m.gout, m.coef, m.ga, m.gb, m.out_d2, a.tg,
                                                             a.lc, m.scale_sp, m.acc, chunk, a.sh);
      note_launch();
      return check_launch();
    };
    if (a.kmode == K_BWD) return launch_stream(ModeArgs<T, K_BWD>(a));
    return launch_stream(ModeArgs<T, K_FUSED>(a));
  }
  if (a.sh.log2w >= 0) return GM_EUNSUPPORTED;  // row-sharded tables: the streaming (training) kernels only
  return launch_by_mode<T>(a, [&](auto m) {
    spd_pair_kernel<Op, T, decltype(m)::kmode><<<grid, block, 0, a.stream>>>(
        op, a.ps, xa, xb, m.gout, m.coef, m.ga, m.gb, m.out_d2, a.tg, a.lc, m.scale_sp, m.acc);
  });
}

template <typename T>
static int launch_typed(const PairArgs& a) {
  constexpr int N = GM_N;
  const bool fe = (a.flags & GM_FAST_EIG) != 0;
  const bool fc = (a.flags & GM_FAST_CHOL) != 0;
  if (a.kind == GM_SPD_AI) {
    if constexpr (N == 2) {
      if (fe && fc) { SpdAI<T, 2, true, true> op{(T)a.wmin, (T)a.wmax}; return launch_op<decltype(op), T>(op, a); }
      if (fe && !fc) { SpdAI<T, 2, true, false> op{(T)a.wmin, (T)a.wmax}; return launch_op<decltype(op), T>(op, a); }
      if (!fe && fc) { SpdAI<T, 2, false, true> op{(T)a.wmin, (T)a.wmax}; return launch_op<decltype(op), T>(op, a); }
    }
    if constexpr (N == 3) {
      if (fe) { SpdAI<T, 3, true, false> op{(T)a.wmin, (T)a.wmax}; return launch_op<decltype(op), T>(op, a); }
    }
    SpdAI<T, N, false, false> op{(T)a.wmin, (T)a.wmax};
    return launch_op<decltype(op), T>(op, a);
  }
  if (a.kind == GM_SPD_STEIN) {
    if constexpr (N == 2) {
      if (fc) { SpdStein<T, 2, true> op{(T)a.wmin, (T)a.wmax}; return launch_op<decltype(op), T>(op, a); }
    }
    SpdStein<T, N, false> op{(T)a.wmin, (T)a.wmax};
    return launch_op<decltype(op), T>(op, a);
  }
  return GM_EINVAL;
}

#define GM_CAT2(a, b) a##b
#define GM_CAT(a, b) GM_CAT2(a, b)
int GM_CAT(spd_launch_, GM_N)(const PairArgs& a) {
  if (a.dtype == GM_F32) return launch_typed<float>(a);
  if (a.dtype == GM_F64) return launch_typed<double>(a);
  return GM_EINVAL;
}

}  // namespace gm
