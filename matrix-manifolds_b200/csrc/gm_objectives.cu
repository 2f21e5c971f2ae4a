// Objective-side kernels that sit between the distance and the gradient kernels:
//   * streamed validation metrics (average distortion, Pearson moments) --
//     TrainingEngine._validate (train.py:230-265), metrics.py:13-17,46-56
//   * the KL-divergence objective with the stochastic-neighbour model --
//     objectives.py:48-76, inference/stochastic_neighbors.py:8-24
#include <cuda_runtime.h>
#include "gm_launch.cuh"

namespace gm {

// ---------------------------------------------------------------------------
// validation metrics
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
pairs_metrics_kernel(int F, FactorPtrs fp, PairSpec ps, TargetSpec tg, int squared, double* __restrict__ acc) {
  __shared__ double red[8];
  double v[7];
  for (int i = 0; i < 7; ++i) v[i] = 0.0;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < ps.P; k += stride) {
    long long ra = 0, rb = 0;
    if (tg.mode == GM_TGT_DENSE) decode_pair(ps, k, ra, rb);
    T g = fetch_target<T>(tg, k, ra, rb);
    T m;
    if (squared) {
      m = Num<T>::sqrt(product_dist2<T>(F, fp, k));  // compute_dists(None).sqrt_()   train.py:232
      g = Num<T>::sqrt(g);                           // graph_dataset[None].sqrt()    train.py:231
    } else {
      m = ((const T*)fp.d2[0])[k];
    }
    double md = (double)m, gd = (double)g;
    v[0] += 1.0;
    v[1] += (double)(Num<T>::abs(m - g) / g);  // metrics.py:56, evaluated in the tensor dtype
    v[2] += md; v[3] += gd; v[4] += md * md; v[5] += gd * gd; v[6] += md * gd;
  }
  for (int i = 0; i < 7; ++i) block_accumulate(v[i], acc + i, red);
}

// ---------------------------------------------------------------------------
// product-manifold loss over F distance vectors
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
product_loss_kernel(int F, FactorPtrs fp, TargetSpec tg, PairSpec ps, LossCfg lc, long long P,
                    double* __restrict__ acc, T* __restrict__ out_g) {
  __shared__ double red[8];
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = k < P;
  double lv = 0.0;
  double gd[8];
  for (int f = 0; f < 8; ++f) gd[f] = 0.0;
  if (active) {
    // sum() of a Python list starts from int 0 and adds left to right (modules.py:84-88)
    T m = (T)0;
    T d2[8];
    for (int f = 0; f < F; ++f) {
      d2[f] = ((const T*)fp.d2[f])[k];
      T term = (T)fp.sp[f] * d2[f];
      m = (f == 0) ? term : m + term;
    }
    long long ra = 0, rb = 0;
    if (tg.mode == GM_TGT_DENSE) decode_pair(ps, k, ra, rb);  // node ids index the dense target matrix
    T g = fetch_target<T>(tg, k, ra, rb);
    T dm;
    lv = (double)loss_term<T>(lc, g, m, dm);
    if (out_g) out_g[k] = dm;
    for (int f = 0; f < F; ++f) gd[f] = (double)dm * (double)d2[f];
  }
  block_accumulate(lv, acc, red);
  for (int f = 0; f < F; ++f) block_accumulate(gd[f], acc + 1 + f, red);
}

// ---------------------------------------------------------------------------
// stochastic-neighbour KL objective
// ---------------------------------------------------------------------------
struct SneCfg {
  long long B;
  double alpha;
  int inclusive;
};

// condensed index of the unordered pair {i, j}, i != j
__device__ __forceinline__ long long cond_index(long long i, long long j, long long B) {
  long long a = i < j ? i : j, b = i < j ? j : i;
  return triu_row_start(a, B) + (b - a - 1);
}

template <typename T>
__device__ __forceinline__ void sne_thetas(int F, const FactorPtrs& fp, const T* __restrict__ g, const SneCfg& c,
                                           long long k, T& tx, T& tz) {
  T tg = -(T)c.alpha * g[k];           // -alpha * gdists   objectives.py:62
  T tm = -product_dist2<T>(F, fp, k);  // -mdists           objectives.py:63
  if (c.inclusive) { tx = tg; tz = tm; } else { tx = tm; tz = tg; }
}

// running (max, sum exp, sum exp*delta) of theta_x and (max, sum exp) of theta_z over part of a row
template <typename T>
struct RowAcc {
  T mx, sx, dx, mz, sz;
  __device__ __forceinline__ void init() { mx = -Num<T>::huge; sx = (T)0; dx = (T)0; mz = -Num<T>::huge; sz = (T)0; }
  __device__ __forceinline__ void add(T tx, T tz) {
    T delta = tz - tx;
    if (tx > mx) { T r = Num<T>::exp(mx - tx); sx *= r; dx *= r; mx = tx; }
    T e = Num<T>::exp(tx - mx);
    sx += e; dx += e * delta;
    if (tz > mz) { sz *= Num<T>::exp(mz - tz); mz = tz; }
    sz += Num<T>::exp(tz - mz);
  }
  __device__ __forceinline__ void merge(const RowAcc& o) {
    T nm = Num<T>::max(mx, o.mx);
    T ra = Num<T>::exp(mx - nm), rb = Num<T>::exp(o.mx - nm);  // exp(-huge - finite) == 0 for empty parts
    sx = sx * ra + o.sx * rb; dx = dx * ra + o.dx * rb; mx = nm;
    T nz = Num<T>::max(mz, o.mz);
    T za = Num<T>::exp(mz - nz), zb = Num<T>::exp(o.mz - nz);
    sz = sz * za + o.sz * zb; mz = nz;
  }
};

// One block per row i: logsumexp of theta_x and theta_z over j != i and the p_x-expectation of theta_z - theta_x.
// Entries (i, j > i) are contiguous in the condensed vector, entries (j < i, i) are strided.
template <typename T>
__global__ void __launch_bounds__(128)
sne_row_stats_kernel(int F, FactorPtrs fp, const T* __restrict__ g, SneCfg c, T* __restrict__ stats) {
  __shared__ RowAcc<T> sh[4];
  const long long i = blockIdx.x;
  RowAcc<T> r;
  r.init();
  for (long long j = threadIdx.x; j < c.B; j += blockDim.x) {
    if (j == i) continue;
    T tx, tz;
    sne_thetas<T>(F, fp, g, c, cond_index(i, j, c.B), tx, tz);
    r.add(tx, tz);
  }
  for (int o = 16; o > 0; o >>= 1) {
    RowAcc<T> t;
    t.mx = __shfl_xor_sync(0xffffffffu, r.mx, o); t.sx = __shfl_xor_sync(0xffffffffu, r.sx, o);
    t.dx = __shfl_xor_sync(0xffffffffu, r.dx, o); t.mz = __shfl_xor_sync(0xffffffffu, r.mz, o);
    t.sz = __shfl_xor_sync(0xffffffffu, r.sz, o);
    r.merge(t);
  }
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) sh[wid] = r;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r.merge(sh[w]);
    stats[i] = r.mx + Num<T>::log(r.sx);
    stats[c.B + i] = r.mz + Num<T>::log(r.sz);
    stats[2 * c.B + i] = r.dx / r.sx;
  }
}

// Per pair k = (a, b): marginals, the loss term and dKL/dm_k; threads k < B also add A_z - A_x of row k.
template <typename T>
__global__ void __launch_bounds__(256)
sne_pair_terms_kernel(int F, FactorPtrs fp, const T* __restrict__ g, SneCfg c, const T* __restrict__ stats,
                      long long P, double* __restrict__ acc, T* __restrict__ out_g) {
  __shared__ double red[8];
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  double lv = 0.0;
  double gd[8];
  for (int f = 0; f < 8; ++f) gd[f] = 0.0;
  if (k < c.B) lv += (double)stats[c.B + k] - (double)stats[k];  // A_z - A_x
  if (k < P) {
    long long a, b;
    triu_decode(k, c.B, a, b);
    T tx, tz;
    sne_thetas<T>(F, fp, g, c, k, tx, tz);
    T delta = tz - tx;
    T pab = Num<T>::exp(tx - stats[a]), pba = Num<T>::exp(tx - stats[b]);  // softmax rows a and b of theta_x
    T margx = pab + pba;
    lv -= (double)(margx * delta);
    T dm;
    if (c.inclusive) {
      // dKL/dtheta_z = margs_z - margs_x, theta_z = -m
      T margz = Num<T>::exp(tz - stats[c.B + a]) + Num<T>::exp(tz - stats[c.B + b]);
      dm = margx - margz;
    } else {
      // dKL/dtheta_x = -[p_ab (delta - D_a) + p_ba (delta - D_b)], theta_x = -m
      dm = pab * (delta - stats[2 * c.B + a]) + pba * (delta - stats[2 * c.B + b]);
    }
    if (out_g) out_g[k] = dm;
    for (int f = 0; f < F; ++f) gd[f] = (double)dm * (double)((const T*)fp.d2[f])[k];
  }
  block_accumulate(lv, acc, red);
  for (int f = 0; f < F; ++f) block_accumulate(gd[f], acc + 1 + f, red);
}

static int fill_factors(FactorPtrs& fp, int F, const void* const* ptrs, const double* sps) {
  if (!ptrs || !sps) return GM_ENULL;
  if (F < 1 || F > 8) return GM_EINVAL;
  for (int f = 0; f < F; ++f) {
    if (!ptrs[f]) return GM_ENULL;
    fp.d2[f] = ptrs[f];
    fp.sp[f] = sps[f];
  }
  return GM_OK;
}

}  // namespace gm

using namespace gm;

extern "C" {
#pragma GCC visibility push(default)

int gm_pairs_metrics(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                     const gm_pairs_t* pairs, const gm_targets_t* targets, int32_t squared_inputs, double* acc,
                     gm_stream_t stream) {
  if (!targets || !acc || !pairs) return GM_ENULL;
  if (dtype != GM_F32 && dtype != GM_F64) return GM_EINVAL;
  FactorPtrs fp{};
  int rc = fill_factors(fp, F, d2_ptrs_host, sp_host);
  if (rc) return rc;
  if (!squared_inputs && F != 1) return GM_EINVAL;
  if (targets->mode < GM_TGT_VECTOR || targets->mode > GM_TGT_HOPS_U16) return GM_EINVAL;
  if (targets->mode == GM_TGT_DENSE) {
    rc = validate_pairs(pairs);
    if (rc) return rc;
    if (pairs->mode == GM_PAIRS_ELEMENTWISE) return GM_EINVAL;
  }
  if (pairs->P < 0) return GM_EINVAL;
  if (pairs->P == 0) return GM_OK;
  if (!targets->data) return GM_ENULL;
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int threads = 256;
  long long want = (pairs->P + threads - 1) / threads;
  long long cap = (long long)sms * 8;  // grid-stride: a few resident blocks per SM, one atomic set per block
  unsigned blocks = (unsigned)(want < cap ? want : cap);
  PairSpec ps = make_pairs(pairs);
  TargetSpec tg = make_targets(targets);
  if (dtype == GM_F32)
    pairs_metrics_kernel<float><<<blocks, threads, 0, (cudaStream_t)stream>>>(F, fp, ps, tg, squared_inputs, acc);
  else
    pairs_metrics_kernel<double><<<blocks, threads, 0, (cudaStream_t)stream>>>(F, fp, ps, tg, squared_inputs, acc);
  note_launch();
  return check_launch();
}

int gm_product_loss(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                    const gm_pairs_t* pairs, const gm_targets_t* targets, const gm_loss_t* loss, int64_t P, double* acc,
                    void* out_g, gm_stream_t stream) {
  if (!d2_ptrs_host || !sp_host || !targets || !loss || !acc) return GM_ENULL;
  if (F < 1 || F > 8 || P < 0) return GM_EINVAL;
  if (dtype != GM_F32 && dtype != GM_F64) return GM_EINVAL;
  if (targets->mode == GM_TGT_HOPS_PACKED) return GM_EINVAL;
  PairSpec ps{};
  if (targets->mode == GM_TGT_DENSE) {  // the pair enumeration gives the node ids that index the target matrix
    int rc = validate_pairs(pairs);
    if (rc) return rc;
    if (pairs->mode == GM_PAIRS_ELEMENTWISE || pairs->P != P) return GM_EINVAL;
    ps = make_pairs(pairs);
  }
  int rc = check_loss(loss);
  if (rc) return rc;
  if (P == 0) return GM_OK;
  FactorPtrs fp{};
  for (int f = 0; f < F; ++f) {
    if (!d2_ptrs_host[f]) return GM_ENULL;
    fp.d2[f] = d2_ptrs_host[f];
    fp.sp[f] = sp_host[f];
  }
  const int threads = 256;
  long long blocks = (P + threads - 1) / threads;
  if (blocks > 0x7fffffffLL) return GM_EINVAL;
  TargetSpec tg = make_targets(targets);
  LossCfg lc = make_loss(loss);
  if (dtype == GM_F32)
    product_loss_kernel<float><<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(F, fp, tg, ps, lc, P, acc,
                                                                                       (float*)out_g);
  else
    product_loss_kernel<double><<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(F, fp, tg, ps, lc, P, acc,
                                                                                        (double*)out_g);
  note_launch();
  return check_launch();
}

int gm_sne_row_stats(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                     const void* g, int64_t B, double alpha, int32_t inclusive, void* row_stats, gm_stream_t stream) {
  if (dtype != GM_F32 && dtype != GM_F64) return GM_EINVAL;
  FactorPtrs fp{};
  int rc = fill_factors(fp, F, d2_ptrs_host, sp_host);
  if (rc) return rc;
  if (B < 0 || B > 0x7fffffffLL) return GM_EINVAL;
  if (B < 2) return GM_OK;
  if (!g || !row_stats) return GM_ENULL;
  SneCfg c{B, alpha, inclusive};
  if (dtype == GM_F32)
    sne_row_stats_kernel<float><<<(unsigned)B, 128, 0, (cudaStream_t)stream>>>(F, fp, (const float*)g, c,
                                                                              (float*)row_stats);
  else
    sne_row_stats_kernel<double><<<(unsigned)B, 128, 0, (cudaStream_t)stream>>>(F, fp, (const double*)g, c,
                                                                               (double*)row_stats);
  note_launch();
  return check_launch();
}

int gm_sne_pair_terms(int32_t dtype, int32_t F, const void* const* d2_ptrs_host, const double* sp_host,
                      const void* g, int64_t B, double alpha, int32_t inclusive, const void* row_stats, double* acc,
                      void* out_g, gm_stream_t stream) {
  if (dtype != GM_F32 && dtype != GM_F64) return GM_EINVAL;
  FactorPtrs fp{};
  int rc = fill_factors(fp, F, d2_ptrs_host, sp_host);
  if (rc) return rc;
  if (B < 0 || B > 0x7fffffffLL) return GM_EINVAL;
  if (B < 2) return GM_OK;
  if (!g || !row_stats || !acc) return GM_ENULL;
  const long long P = B * (B - 1) / 2;
  const long long work = P > B ? P : B;
  const int threads = 256;
  long long blocks = (work + threads - 1) / threads;
  if (blocks > 0x7fffffffLL) return GM_EINVAL;
  SneCfg c{B, alpha, inclusive};
  if (dtype == GM_F32)
    sne_pair_terms_kernel<float><<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
        F, fp, (const float*)g, c, (const float*)row_stats, P, acc, (float*)out_g);
  else
    sne_pair_terms_kernel<double><<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
        F, fp, (const double*)g, c, (const double*)row_stats, P, acc, (double*)out_g);
  note_launch();
  return check_launch();
}

#pragma GCC visibility pop
}  // extern "C"
