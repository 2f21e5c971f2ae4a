// Pair kernels for the vector manifolds (Lorentz, Sphere, Euclidean, Universal)
// and the Grassmannian.  One pair per thread; points have a run-time length and are
// streamed from global memory (rows are short, the second pass hits L1).
//
// Replaces Lorentz.dist (manifolds/lorentz.py:72-77 + LorentzDot/Acosh :101-141),
// Sphere.dist (manifolds/sphere.py:68-74), the Euclidean distance obtained from
// base.py:56-57, Universal.dist (manifolds/universal.py:76-81 + impl/math.py:567-572),
// Grassmann.dist (manifolds/grassmann.py:91-96), each fused with the pair gather
// (base.py:59-63), the loss and the gradient scatter-add.
#include "gm_product.cuh"

namespace gm {

template <typename T, int KIND, int KMODE>
__global__ void __launch_bounds__(128)
vec_pair_kernel(VecMan<T, KIND> op, int n, PairSpec ps, const T* __restrict__ xa, const T* __restrict__ xb,
                const T* __restrict__ gout, T coef, T* __restrict__ ga, T* __restrict__ gb,
                T* __restrict__ out_d2, TargetSpec tg, LossCfg lc, T scale_sp, double* __restrict__ acc,
                double* __restrict__ c_grad) {
  __shared__ double red[3][4];
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = k < ps.P;
  long long ra = -1, rb = -1;
  double loss_v = 0.0, gd2_v = 0.0;
  VecCoef<T> c{};
  T w = (T)0;
  const T* px = xa;
  const T* py = xb;
  if (active) {
    decode_pair(ps, k, ra, rb);
    px = xa + ra * n;
    py = xb + rb * n;
    T d2 = op.value(px, py, n, c);
    if constexpr (KMODE == K_FWD) {
      out_d2[k] = d2;
    } else if constexpr (KMODE == K_BWD) {
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
  }
  if constexpr (KMODE != K_FWD) {
    if (ps.mode == GM_PAIRS_ELEMENTWISE) {
      if (active) {
        for (int e = 0; e < n; ++e) {
          T gxe, gye;
          op.grad_elem(e, px[e], py[e], c, gxe, gye);
          ga[ra * n + e] = w * gxe;
          gb[rb * n + e] = w * gye;
        }
      }
    } else {
      vec_scatter<T>(op, n, px, py, c, w, ga, gb, ra, rb, active);
    }
  }
  if constexpr (KMODE == K_FUSED) {
    block_accumulate(loss_v, acc, red[0]);
    block_accumulate(gd2_v, acc + 1, red[1]);
  }
  if constexpr (KIND == VEC_UNIVERSAL && KMODE != K_FWD) {  // d(loss)/dc (block-uniform branch)
    if (c_grad) block_accumulate(active ? (double)w * (double)c.dc : 0.0, c_grad, red[2]);
  }
}

template <typename T, int P, bool FAST, int KMODE>
__global__ void __launch_bounds__(128)
grassmann_pair_kernel(GrassmannCore<T, P, FAST> op, int n, PairSpec ps, const T* __restrict__ xa,
                      const T* __restrict__ xb, const T* __restrict__ gout, T coef, T* __restrict__ ga,
                      T* __restrict__ gb, T* __restrict__ out_d2, TargetSpec tg, LossCfg lc, T scale_sp,
                      double* __restrict__ acc, double* __restrict__ /*c_grad: Universal only*/) {
  __shared__ double red[2][4];
  long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = k < ps.P;
  long long ra = -1, rb = -1;
  double loss_v = 0.0, gd2_v = 0.0;
  T w = (T)0;
  T gA[P * P];
  GM_UNROLL for (int i = 0; i < P * P; ++i) gA[i] = (T)0;
  const T* px = xa;
  const T* py = xb;
  if (active) {
    decode_pair(ps, k, ra, rb);
    px = xa + ra * (long long)n * P;
    py = xb + rb * (long long)n * P;
    T a[P * P];
    GM_UNROLL for (int i = 0; i < P * P; ++i) a[i] = (T)0;
    for (int r = 0; r < n; ++r) {
      T xr[P], yr[P];
      GM_UNROLL for (int i = 0; i < P; ++i) { xr[i] = px[r * P + i]; yr[i] = py[r * P + i]; }
      GM_UNROLL for (int i = 0; i < P; ++i)
        GM_UNROLL for (int j = 0; j < P; ++j) a[i * P + j] += xr[i] * yr[j];
    }
    T d2 = op.run(a, KMODE != K_FWD, gA);
    if constexpr (KMODE == K_FWD) {
      out_d2[k] = d2;
    } else if constexpr (KMODE == K_BWD) {
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
  }
  if constexpr (KMODE != K_FWD) {
    const unsigned full = 0xffffffffu;
    const bool elementwise = ps.mode == GM_PAIRS_ELEMENTWISE;
    long long ra0 = __shfl_sync(full, ra, 0);
    bool uni_a = !elementwise && __all_sync(full, ra == ra0) && ra0 >= 0;
    for (int r = 0; r < n; ++r) {
      T xr[P], yr[P];
      GM_UNROLL for (int i = 0; i < P; ++i) {
        xr[i] = active ? px[r * P + i] : (T)0;
        yr[i] = active ? py[r * P + i] : (T)0;
      }
      GM_UNROLL for (int i = 0; i < P; ++i) {
        // gx = y gA^T, gy = x gA
        T sx = (T)0, sy = (T)0;
        GM_UNROLL for (int j = 0; j < P; ++j) {
          sx += yr[j] * gA[i * P + j];
          sy += xr[j] * gA[j * P + i];
        }
        sx *= w; sy *= w;
        if (elementwise) {
          if (active) {
            ga[(ra * n + r) * P + i] = sx;
            gb[(rb * n + r) * P + i] = sy;
          }
        } else {
          warp_accumulate_elem<T>(ga + ((uni_a ? ra0 : ra) * n + r) * P + i, sx, uni_a, active);
          if (active) atomicAdd(gb + (rb * n + r) * P + i, sy);
        }
      }
    }
  }
  if constexpr (KMODE == K_FUSED) {
    block_accumulate(loss_v, acc, red[0]);
    block_accumulate(gd2_v, acc + 1, red[1]);
  }
}

template <typename T>
static T one_minus_eps2() {
  // `1 - EPS[dtype]**2` is evaluated by Python in double and then cast by torch's
  // clamp_ to the tensor dtype (sphere.py:70, grassmann.py:94)
  return (T)(1.0 - 1e-8 * 1e-8);
}

template <typename T, int KIND>
static int launch_vec(const PairArgs& a, dim3 grid, dim3 block, VecMan<T, KIND> op) {
  return launch_by_mode<T>(a, [&](auto m) {
    vec_pair_kernel<T, KIND, decltype(m)::kmode><<<grid, block, 0, a.stream>>>(
        op, a.n, a.ps, (const T*)a.xa, (const T*)a.xb, m.gout, m.coef, m.ga, m.gb, m.out_d2, a.tg, a.lc, m.scale_sp,
        m.acc, m.c_grad);
  });
}

template <typename T, int P, bool FAST>
static int launch_grassmann(const PairArgs& a, dim3 grid, dim3 block) {
  GrassmannCore<T, P, FAST> op{one_minus_eps2<T>()};
  return launch_by_mode<T>(a, [&](auto m) {
    grassmann_pair_kernel<T, P, FAST, decltype(m)::kmode><<<grid, block, 0, a.stream>>>(
        op, a.n, a.ps, (const T*)a.xa, (const T*)a.xb, m.gout, m.coef, m.ga, m.gb, m.out_d2, a.tg, a.lc, m.scale_sp,
        m.acc, m.c_grad);
  });
}

template <typename T>
static int vec_launch_typed(const PairArgs& a) {
  if (a.ps.P <= 0) return 0;
  const int threads = 128;
  long long blocks = (a.ps.P + threads - 1) / threads;
  if (blocks > 0x7fffffffLL) return GM_EINVAL;
  dim3 grid((unsigned)blocks), block(threads);
  const T eps = (T)1e-8;
  switch (a.kind) {
    case GM_LORENTZ: return launch_vec(a, grid, block, VecMan<T, VEC_LORENTZ>{eps, one_minus_eps2<T>(), nullptr});
    case GM_SPHERE: return launch_vec(a, grid, block, VecMan<T, VEC_SPHERE>{eps, one_minus_eps2<T>(), nullptr});
    case GM_EUCLIDEAN: return launch_vec(a, grid, block, VecMan<T, VEC_EUCLIDEAN>{eps, one_minus_eps2<T>(), nullptr});
    case GM_UNIVERSAL:  // value floor: wmin
      return launch_vec(a, grid, block, VecMan<T, VEC_UNIVERSAL>{(T)a.wmin, one_minus_eps2<T>(), (const T*)a.c_dev});
    case GM_GRASSMANN:
      if (a.p == 2 && (a.flags & GM_FAST_SVD)) return launch_grassmann<T, 2, true>(a, grid, block);
      switch (a.p) {
        case 1: return launch_grassmann<T, 1, false>(a, grid, block);
        case 2: return launch_grassmann<T, 2, false>(a, grid, block);
        case 3: return launch_grassmann<T, 3, false>(a, grid, block);
        case 4: return launch_grassmann<T, 4, false>(a, grid, block);
        case 5: return launch_grassmann<T, 5, false>(a, grid, block);
        default: return GM_EUNSUPPORTED;
      }
    default: return GM_EINVAL;
  }
}

int vec_launch(const PairArgs& a) {
  if (a.px) {  // product of vector manifolds only: every factor travels in a.px
    if (a.dtype == GM_F32) return launch_product<NoLead<float>, float>(NoLead<float>{}, a);
    if (a.dtype == GM_F64) return launch_product<NoLead<double>, double>(NoLead<double>{}, a);
    return GM_EINVAL;
  }
  if (a.dtype == GM_F32) return vec_launch_typed<float>(a);
  if (a.dtype == GM_F64) return vec_launch_typed<double>(a);
  return GM_EINVAL;
}

}  // namespace gm
