// Register-resident small-matrix math for the pair / optimizer kernels (sm_100a).
//
// Everything here is templated on the scalar type T (float | double) and the
// compile-time matrix size N so that every loop fully unrolls and every matrix
// element lives in a register.  No shared memory, no local-memory arrays (as
// long as N is small enough for ptxas to keep the working set in 255 regs).
//
// The functions are __host__ __device__ only so that tests/hostcheck can compile
// the *same* arithmetic for x86 and compare it with the oracle in a container
// that has no GPU; the shipped library never runs them on the host.
//
// Reference semantics being restated (never copied) are cited per function as
// graphembed/<file>:<line> relative to /root/reference/graphembed/.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <float.h>

#define GM_HD __host__ __device__ __forceinline__
#ifndef GM_ROT_NEWTON
#define GM_ROT_NEWTON 1
#endif

namespace gm {

// ---------------------------------------------------------------------------
// scalar helpers
// ---------------------------------------------------------------------------
template <typename T> struct Num;
template <> struct Num<float> {
  static constexpr float eps = FLT_EPSILON;
  static constexpr float tiny = FLT_MIN;
  static constexpr float huge = FLT_MAX;
  GM_HD static float sqrt(float x) { return sqrtf(x); }
  GM_HD static float rsqrt(float x) {
#ifdef __CUDA_ARCH__
    return rsqrtf(x);
#else
    return 1.0f / sqrtf(x);
#endif
  }
  // Raw special-function-unit approximations (MUFU.RSQ / MUFU.RCP, <= 2 ulp, flush-to-zero, no denormal or
  // IEEE slow paths): one instruction each instead of the 4-10 the C library forms expand to.
  GM_HD static float rsqrt_raw(float x) {
#ifdef __CUDA_ARCH__
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / sqrtf(x);
#endif
  }
  GM_HD static float rcp_raw(float x) {
#ifdef __CUDA_ARCH__
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
  }
  // a / b to ~2 ulp; for coefficients whose consumers tolerate 1e-6 relative error (never for values the
  // reference clamps or compares).
  GM_HD static float div_fast(float a, float b) { return a * rcp_raw(b); }
  // 1 / x to <= 1 ulp: MUFU.RCP + one Newton step (no IEEE slow path; x normal, finite, non-zero)
  GM_HD static float recip(float x) {
#ifdef __CUDA_ARCH__
    float r = rcp_raw(x);
    return fmaf(r, fmaf(-x, r, 1.0f), r);
#else
    return 1.0f / x;
#endif
  }
  // sign(d) * v with sign(+-0) = +-1: one LOP3
  GM_HD static float mul_sign(float v, float d) {
#ifdef __CUDA_ARCH__
    return __uint_as_float(__float_as_uint(v) ^ (__float_as_uint(d) & 0x80000000u));
#else
    return std::signbit(d) ? -v : v;
#endif
  }
  // Jacobi rotation (c, s, t = s/c) annihilating a_pq given d = a_qq - a_pp.  The rotation ANGLE may be inexact
  // (it only affects the convergence rate) but (c, s) must be orthonormal to rounding: approximate rsqrt / rcp for
  // tan(theta), one Newton step on the rsqrt that normalises (c, s).
  //   t = sgn(d) 2 a_pq / (|d| + sqrt(d^2 + 4 a_pq^2))   (smaller root; a_pq == 0 -> t == 0)
  GM_HD static void rotation(float d, float apq, float& t, float& c, float& s) {
    float two = apq + apq;
    float h2 = fmaf(two, two, fmaf(d, d, FLT_MIN));  // + FLT_MIN: d == a_pq == 0 must give t == 0, not 0 * inf
    float h = h2 * rsqrt_raw(h2);
    float den = fabsf(d) + h;
    t = mul_sign(two, d) * rcp_raw(den);
    float x = fmaf(t, t, 1.0f);
    float r = rsqrt_raw(x);
#if GM_ROT_NEWTON
    c = r * fmaf(-0.5f * x, r * r, 1.5f);
#else
    c = r;
#endif
    s = t * c;
  }
  GM_HD static float log(float x) { return logf(x); }
  // log(x) for x that is positive, normal and finite or NaN -- what remains after the reference's eigenvalue clamp
  // to [wmin, wmax] (spd.py:163-169).  Same scheme as logf (x = 2^e m, m in [2/3, 4/3), log m = f + f^2 g(f),
  // f = m - 1, g a degree-8 near-minimax fit; <= 1.3 ulp over the range) minus the denormal / zero / infinity
  // handling logf carries: 17 instructions instead of ~33.  NaN stays NaN.
  GM_HD static float log_pos(float x) {
#ifdef __CUDA_ARCH__
    int ix = __float_as_int(x);
    int e = (ix - 0x3f2aaaab) & 0xff800000;
    float m = fmaf(x, 0.0f, __int_as_float(ix - e));  // x * 0 keeps a NaN input alive
    float f = m - 1.0f;
    float g = -0.12734152376651764f;
    g = fmaf(g, f, 0.13756538927555084f);
    g = fmaf(g, f, -0.12219617515802383f);
    g = fmaf(g, f, 0.1405421793460846f);
    g = fmaf(g, f, -0.16678093373775482f);
    g = fmaf(g, f, 0.2000732272863388f);
    g = fmaf(g, f, -0.24999839067459106f);
    g = fmaf(g, f, 0.33333271741867065f);
    g = fmaf(g, f, -0.5f);
    float r = fmaf(f, f * g, f);
    return fmaf((float)e, 1.1920928955078125e-07f * 0.693147180559945309f, r);
#else
    return logf(x);
#endif
  }
  GM_HD static float log1p(float x) { return log1pf(x); }
  GM_HD static float exp(float x) { return expf(x); }
  GM_HD static float acos(float x) { return acosf(x); }
  GM_HD static float atan(float x) { return atanf(x); }
  GM_HD static float tan(float x) { return tanf(x); }
  GM_HD static float tanh(float x) { return tanhf(x); }
  GM_HD static float cos(float x) { return cosf(x); }
  GM_HD static float sin(float x) { return sinf(x); }
  GM_HD static float cosh(float x) { return coshf(x); }
  GM_HD static float sinh(float x) { return sinhf(x); }
  GM_HD static float abs(float x) { return fabsf(x); }
  GM_HD static float fma(float a, float b, float c) { return fmaf(a, b, c); }
  GM_HD static float max(float a, float b) { return fmaxf(a, b); }
  GM_HD static float min(float a, float b) { return fminf(a, b); }
  GM_HD static float copysign(float a, float b) { return copysignf(a, b); }
};
template <> struct Num<double> {
  static constexpr double eps = DBL_EPSILON;
  static constexpr double tiny = DBL_MIN;
  static constexpr double huge = DBL_MAX;
  GM_HD static double sqrt(double x) { return ::sqrt(x); }
  GM_HD static double rsqrt(double x) { return 1.0 / ::sqrt(x); }
  GM_HD static double div_fast(double a, double b) { return a / b; }
  GM_HD static double recip(double x) { return 1.0 / x; }
  GM_HD static void rotation(double d, double apq, double& t, double& c, double& s) {
    double two = apq + apq;
    double den = fabs(d) + ::sqrt(d * d + two * two);
    t = (den > 0.0) ? (d >= 0.0 ? two : -two) / den : 0.0;
    c = 1.0 / ::sqrt(t * t + 1.0);
    s = t * c;
  }
  GM_HD static double log(double x) { return ::log(x); }
  GM_HD static double log_pos(double x) { return ::log(x); }
  GM_HD static double log1p(double x) { return ::log1p(x); }
  GM_HD static double exp(double x) { return ::exp(x); }
  GM_HD static double acos(double x) { return ::acos(x); }
  GM_HD static double atan(double x) { return ::atan(x); }
  GM_HD static double tan(double x) { return ::tan(x); }
  GM_HD static double tanh(double x) { return ::tanh(x); }
  GM_HD static double cos(double x) { return ::cos(x); }
  GM_HD static double sin(double x) { return ::sin(x); }
  GM_HD static double cosh(double x) { return ::cosh(x); }
  GM_HD static double sinh(double x) { return ::sinh(x); }
  GM_HD static double abs(double x) { return fabs(x); }
  GM_HD static double fma(double a, double b, double c) { return ::fma(a, b, c); }
  GM_HD static double max(double a, double b) { return fmax(a, b); }
  GM_HD static double min(double a, double b) { return fmin(a, b); }
  GM_HD static double copysign(double a, double b) { return ::copysign(a, b); }
};

// torch.clamp semantics on a *value* (NaN propagates like torch: clamp(NaN)=NaN)
template <typename T>
GM_HD T clampv(T x, T lo, T hi) {
  return x < lo ? lo : (x > hi ? hi : x);
}
template <typename T>
GM_HD T clamp_min(T x, T lo) { return x < lo ? lo : x; }
template <typename T>
GM_HD T clamp_max(T x, T hi) { return x > hi ? hi : x; }
// torch.sign / abs-backward convention: sign(0) == 0
template <typename T>
GM_HD T sgn0(T x) { return (T)((x > (T)0) - (x < (T)0)); }

// ---------------------------------------------------------------------------
// N x N matrices held as flat register arrays (row-major, index i*N+j)
// ---------------------------------------------------------------------------
#define GM_UNROLL _Pragma("unroll")

// Lower Cholesky factor of a symmetric matrix (reads the lower triangle of x).
// Non-PD input yields NaN (sqrt of a negative pivot), mirroring the reference's
// "NaNs are not detected" behaviour (torch.cholesky would raise on CPU;
// graphembed/linalg/torch_batch.py:43-67).
template <typename T, int N>
GM_HD void chol_lower(const T (&x)[N * N], T (&l)[N * N]) {
  GM_UNROLL for (int j = 0; j < N; ++j) {
    T s = x[j * N + j];
    GM_UNROLL for (int k = 0; k < j; ++k) s -= l[j * N + k] * l[j * N + k];
    T d = Num<T>::sqrt(s);
    l[j * N + j] = d;
    T inv = (T)1 / d;
    GM_UNROLL for (int i = j + 1; i < N; ++i) {
      T t = x[i * N + j];
      GM_UNROLL for (int k = 0; k < j; ++k) t -= l[i * N + k] * l[j * N + k];
      l[i * N + j] = t * inv;
    }
    GM_UNROLL for (int i = 0; i < j; ++i) l[i * N + j] = (T)0;
  }
}

// a = l^{-1} for lower-triangular l (forward substitution against I;
// graphembed/manifolds/spd.py:55-61).
template <typename T, int N>
GM_HD void tri_inv_lower(const T (&l)[N * N], T (&a)[N * N]) {
  GM_UNROLL for (int j = 0; j < N; ++j) {
    GM_UNROLL for (int i = 0; i < j; ++i) a[i * N + j] = (T)0;
    a[j * N + j] = (T)1 / l[j * N + j];
    GM_UNROLL for (int i = j + 1; i < N; ++i) {
      T s = (T)0;
      GM_UNROLL for (int k = j; k < i; ++k) s += l[i * N + k] * a[k * N + j];
      a[i * N + j] = -s / l[i * N + i];
    }
  }
}

// m = a y a^T for lower-triangular a and symmetric y; m is produced exactly
// symmetric (upper computed, mirrored).  graphembed/linalg/torch_batch.py:30-34.
template <typename T, int N>
GM_HD void congr_lower(const T (&a)[N * N], const T (&y)[N * N], T (&m)[N * N]) {
  T t[N * N];
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = 0; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k <= i; ++k) s += a[i * N + k] * y[k * N + j];
      t[i * N + j] = s;
    }
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = i; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k <= j; ++k) s += t[i * N + k] * a[j * N + k];
      m[i * N + j] = s;
      m[j * N + i] = s;
    }
}

// m = a y a^T for general (full) a and symmetric y.
template <typename T, int N>
GM_HD void congr_full(const T (&a)[N * N], const T (&y)[N * N], T (&m)[N * N]) {
  T t[N * N];
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = 0; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k < N; ++k) s += a[i * N + k] * y[k * N + j];
      t[i * N + j] = s;
    }
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = i; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k < N; ++k) s += t[i * N + k] * a[j * N + k];
      m[i * N + j] = s;
      m[j * N + i] = s;
    }
}

// w = a^T v for lower-triangular a.
template <typename T, int N>
GM_HD void lowerT_mul(const T (&a)[N * N], const T (&v)[N * N], T (&w)[N * N]) {
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = 0; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = i; k < N; ++k) s += a[k * N + i] * v[k * N + j];
      w[i * N + j] = s;
    }
}

// w = l v for lower-triangular l.
template <typename T, int N>
GM_HD void lower_mul(const T (&l)[N * N], const T (&v)[N * N], T (&w)[N * N]) {
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = 0; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k <= i; ++k) s += l[i * N + k] * v[k * N + j];
      w[i * N + j] = s;
    }
}

// g = w diag(c) w^T (symmetric; upper computed, mirrored).
// graphembed/linalg/torch_batch.py:84-91,138-142 (mvmt / hgie).
template <typename T, int N>
GM_HD void wdwt(const T (&w)[N * N], const T (&c)[N], T (&g)[N * N]) {
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = i; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k < N; ++k) s += (w[i * N + k] * c[k]) * w[j * N + k];
      g[i * N + j] = s;
      g[j * N + i] = s;
    }
}

template <typename T, int N>
GM_HD void matmul(const T (&a)[N * N], const T (&b)[N * N], T (&c)[N * N]) {
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = 0; j < N; ++j) {
      T s = (T)0;
      GM_UNROLL for (int k = 0; k < N; ++k) s += a[i * N + k] * b[k * N + j];
      c[i * N + j] = s;
    }
}

// ---------------------------------------------------------------------------
// Cyclic Jacobi eigensolver for a symmetric N x N matrix held in registers.
// On exit w[k] are the eigenvalues and the columns of v the eigenvectors
// (a = v diag(w) v^T).  Replaces torch.symeig(eigenvectors=True), i.e. LAPACK
// syevd, at graphembed/linalg/torch_batch.py:127-135 / manifolds/spd.py:63-64.
// Order and sign of eigenpairs are unspecified; every caller uses only
// permutation/sign-invariant combinations (sum f(w), v f(w) v^T).
// ---------------------------------------------------------------------------
template <typename T> struct JacobiCfg;
// off_factor: the iteration stops when ||off(A)||_F^2 <= eps^2 * off_factor * ||diag(A)||_F^2.  fp64: off-diagonal mass
// a quarter of an ulp of the diagonal (1e-10 parity with LAPACK's eigenvectors).  fp32: 4 ulp (GM_JACOBI_F32_OFF = 16)
// -- the error a residual off-diagonal E leaves in V f(Lambda) V^T is |E| max|f'| (the eigenvalue gaps cancel for a
// smooth matrix function), i.e. 5e-7 relative, below the 2e-6 mean / 2e-5 worst-case error the fp32 Cholesky +
// congruence in front of the solver already carry (tools/eig_lab.cu: accuracy against fp64 unchanged from 1/4 ulp up
// to 4 ulp, while the share of 4x4 pair matrices done after 3 sweeps goes 95.2 -> 98.5 %).
// Applied to n <= 4 only (GM_JACOBI_F32_OFF_MAX_N): there the solver runs inside warps that stop together, and the
// looser test lets most warps stop after 3 sweeps (pair kernel 0.962 -> 0.902 ms).  For n = 6 the same change measured
// 9 % SLOWER (BASELINE config 4: 57.6 -> 62.5 ms per epoch, profiles/r02_pair_kernel_ab.txt run 12), so n >= 5 keep 1/4 ulp.
#ifndef GM_JACOBI_F32_OFF
#define GM_JACOBI_F32_OFF 16.0f
#endif
#ifndef GM_JACOBI_F32_OFF_MAX_N
#define GM_JACOBI_F32_OFF_MAX_N 4
#endif
template <> struct JacobiCfg<float> {
  static constexpr int max_sweeps = 10;
  static constexpr float off_factor = GM_JACOBI_F32_OFF;
};
template <> struct JacobiCfg<double> {
  static constexpr int max_sweeps = 16;
  static constexpr double off_factor = 0.0625;
};

// Rotation schedule of one sweep (inside jacobi_eigh).  N == 4 uses the round-robin ("tournament") order (0,1)(2,3) (0,2)(1,3)
// (0,3)(1,2): the two rotations of a round touch disjoint rows/columns, so their parameter chains are independent
// (instruction-level parallelism 2), and it needs fewer sweeps than the row-cyclic order on the pair workload
// (tools/eig_lab.cu: 92 % vs 52 % of 4x4 pair matrices done after 3 sweeps).  Other sizes: row-cyclic.
// No sweep before this one is ever the last on non-trivial input (eig_lab: < 0.1 % of 4x4 matrices converge in
// fewer than 3 sweeps), so the convergence test is skipped for them; an already diagonal matrix just sees identity
// rotations.
template <int N>
struct JacobiFirstCheck { static constexpr int value = N >= 4 ? 3 : (N == 3 ? 2 : 1); };

// INIT_V: start from v = I (eigenvectors).  With INIT_V == false the caller passes any matrix B in v and gets
// B * V back -- the pair kernels pass L^-T so that W = L^-T V comes out of the sweeps directly.
// max_sweeps (<= JacobiCfg<T>::max_sweeps) caps the number of sweeps; the return value says whether the convergence
// test passed (always evaluated once the cap is reached, so a caller can run a fixed number of sweeps and hand the
// few matrices that need more to a second pass -- the streaming pair kernel does, see gm_pairs_spd.cu).
template <typename T, int N, bool WANT_V = true, bool INIT_V = true>
GM_HD bool jacobi_eigh(T (&a)[N * N], T (&v)[N * N], T (&w)[N], int max_sweeps = JacobiCfg<T>::max_sweeps) {
  if (WANT_V && INIT_V) {
    GM_UNROLL for (int i = 0; i < N; ++i)
      GM_UNROLL for (int j = 0; j < N; ++j) v[i * N + j] = (i == j) ? (T)1 : (T)0;
  }
  if (N == 1) { w[0] = a[0]; return true; }
  auto rotate = [&](const int p, const int q) {
    T apq = a[p * N + q];
    T t, c, s;
    Num<T>::rotation(a[q * N + q] - a[p * N + p], apq, t, c, s);
    if constexpr (N >= 5) {
      // The diagonal from the same rounded (c, s) that rotates the off-diagonal rows below.  The cheaper
      // a_pp - t a_pq assumes the exact rotation; with the rounded one it is not a congruence, and on spectra over
      // 4 decades (6x6 fp32, condition up to 1e8) that mismatch biases every eigenvalue sum inward: d2 -1.1e-5 on
      // average, the loss summed over such pairs 1.4e-5 low (tests/test_gpu_spd_hotpath.py, class C), against
      // 3e-8 with this form.  n <= 4 keep a_pp - t a_pq: there the same bars hold and it is the bench.py path.
      const T app = a[p * N + p], aqq = a[q * N + q], cs2 = (T)2 * c * s * apq;
      a[p * N + p] = c * c * app - cs2 + s * s * aqq;
      a[q * N + q] = s * s * app + cs2 + c * c * aqq;
    } else {
      a[p * N + p] = Num<T>::fma(-t, apq, a[p * N + p]);
      a[q * N + q] = Num<T>::fma(t, apq, a[q * N + q]);
    }
    a[p * N + q] = (T)0;
    a[q * N + p] = (T)0;
    GM_UNROLL for (int r = 0; r < N; ++r) {
      if (r != p && r != q) {
        T arp = a[r * N + p], arq = a[r * N + q];
        T nrp = c * arp - s * arq;
        T nrq = s * arp + c * arq;
        a[r * N + p] = nrp; a[p * N + r] = nrp;
        a[r * N + q] = nrq; a[q * N + r] = nrq;
      }
    }
    if (WANT_V) {
      GM_UNROLL for (int r = 0; r < N; ++r) {
        T vrp = v[r * N + p], vrq = v[r * N + q];
        v[r * N + p] = c * vrp - s * vrq;
        v[r * N + q] = s * vrp + c * vrq;
      }
    }
  };
  bool converged = false;
  for (int sweep = 0;; ++sweep) {
    if (sweep >= JacobiFirstCheck<N>::value || sweep >= max_sweeps) {
      T off = (T)0, dia = (T)0;
      GM_UNROLL for (int i = 0; i < N; ++i) {
        dia += a[i * N + i] * a[i * N + i];
        GM_UNROLL for (int j = i + 1; j < N; ++j) off += a[i * N + j] * a[i * N + j];
      }
      // converged when the off-diagonal mass is below rounding level of the diagonal
      // (n <= 4 in fp32: 4 ulp; everything else 1/4 ulp -- see JacobiCfg)
      constexpr T off_factor = (N <= GM_JACOBI_F32_OFF_MAX_N) ? JacobiCfg<T>::off_factor : (T)0.0625;
      converged = off <= (Num<T>::eps * Num<T>::eps * off_factor) * dia || off < Num<T>::tiny;
      if (converged || sweep >= max_sweeps) break;
    }
    if constexpr (N == 4) {
      rotate(0, 1); rotate(2, 3);
      rotate(0, 2); rotate(1, 3);
      rotate(0, 3); rotate(1, 2);
    } else {
      GM_UNROLL for (int p = 0; p < N - 1; ++p)
        GM_UNROLL for (int q = p + 1; q < N; ++q) rotate(p, q);
    }
  }
  GM_UNROLL for (int i = 0; i < N; ++i) w[i] = a[i * N + i];
  return converged;
}

// ---------------------------------------------------------------------------
// One-sided (Hestenes) Jacobi SVD of an R x C matrix (R >= C) held in
// registers: on exit the columns of `a` are u_k * s_k, `v` (C x C) holds the right
// singular vectors and s[k] >= 0 the singular values (unsorted).  Replaces
// torch.svd (LAPACK gesdd) at graphembed/linalg/torch_batch.py:109-112.
// ---------------------------------------------------------------------------
template <typename T, int R, int C>
GM_HD void jacobi_svd(T (&a)[R * C], T (&v)[C * C], T (&s)[C]) {
  GM_UNROLL for (int i = 0; i < C; ++i)
    GM_UNROLL for (int j = 0; j < C; ++j) v[i * C + j] = (i == j) ? (T)1 : (T)0;
  for (int sweep = 0; sweep < JacobiCfg<T>::max_sweeps + 4; ++sweep) {
    bool rotated = false;
    GM_UNROLL for (int p = 0; p < C - 1; ++p) {
      GM_UNROLL for (int q = p + 1; q < C; ++q) {
        T alpha = (T)0, beta = (T)0, gamma = (T)0;
        GM_UNROLL for (int r = 0; r < R; ++r) {
          alpha += a[r * C + p] * a[r * C + p];
          beta += a[r * C + q] * a[r * C + q];
          gamma += a[r * C + p] * a[r * C + q];
        }
        if (Num<T>::abs(gamma) > (Num<T>::eps * (T)0.25) * Num<T>::sqrt(alpha * beta) &&
            Num<T>::abs(gamma) > Num<T>::tiny) {
          rotated = true;
          T t, c, sn;
          Num<T>::rotation(beta - alpha, gamma, t, c, sn);
          GM_UNROLL for (int r = 0; r < R; ++r) {
            T x = a[r * C + p], y = a[r * C + q];
            a[r * C + p] = c * x - sn * y;
            a[r * C + q] = sn * x + c * y;
          }
          GM_UNROLL for (int r = 0; r < C; ++r) {
            T x = v[r * C + p], y = v[r * C + q];
            v[r * C + p] = c * x - sn * y;
            v[r * C + q] = sn * x + c * y;
          }
        }
      }
    }
    if (!rotated) break;
  }
  GM_UNROLL for (int k = 0; k < C; ++k) {
    T n2 = (T)0;
    GM_UNROLL for (int r = 0; r < R; ++r) n2 += a[r * C + k] * a[r * C + k];
    s[k] = Num<T>::sqrt(n2);
  }
}

// ---------------------------------------------------------------------------
// warp / block reductions
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
  GM_UNROLL for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum `v` over the block and add it to *dst (one atomic per block).  `red` must
// hold blockDim.x/32 doubles of shared memory.
__device__ __forceinline__ void block_accumulate(double v, double* dst, double* red) {
  v = warp_sum(v);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    int nw = (blockDim.x + 31) >> 5;
    double s = lane < nw ? red[lane] : 0.0;
    s = warp_sum(s);
    if (lane == 0 && dst != nullptr) atomicAdd(dst, s);
  }
  __syncthreads();
}

}  // namespace gm
