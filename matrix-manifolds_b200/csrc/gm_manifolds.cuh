// Per-pair manifold arithmetic: squared distance and its Euclidean gradient
// with respect to both endpoints, one pair per thread, everything in registers.
//
// Each `struct` restates one reference distance (file:line cited) including the
// reference's value-only ("straight-through") clamps: `t.data.clamp_()` changes
// the value autograd later differentiates *at*, never the derivative itself
// (SURVEY.md Appendix A.1).  Gradients are the analytic ones of SURVEY.md
// Appendix B; for SPD they are returned symmetrised, which is what the
// reference's optimizers consume (egrad2rgrad applies sym(), spd.py:134-135).
#pragma once
#include "gm_math.cuh"

namespace gm {

// ===========================================================================
// SPD building blocks
// ===========================================================================

// Inverse Cholesky factor a = chol(x)^{-1} (lower) and optionally l = chol(x).
// FAST_CHOL (n == 2 only) restates fast.invcholesky2x2 (linalg/fast.py:110-134):
//   x00 clamped >= eps, a = sqrt(x00), b = x01/a, c = sqrt(x11 - b^2 + eps),
//   det = a c clamped >= eps, l^{-1} = [[c, 0], [-b, a]] / det.
// otherwise torch.cholesky + triangular_solve against I (spd.py:55-61).
template <typename T, int N, bool FAST_CHOL>
struct InvChol {
  T a[N * N];
  T l[N * N];
  // closed-form intermediates kept for the backward pass
  T fa, fb, fc, fdet;
  GM_HD void run(const T (&x)[N * N]) {
    if constexpr (FAST_CHOL) {
      static_assert(N == 2, "closed-form Cholesky exists for 2x2 only");
      const T eps = (T)1e-8;
      T x00 = clamp_min(x[0], eps);
      fa = Num<T>::sqrt(x00);
      fb = x[1] / fa;  // upper entry x01, as the reference reads it
      fc = Num<T>::sqrt(x[3] - fb * fb + eps);
      fdet = clamp_min(fa * fc, eps);
      a[0] = fc / fdet; a[1] = (T)0; a[2] = -fb / fdet; a[3] = fa / fdet;
      l[0] = fa; l[1] = (T)0; l[2] = fb; l[3] = fc;
    } else {
      chol_lower<T, N>(x, l);
      tri_inv_lower<T, N>(l, a);
    }
  }
  // Given abar = d f / d a (only the lower triangle is used), return the
  // symmetrised gradient with respect to x.
  GM_HD void backward_closed(const T (&abar)[N * N], T (&gx)[N * N]) const {
    static_assert(N == 2, "");
    T cbar = abar[0] / fdet;
    T bbar = -abar[2] / fdet;
    T abar_ = abar[3] / fdet;
    T detbar = -(abar[0] * fc - abar[2] * fb + abar[3] * fa) / (fdet * fdet);
    abar_ += detbar * fc;
    cbar += detbar * fa;
    T sbar = cbar / (fc + fc);
    T x11bar = sbar;
    bbar -= (fb + fb) * sbar;
    T x01bar = bbar / fa;
    abar_ -= bbar * fb / fa;
    T x00bar = abar_ / (fa + fa);
    gx[0] = x00bar; gx[3] = x11bar;
    gx[1] = gx[2] = (T)0.5 * x01bar;
  }
};

// g = a^T s a for lower-triangular a and symmetric s (result symmetric).
template <typename T, int N>
GM_HD void congr_lowerT(const T (&a)[N * N], const T (&s)[N * N], T (&g)[N * N]) {
  T t[N * N];  // t = s a
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = 0; j < N; ++j) {
      T acc = (T)0;
      GM_UNROLL for (int k = j; k < N; ++k) acc += s[i * N + k] * a[k * N + j];
      t[i * N + j] = acc;
    }
  GM_UNROLL for (int i = 0; i < N; ++i)
    GM_UNROLL for (int j = i; j < N; ++j) {
      T acc = (T)0;
      GM_UNROLL for (int k = i; k < N; ++k) acc += a[k * N + i] * t[k * N + j];
      g[i * N + j] = acc;
      g[j * N + i] = acc;
    }
}

// Closed-form eigenvalue functional phi(m) = sum log^2(clamp(eig(m))) and the
// symmetrised derivative g = sym(d phi / d m), differentiating the reference's
// closed forms themselves (eps terms included) -- linalg/fast.py:53-70 (2x2),
// :75-91 (3x3); clamp/log/sum from spd.py:163-169.
template <typename T, int N>
struct ClosedEig;

template <typename T>
struct ClosedEig<T, 2> {
  GM_HD static T run(const T (&m)[4], T wmin, T wmax, bool want_grad, T (&g)[4]) {
    const T eps = (T)1e-8;
    T a = m[0], b = m[3], c = m[1];
    T det = a * b - c * c;
    T h = (T)0.5 * (a + b);
    T delta = clamp_min(h * h - det, eps);
    T r = Num<T>::sqrt(delta);
    T e1 = clampv(h - r, wmin, wmax), e2 = clampv(h + r, wmin, wmax);
    T l1 = Num<T>::log(e1), l2 = Num<T>::log(e2);
    T phi = l1 * l1 + l2 * l2;
    if (want_grad) {
      T g1 = (T)2 * l1 / e1, g2 = (T)2 * l2 / e2;
      T sh = (T)0.5 * (g1 + g2);
      T dr = (g2 - g1) / (r + r);  // d phi / d delta
      g[0] = sh + dr * (h - b);
      g[3] = sh + dr * (h - a);
      g[1] = g[2] = dr * c;  // (2 c dr) on the upper entry, halved by sym()
    }
    return phi;
  }
};

template <typename T>
struct ClosedEig<T, 3> {
  GM_HD static T run(const T (&m)[9], T wmin, T wmax, bool want_grad, T (&g)[9]) {
    const T eps = (T)1e-8;
    const T two_pi_3 = (T)2.0943951023931954923084289221863;
    T q = (m[0] + m[4] + m[8]) / (T)3;
    T y00 = m[0] - q, y11 = m[4] - q, y22 = m[8] - q;
    T y01 = m[1], y02 = m[2], y12 = m[5];
    T y10 = m[3], y20 = m[6], y21 = m[7];
    T ss = y00 * y00 + y01 * y01 + y02 * y02 + y10 * y10 + y11 * y11 + y12 * y12 + y20 * y20 + y21 * y21 +
           y22 * y22;
    T p = clamp_min(Num<T>::sqrt(ss / (T)6), eps);
    T det = y00 * y11 * y22 + (T)2 * y01 * y02 * y12 - y11 * y02 * y02 - y00 * y12 * y12 - y22 * y01 * y01;
    T den = (T)2 * p * p * p + eps;
    T r = clampv(det / den, (T)-1 + eps, (T)1 - eps);
    T phi3 = Num<T>::acos(r) / (T)3;
    T c1 = Num<T>::cos(phi3), c2 = Num<T>::cos(phi3 + two_pi_3);
    T e1 = q + (T)2 * p * c1;
    T e2 = q + (T)2 * p * c2;
    T e3 = (T)3 * q - e1 - e2;
    T f1 = clampv(e1, wmin, wmax), f2 = clampv(e2, wmin, wmax), f3 = clampv(e3, wmin, wmax);
    T l1 = Num<T>::log(f1), l2 = Num<T>::log(f2), l3 = Num<T>::log(f3);
    T phi = l1 * l1 + l2 * l2 + l3 * l3;
    if (want_grad) {
      T g1 = (T)2 * l1 / f1, g2 = (T)2 * l2 / f2, g3 = (T)2 * l3 / f3;
      // e3 = 3q - e1 - e2
      T e1b = g1 - g3, e2b = g2 - g3;
      T qb = (T)3 * g3 + e1b + e2b;
      T pb = (T)2 * (e1b * c1 + e2b * c2);
      T s1 = Num<T>::sin(phi3), s2 = Num<T>::sin(phi3 + two_pi_3);
      T phib = -(T)2 * p * (e1b * s1 + e2b * s2);
      T rb = -phib / ((T)3 * Num<T>::sqrt((T)1 - r * r));
      T detb = rb / den;
      pb += -rb * (det / den) / den * (T)6 * p * p;  // d(det/den)/dp with r's *unclamped* quotient
      T ssb = pb / ((T)2 * p) / (T)6;
      T two_ssb = ssb + ssb;
      T b00 = two_ssb * y00 + detb * (y11 * y22 - y12 * y12);
      T b11 = two_ssb * y11 + detb * (y00 * y22 - y02 * y02);
      T b22 = two_ssb * y22 + detb * (y00 * y11 - y01 * y01);
      T b01 = two_ssb * y01 + detb * ((T)2 * y02 * y12 - (T)2 * y22 * y01);
      T b02 = two_ssb * y02 + detb * ((T)2 * y01 * y12 - (T)2 * y11 * y02);
      T b12 = two_ssb * y12 + detb * ((T)2 * y01 * y02 - (T)2 * y00 * y12);
      T b10 = two_ssb * y10, b20 = two_ssb * y20, b21 = two_ssb * y21;
      T dq = (qb - (b00 + b11 + b22)) / (T)3;
      g[0] = b00 + dq; g[4] = b11 + dq; g[8] = b22 + dq;
      g[1] = g[3] = (T)0.5 * (b01 + b10);
      g[2] = g[6] = (T)0.5 * (b02 + b20);
      g[5] = g[7] = (T)0.5 * (b12 + b21);
    }
    return phi;
  }
};

// ===========================================================================
// SPD, affine-invariant metric: d^2(x, y) = sum_k log^2 lambda_k(L^-1 y L^-T)
// spd.py:171-181 (dist/pdist), :163-169 (_norm_log), :108-111 (_lult).
// ===========================================================================
template <typename T, int N, bool FAST_EIG, bool FAST_CHOL>
struct SpdAI {
  static constexpr int E = N * N;
  T wmin, wmax;

  GM_HD T dist2(const T (&x)[E], const T (&y)[E]) const {
    InvChol<T, N, FAST_CHOL> ic;
    ic.run(x);
    T m[E];
    congr_lower<T, N>(ic.a, y, m);
    T phi;
    if constexpr (FAST_EIG) {
      T dummy[E];
      phi = ClosedEig<T, N>::run(m, wmin, wmax, false, dummy);
    } else {
      T v[E], w[N];
      jacobi_eigh<T, N, false>(m, v, w);
      phi = (T)0;
      if constexpr (FAST_CHOL) {
        GM_UNROLL for (int k = 0; k < N; ++k) {
          T lg = Num<T>::log(clampv(w[k], wmin, wmax));
          phi += lg * lg;
        }
      } else {  // same arithmetic as eig_forward, so that forward-only and fused launches agree bit for bit
        const T lo = Num<T>::max(wmin, Num<T>::tiny), hi = Num<T>::min(wmax, Num<T>::huge);
        GM_UNROLL for (int k = 0; k < N; ++k) {
          T lg = Num<T>::log_pos(clampv(w[k], lo, hi));
          phi += lg * lg;
        }
      }
    }
    return clamp_min(phi, wmin);
  }

  // The exact path (LAPACK-equivalent Cholesky + Jacobi) depends on x only through a = chol(x)^-1, which a
  // caller that visits many pairs with the same first endpoint can compute once (spd.py:178 does the same per node).
  // It is split in two so that the caller can fold its loss weight into the N gradient coefficients instead of
  // scaling 2 N^2 gradient entries afterwards:
  //   eig_forward : m = a y a^T, Jacobi sweeps started from W0 = a^T so that W = L^-T V (which diagonalises both:
  //                 W^T x W = I, W^T y W = diag(lambda)) comes out of the sweeps directly; returns phi = sum log^2.
  //   eig_backward: gx = wgt * d(phi)/dx = W diag(-2 wgt log l_k) W^T,  gy = W diag(2 wgt log l_k / l_k) W^T.
  static constexpr bool kCanPrep = !FAST_EIG && !FAST_CHOL;
  static constexpr int kPrepSize = N * (N + 1) / 2;
  struct EigState {
    T wm[E];
    T cx[N], cy[N];
  };
  GM_HD void prep(const T (&x)[E], T (&ap)[kPrepSize]) const {
    InvChol<T, N, false> ic;
    ic.run(x);
    GM_UNROLL for (int i = 0; i < N; ++i)
      GM_UNROLL for (int j = 0; j <= i; ++j) ap[i * (i + 1) / 2 + j] = ic.a[i * N + j];
  }
  // max_sweeps / converged / PACK: see jacobi_eigh.  With the default cap `converged` is of no interest.
  template <bool PACK = false>
  GM_HD T eig_forward(const T (&a)[E], const T (&y)[E], EigState& st, int max_sweeps = JacobiCfg<T>::max_sweeps,
                      bool* converged = nullptr) const {
    T m[E], w[N];
    congr_lower<T, N>(a, y, m);
    GM_UNROLL for (int i = 0; i < N; ++i)
      GM_UNROLL for (int j = 0; j < N; ++j) st.wm[i * N + j] = (j >= i) ? a[j * N + i] : (T)0;
    const bool conv = jacobi_eigh<T, N, true, false, PACK>(m, st.wm, w, max_sweeps);
    if (converged) *converged = conv;
    T phi = (T)0;
    // log_pos needs a positive normal finite argument: guaranteed by the clamp for every sane [wmin, wmax]
    // (default [1e-8, 1e8]); a caller-supplied wmin below the smallest normal is raised to it.
    const T lo = Num<T>::max(wmin, Num<T>::tiny), hi = Num<T>::min(wmax, Num<T>::huge);
    GM_UNROLL for (int k = 0; k < N; ++k) {
      T wc = clampv(w[k], lo, hi);
      T lg = Num<T>::log_pos(wc);
      phi += lg * lg;
      T c = Num<T>::div_fast(lg + lg, wc);
      st.cy[k] = c;
      st.cx[k] = -c * w[k];
    }
    return clamp_min(phi, wmin);
  }
  template <bool PACK = false>
  GM_HD T eig_forward_prepped(const T (&ap)[kPrepSize], const T (&y)[E], EigState& st,
                              int max_sweeps = JacobiCfg<T>::max_sweeps, bool* converged = nullptr) const {
    T a[E];
    GM_UNROLL for (int i = 0; i < N; ++i)
      GM_UNROLL for (int j = 0; j < N; ++j) a[i * N + j] = (j <= i) ? ap[i * (i + 1) / 2 + j] : (T)0;
    return eig_forward<PACK>(a, y, st, max_sweeps, converged);
  }
  GM_HD void eig_backward(const EigState& st, T wgt, T (&gx)[E], T (&gy)[E]) const {
    T cx[N], cy[N];
    GM_UNROLL for (int k = 0; k < N; ++k) { cx[k] = st.cx[k] * wgt; cy[k] = st.cy[k] * wgt; }
    wdwt<T, N>(st.wm, cx, gx);
    wdwt<T, N>(st.wm, cy, gy);
  }

  // Returns d2 and fills gx = d(d2)/dx, gy = d(d2)/dy (both symmetric).
  GM_HD T dist2_grad(const T (&x)[E], const T (&y)[E], T (&gx)[E], T (&gy)[E]) const {
    InvChol<T, N, FAST_CHOL> ic;
    ic.run(x);
    T m[E];
    congr_lower<T, N>(ic.a, y, m);
    T phi = (T)0;
    if constexpr (!FAST_EIG && !FAST_CHOL) {
      EigState st;
      T d2 = eig_forward(ic.a, y, st);
      eig_backward(st, (T)1, gx, gy);
      return d2;
    } else {
      T g[E];  // sym(d phi / d m)
      if constexpr (FAST_EIG) {
        phi = ClosedEig<T, N>::run(m, wmin, wmax, true, g);
      } else {
        T mm[E], v[E], w[N], c[N];
        GM_UNROLL for (int k = 0; k < E; ++k) mm[k] = m[k];
        jacobi_eigh<T, N, true>(mm, v, w);
        phi = (T)0;
        GM_UNROLL for (int k = 0; k < N; ++k) {
          T wc = clampv(w[k], wmin, wmax);
          T lg = Num<T>::log(wc);
          phi += lg * lg;
          c[k] = (T)2 * lg / wc;
        }
        wdwt<T, N>(v, c, g);
      }
      congr_lowerT<T, N>(ic.a, g, gy);
      if constexpr (FAST_CHOL) {
        // abar = 2 g a y, pushed through the closed-form inverse Cholesky
        T ga[E], abar[E];
        matmul<T, N>(g, ic.a, ga);
        matmul<T, N>(ga, y, abar);
        GM_UNROLL for (int k = 0; k < E; ++k) abar[k] *= (T)2;
        ic.backward_closed(abar, gx);
      } else {
        // exact Cholesky: gx = -a^T P a with P the symmetric matrix whose lower
        // triangle (diagonal included) is that of k = g m (torch's
        // cholesky_backward keeps tril(L^T gL), halves the diagonal, symmetrises).
        T k[E], pm[E];
        matmul<T, N>(g, m, k);
        GM_UNROLL for (int i = 0; i < N; ++i)
          GM_UNROLL for (int j = 0; j <= i; ++j) {
            pm[i * N + j] = -k[i * N + j];
            pm[j * N + i] = -k[i * N + j];
          }
        congr_lowerT<T, N>(ic.a, pm, gx);
      }
    }
    return clamp_min(phi, wmin);
  }
};

// ===========================================================================
// SPD, symmetric Stein divergence S = logdet((x+y)/2) - (logdet x + logdet y)/2
// spd.py:183-194 (stein_div / stein_pdiv), :246-295 (PairwiseSteinDivergence),
// linalg/torch_batch.py:173-197 (PLogDet).  d S/dx = ((x+y)/2)^-1/2 - x^-1/2.
// With FAST_CHOL the eps-perturbed closed-form factor is used for both the
// log-determinant and the inverse, as the reference's `chol` argument does.
// ===========================================================================
template <typename T, int N, bool FAST_CHOL>
struct SpdStein {
  static constexpr int E = N * N;
  static constexpr bool kCanPrep = false;
  static constexpr int kPrepSize = 1;
  T wmin, wmax;
  struct EigState {};
  GM_HD void prep(const T (&)[E], T (&)[1]) const {}
  template <bool PACK = false>
  GM_HD T eig_forward_prepped(const T (&)[1], const T (&)[E], EigState&, int = 0, bool* = nullptr) const { return (T)0; }
  GM_HD void eig_backward(const EigState&, T, T (&)[E], T (&)[E]) const {}

  template <bool WANT_INV>
  GM_HD static T logdet_inv(const T (&x)[E], T (&inv)[E]) {
    InvChol<T, N, FAST_CHOL> ic;
    ic.run(x);
    T ld = (T)0;
    GM_UNROLL for (int k = 0; k < N; ++k) ld += Num<T>::log(Num<T>::abs(ic.l[k * N + k]));
    if (WANT_INV) {
      // (l l^T)^-1 = a^T a
      GM_UNROLL for (int i = 0; i < N; ++i)
        GM_UNROLL for (int j = i; j < N; ++j) {
          T s = (T)0;
          GM_UNROLL for (int k = j; k < N; ++k) s += ic.a[k * N + i] * ic.a[k * N + j];
          inv[i * N + j] = s;
          inv[j * N + i] = s;
        }
    }
    return (T)2 * ld;
  }

  GM_HD T dist2(const T (&x)[E], const T (&y)[E]) const {
    T z[E], dummy[E];
    GM_UNROLL for (int k = 0; k < E; ++k) z[k] = (T)0.5 * (x[k] + y[k]);
    T lz = logdet_inv<false>(z, dummy);
    T lx = logdet_inv<false>(x, dummy);
    T ly = logdet_inv<false>(y, dummy);
    return clamp_min(lz - (T)0.5 * (lx + ly), wmin);
  }

  GM_HD T dist2_grad(const T (&x)[E], const T (&y)[E], T (&gx)[E], T (&gy)[E]) const {
    T z[E], zi[E];
    GM_UNROLL for (int k = 0; k < E; ++k) z[k] = (T)0.5 * (x[k] + y[k]);
    T lz = logdet_inv<true>(z, zi);
    T lx = logdet_inv<true>(x, gx);
    T ly = logdet_inv<true>(y, gy);
    GM_UNROLL for (int k = 0; k < E; ++k) {
      gx[k] = (T)0.5 * (zi[k] - gx[k]);
      gy[k] = (T)0.5 * (zi[k] - gy[k]);
    }
    return clamp_min(lz - (T)0.5 * (lx + ly), wmin);
  }
};

// ===========================================================================
// Grassmann Gr(n, P): d^2 = sum acos^2 sigma_k(x^T y)
// grassmann.py:91-96 (dist), :27-30, linalg/fast.py:138-159 (closed-form 2x2).
// Only the P x P core lives in registers; the n x P points are streamed from
// memory by the kernel (n is a run-time value).
// ===========================================================================
template <typename T, int P, bool FAST_SVD>
struct GrassmannCore {
  T one_m;  // 1 - EPS^2 evaluated in T (== 1 in fp32, SURVEY A.3)

  // d2 and (optionally) ga = d(d2)/d(a) for a = x^T y
  GM_HD T run(const T (&a)[P * P], bool want_grad, T (&ga)[P * P]) const {
    T d2 = (T)0;
    if constexpr (FAST_SVD) {
      static_assert(P == 2, "closed-form singular values exist for 2x2 only");
      const T eps = (T)1e-8;
      T aa = a[0], bb = a[1], cc = a[2], dd = a[3];
      T S1 = aa * aa + bb * bb + cc * cc + dd * dd;
      T e = aa * aa + bb * bb - cc * cc - dd * dd;
      T f = aa * cc + bb * dd;
      T S2 = Num<T>::sqrt(clamp_min(e * e + (T)4 * f * f, eps));
      T s1 = clamp_min((T)0.5 * (S1 + S2), eps);
      T s2 = clamp_min((T)0.5 * (S1 - S2), eps);
      T sg1 = Num<T>::sqrt(s1), sg2 = Num<T>::sqrt(s2);
      T t1 = clampv(sg1, -one_m, one_m), t2 = clampv(sg2, -one_m, one_m);
      T a1 = Num<T>::acos(t1), a2 = Num<T>::acos(t2);
      d2 = a1 * a1 + a2 * a2;
      if (want_grad) {
        T h1 = -(T)2 * a1 / Num<T>::sqrt((T)1 - t1 * t1);
        T h2 = -(T)2 * a2 / Num<T>::sqrt((T)1 - t2 * t2);
        T s1b = h1 / (sg1 + sg1), s2b = h2 / (sg2 + sg2);
        T S1b = (T)0.5 * (s1b + s2b), S2b = (T)0.5 * (s1b - s2b);
        T qb = S2b / (S2 + S2);
        T eb = (T)2 * e * qb, fb = (T)8 * f * qb;
        ga[0] = (T)2 * aa * (S1b + eb) + cc * fb;
        ga[1] = (T)2 * bb * (S1b + eb) + dd * fb;
        ga[2] = (T)2 * cc * (S1b - eb) + aa * fb;
        ga[3] = (T)2 * dd * (S1b - eb) + bb * fb;
      }
    } else {
      T us[P * P], v[P * P], s[P], h[P];
      GM_UNROLL for (int k = 0; k < P * P; ++k) us[k] = a[k];
      jacobi_svd<T, P, P>(us, v, s);
      GM_UNROLL for (int k = 0; k < P; ++k) {
        T t = clampv(s[k], -one_m, one_m);
        T ac = Num<T>::acos(t);
        d2 += ac * ac;
        // u_k = us[:,k]/s_k  ->  fold 1/s_k into the coefficient
        h[k] = -(T)2 * ac / Num<T>::sqrt((T)1 - t * t) / clamp_min(s[k], Num<T>::tiny);
      }
      if (want_grad) {
        GM_UNROLL for (int i = 0; i < P; ++i)
          GM_UNROLL for (int j = 0; j < P; ++j) {
            T acc = (T)0;
            GM_UNROLL for (int k = 0; k < P; ++k) acc += us[i * P + k] * h[k] * v[j * P + k];
            ga[i * P + j] = acc;
          }
      }
    }
    return d2;
  }
};

// ===========================================================================
// Vector manifolds (run-time length n): the distance is a function of one dot
// product; the gradient is a scalar times a (signed) copy of the other endpoint.
//   value(x, y, n, c): returns d^2 and the scalar c = d(d^2)/d(dot-like quantity)
//   gx[k] = c * sx(k) * y[k]  (Lorentz/Sphere),  Euclidean: gx = -2 (y - x).
// ===========================================================================
enum VecKind { VEC_LORENTZ = 0, VEC_SPHERE = 1, VEC_EUCLIDEAN = 2, VEC_UNIVERSAL = 3 };

// Per-pair gradient coefficients.  Lorentz / Sphere / Euclidean use `c` only; Universal:
//   z_k = zA x_k + zB y_k,  gx_k = p1 z_k + p2 x_k + p3 y_k,  gy_k = q1 z_k + q2 y_k + p3 x_k,  dc = d(d^2)/d(c)
template <typename T>
struct VecCoef {
  T c;
  T zA, zB, p1, p2, p3, q1, q2, dc;
};

// ---------------------------------------------------------------------------
// kappa-stereographic ("Universal") model: manifolds/universal.py + manifolds/impl/math.py.
// c > 0: Poincare ball (tanh / artanh), c < 0: stereographic sphere (tan / atan).
// ---------------------------------------------------------------------------
template <typename T>
struct Kappa {
  static constexpr double kMinNorm = 1e-15;  // math.py:15 MIN_NORM
  // math.py:21-22
  GM_HD static T tanh_clamped(T x) { return Num<T>::tanh(clampv(x, (T)-15, (T)15)); }
  // Artanh.forward (math.py:25-35): clamp in T, evaluate in double, cast back.  `xc` returns the clamped input the
  // backward divides by (math.py:37-40).
  GM_HD static T artanh(T x, T& xc) {
    xc = clampv(x, (T)(-1.0 + 1e-15), (T)(1.0 - 1e-15));
    double xd = (double)xc;
    return (T)((::log(1.0 + xd) - ::log(1.0 - xd)) * 0.5);
  }
  GM_HD static T tan_func(T x, T c) { return c > (T)0 ? tanh_clamped(x) : Num<T>::tan(x); }  // math.py:73-85
  // arctan_func (math.py:88-99) and its derivative at x
  GM_HD static T arctan_func(T x, T c, T& dphi) {
    if (c > (T)0) {
      T xc;
      T r = artanh(x, xc);
      dphi = (T)1 / ((T)1 - xc * xc);
      return r;
    }
    dphi = (T)1 / ((T)1 + x * x);
    return Num<T>::atan(x);
  }
  GM_HD static T lambda_x(T x2, T c) { return (T)2 / clamp_min((T)1 - c * x2, (T)kMinNorm); }  // math.py:187-190
  // out = x (+)_c y  (math.py:326-345)
  GM_HD static void mobius_add(const T* x, const T* y, int n, T c, T* out) {
    T x2 = (T)0, y2 = (T)0, xy = (T)0;
    for (int k = 0; k < n; ++k) { x2 += x[k] * x[k]; y2 += y[k] * y[k]; xy += x[k] * y[k]; }
    T a = (T)1 + (T)2 * c * xy + c * y2;
    T b = (T)1 - c * x2;
    T den = clamp_min((T)1 + (T)2 * c * xy + c * c * x2 * y2, (T)kMinNorm);
    for (int k = 0; k < n; ++k) out[k] = (a * x[k] + b * y[k]) / den;
  }
  // project (math.py:142-156): only the ball (c > 0) has a boundary
  GM_HD static void project(const T* x, int n, T c, T ball_eps, T* out) {
    T s = (T)0;
    for (int k = 0; k < n; ++k) s += x[k] * x[k];
    T nrm = clamp_min(Num<T>::sqrt(s), (T)kMinNorm);
    T maxnorm = ((T)1 - ball_eps) / Num<T>::sqrt(Num<T>::abs(c));
    bool cond = (c > (T)0) && (nrm > maxnorm);
    for (int k = 0; k < n; ++k) out[k] = cond ? (x[k] / nrm) * maxnorm : x[k];
  }
};

template <typename T, int KIND>
struct VecMan {
  T eps;    // EPS[dtype] = 1e-8 (utils.py:13)
  T one_m;  // 1 - EPS^2 in T
  const T* c_dev;  // Universal: device scalar c = get_c() (universal.py:28-32)

  // Lorentz (lorentz.py:72-77,101-141): z = x0 y0 - sum_{k>=1} xk yk, clamp z >= 1,
  //   d = log(z + sqrt(z^2-1)) clamped >= EPS; Acosh backward divides by max(sqrt(z^2-1), EPS).
  // Sphere (sphere.py:68-74): s = <x,y> clamped to +-(1-EPS^2), d = acos(s) clamped >= EPS.
  // Euclidean (euclidean.py:46-50 + base.py:29-32): d^2 = max(|y-x|^2, EPS).
  // Universal (universal.py:76-81, math.py:567-572): z = (-x) (+)_c y, d = 2 arctan_c(sqrt|c| |z|) / sqrt|c|,
  //   d^2 clamped >= EPS (value only).  The gradient is taken through the vector z exactly as autograd does
  //   (z_k has no cancellation when x ~ y; a closed form in <x,x>, <y,y>, <x,y> would).
  GM_HD T value(const T* __restrict__ x, const T* __restrict__ y, int n, VecCoef<T>& co) const {
    T& c = co.c;
    if constexpr (KIND == VEC_LORENTZ) {
      T s = -(x[0] * y[0]);
      for (int k = 1; k < n; ++k) s += x[k] * y[k];
      T z = clamp_min(-s, (T)1);
      T w = Num<T>::sqrt(z * z - (T)1);
      T d = clamp_min(Num<T>::log(z + w), eps);
      c = (T)2 * d / clamp_min(w, eps);
      return d * d;
    } else if constexpr (KIND == VEC_SPHERE) {
      T s = (T)0;
      for (int k = 0; k < n; ++k) s += x[k] * y[k];
      s = clampv(s, -one_m, one_m);
      T d = clamp_min(Num<T>::acos(s), eps);
      c = -(T)2 * d / Num<T>::sqrt((T)1 - s * s);
      return d * d;
    } else if constexpr (KIND == VEC_EUCLIDEAN) {
      T s = (T)0;
      for (int k = 0; k < n; ++k) { T d = y[k] - x[k]; s += d * d; }
      c = (T)2;
      return clamp_min(s, eps);
    } else {
      const T cc = *c_dev;
      c = cc;
      T x2 = (T)0, y2 = (T)0, xy = (T)0;
      for (int k = 0; k < n; ++k) { x2 += x[k] * x[k]; y2 += y[k] * y[k]; xy += x[k] * y[k]; }
      // mobius_add(-x, y): num = A (-x) + B y, denom = D  (math.py:326-345 with <-x, y> = -xy)
      const T A = (T)1 - (T)2 * cc * xy + cc * y2;
      const T B = (T)1 - cc * x2;
      const T D = (T)1 - (T)2 * cc * xy + cc * cc * x2 * y2;
      const bool d_free = D >= (T)Kappa<T>::kMinNorm;  // clamp_min passes the gradient only where it is inactive
      const T invD = (T)1 / clamp_min(D, (T)Kappa<T>::kMinNorm);
      co.zA = -A * invD;
      co.zB = B * invD;
      T r2 = (T)0, zx = (T)0, zy = (T)0;
      for (int k = 0; k < n; ++k) {
        T z = co.zA * x[k] + co.zB * y[k];
        r2 += z * z; zx += z * x[k]; zy += z * y[k];
      }
      const T r = Num<T>::sqrt(r2);
      const T sc = Num<T>::sqrt(Num<T>::abs(cc));
      T dphi;
      const T phi = Kappa<T>::arctan_func(sc * r, cc, dphi);
      const T d = phi * (T)2 / sc;
      const T d2 = d * d;
      // d(d^2)/dz_k = gz z_k, gz = 4 d phi' / r (torch.norm's subgradient at r == 0 is 0)
      const T gz = (r > (T)0) ? (T)4 * d * dphi / r : (T)0;
      const T dA = -(gz * zx) * invD;
      const T dB = (gz * zy) * invD;
      const T dD = d_free ? -(gz * r2) * invD : (T)0;
      const T g_xy = -(T)2 * cc * (dA + dD);
      const T g_x2 = -cc * dB + cc * cc * y2 * dD;
      const T g_y2 = cc * dA + cc * cc * x2 * dD;
      co.p1 = co.zA * gz; co.p2 = (T)2 * g_x2; co.p3 = g_xy;
      co.q1 = co.zB * gz; co.q2 = (T)2 * g_y2;
      // d(d^2)/dc: through A, B, D and through sqrt|c| (u = sc r and the 2/sc factor)
      // The explicit part is 2 d * sgn(c) h(u) / sc^3 with u = sc r and h(u) = u phi'(u) - phi(u): for small u both
      // terms of h are ~u and their difference ~(2/3) u^3, so the closed form loses log10(1/u^2) digits (all of them
      // in fp32 at the default init, |c| r^2 ~ 1e-6).  There h is summed as its power series, which in w = c r^2 is
      // sgn(c) h / sc^3 = r^3 sum_{k>=1} 2k/(2k+1) w^(k-1), valid for either sign of c.  fp32 only: in fp64 the closed
      // form is evaluated exactly as the reference's autograd evaluates it, so that the two agree to 1e-10 (the
      // reference's own fp64 value carries the cancellation noise, ~1e-9 relative at the default init).
      const T sgn = cc > (T)0 ? (T)1 : (T)-1;
      const T w = cc * r2;
      T explicit_c;
      if (sizeof(T) == 4 && Num<T>::abs(w) < (T)0.1) {
        T sres = (T)0;
        GM_UNROLL for (int k = 8; k >= 1; --k) sres = sres * w + (T)(2.0 * k / (2.0 * k + 1.0));
        explicit_c = (T)2 * d * r * r2 * sres;
      } else {
        explicit_c = ((T)4 * d * dphi * r - (T)2 * d2) / sc * (sgn * (T)0.5 / sc);
      }
      co.dc = dA * (y2 - (T)2 * xy) - dB * x2 + dD * ((T)2 * cc * x2 * y2 - (T)2 * xy) + explicit_c;
      return clamp_min(d2, eps);
    }
  }
  // gradient element k of d^2 w.r.t. x and y
  GM_HD void grad_elem(int k, T xk, T yk, const VecCoef<T>& co, T& gxk, T& gyk) const {
    const T c = co.c;
    if constexpr (KIND == VEC_LORENTZ) {
      T sg = (k == 0) ? c : -c;
      gxk = sg * yk; gyk = sg * xk;
    } else if constexpr (KIND == VEC_SPHERE) {
      gxk = c * yk; gyk = c * xk;
    } else if constexpr (KIND == VEC_EUCLIDEAN) {
      T d = yk - xk;
      gxk = -c * d; gyk = c * d;
    } else {
      T z = co.zA * xk + co.zB * yk;
      gxk = co.p1 * z + co.p2 * xk + co.p3 * yk;
      gyk = co.q1 * z + co.q2 * yk + co.p3 * xk;
    }
  }
};

// ===========================================================================
// Loss terms (objectives.py:16-45): value and derivative with respect to m.
// torch.abs backward is sign() with sign(0) = 0.
// ===========================================================================
struct LossCfg {
  int kind, inc_l1, inc_l2;
  double alpha, eps;
};

// FAST: reciprocals through Num<T>::div_fast (fp32: MUFU.RCP, ~2 ulp) instead of IEEE division -- used by the
// streaming training kernel, whose loss and gradient are checked at 1e-5 relative.
template <typename T, bool FAST = false>
GM_HD T loss_term(const LossCfg& c, T g, T m, T& dm) {
  if (c.kind == 1) {  // StressLoss: (m - g)^2
    T d = m - g;
    dm = (T)2 * d;
    return d * d;
  }
  T t = g * (T)c.alpha;
  T v = (T)0;
  dm = (T)0;
  if (c.inc_l1) {
    T rt = FAST ? Num<T>::div_fast((T)1, t) : (T)1 / t;
    T q = FAST ? m * rt - (T)1 : m / t - (T)1;
    v += Num<T>::abs(q);
    dm += sgn0(q) * rt;
  }
  if (c.inc_l2) {
    T den = m + (T)c.eps;
    T rd = FAST ? Num<T>::div_fast((T)1, den) : (T)1 / den;
    T q = FAST ? t * rd - (T)1 : t / den - (T)1;
    v += Num<T>::abs(q);
    dm -= FAST ? sgn0(q) * t * rd * rd : sgn0(q) * t / (den * den);
  }
  return v;
}

}  // namespace gm
