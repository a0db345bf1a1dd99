// =====================================================================================
// ORACLE — TEST INFRASTRUCTURE ONLY.  Not part of the product.
//
// CPU restatement of the MLS-MPM substep hot path of yuanming-hu/taichi_mpm, written
// from the reference's *behaviour* (citations are path:line under /root/reference).
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
// legs may load this library.  The product (libmpmb.so) never links or calls it.
//
// PARITY STATUS (what is pinned against the reference's OWN code executed here, `make -C oracle ref`):
//   * mpm88_advance (2-D, BASELINE config 1): against mls-mpm88.cpp:16-69 (oracle/mpm88_ref.cpp);
//   * calculate_force / plasticity of the five 3-D materials and friction_project: against
//     src/particles.cpp and src/mpm_fwd.h:25-57 (oracle/particles_ref.cpp);
//   both compile the reference's translation units where they lie against stand-ins for the
//   un-vendored taichi core headers (oracle/taichi_stub/: vector/matrix vocabulary, Config, svd/polar —
//   the stand-in's header states what it restates), golden vectors under tests/golden/;
//   * the B-spline weights (quadratic, cubic, the 27-product fast kernel): against src/kernel.h
//     (oracle/kernel_ref.cpp), and the reference's own weight tests (src/tests.cpp:10-51,
//     src/transfer.cpp:353-359,975-989) restated against this file (tests/test_oracle_kat.py).
//   * the 3-D transfers (P2G and G2P, fast SSE path and scalar path): against src/transfer.cpp
//     rasterize_optimized / resample_optimized / rasterize / resample with src/mpm.h,
//     particle_allocator.h and the vendored SPGrid (oracle/transfer_ref.cpp).
//   * the rest of the substep — grid normalisation, level-set boundary condition, ordering, boundary
//     deletion — and MPM<3>::substep() as a whole: against src/mpm.cpp compiled the same way
//     (oracle/transfer_ref.cpp): same survivors, same trajectories over 10-25 substeps.
// What the stand-in core supplies instead of the reference is stated in oracle/taichi_stub/taichi/util.h;
// the one piece with a free convention is svd()/polar_decomp() (call sites src/particles.cpp:212,227,
// 394,630,642): this file has its own one-sided-Jacobi SVD and only convention-invariant quantities are
// compared (det F > 0).
//
// Two precisions are instantiated: float (same operation order / FMA placement as the
// reference's SSE path) and double (the accuracy arbiter for the GPU kernels).
// Matrices are column-major 3x3: m[c*3+r] is row r of column c (README.md:314,
// src/transfer.cpp:503,929: `M[i]` is column i).
// =====================================================================================
#include <immintrin.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <numeric>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace {

enum MaterialKind { MAT_LINEAR = 0, MAT_JELLY = 1, MAT_SNOW = 2, MAT_WATER = 3, MAT_SAND = 4, MAT_ELASTIC = 5, MAT_VON_MISES = 6, MAT_VISCO = 7 };
constexpr int kMatParams = 8;
// params layout (all kinds, unused = 0):
//  LINEAR/JELLY: [0]=mu [1]=lambda
//  SNOW        : [0]=mu_0 [1]=lambda_0 [2]=hardening [3]=theta_c [4]=theta_s [5]=min_Jp [6]=max_Jp
//  WATER       : [0]=k [1]=gamma
//  SAND        : [0]=mu_0 [1]=lambda_0 [2]=alpha [3]=cohesion [4]=beta
//  ELASTIC     : [0]=mu_0 [1]=lambda_0                                  (src/particles.cpp:764-841)
//  VON_MISES   : [0]=mu_0 [1]=lambda_0 [2]=yield_stress                 (src/particles.cpp:679-761)
//  VISCO       : [0]=mu_0 [1]=lambda_0 [2]=visco_nu [3]=visco_kappa [4]=dt (the particle's own copy of base_delta_t,
//                src/particles.cpp:66) ; scalar = visco_tau             (src/particles.cpp:40-163)

// ---------------------------------------------------------------- small 3x3 algebra
template <class R> inline R &at(R *m, int r, int c) { return m[c * 3 + r]; }
template <class R> inline R at(const R *m, int r, int c) { return m[c * 3 + r]; }

template <class R> inline void mat_mul(const R *a, const R *b, R *out) {  // out = a*b
  R t[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++) {
      R s = 0;
      for (int k = 0; k < 3; k++) s += at(a, r, k) * at(b, k, c);
      at(t, r, c) = s;
    }
  std::memcpy(out, t, sizeof(t));
}
template <class R> inline void mat_transpose(const R *a, R *out) {
  R t[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++) at(t, c, r) = at(a, r, c);
  std::memcpy(out, t, sizeof(t));
}
template <class R> inline R mat_det(const R *a) {
  return at(a, 0, 0) * (at(a, 1, 1) * at(a, 2, 2) - at(a, 1, 2) * at(a, 2, 1)) -
         at(a, 0, 1) * (at(a, 1, 0) * at(a, 2, 2) - at(a, 1, 2) * at(a, 2, 0)) +
         at(a, 0, 2) * (at(a, 1, 0) * at(a, 2, 1) - at(a, 1, 1) * at(a, 2, 0));
}
template <class R> inline void mat_inverse(const R *a, R *out) {
  R d = mat_det(a), id = R(1) / d, t[9];
  at(t, 0, 0) = (at(a, 1, 1) * at(a, 2, 2) - at(a, 1, 2) * at(a, 2, 1)) * id;
  at(t, 0, 1) = (at(a, 0, 2) * at(a, 2, 1) - at(a, 0, 1) * at(a, 2, 2)) * id;
  at(t, 0, 2) = (at(a, 0, 1) * at(a, 1, 2) - at(a, 0, 2) * at(a, 1, 1)) * id;
  at(t, 1, 0) = (at(a, 1, 2) * at(a, 2, 0) - at(a, 1, 0) * at(a, 2, 2)) * id;
  at(t, 1, 1) = (at(a, 0, 0) * at(a, 2, 2) - at(a, 0, 2) * at(a, 2, 0)) * id;
  at(t, 1, 2) = (at(a, 0, 2) * at(a, 1, 0) - at(a, 0, 0) * at(a, 1, 2)) * id;
  at(t, 2, 0) = (at(a, 1, 0) * at(a, 2, 1) - at(a, 1, 1) * at(a, 2, 0)) * id;
  at(t, 2, 1) = (at(a, 0, 1) * at(a, 2, 0) - at(a, 0, 0) * at(a, 2, 1)) * id;
  at(t, 2, 2) = (at(a, 0, 0) * at(a, 1, 1) - at(a, 0, 1) * at(a, 1, 0)) * id;
  std::memcpy(out, t, sizeof(t));
}

// One-sided Jacobi (Hestenes) SVD, A = U diag(s) V^T, s >= 0.  Stands in for the
// taichi core's svd() (call sites src/particles.cpp:227,630,642).  Sign/ordering
// conventions are NOT those of the core; only invariant results are compared.
inline void svd3_fast(const float *A, float *U, float *s, float *V);
template <class R> inline bool svd3_try_fast(const R *, R *, R *, R *) { return false; }
template <> inline bool svd3_try_fast<float>(const float *A, float *U, float *s, float *V);
template <class R> void svd3(const R *A, R *U, R *s, R *V) {
  if (svd3_try_fast<R>(A, U, s, V)) return;
  R a[9];
  std::memcpy(a, A, sizeof(a));
  for (int i = 0; i < 9; i++) V[i] = (i % 4 == 0) ? R(1) : R(0);
  const R eps = std::is_same<R, float>::value ? R(1e-7) : R(1e-15);
  for (int sweep = 0; sweep < 60; sweep++) {
    bool rotated = false;
    for (int p = 0; p < 2; p++)
      for (int q = p + 1; q < 3; q++) {
        R alpha = 0, beta = 0, gamma = 0;
        for (int r = 0; r < 3; r++) {
          alpha += at(a, r, p) * at(a, r, p);
          beta += at(a, r, q) * at(a, r, q);
          gamma += at(a, r, p) * at(a, r, q);
        }
        if (std::abs(gamma) <= eps * std::sqrt(alpha * beta) || gamma == R(0)) continue;
        rotated = true;
        R zeta = (beta - alpha) / (R(2) * gamma);
        R t = (zeta >= 0 ? R(1) : R(-1)) / (std::abs(zeta) + std::sqrt(R(1) + zeta * zeta));
        R c = R(1) / std::sqrt(R(1) + t * t), sn = c * t;
        for (int r = 0; r < 3; r++) {
          R ap = at(a, r, p), aq = at(a, r, q);
          at(a, r, p) = c * ap - sn * aq;
          at(a, r, q) = sn * ap + c * aq;
          R vp = at(V, r, p), vq = at(V, r, q);
          at(V, r, p) = c * vp - sn * vq;
          at(V, r, q) = sn * vp + c * vq;
        }
      }
    if (!rotated) break;
  }
  for (int c = 0; c < 3; c++) {
    R n = std::sqrt(at(a, 0, c) * at(a, 0, c) + at(a, 1, c) * at(a, 1, c) + at(a, 2, c) * at(a, 2, c));
    s[c] = n;
    if (n > R(0))
      for (int r = 0; r < 3; r++) at(U, r, c) = at(a, r, c) / n;
  }
  // Degenerate (rank-deficient) columns: complete U to an orthonormal basis.
  for (int c = 0; c < 3; c++)
    if (!(s[c] > R(0))) {
      int c1 = (c + 1) % 3, c2 = (c + 2) % 3;
      if (s[c1] > 0 && s[c2] > 0) {
        at(U, 0, c) = at(U, 1, c1) * at(U, 2, c2) - at(U, 2, c1) * at(U, 1, c2);
        at(U, 1, c) = at(U, 2, c1) * at(U, 0, c2) - at(U, 0, c1) * at(U, 2, c2);
        at(U, 2, c) = at(U, 0, c1) * at(U, 1, c2) - at(U, 1, c1) * at(U, 0, c2);
      } else {
        for (int r = 0; r < 3; r++) at(U, r, c) = (r == c) ? R(1) : R(0);
      }
    }
  // Make U and V proper rotations when det(A) > 0 (matches "A = U S V^T" with s>0);
  // for det(A) < 0 flip the sign of the smallest singular value (the usual
  // rotation-variant convention).  det(A) == 0 keeps s >= 0.
  R dU = mat_det(U), dV = mat_det(V);
  if (dU < 0 || dV < 0) {
    int k = 0;
    for (int c = 1; c < 3; c++)
      if (s[c] < s[k]) k = c;
    if (dU < 0 && dV < 0) {
      for (int r = 0; r < 3; r++) { at(U, r, k) = -at(U, r, k); at(V, r, k) = -at(V, r, k); }
    } else if (dU < 0) {
      for (int r = 0; r < 3; r++) at(U, r, k) = -at(U, r, k);
      s[k] = -s[k];
    } else {
      for (int r = 0; r < 3; r++) at(V, r, k) = -at(V, r, k);
      s[k] = -s[k];
    }
  }
}


// ---- faster 3x3 SVD for the TIMED fast path only (the checker paths above keep the one-sided
// Jacobi).  Stands in for the core's optimized svd() so that the CPU baseline is not dominated by
// an unoptimised factorisation: symmetric cyclic Jacobi on F^T F (V, s^2), then U = F V S^-1.
inline void svd3_fast(const float *A, float *U, float *s, float *V) {
  float c00 = 0, c11 = 0, c22 = 0, c01 = 0, c02 = 0, c12 = 0;
  for (int r = 0; r < 3; r++) {
    const float a0 = at(A, r, 0), a1 = at(A, r, 1), a2 = at(A, r, 2);
    c00 += a0 * a0; c11 += a1 * a1; c22 += a2 * a2; c01 += a0 * a1; c02 += a0 * a2; c12 += a1 * a2;
  }
  float v[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  auto rot = [&](float &app, float &aqq, float &apq, float &arp, float &arq, int p, int q) {
    if (apq == 0.f) return;
    const float d = aqq - app, b = 2.f * apq;
    const float h = std::sqrt(d * d + b * b);
    if (!(h > 0.f)) return;  // d == 0 and b*b underflowed: already diagonal to working precision
    const float t = b / (d + (d >= 0.f ? h : -h));
    const float c = 1.f / std::sqrt(t * t + 1.f), sn = t * c;
    app -= t * apq; aqq += t * apq; apq = 0.f;
    const float nrp = c * arp - sn * arq, nrq = sn * arp + c * arq;
    arp = nrp; arq = nrq;
    for (int r = 0; r < 3; r++) {
      const float vp = at(v, r, p), vq = at(v, r, q);
      at(v, r, p) = c * vp - sn * vq;
      at(v, r, q) = sn * vp + c * vq;
    }
  };
  for (int sweep = 0; sweep < 6; sweep++) {
    rot(c00, c11, c01, c02, c12, 0, 1);
    rot(c00, c22, c02, c01, c12, 0, 2);
    rot(c11, c22, c12, c01, c02, 1, 2);
    const float off = c01 * c01 + c02 * c02 + c12 * c12, nrm = c00 * c00 + c11 * c11 + c22 * c22;
    if (off <= 1e-14f * nrm) break;
  }
  s[0] = std::sqrt(std::max(c00, 0.f)); s[1] = std::sqrt(std::max(c11, 0.f)); s[2] = std::sqrt(std::max(c22, 0.f));
  for (int i = 0; i < 9; i++) V[i] = v[i];
  for (int c = 0; c < 3; c++) {
    const float inv = s[c] > 1e-20f ? 1.f / s[c] : 0.f;
    for (int r = 0; r < 3; r++) at(U, r, c) = (at(A, r, 0) * at(v, 0, c) + at(A, r, 1) * at(v, 1, c) + at(A, r, 2) * at(v, 2, c)) * inv;
  }
}
// thread-local switch: the fast path routes svd3<float> through svd3_fast
static thread_local bool g_use_fast_svd = false;
template <> inline bool svd3_try_fast<float>(const float *A, float *U, float *s, float *V) {
  if (!g_use_fast_svd) return false;
  svd3_fast(A, U, s, V);
  return true;
}

// polar_decomp(A, R, S): A = R S (usage src/particles.cpp:212-215,394; mls-mpm88.cpp:26)
template <class R> void polar3(const R *A, R *Rm, R *S) {
  R U[9], s[3], V[9], Vt[9];
  svd3(A, U, s, V);
  mat_transpose(V, Vt);
  mat_mul(U, Vt, Rm);
  R SV[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++) at(SV, r, c) = at(V, r, c) * s[c];
  mat_mul(SV, Vt, S);
}

// ------------------------------------------------------------------- B-spline weights
// MPMKernel<dim,2>::calculate_kernel (src/kernel.h:122-134): p_fract = fract(pos-0.5),
// t = p_fract - (-0.5,0.5,1.5); w = (0.5,-1,0.5) t^2 + (-1.5,0,1.5) t + (1.125,0.75,1.125);
// dw = (1,-2,1) t + (-1.5,0,1.5).
template <class R> void quadratic_kernel_axis(R x, R *w, R *dw) {
  R s = x - R(0.5);
  R f = s - std::floor(s);
  const R off[3] = {R(-0.5), R(0.5), R(1.5)};
  const R a2[3] = {R(0.5), R(-1), R(0.5)}, a1[3] = {R(-1.5), R(0), R(1.5)}, a0[3] = {R(1.125), R(0.75), R(1.125)};
  const R d1[3] = {R(1), R(-2), R(1)}, d0[3] = {R(-1.5), R(0), R(1.5)};
  for (int k = 0; k < 3; k++) {
    R t = f - off[k];
    w[k] = a2[k] * (t * t) + a1[k] * t + a0[k];
    dw[k] = d1[k] * t + d0[k];
  }
}
// Cubic kernel weights for the reference's order-3 KAT (src/kernel.h:137-166).
template <class R> void cubic_kernel_axis(R x, R *w, R *dw) {
  R f = x - std::floor(x);
  const R off[4] = {R(-1), R(0), R(1), R(2)};
  const R a3[4] = {R(-1) / 6, R(0.5), R(-0.5), R(1) / 6}, a2[4] = {R(1), R(-1), R(-1), R(1)},
          a1[4] = {R(-2), R(0), R(0), R(2)}, a0[4] = {R(4) / 3, R(2) / 3, R(2) / 3, R(4) / 3};
  const R d2[4] = {R(-0.5), R(1.5), R(-1.5), R(0.5)}, d1[4] = {R(2), R(-2), R(-2), R(2)}, d0[4] = {R(-2), R(0), R(0), R(2)};
  for (int k = 0; k < 4; k++) {
    R t = f - off[k], tt = t * t;
    w[k] = a3[k] * (tt * t) + a2[k] * tt + a1[k] * t + a0[k];
    dw[k] = d2[k] * tt + d1[k] * t + d0[k];
  }
}

// MLSMPMFastKernel32 (src/transfer.cpp:162-186): input = pos/dx - base in [0.5,1.5)^3;
// p_fract = rel - 0.5; t = p_fract - (-0.5,0.5,1.5);
// w = fma((0.5,-1,0.5), t*t, fma((-1.5,0,1.5), t, (1.125,0.75,1.125)));
// kernels[i][j][k] = (w0[i]*w1[j]) * w2[k].
template <class R> inline void mls_axis_weights(R rel, R *w) {
  R pf = rel - R(0.5);
  const R off[3] = {R(-0.5), R(0.5), R(1.5)};
  const R a2[3] = {R(0.5), R(-1), R(0.5)}, a1[3] = {R(-1.5), R(0), R(1.5)}, a0[3] = {R(1.125), R(0.75), R(1.125)};
  for (int k = 0; k < 3; k++) {
    R t = pf - off[k];
    R tt = t * t;
    w[k] = std::fma(a2[k], tt, std::fma(a1[k], t, a0[k]));
  }
}
template <class R> inline void mls_fast_kernel(const R *rel, R *w27) {
  R w[3][3];
  for (int d = 0; d < 3; d++) mls_axis_weights(rel[d], w[d]);
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) {
      R wij = w[0][i] * w[1][j];
      for (int k = 0; k < 3; k++) w27[i * 9 + j * 3 + k] = wij * w[2][k];
    }
}

// ------------------------------------------------------------------ constitutive models
// calculate_force() returns -vol * P(F) * F^T (src/particles.cpp:216-218,335-337,409-411,
// 463-467,628-637).  plasticity(cdg) updates F and the plastic scalar.
template <class R> void first_piola_fixed_corotated(const R *F, R mu, R lambda, R *P) {
  // src/particles.cpp:391-398 (jelly) / 207-214 (snow): 2mu(F-R) + lambda(J-1)J F^-T
  R j = mat_det(F);
  R r[9], s[9];
  polar3(F, r, s);
  R Ft[9], FinvT[9];
  mat_transpose(F, Ft);
  mat_inverse(Ft, FinvT);
  for (int i = 0; i < 9; i++) P[i] = R(2) * mu * (F[i] - r[i]) + lambda * (j - R(1)) * j * FinvT[i];
}

template <class R> void calculate_force(int kind, const R *prm, const R *F, R ps, R vol, R *out) {
  R P[9], Ft[9], PFt[9];
  switch (kind) {
    case MAT_LINEAR: {  // src/particles.cpp:329-337
      R mu = prm[0], lambda = prm[1];
      R tr = at(F, 0, 0) + at(F, 1, 1) + at(F, 2, 2);
      for (int c = 0; c < 3; c++)
        for (int r = 0; r < 3; r++)
          at(P, r, c) = mu * (at(F, r, c) + at(F, c, r) - (r == c ? R(2) : R(0))) + (r == c ? lambda * (tr - R(3)) : R(0));
      mat_transpose(F, Ft);
      mat_mul(P, Ft, PFt);
      for (int i = 0; i < 9; i++) out[i] = -vol * PFt[i];
      return;
    }
    case MAT_JELLY: {  // src/particles.cpp:391-411
      first_piola_fixed_corotated(F, prm[0], prm[1], P);
      mat_transpose(F, Ft);
      mat_mul(P, Ft, PFt);
      for (int i = 0; i < 9; i++) out[i] = -vol * PFt[i];
      return;
    }
    case MAT_SNOW: {  // src/particles.cpp:207-218,244-252: mu,lambda *= exp(h(1-Jp))
      R e = std::exp(prm[2] * (R(1) - ps));
      first_piola_fixed_corotated(F, prm[0] * e, prm[1] * e, P);
      mat_transpose(F, Ft);
      mat_mul(P, Ft, PFt);
      for (int i = 0; i < 9; i++) out[i] = -vol * PFt[i];
      return;
    }
    case MAT_WATER: {  // src/particles.cpp:463-467: p = k(j^-gamma - 1); -vol*j*(-p I)
      R j = ps;
      R p = prm[0] * (std::pow(j, -prm[1]) - R(1));
      for (int i = 0; i < 9; i++) out[i] = R(0);
      for (int d = 0; d < 3; d++) at(out, d, d) = -vol * j * (-p);
      return;
    }
    case MAT_VISCO: {  // src/particles.cpp:69-82: fixed corotated with the constant mu_0, lambda_0
      first_piola_fixed_corotated(F, prm[0], prm[1], P);
      mat_transpose(F, Ft);
      mat_mul(P, Ft, PFt);
      for (int i = 0; i < 9; i++) out[i] = -vol * PFt[i];
      return;
    }
    case MAT_ELASTIC:    // src/particles.cpp:800-809  (the same Hencky stress, word for word)
    case MAT_VON_MISES:  // src/particles.cpp:703-712
    case MAT_SAND: {     // src/particles.cpp:628-637
      R mu0 = prm[0], lambda0 = prm[1];
      R U[9], s[3], V[9];
      svd3(F, U, s, V);
      R ls[3], is[3], center[3];
      for (int d = 0; d < 3; d++) { ls[d] = std::log(s[d]); is[d] = R(1) / s[d]; }
      R trl = ls[0] + ls[1] + ls[2];
      for (int d = 0; d < 3; d++) center[d] = R(2) * mu0 * is[d] * ls[d] + lambda0 * trl * is[d];
      R UC[9], Vt[9], UCVt[9];
      for (int c = 0; c < 3; c++)
        for (int r = 0; r < 3; r++) at(UC, r, c) = at(U, r, c) * center[c];
      mat_transpose(V, Vt);
      mat_mul(UC, Vt, UCVt);
      mat_transpose(F, Ft);
      mat_mul(UCVt, Ft, PFt);
      for (int i = 0; i < 9; i++) out[i] = -vol * PFt[i];
      return;
    }
  }
}

template <class R> void sand_project(const R *prm, const R *sigma, R &logJp, R *sigma_out) {
  // src/particles.cpp:599-626
  const R d = 3;
  R mu0 = prm[0], lambda0 = prm[1], alpha = prm[2], cohesion = prm[3], beta = prm[4];
  R eps[3], tr = 0;
  for (int i = 0; i < 3; i++) {
    eps[i] = std::log(std::max(std::abs(sigma[i]), R(1e-4))) - cohesion;
    tr += eps[i];
  }
  R eps_sum = tr;
  tr += logJp;
  R hat[3], hat_n2 = 0;
  for (int i = 0; i < 3; i++) { hat[i] = eps[i] - tr / d; hat_n2 += hat[i] * hat[i]; }
  R hat_n = std::sqrt(hat_n2);
  if (tr >= R(0)) {
    for (int i = 0; i < 3; i++) sigma_out[i] = std::exp(cohesion);
    logJp = beta * eps_sum + logJp;
  } else {
    logJp = 0;
    R dgamma = hat_n + (d * lambda0 + R(2) * mu0) / (R(2) * mu0) * tr * alpha;
    if (dgamma <= 0) {
      for (int i = 0; i < 3; i++) sigma_out[i] = std::exp(eps[i] + cohesion);
    } else {
      for (int i = 0; i < 3; i++) sigma_out[i] = std::exp(eps[i] - dgamma / hat_n * hat[i] + cohesion);
    }
  }
}

// ViscoParticle::approximate_exponent (src/particles.cpp:89-102): r = (s/2 + I) s + I with s = m dt; if det r <= 0
// the step is halved and the result squared.
template <class R> void visco_approximate_exponent(R dt, const R *m, R *out, int depth = 0) {
  R s[9], h[9], r[9];
  for (int i = 0; i < 9; i++) { s[i] = m[i] * dt; h[i] = s[i] * R(0.5); }
  for (int d = 0; d < 3; d++) at(h, d, d) += R(1);
  mat_mul(h, s, r);
  for (int d = 0; d < 3; d++) at(r, d, d) += R(1);
  if (mat_det(r) > R(0) || depth >= 16) {
    std::memcpy(out, r, sizeof(r));
    return;
  }
  R tmp[9];
  visco_approximate_exponent(dt / R(2), m, tmp, depth + 1);
  mat_mul(tmp, tmp, out);
}

// ViscoParticle::plasticity (src/particles.cpp:104-137).  ps = visco_tau.
template <class R> void visco_plasticity(const R *prm, const R *cdg, R *F, R &ps) {
  const R mu0 = prm[0], lambda0 = prm[1], nu = prm[2], kappa = prm[3], dt = prm[4];
  R m[9], ex[9], Fh[9];
  for (int i = 0; i < 9; i++) m[i] = cdg[i];
  for (int d = 0; d < 3; d++) at(m, d, d) -= R(1);
  for (int i = 0; i < 9; i++) m[i] *= (R(1) / dt);
  visco_approximate_exponent(dt, m, ex);
  mat_mul(ex, F, Fh);
  R U[9], sg[3], V[9], Vt[9];
  svd3(Fh, U, sg, V);
  mat_transpose(V, Vt);
  R P[9], pn2 = 0;
  first_piola_fixed_corotated(F, mu0, lambda0, P);  // of the OLD dg_e (111: this->dg_e is not yet updated)
  for (int i = 0; i < 9; i++) pn2 += P[i] * P[i];
  const R pnorm = std::sqrt(pn2);
  R gamma = 0;
  if (pnorm > R(1e-5)) gamma = std::min(std::max(dt * nu * (pnorm - ps) / pnorm, R(0)), R(1));
  const R det = sg[0] * sg[1] * sg[2];
  R scale = 1;
  if (std::abs(det) > R(1e-5)) scale = R(1) / std::pow(det, R(1) / R(3));
  R snew[3];
  for (int d = 0; d < 3; d++) {
    const R mid = std::pow(sg[d] * scale, gamma);
    const R mid_inv = std::abs(mid) > R(1e-5) ? R(1) / mid : R(1);
    snew[d] = sg[d] * mid_inv;
  }
  // the second svd (127-130) of U diag(snew) V^T returns the same factors: clamp the singular values in place
  for (int d = 0; d < 3; d++) snew[d] = std::min(std::max(snew[d], R(0.1)), R(10));
  R US[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++) at(US, r, c) = at(U, r, c) * snew[c];
  mat_mul(US, Vt, F);
  ps += kappa * gamma * pnorm;
}

template <class R> void plasticity(int kind, const R *prm, const R *cdg, R *F, R &ps) {
  if (kind == MAT_WATER) {  // src/particles.cpp:469-478: j *= tr(cdg) - (dim-1); floor 0.1
    ps *= (at(cdg, 0, 0) + at(cdg, 1, 1) + at(cdg, 2, 2)) - R(2);
    if (ps < R(0.1)) ps = R(0.1);
    return;
  }
  if (kind == MAT_VISCO) {
    visco_plasticity(prm, cdg, F, ps);
    return;
  }
  R Fn[9];
  mat_mul(cdg, F, Fn);  // dg_e = cdg * dg_e (src/particles.cpp:223,342,414,640,715,812)
  if (kind == MAT_LINEAR || kind == MAT_JELLY || kind == MAT_ELASTIC) {
    std::memcpy(F, Fn, sizeof(Fn));
    return;
  }
  R U[9], s[3], V[9], Vt[9];
  svd3(Fn, U, s, V);
  mat_transpose(V, Vt);
  R snew[3];
  if (kind == MAT_VON_MISES) {  // src/particles.cpp:714-734
    R mu0 = prm[0], yield_stress = prm[2];
    R eps[3], tr = 0;
    for (int i = 0; i < 3; i++) { eps[i] = std::log(s[i]); tr += eps[i]; }
    R hat[3], n2 = 0;
    for (int i = 0; i < 3; i++) { hat[i] = eps[i] - tr / R(3); n2 += hat[i] * hat[i]; }
    // NB `epsilon_hat.frobenius_norm2()` (724): the SQUARED Frobenius norm enters both the yield test and the scaling
    R dgamma = n2 - yield_stress / (R(2) * mu0);
    if (dgamma <= 0) {  // case I: dg_e = cdg * dg_e is kept as it is (no rebuild from the factors)
      std::memcpy(F, Fn, sizeof(Fn));
      return;
    }
    for (int i = 0; i < 3; i++) snew[i] = std::exp(eps[i] - (dgamma / n2) * hat[i]);
  } else if (kind == MAT_SNOW) {  // src/particles.cpp:222-242
    R theta_c = prm[3], theta_s = prm[4], minJp = prm[5], maxJp = prm[6];
    R det_orig = 1, det_new = 1;
    for (int i = 0; i < 3; i++) {
      det_orig *= s[i];
      snew[i] = std::min(std::max(s[i], R(1) - theta_c), R(1) + theta_s);
      det_new *= snew[i];
    }
    R Jp_new = ps * det_orig / det_new;
    if (!(Jp_new <= maxJp)) Jp_new = maxJp;
    if (!(Jp_new >= minJp)) Jp_new = minJp;
    ps = Jp_new;
  } else {  // MAT_SAND, src/particles.cpp:639-647
    sand_project(prm, s, ps, snew);
  }
  R US[9];
  for (int c = 0; c < 3; c++)
    for (int r = 0; r < 3; r++) at(US, r, c) = at(U, r, c) * snew[c];
  mat_mul(US, Vt, F);
}

// ------------------------------------------------------------------ grid boundary op
// friction_project (src/mpm_fwd.h:25-57)
template <class R> void friction_project(const R *vel, const R *base, const R *n, R friction, R *out) {
  R rel[3] = {vel[0] - base[0], vel[1] - base[1], vel[2] - base[2]};
  if (friction == R(-1)) { out[0] = base[0]; out[1] = base[1]; out[2] = base[2]; return; }
  bool slip = friction <= R(-2);
  if (slip) friction = -friction - R(2);
  R nn = n[0] * rel[0] + n[1] * rel[1] + n[2] * rel[2];
  R tang[3] = {rel[0] - nn * n[0], rel[1] - nn * n[1], rel[2] - nn * n[2]};
  R tn = std::sqrt(tang[0] * tang[0] + tang[1] * tang[1] + tang[2] * tang[2]);
  R scale = std::max(tn + std::min(nn, R(0)) * friction, R(0)) / std::max(R(1e-30), tn);
  R keep = std::max(R(0), nn * R(!slip));
  for (int d = 0; d < 3; d++) out[d] = scale * tang[d] + keep * n[d] + base[d];
}

// ------------------------------------------------------------------ scene description
template <class R> struct Scene {
  int res[3];            // cells per axis; nodes = res+1 (src/mpm.cpp:66)
  R dx, inv_dx, dt;
  R gravity[3];
  int particle_gravity;  // default true (src/mpm.cpp:47)
  const int32_t *mat_kind;  // [n_groups]
  const R *mat_params;      // [n_groups][kMatParams]
  const R *sdf;             // dense node array [nx][ny][nz][4] = (n_x,n_y,n_z,phi) in grid units, or null
  R friction;               // levelset0->friction
  int nx() const { return res[0] + 1; }
  int ny() const { return res[1] + 1; }
  int nz() const { return res[2] + 1; }
  size_t node(int i, int j, int k) const { return (size_t(i) * ny() + j) * nz() + k; }
  size_t n_nodes() const { return size_t(nx()) * ny() * nz(); }
};

template <class R> struct Particles {
  int64_t n;
  R *x, *v, *F, *b;      // [n][3], [n][3], [n][9], [n][9] (b = apic_b)
  const R *mass, *vol;   // [n]
  R *ps;                 // plastic scalar: Jp (snow), j (water), logJp (sand)
  const int32_t *group;  // material group per particle
};

template <class R> inline void base_and_rel(const Scene<R> &sc, const R *x, int *base, R *rel) {
  // pos_ = p.pos * inv_delta_x (src/transfer.cpp:490); base = int(x - 0.5) (src/kernel.h:119-121)
  for (int d = 0; d < 3; d++) {
    R X = x[d] * sc.inv_dx;
    base[d] = int(X - R(0.5));
    rel[d] = X - R(base[d]);
  }
}

// Order in which the reference visits particles: sorted by (SPGrid block of the base
// node, node-in-block, particle index) (src/mpm.cpp:783-795).  Only the fp32 summation
// order depends on it.  Blocks are 4x4x8 (x,y,z) (src/mpm_fwd.h:69-119); we order
// blocks lexicographically instead of by the SPGrid Morton offset.
template <class R> std::vector<int64_t> visit_order(const Scene<R> &sc, const Particles<R> &P, const uint8_t *alive) {
  std::vector<std::pair<uint64_t, int64_t>> keys;
  keys.reserve(P.n);
  for (int64_t i = 0; i < P.n; i++) {
    if (alive && !alive[i]) continue;
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * i, base, rel);
    uint64_t bx = base[0] >> 2, by = base[1] >> 2, bz = base[2] >> 3;
    uint64_t in = (base[0] & 3) * 32 + (base[1] & 3) * 8 + (base[2] & 7);
    uint64_t blk = (bx * 4096 + by) * 4096 + bz;
    keys.push_back({(blk << 7) | in, i});
  }
  std::sort(keys.begin(), keys.end());
  std::vector<int64_t> order(keys.size());
  for (size_t i = 0; i < keys.size(); i++) order[i] = keys[i].second;
  return order;
}

// ----------------------------------------------------------------------------- P2G
// MPM<3>::rasterize_optimized / block_op_normal (src/transfer.cpp:467-569).
// grid: dense [nodes][4] = (p_x,p_y,p_z,m), must be zeroed by the caller
// (sort_particles_and_populate_grid memsets the active blocks, src/mpm.cpp:868-874).
template <class R> void p2g(const Scene<R> &sc, Particles<R> &P, const std::vector<int64_t> &order, R *grid) {
  const R S = R(-4) * sc.inv_dx * sc.dt;  // src/transfer.cpp:465
  for (int64_t i : order) {
    R *v = P.v + 3 * i;
    if (sc.particle_gravity)  // src/transfer.cpp:485-487 (stored back)
      for (int d = 0; d < 3; d++) v[d] = v[d] + sc.gravity[d] * sc.dt;
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * i, base, rel);
    R w27[27];
    mls_fast_kernel(rel, w27);
    const R mass = P.mass[i];
    const int g = P.group[i];
    R stress[9];
    calculate_force(sc.mat_kind[g], sc.mat_params + g * kMatParams, P.F + 9 * i, P.ps[i], P.vol[i], stress);
    R affine[9];  // affine[c] = fma(stress[c], S, apic_b[c] * (inv_D*mass)) (src/transfer.cpp:503,521-522)
    const R bm = R(4) * mass;  // Kernel::inv_D() = 6 - order = 4 (src/kernel.h:68-70)
    for (int k = 0; k < 9; k++) affine[k] = std::fma(stress[k], S, P.b[9 * i + k] * bm);
    R mv[3] = {mass * v[0], mass * v[1], mass * v[2]};
    for (int a = 0; a < 3; a++)
      for (int bb = 0; bb < 3; bb++)
        for (int c = 0; c < 3; c++) {
          R d[3] = {rel[0] - R(a), rel[1] - R(bb), rel[2] - R(c)};  // particle - node, grid units (528)
          R w = w27[a * 9 + bb * 3 + c];
          R *gn = grid + 4 * sc.node(base[0] + a, base[1] + bb, base[2] + c);
          for (int r = 0; r < 3; r++) {
            // fma(affine[2], d2, fma(affine[1], d1, fma(affine[0], d0, mass_v)))  (533-536)
            R ap = std::fma(at(affine, r, 2), d[2], std::fma(at(affine, r, 1), d[1], std::fma(at(affine, r, 0), d[0], mv[r])));
            gn[r] = gn[r] + w * ap;
          }
          gn[3] = gn[3] + w * mass;
        }
  }
}

// ---------------------------------------------------------------------- grid update
// normalize_grid_and_apply_external_force (src/mpm.cpp:277-294) then
// apply_grid_boundary_conditions (src/mpm.cpp:296-372), static level set.
template <class R> void grid_update(const Scene<R> &sc, R *grid) {
  R incr[3] = {0, 0, 0};
  if (!sc.particle_gravity)
    for (int d = 0; d < 3; d++) incr[d] = sc.gravity[d] * sc.dt;  // src/mpm.cpp:526-530
  const size_t nn = sc.n_nodes();
#pragma omp parallel for schedule(static)
  for (size_t n = 0; n < nn; n++) {
    R *g = grid + 4 * n;
    R mass = g[3];
    if (mass > 0) {
      R inv = R(1) / mass;
      for (int d = 0; d < 3; d++) g[d] = std::fma(g[d], inv, incr[d]);
    }
    if (sc.sdf && mass != R(0)) {
      const R *s = sc.sdf + 4 * n;
      R phi = s[3];
      if (phi < R(-3) || R(0) < phi) continue;
      R vb[3] = {0, 0, 0};  // static level set: -d(phi)/dt * n * dx = 0
      R out[3];
      friction_project(g, vb, s, sc.friction, out);
      g[0] = out[0]; g[1] = out[1]; g[2] = out[2];
    }
  }
}

// ----------------------------------------------------------------------------- G2P
// MPM<3>::resample_optimized / block_op_normal (src/transfer.cpp:837-954).
template <class R> void g2p(const Scene<R> &sc, Particles<R> &P, const std::vector<int64_t> &order, const R *grid) {
  const R scale = R(-4) * sc.inv_dx * sc.dt;  // src/transfer.cpp:938
  const int64_t m = (int64_t)order.size();
#pragma omp parallel for schedule(static)
  for (int64_t oi = 0; oi < m; oi++) {
    int64_t i = order[oi];
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * i, base, rel);
    R w27[27];
    mls_fast_kernel(rel, w27);
    R vacc[3] = {0, 0, 0}, b[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int a = 0; a < 3; a++)
      for (int bb = 0; bb < 3; bb++)
        for (int c = 0; c < 3; c++) {
          R d[3] = {rel[0] - R(a), rel[1] - R(bb), rel[2] - R(c)};
          R w = w27[a * 9 + bb * 3 + c];
          const R *gn = grid + 4 * sc.node(base[0] + a, base[1] + bb, base[2] + c);
          for (int r = 0; r < 3; r++) {
            vacc[r] = std::fma(gn[r], w, vacc[r]);             // v_ = fma(grid_vel, w, v_)
            R wg = w * gn[r];                                   // w_grid_vel
            for (int cc = 0; cc < 3; cc++) at(b, r, cc) = std::fma(wg, d[cc], at(b, r, cc));  // b_[cc] (900-903)
          }
        }
    std::memcpy(P.b + 9 * i, b, sizeof(b));        // apic_b <- b (928-930; damping branch not taken)
    for (int d = 0; d < 3; d++) P.v[3 * i + d] = vacc[d];  // set_velocity (933)
    R cdg[9];
    for (int c = 0; c < 3; c++)
      for (int r = 0; r < 3; r++) at(cdg, r, c) = std::fma(scale, at(b, r, c), r == c ? R(1) : R(0));  // 940-942
    const int g = P.group[i];
    plasticity(sc.mat_kind[g], sc.mat_params + g * kMatParams, cdg, P.F + 9 * i, P.ps[i]);  // 950
    for (int d = 0; d < 3; d++) P.x[3 * i + d] = std::fma(vacc[d], sc.dt, P.x[3 * i + d]);    // 951
  }
}

// clear_boundary_particles + near_boundary (src/mpm.cpp:583-633, src/mpm.h:269-276)
template <class R> void clear_boundary(const Scene<R> &sc, const Particles<R> &P, uint8_t *alive) {
  for (int64_t i = 0; i < P.n; i++) {
    if (!alive[i]) continue;
    const R *x = P.x + 3 * i, *v = P.v + 3 * i;
    R pmin = x[0] * sc.inv_dx, pmax = x[0] * sc.inv_dx - R(sc.res[0]);
    bool bad = false;
    for (int d = 0; d < 3; d++) {
      R X = x[d] * sc.inv_dx;
      pmin = std::min(pmin, X);
      pmax = std::max(pmax, X - R(sc.res[d]));
      if (!std::isfinite(x[d]) || !std::isfinite(v[d])) bad = true;
    }
    if (pmin < R(7) || pmax > R(-7)) bad = true;
    if (bad) alive[i] = 0;
  }
}

template <class R>
void substep(const Scene<R> &sc, Particles<R> &P, uint8_t *alive, R *grid_out /* may be null */, R *grid_rast_out /* may be null */) {
  std::vector<R> grid_local;
  R *grid = grid_out;
  if (!grid) { grid_local.assign(sc.n_nodes() * 4, R(0)); grid = grid_local.data(); }
  else std::fill(grid, grid + sc.n_nodes() * 4, R(0));
  auto order = visit_order(sc, P, alive);
  p2g(sc, P, order, grid);
  if (grid_rast_out) std::memcpy(grid_rast_out, grid, sizeof(R) * sc.n_nodes() * 4);
  grid_update(sc, grid);
  g2p(sc, P, order, grid);
  clear_boundary(sc, P, alive);
}

// ================================================================================
// CPIC rigid-coupled path (SURVEY §8f row 2): rasterize_rigid_boundary + gather_cdf (src/rigid_transfer.cpp:18-113,
// 120-274), update_rigid_page_map (src/mpm.cpp:1026-1076), block_op_rigid of rasterize_optimized / resample_optimized
// (src/transfer.cpp:367-463, 706-835).  PARITY STATUS: the MPM side follows those lines; what they call in the
// un-vendored core is ASSUMED and stated here once (SURVEY appendix C):
//   RigidBody::get_velocity_at(p)        = velocity + angular_velocity x (p - position)
//   RigidBody::apply_tmp_impulse(j, p)   : tmp_velocity += inv_mass j ; tmp_angular_velocity += Iw^-1 ((p - position) x j)
//   reset_tmp_velocity / apply_tmp_velocity : zero the two accumulators / add them to velocity, angular_velocity
//   get_mesh_to_world() = get_centroid_to_world() = x -> position + Rot x   (the mesh is re-centred on the centre of
//                                                    mass at creation, src/mpm_rigid_body.cpp:190-207)
//   Element::get_transformed(M)          : the three vertices mapped by M
//   world_to_element(e)                  = [v1 - v0, v2 - v0, n]^-1, n = unit normal (v1-v0) x (v2-v0)
//   VectorI(ind) for a Region index      = the index's integer coordinates — with which update_rigid_page_map's range test
//                                          (src/mpm.cpp:1062) admits only the offsets {0,1}^3 of the 27 it loops over
// Rigid ids index MPM::rigids; 0 is the background body (src/mpm.cpp:72-74), so real bodies are 1..11.
// ================================================================================
constexpr uint32_t kStateMask = 0xAAAAAAAAu;       // src/mpm.h:36 (the particle / node words are 32-bit)
constexpr int kTagBits = 24;                       // GridState::tag_bits = 12 bodies x 2 (src/mpm_fwd.h:79-85)
constexpr uint32_t kTagMask = (1u << kTagBits) - 1u;

template <class R> struct Rigid {
  int n_rigid;                      // length of the per-body arrays (body 0 = background, never referenced)
  const R *position, *rot;          // [n_rigid][3], [n_rigid][9] column-major
  R *velocity, *angular_velocity;   // [n_rigid][3]; updated by apply_tmp_velocity after each transfer
  const R *inv_mass, *inv_inertia;  // [n_rigid], [n_rigid][9] world-space, column-major
  const R *frictions;               // [n_rigid][2]
  int64_t n_samples;                // RigidBoundaryParticles (src/boundary_particle.h)
  const R *offset, *tri;            // [ns][3] anchor in the centroid frame, [ns][9] untransformed_element (v0,v1,v2)
  const int32_t *sample_rigid;      // [ns]
  R penalty, pushing_force;         // src/mpm.cpp:35,40
  uint32_t *states;                 // [n] MPMParticle::states (persists)
  R *bnormal, *bdist;               // [n][3], [n]   boundary_normal, boundary_distance (rewritten every substep)
  uint8_t *near;                    // [n]           near_boundary_
  // scratch
  std::vector<uint32_t> node_state; // tags | (rigid id + 1) << 24   (GridState::states)
  std::vector<R> node_dist;         // GridState::distance
  std::vector<uint8_t> page;        // rigid_page_map over 4x4x8 blocks
  std::vector<R> tmp_v, tmp_w;
  int nb[3];
};

template <class R> inline void cross3(const R *a, const R *b, R *o) {
  o[0] = a[1] * b[2] - a[2] * b[1];
  o[1] = a[2] * b[0] - a[0] * b[2];
  o[2] = a[0] * b[1] - a[1] * b[0];
}
template <class R> inline void rigid_to_world(const Rigid<R> &rg, int id, const R *local, R *out) {
  const R *c = rg.position + 3 * id, *M = rg.rot + 9 * id;
  for (int r = 0; r < 3; r++) out[r] = c[r] + (at(M, r, 0) * local[0] + at(M, r, 1) * local[1] + at(M, r, 2) * local[2]);
}
template <class R> inline void rigid_velocity_at(const Rigid<R> &rg, int id, const R *p, R *out) {
  R d[3] = {p[0] - rg.position[3 * id], p[1] - rg.position[3 * id + 1], p[2] - rg.position[3 * id + 2]}, w[3];
  cross3(rg.angular_velocity + 3 * id, d, w);
  for (int k = 0; k < 3; k++) out[k] = rg.velocity[3 * id + k] + w[k];
}
template <class R> inline void rigid_apply_tmp_impulse(Rigid<R> &rg, int id, const R *j, const R *p) {
  R d[3] = {p[0] - rg.position[3 * id], p[1] - rg.position[3 * id + 1], p[2] - rg.position[3 * id + 2]}, t[3];
  cross3(d, j, t);
  const R *I = rg.inv_inertia + 9 * id;
  for (int k = 0; k < 3; k++) {
    rg.tmp_v[3 * id + k] += rg.inv_mass[id] * j[k];
    rg.tmp_w[3 * id + k] += at(I, k, 0) * t[0] + at(I, k, 1) * t[1] + at(I, k, 2) * t[2];
  }
}
template <class R> inline void rigid_reset_tmp(Rigid<R> &rg) {
  rg.tmp_v.assign(size_t(rg.n_rigid) * 3, R(0));
  rg.tmp_w.assign(size_t(rg.n_rigid) * 3, R(0));
}
template <class R> inline void rigid_apply_tmp(Rigid<R> &rg) {
  for (int k = 0; k < rg.n_rigid * 3; k++) { rg.velocity[k] += rg.tmp_v[k]; rg.angular_velocity[k] += rg.tmp_w[k]; }
}
template <class R> inline bool rigid_page_of_block(const Rigid<R> &rg, int bx, int by, int bz) {
  if (bx < 0 || by < 0 || bz < 0 || bx >= rg.nb[0] || by >= rg.nb[1] || bz >= rg.nb[2]) return false;
  return rg.page[(size_t(bx) * rg.nb[1] + by) * rg.nb[2] + bz] != 0;
}

// sample s: world position of its anchor (align_with_rigid_body, src/boundary_particle.h:48-53)
template <class R> inline void sample_world(const Rigid<R> &rg, int64_t s, R *pos) { rigid_to_world(rg, rg.sample_rigid[s], rg.offset + 3 * s, pos); }

// update_rigid_page_map (src/mpm.cpp:1026-1076): blocks that hold a rigid particle (by its base node) and — because of the
// range test on the OFFSET at 1062 — their {0,1}^3 upper neighbours.
template <class R> void rigid_pages(const Scene<R> &sc, Rigid<R> &rg) {
  rg.nb[0] = (sc.nx() + 3) / 4 + 1; rg.nb[1] = (sc.ny() + 3) / 4 + 1; rg.nb[2] = (sc.nz() + 7) / 8 + 1;
  rg.page.assign(size_t(rg.nb[0]) * rg.nb[1] * rg.nb[2], 0);
  for (int64_t s = 0; s < rg.n_samples; s++) {
    R pos[3]; int base[3]; R rel[3];
    sample_world(rg, s, pos);
    base_and_rel(sc, pos, base, rel);
    const int bx = base[0] >> 2, by = base[1] >> 2, bz = base[2] >> 3;
    for (int i = 0; i < 2; i++) for (int j = 0; j < 2; j++) for (int k = 0; k < 2; k++) {
      const int x = bx + i, y = by + j, z = bz + k;
      if (x < rg.nb[0] && y < rg.nb[1] && z < rg.nb[2]) rg.page[(size_t(x) * rg.nb[1] + y) * rg.nb[2] + z] = 1;
    }
  }
}

// rasterize_rigid_boundary (src/rigid_transfer.cpp:18-77), 3-D branch.
template <class R> void cdf_rasterize(const Scene<R> &sc, Rigid<R> &rg) {
  rg.node_state.assign(sc.n_nodes(), 0u);
  rg.node_dist.assign(sc.n_nodes(), R(0));
  for (int64_t s = 0; s < rg.n_samples; s++) {
    const int id = rg.sample_rigid[s];
    R pos[3]; int base[3]; R rel[3];
    sample_world(rg, s, pos);
    base_and_rel(sc, pos, base, rel);                 // get_grid_base_pos_with<3> (29-30)
    R v0[3], v1[3], v2[3];                            // get_world_space_element (32)
    rigid_to_world(rg, id, rg.tri + 9 * s, v0);
    rigid_to_world(rg, id, rg.tri + 9 * s + 3, v1);
    rigid_to_world(rg, id, rg.tri + 9 * s + 6, v2);
    R M[9], Minv[9], e1[3], e2[3], n[3];              // world_to_element (33)
    for (int k = 0; k < 3; k++) { e1[k] = v1[k] - v0[k]; e2[k] = v2[k] - v0[k]; }
    cross3(e1, e2, n);
    const R nl = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    for (int k = 0; k < 3; k++) { n[k] /= nl; at(M, k, 0) = e1[k]; at(M, k, 1) = e2[k]; at(M, k, 2) = n[k]; }
    mat_inverse(M, Minv);
    for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) for (int c = 0; c < 3; c++) {
      const int i[3] = {base[0] + a, base[1] + b, base[2] + c};
      if (i[0] < 0 || i[1] < 0 || i[2] < 0 || i[0] >= sc.nx() || i[1] >= sc.ny() || i[2] >= sc.nz()) continue;
      R d[3] = {R(i[0]) * sc.dx - v0[0], R(i[1]) * sc.dx - v0[1], R(i[2]) * sc.dx - v0[2]};
      R coord[3];
      for (int r = 0; r < 3; r++) coord[r] = at(Minv, r, 0) * d[0] + at(Minv, r, 1) * d[1] + at(Minv, r, 2) * d[2];
      const bool negative = coord[2] < 0;
      R dist = std::abs(coord[2]);
      if (!(R(0) <= coord[0] && R(0) <= coord[1] && coord[0] + coord[1] <= R(1))) continue;   // 50-53
      dist *= sc.inv_dx;                                                                           // 60
      const size_t node = sc.node(i[0], i[1], i[2]);
      uint32_t &st = rg.node_state[node];
      if ((st >> kTagBits) == 0u || dist < rg.node_dist[node]) {                                  // 65-69
        rg.node_dist[node] = dist;
        st = (st & kTagMask) | (uint32_t(id + 1) << kTagBits);
      }
      st |= uint32_t(2 + int(negative)) << (id * 2);                                              // 73-74
    }
  }
  for (auto &d : rg.node_dist) d *= sc.dx;                                                        // 77-78
}

template <class R> R det4(const R *m) {  // m[c*4+r]
  auto a = [&](int r, int c) { return m[c * 4 + r]; };
  R det = 0;
  for (int c = 0; c < 4; c++) {
    int cc[3], k = 0;
    for (int j = 0; j < 4; j++) if (j != c) cc[k++] = j;
    R minor = a(1, cc[0]) * (a(2, cc[1]) * a(3, cc[2]) - a(2, cc[2]) * a(3, cc[1])) - a(1, cc[1]) * (a(2, cc[0]) * a(3, cc[2]) - a(2, cc[2]) * a(3, cc[0])) +
              a(1, cc[2]) * (a(2, cc[0]) * a(3, cc[1]) - a(2, cc[1]) * a(3, cc[0]));
    det += ((c & 1) ? R(-1) : R(1)) * a(0, c) * minor;
  }
  return det;
}
// solves m x = y for symmetric-positive 4x4 m by Gaussian elimination with partial pivoting (inversed(XtX) * XtY, 252)
template <class R> void solve4(const R *m, const R *y, R *x) {
  R a[4][5];
  for (int r = 0; r < 4; r++) { for (int c = 0; c < 4; c++) a[r][c] = m[c * 4 + r]; a[r][4] = y[r]; }
  for (int c = 0; c < 4; c++) {
    int p = c;
    for (int r = c + 1; r < 4; r++) if (std::abs(a[r][c]) > std::abs(a[p][c])) p = r;
    for (int k = 0; k < 5; k++) std::swap(a[c][k], a[p][k]);
    for (int r = c + 1; r < 4; r++) { const R f = a[r][c] / a[c][c]; for (int k = c; k < 5; k++) a[r][k] -= f * a[c][k]; }
  }
  for (int r = 3; r >= 0; r--) { R sum = a[r][4]; for (int c = r + 1; c < 4; c++) sum -= a[r][c] * x[c]; x[r] = sum / a[r][r]; }
}

// gather_cdf (src/rigid_transfer.cpp:120-274), 3-D, mpm_use_weighted_reconstruction = cdf_use_negative = true.
template <class R> void gather_cdf(const Scene<R> &sc, Rigid<R> &rg, const Particles<R> &P, const uint8_t *alive) {
  for (int64_t p = 0; p < P.n; p++) {
    if (alive && !alive[p]) continue;
    rg.bdist[p] = 0; rg.bnormal[3 * p] = rg.bnormal[3 * p + 1] = rg.bnormal[3 * p + 2] = 0; rg.near[p] = 0;   // 138-140
    R pos[3] = {P.x[3 * p] * sc.inv_dx, P.x[3 * p + 1] * sc.inv_dx, P.x[3 * p + 2] * sc.inv_dx};
    if (!rigid_page_of_block(rg, int(pos[0]) >> 2, int(pos[1]) >> 2, int(pos[2]) >> 3)) continue;           // 142-146: the CELL's page
    uint32_t &pst = rg.states[p];
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * p, base, rel);
    R w[3][3], dw[3][3];
    for (int d = 0; d < 3; d++) quadratic_kernel_axis(pos[d], w[d], dw[d]);
    uint32_t all_boundaries = 0;
    for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) for (int c = 0; c < 3; c++)
      all_boundaries |= rg.node_state[sc.node(base[0] + a, base[1] + b, base[2] + c)] & kTagMask & kStateMask;   // 155-159
    pst &= (all_boundaries + (all_boundaries >> 1));                                                           // 162
    uint32_t to_add = all_boundaries & ~pst;                                                                   // 164
    while (to_add) {
      const uint32_t bit = to_add & (0u - to_add);
      to_add ^= bit;
      R wd[2] = {0, 0};
      for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) for (int c = 0; c < 3; c++) {
        const size_t node = sc.node(base[0] + a, base[1] + b, base[2] + c);
        const uint32_t gs = rg.node_state[node];
        if ((gs >> kTagBits) == 0u) continue;                                                                  // 182-184
        const R d = rg.node_dist[node] * sc.inv_dx;
        const R weight = (w[0][a] * w[1][b]) * w[2][c];
        if ((gs & kTagMask) & bit) wd[((gs & kTagMask) & (bit >> 1)) != 0 ? 1 : 0] += d * weight;              // 195-198
      }
      if (wd[0] + wd[1] > R(1e-7)) pst |= bit | ((bit >> 1) * uint32_t(wd[0] < wd[1]));                        // 200-205
    }
    if (pst == 0) continue;
    R XtX[16] = {0}, XtY[4] = {0};
    for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) for (int c = 0; c < 3; c++) {
      const size_t node = sc.node(base[0] + a, base[1] + b, base[2] + c);
      const uint32_t word = rg.node_state[node];
      if ((word >> kTagBits) == 0u) continue;                                                                  // 217-219
      const uint32_t gs = word & kTagMask;
      const R dpos[3] = {pos[0] - R(base[0] + a), pos[1] - R(base[1] + b), pos[2] - R(base[2] + c)};
      const uint32_t mask = (gs & pst & kStateMask) >> 1;
      const R d = rg.node_dist[node] * sc.inv_dx;
      const R xp[4] = {-dpos[0], -dpos[1], -dpos[2], R(1)};
      const R weight = (w[0][a] * w[1][b]) * w[2][c];
      if (gs == 0) continue;
      R sgn;
      if ((gs & mask) == (pst & mask)) sgn = R(1);                                                             // 232-236: same colour
      else {
        const uint32_t diff = (gs & mask) ^ (pst & mask);                                                      // 239-243: exactly one colour differs
        if (diff > 0 && (diff & (diff - 1)) == 0) sgn = R(-1); else continue;
      }
      for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) XtX[j * 4 + i] += xp[i] * xp[j] * weight;
      const R y[4] = {-d * dpos[0], -d * dpos[1], -d * dpos[2], d};
      for (int i = 0; i < 4; i++) XtY[i] += sgn * y[i] * weight;
    }
    if (std::abs(det4(XtX)) > R(1e-4)) {                                                                       // 251: mpm_reconstruction_guard<3>
      R r[4];
      solve4(XtX, XtY, r);
      rg.near[p] = 1;
      rg.bdist[p] = r[3] * sc.dx;
      const R l2 = r[0] * r[0] + r[1] * r[1] + r[2] * r[2];
      if (l2 > R(1e-4)) { const R il = R(1) / std::sqrt(l2); for (int k = 0; k < 3; k++) rg.bnormal[3 * p + k] = r[k] * il; }
    }
  }
}

template <class R> inline bool particle_in_rigid_page(const Scene<R> &sc, const Rigid<R> &rg, const R *x) {
  int base[3]; R rel[3];
  base_and_rel(sc, x, base, rel);   // block_op_switch tests the page of the block the particle is SORTED into: its base node's
  return rigid_page_of_block(rg, base[0] >> 2, base[1] >> 2, base[2] >> 3);
}

// colour test of block_op_rigid (src/transfer.cpp:416-420, 757-761): true = compatible
inline bool cdf_compatible(uint32_t node_word, uint32_t pst) {
  const uint32_t gs = node_word & kTagMask;
  const uint32_t mask = (gs & pst & kStateMask) >> 1;
  return (gs & mask) == (pst & mask);
}

// the 27 dw_w of MPMFastKernel32 (src/kernel.h:168-189): lanes (dw_x w_y w_z, w_x dw_y w_z, w_x w_y dw_z, w_x w_y w_z),
// dw in world units (shuffle() multiplies by inv_delta_x)
template <class R> inline void dw_w27(const Scene<R> &sc, const R *pos_grid, R (*out)[4]) {
  R w[3][3], dw[3][3];
  for (int d = 0; d < 3; d++) { quadratic_kernel_axis(pos_grid[d], w[d], dw[d]); for (int k = 0; k < 3; k++) dw[d][k] *= sc.inv_dx; }
  for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) for (int c = 0; c < 3; c++) {
    R *o = out[a * 9 + b * 3 + c];
    o[0] = (dw[0][a] * w[1][b]) * w[2][c];
    o[1] = (w[0][a] * dw[1][b]) * w[2][c];
    o[2] = (w[0][a] * w[1][b]) * dw[2][c];
    o[3] = (w[0][a] * w[1][b]) * w[2][c];
  }
}

// rasterize_optimized with block_op_switch (src/transfer.cpp:361-581): block_op_rigid for particles of rigid pages
// (367-463), block_op_normal (p2g above) for the others.
template <class R> void p2g_coupled(const Scene<R> &sc, Rigid<R> &rg, Particles<R> &P, const std::vector<int64_t> &order, R *grid) {
  rigid_reset_tmp(rg);
  std::vector<int64_t> normal, rigid;
  for (int64_t i : order) (particle_in_rigid_page(sc, rg, P.x + 3 * i) ? rigid : normal).push_back(i);
  p2g(sc, P, normal, grid);
  for (int64_t i : rigid) {
    R *v = P.v + 3 * i;
    if (sc.particle_gravity) for (int d = 0; d < 3; d++) v[d] = v[d] + sc.gravity[d] * sc.dt;   // 383-385
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * i, base, rel);
    const R pos[3] = {P.x[3 * i] * sc.inv_dx, P.x[3 * i + 1] * sc.inv_dx, P.x[3 * i + 2] * sc.inv_dx};
    R k27[27][4];
    dw_w27(sc, pos, k27);
    const R mass = P.mass[i];
    const int g = P.group[i];
    R binv[9], mv[3], tf[9];
    for (int k = 0; k < 9; k++) binv[k] = P.b[9 * i + k] * (R(4) * mass);                       // 401
    for (int d = 0; d < 3; d++) mv[d] = mass * v[d];
    calculate_force(sc.mat_kind[g], sc.mat_params + g * kMatParams, P.F + 9 * i, P.ps[i], P.vol[i], tf);
    for (int k = 0; k < 9; k++) tf[k] *= sc.dt;                                                 // 404
    const uint32_t pst = rg.states[i];
    for (int a = 0; a < 3; a++) for (int b = 0; b < 3; b++) for (int c = 0; c < 3; c++) {
      const int ni[3] = {base[0] + a, base[1] + b, base[2] + c};
      const R dpos[3] = {pos[0] - R(ni[0]), pos[1] - R(ni[1]), pos[2] - R(ni[2])};
      const size_t node = sc.node(ni[0], ni[1], ni[2]);
      const R *dw_w = k27[a * 9 + b * 3 + c];
      const uint32_t word = rg.node_state[node];
      if (!cdf_compatible(word, pst)) {                                                         // 420-446
        const int rid = int(word >> kTagBits) - 1;
        if (rid < 0) continue;
        const R gp[3] = {sc.dx * R(ni[0]), sc.dx * R(ni[1]), sc.dx * R(ni[2])};
        R rv[3], proj[3], imp[3];
        rigid_velocity_at(rg, rid, gp, rv);
        friction_project(v, rv, rg.bnormal + 3 * i, rg.frictions[2 * rid + ((pst >> (2 * rid)) & 1u)], proj);
        for (int r = 0; r < 3; r++)
          imp[r] = mass * dw_w[3] * (v[r] - proj[r]) + (at(tf, r, 0) * dw_w[0] + at(tf, r, 1) * dw_w[1] + at(tf, r, 2) * dw_w[2]);
        rigid_apply_tmp_impulse(rg, rid, imp, gp);
        continue;
      }
      R *gn = grid + 4 * node;                                                                  // 451-459 (MLSMPM)
      for (int r = 0; r < 3; r++) {
        const R ap = mv[r] + (at(binv, r, 0) * dpos[0] + at(binv, r, 1) * dpos[1] + at(binv, r, 2) * dpos[2]);
        const R st = -(at(tf, r, 0) * dpos[0] + at(tf, r, 1) * dpos[1] + at(tf, r, 2) * dpos[2]) * R(4) * sc.inv_dx;
        gn[r] += dw_w[3] * (ap + st);
      }
      gn[3] += dw_w[3] * mass;
    }
  }
  rigid_apply_tmp(rg);                                                                          // 578-580
}

// resample_optimized with block_op_switch (src/transfer.cpp:702-970): block_op_rigid (706-835) / block_op_normal (g2p above).
template <class R> void g2p_coupled(const Scene<R> &sc, Rigid<R> &rg, Particles<R> &P, const std::vector<int64_t> &order, const R *grid) {
  rigid_reset_tmp(rg);                                                                          // 956-958
  std::vector<int64_t> normal, rigid;
  for (int64_t i : order) (particle_in_rigid_page(sc, rg, P.x + 3 * i) ? rigid : normal).push_back(i);
  g2p(sc, P, normal, grid);
  for (int64_t i : rigid) {
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * i, base, rel);
    const R pos[3] = {P.x[3 * i] * sc.inv_dx, P.x[3 * i + 1] * sc.inv_dx, P.x[3 * i + 2] * sc.inv_dx};
    R k27[27][4];
    dw_w27(sc, pos, k27);
    const uint32_t pst = rg.states[i];
    const R *pv = P.v + 3 * i, *bn = rg.bnormal + 3 * i;
    R v[3] = {0, 0, 0}, b[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int rigid_id = -1;
    for (int a = 0; a < 3; a++) for (int bb = 0; bb < 3; bb++) for (int c = 0; c < 3; c++) {
      const int ni[3] = {base[0] + a, base[1] + bb, base[2] + c};
      const R dpos[3] = {pos[0] - R(ni[0]), pos[1] - R(ni[1]), pos[2] - R(ni[2])};
      const size_t node = sc.node(ni[0], ni[1], ni[2]);
      const R w = k27[a * 9 + bb * 3 + c][3];
      R gv[3] = {grid[4 * node], grid[4 * node + 1], grid[4 * node + 2]};
      const uint32_t word = rg.node_state[node];
      if (!cdf_compatible(word, pst)) {                                                         // 761-785
        R fake[3] = {pv[0], pv[1], pv[2]}, vg[3] = {0, 0, 0};
        R friction = 0;
        const int rid = int(word >> kTagBits) - 1;
        if (rid >= 0) {
          const R gp[3] = {R(ni[0]) * sc.dx, R(ni[1]) * sc.dx, R(ni[2]) * sc.dx};
          rigid_velocity_at(rg, rid, gp, vg);
          rigid_id = rid;
          friction = rg.frictions[2 * rid + ((pst >> (2 * rid)) & 1u)];
        }
        if (rg.near[i]) {
          friction_project(pv, vg, bn, friction, fake);
          const R push = sc.dt * sc.dx * rg.pushing_force;
          for (int r = 0; r < 3; r++) fake[r] += bn[r] * push;
        }
        for (int r = 0; r < 3; r++) gv[r] = fake[r];
      }
      for (int r = 0; r < 3; r++) {
        v[r] = std::fma(gv[r], w, v[r]);                                                        // 788
        const R wg = w * gv[r];
        for (int cc = 0; cc < 3; cc++) at(b, r, cc) = std::fma(wg, dpos[cc], at(b, r, cc));     // 793-795
      }
    }
    if (rg.near[i]) {                                                                           // 800-804
      for (int k = 0; k < 9; k++) P.b[9 * i + k] = 0;
    } else {                                                                                    // damp_affine_momemtum with zero damping (src/mpm.h:465-469)
      for (int c = 0; c < 3; c++) for (int r = 0; r < 3; r++) {
        const R sym = R(0.5) * (at(b, r, c) + at(b, c, r));
        at(P.b + 9 * i, r, c) = sym + (at(b, r, c) - sym);
      }
    }
    for (int d = 0; d < 3; d++) P.v[3 * i + d] = v[d];
    R cdg[9];
    for (int c = 0; c < 3; c++) for (int r = 0; r < 3; r++) at(cdg, r, c) = std::fma(sc.dt, at(b, r, c) * (R(-4) * sc.inv_dx), r == c ? R(1) : R(0));   // 810-815
    const int g = P.group[i];
    plasticity(sc.mat_kind[g], sc.mat_params + g * kMatParams, cdg, P.F + 9 * i, P.ps[i]);
    for (int d = 0; d < 3; d++) P.x[3 * i + d] = std::fma(v[d], sc.dt, P.x[3 * i + d]);        // 819
    if (rg.near[i] && rg.bdist[i] < R(-0.05) * sc.dx && rg.bdist[i] > -sc.dx * R(0.3)) {         // 823-832: position correction
      R dv[3], imp[3];
      for (int d = 0; d < 3; d++) { dv[d] = rg.bdist[i] * bn[d] * rg.penalty; P.v[3 * i + d] -= dv[d]; imp[d] = dv[d] * P.mass[i]; }
      if (rigid_id != -1) rigid_apply_tmp_impulse(rg, rigid_id, imp, P.x + 3 * i);
    }
  }
  rigid_apply_tmp(rg);                                                                          // 967-969
}

// MPM<3>::substep with rigid bodies (src/mpm.cpp:452-575), without the host-side rigid dynamics (rigidify, articulate,
// advect_rigid_bodies): one substep at a fixed pose; velocity / angular_velocity return with the impulses of both transfers.
template <class R>
void substep_coupled(const Scene<R> &sc, Rigid<R> &rg, Particles<R> &P, uint8_t *alive, R *grid_out, R *grid_rast_out, uint32_t *node_state_out,
                     R *node_dist_out) {
  std::vector<R> grid_local;
  R *grid = grid_out;
  if (!grid) { grid_local.assign(sc.n_nodes() * 4, R(0)); grid = grid_local.data(); }
  else std::fill(grid, grid + sc.n_nodes() * 4, R(0));
  auto order = visit_order(sc, P, alive);
  rigid_pages(sc, rg);
  cdf_rasterize(sc, rg);
  if (node_state_out) std::memcpy(node_state_out, rg.node_state.data(), sizeof(uint32_t) * sc.n_nodes());
  if (node_dist_out) std::memcpy(node_dist_out, rg.node_dist.data(), sizeof(R) * sc.n_nodes());
  gather_cdf(sc, rg, P, alive);
  p2g_coupled(sc, rg, P, order, grid);
  if (grid_rast_out) std::memcpy(grid_rast_out, grid, sizeof(R) * sc.n_nodes() * 4);
  grid_update(sc, grid);
  g2p_coupled(sc, rg, P, order, grid);
  clear_boundary(sc, P, alive);
}

// ================================================================================
// FAST fp32 path: the timed CPU baseline.  Mirrors the *structure* of the reference's
// optimized path: sort by (block,node) (src/mpm.cpp:770-918), per-block tile cache
// [6][6][10] (GridCache, src/transfer.cpp:52-156), 8-colour block passes for P2G
// (src/mpm.h:447-461), blocked grid, OpenMP over blocks.  Same arithmetic as above.
// ================================================================================
struct FastState {
  int res[3];
  int nb[3];                      // blocks per axis (4,4,8)
  std::vector<float> grid;        // [block][128][4]
  std::vector<uint64_t> keys, keys_tmp;
  std::vector<int32_t> order;
  std::vector<int32_t> block_ids; // occupied blocks
  std::vector<int32_t> block_off; // particle offsets per occupied block (+sentinel)
  std::vector<uint8_t> fat;       // dilated block flags
  std::vector<int32_t> fat_ids;
  double t_sort = 0, t_p2g = 0, t_grid = 0, t_g2p = 0;
  // Physical re-ordering of the particle storage (sort_allocator, src/mpm.cpp:753-768, called when
  // substep_counter % reorder_interval == 0, src/mpm.cpp:811-813).  0 = never (the parity tests:
  // storage index == caller index, so ties in the sort break exactly as in the scalar oracle).
  int reorder_interval = 0;
  int64_t step = 0;
  std::vector<int32_t> origin;  // storage slot -> caller index
  std::vector<float> sx, sv, sF, sb, smass, svol, sps, stmp;
  std::vector<int32_t> sgroup, itmp;
  std::vector<uint8_t> salive, atmp;
};

inline double now_s() {
#ifdef _OPENMP
  return omp_get_wtime();
#else
  return 0.0;
#endif
}

inline size_t fast_node_index(const FastState &st, int i, int j, int k) {
  int bx = i >> 2, by = j >> 2, bz = k >> 3;
  size_t b = (size_t(bx) * st.nb[1] + by) * st.nb[2] + bz;
  return b * 128 + (i & 3) * 32 + (j & 3) * 8 + (k & 7);
}

// Gather `width` floats per particle through `perm` (parallel); dst/src must not alias.
template <typename T>
inline void permute_rows(const std::vector<int32_t> &perm, int width, const T *src, T *dst) {
  const int64_t n = int64_t(perm.size());
#pragma omp parallel for schedule(static)
  for (int64_t j = 0; j < n; j++) {
    const T *s = src + size_t(perm[j]) * width;
    T *d = dst + size_t(j) * width;
    for (int c = 0; c < width; c++) d[c] = s[c];
  }
}

// sort_allocator (src/mpm.cpp:753-768): storage slot j receives the particle the sort put at rank j
// (dead particles, which the reference has already dropped, go to the tail); afterwards order = iota.
inline void fast_reorder_storage(FastState &st, std::vector<uint8_t> &alive) {
  const int64_t n = int64_t(alive.size()), na = int64_t(st.order.size());
  std::vector<int32_t> perm(n);
  std::copy(st.order.begin(), st.order.end(), perm.begin());
  int64_t k = na;
  for (int64_t i = 0; i < n; i++)
    if (!alive[i]) perm[k++] = int32_t(i);
  st.stmp.resize(size_t(n) * 9);
  auto rows = [&](std::vector<float> &a, int w) {
    permute_rows(perm, w, a.data(), st.stmp.data());
    std::memcpy(a.data(), st.stmp.data(), size_t(n) * w * sizeof(float));
  };
  rows(st.sx, 3); rows(st.sv, 3); rows(st.sF, 9); rows(st.sb, 9); rows(st.smass, 1); rows(st.svol, 1); rows(st.sps, 1);
  st.itmp.resize(n);
  permute_rows(perm, 1, st.sgroup.data(), st.itmp.data());
  std::memcpy(st.sgroup.data(), st.itmp.data(), size_t(n) * sizeof(int32_t));  // in place: Particles views stay valid
  permute_rows(perm, 1, st.origin.data(), st.itmp.data()); st.origin.swap(st.itmp);
  st.atmp.resize(n);
  permute_rows(perm, 1, alive.data(), st.atmp.data()); alive.swap(st.atmp);
#pragma omp parallel for schedule(static)
  for (int64_t j = 0; j < na; j++) st.order[j] = int32_t(j);
}

void fast_substep(FastState &st, const Scene<float> &sc, Particles<float> &P, std::vector<uint8_t> &alive, bool reorder_now = false) {
  using R = float;
  const int64_t n = P.n;
  double t0 = now_s();
  // ---- sort_particles_and_populate_grid (src/mpm.cpp:770-918)
  st.keys.resize(n);
  int64_t n_alive = 0;
#pragma omp parallel for schedule(static) reduction(+ : n_alive)
  for (int64_t i = 0; i < n; i++) {
    if (!alive[i]) { st.keys[i] = ~0ull; continue; }
    int base[3]; R rel[3];
    base_and_rel(sc, P.x + 3 * i, base, rel);
    uint64_t b = (uint64_t(base[0] >> 2) * st.nb[1] + (base[1] >> 2)) * st.nb[2] + (base[2] >> 3);
    uint64_t in = (base[0] & 3) * 32 + (base[1] & 3) * 8 + (base[2] & 7);
    st.keys[i] = (((b << 7) | in) << 26) | uint64_t(i);
    n_alive++;
  }
  // parallel sort (stand-in for tbb::parallel_sort, src/mpm.cpp:793-795): the keys carry the particle
  // index in their low 26 bits and arrive in index order, so a STABLE LSD radix sort over the
  // (block,node) bits alone yields the same order as sorting the full 64-bit keys.
  {
    int nt = 1;
#ifdef _OPENMP
    nt = omp_get_max_threads();
#endif
    const int RB = 11, NB = 1 << RB;
    int top = 26 + 7;  // highest significant bit: block index range
    {
      uint64_t nblk = uint64_t(st.nb[0]) * st.nb[1] * st.nb[2];
      while ((1ull << (top - 26 - 7)) < nblk) top++;
      top += 1;  // dead keys (~0) must still sort last: handled by the clamp below
    }
    st.keys_tmp.resize(n);
    std::vector<uint32_t> hist(size_t(nt) * NB);
    uint64_t *src = st.keys.data(), *dst = st.keys_tmp.data();
    auto digit = [&](uint64_t k, int shift, bool last) -> uint32_t {
      if (k == ~0ull) return last ? NB - 1 : (NB - 1);  // dead: always the last bucket
      return uint32_t(k >> shift) & (NB - 1);
    };
    for (int shift = 26; shift < top; shift += RB) {
      const bool last = shift + RB >= top;
      std::fill(hist.begin(), hist.end(), 0u);
#pragma omp parallel for schedule(static, 1)
      for (int t = 0; t < nt; t++) {
        uint32_t *h = &hist[size_t(t) * NB];
        for (size_t i = size_t(n) * t / nt, e = size_t(n) * (t + 1) / nt; i < e; i++) h[digit(src[i], shift, last)]++;
      }
      uint32_t run = 0;
      for (int d = 0; d < NB; d++)
        for (int t = 0; t < nt; t++) { uint32_t c = hist[size_t(t) * NB + d]; hist[size_t(t) * NB + d] = run; run += c; }
#pragma omp parallel for schedule(static, 1)
      for (int t = 0; t < nt; t++) {
        uint32_t *h = &hist[size_t(t) * NB];
        for (size_t i = size_t(n) * t / nt, e = size_t(n) * (t + 1) / nt; i < e; i++) dst[h[digit(src[i], shift, last)]++] = src[i];
      }
      std::swap(src, dst);
    }
    if (src != st.keys.data()) st.keys.swap(st.keys_tmp);
  }
  st.order.resize(n_alive);
  st.block_ids.clear();
  st.block_off.clear();
  {
    uint64_t last = ~0ull;
    for (int64_t i = 0; i < n_alive; i++) {
      st.order[i] = int32_t(st.keys[i] & ((1ull << 26) - 1));
      uint64_t b = st.keys[i] >> (26 + 7);
      if (b != last) { st.block_ids.push_back(int32_t(b)); st.block_off.push_back(int32_t(i)); last = b; }
    }
    st.block_off.push_back(int32_t(n_alive));
  }
  if (reorder_now) fast_reorder_storage(st, alive);
  // fat page map = 3x3x3 dilation, then memset (src/mpm.cpp:831-874)
  const size_t nblocks = size_t(st.nb[0]) * st.nb[1] * st.nb[2];
  if (st.fat.size() != nblocks) st.fat.assign(nblocks, 0);
  for (int32_t id : st.fat_ids) st.fat[id] = 0;
  st.fat_ids.clear();
  for (int32_t b : st.block_ids) {
    int bz = b % st.nb[2], by = (b / st.nb[2]) % st.nb[1], bx = b / (st.nb[2] * st.nb[1]);
    for (int dx = -1; dx <= 1; dx++)
      for (int dy = -1; dy <= 1; dy++)
        for (int dz = -1; dz <= 1; dz++) {
          int x = bx + dx, y = by + dy, z = bz + dz;
          if (x < 0 || y < 0 || z < 0 || x >= st.nb[0] || y >= st.nb[1] || z >= st.nb[2]) continue;
          size_t id = (size_t(x) * st.nb[1] + y) * st.nb[2] + z;
          if (!st.fat[id]) { st.fat[id] = 1; st.fat_ids.push_back(int32_t(id)); }
        }
  }
  if (st.grid.size() != nblocks * 512) st.grid.assign(nblocks * 512, 0.f);
#pragma omp parallel for schedule(static)
  for (size_t f = 0; f < st.fat_ids.size(); f++) std::memset(&st.grid[size_t(st.fat_ids[f]) * 512], 0, 512 * sizeof(float));
  double t1 = now_s();

  // ---- P2G, 8 colours (src/mpm.h:447-461), tile cache [6][6][10] (src/transfer.cpp:59-63)
  const R S = R(-4) * sc.inv_dx * sc.dt;
  const int nocc = (int)st.block_ids.size();
  auto tile_io = [&](int b, float (*tile)[4], bool store) {
    int bz = b % st.nb[2], by = (b / st.nb[2]) % st.nb[1], bx = b / (st.nb[2] * st.nb[1]);
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 6; j++)
        for (int k = 0; k < 10; k++) {
          int gi = bx * 4 + i, gj = by * 4 + j, gk = bz * 8 + k;
          if (gi >= st.nb[0] * 4 || gj >= st.nb[1] * 4 || gk >= st.nb[2] * 8) continue;
          float *g = &st.grid[fast_node_index(st, gi, gj, gk) * 4];
          float *t = tile[(i * 6 + j) * 10 + k];
          if (store) std::memcpy(g, t, 16); else std::memcpy(t, g, 16);
        }
  };
  for (int colour = 0; colour < 8; colour++) {
#pragma omp parallel for schedule(dynamic, 4)
    for (int ob = 0; ob < nocc; ob++) {
      int b = st.block_ids[ob];
      int bz = b % st.nb[2], by = (b / st.nb[2]) % st.nb[1], bx = b / (st.nb[2] * st.nb[1]);
      if ((((bx & 1) << 2) | ((by & 1) << 1) | (bz & 1)) != colour) continue;
      alignas(64) float tile[360][4];
      std::memset(tile, 0, sizeof(tile));
      tile_io(b, tile, false);
      g_use_fast_svd = true;
      for (int32_t pi = st.block_off[ob]; pi < st.block_off[ob + 1]; pi++) {
        int64_t i = st.order[pi];
        R *v = P.v + 3 * i;
        if (sc.particle_gravity)
          for (int d = 0; d < 3; d++) v[d] = v[d] + sc.gravity[d] * sc.dt;
        int base[3]; R rel[3];
        base_and_rel(sc, P.x + 3 * i, base, rel);
        R w27[27];
        mls_fast_kernel(rel, w27);
        const R mass = P.mass[i];
        const int g = P.group[i];
        R stress[9];
        calculate_force(sc.mat_kind[g], sc.mat_params + g * kMatParams, P.F + 9 * i, P.ps[i], P.vol[i], stress);
        R affine[9];
        const R bm = R(4) * mass;
        for (int k = 0; k < 9; k++) affine[k] = std::fma(stress[k], S, P.b[9 * i + k] * bm);
        R mv[3] = {mass * v[0], mass * v[1], mass * v[2]};
        int li = base[0] - bx * 4, lj = base[1] - by * 4, lk = base[2] - bz * 8;
        // 4-wide SSE/FMA, one __m128 = (x,y,z,mass) per node, as the reference's LOOP macro
        // (src/transfer.cpp:526-547): affine_prod = fmadd(A2,d2, fmadd(A1,d1, fmadd(A0,d0, mass_v)));
        // contrib = blend(mass, affine_prod); g += weight * contrib.  Same rounding as the scalar form.
        const __m128 A0 = _mm_set_ps(0.f, at(affine, 2, 0), at(affine, 1, 0), at(affine, 0, 0));
        const __m128 A1 = _mm_set_ps(0.f, at(affine, 2, 1), at(affine, 1, 1), at(affine, 0, 1));
        const __m128 A2 = _mm_set_ps(0.f, at(affine, 2, 2), at(affine, 1, 2), at(affine, 0, 2));
        const __m128 MV = _mm_set_ps(mass, mv[2], mv[1], mv[0]);
        for (int a = 0; a < 3; a++)
          for (int bb = 0; bb < 3; bb++)
            for (int c = 0; c < 3; c++) {
              const __m128 d0 = _mm_set1_ps(rel[0] - R(a)), d1 = _mm_set1_ps(rel[1] - R(bb)), d2 = _mm_set1_ps(rel[2] - R(c));
              const __m128 w = _mm_set1_ps(w27[a * 9 + bb * 3 + c]);
              float *gn = tile[((li + a) * 6 + (lj + bb)) * 10 + (lk + c)];
              const __m128 contrib = _mm_fmadd_ps(A2, d2, _mm_fmadd_ps(A1, d1, _mm_fmadd_ps(A0, d0, MV)));
              _mm_store_ps(gn, _mm_add_ps(_mm_load_ps(gn), _mm_mul_ps(w, contrib)));
            }
      }
      g_use_fast_svd = false;  // the switch is per thread: later svd3<float> calls on this thread take the checker path again
      tile_io(b, tile, true);
    }
  }
  double t2 = now_s();

  // ---- normalise + boundary on fat blocks (src/mpm.cpp:277-372)
  R incr[3] = {0, 0, 0};
  if (!sc.particle_gravity)
    for (int d = 0; d < 3; d++) incr[d] = sc.gravity[d] * sc.dt;
#pragma omp parallel for schedule(static)
  for (size_t f = 0; f < st.fat_ids.size(); f++) {
    int b = st.fat_ids[f];
    int bz = b % st.nb[2], by = (b / st.nb[2]) % st.nb[1], bx = b / (st.nb[2] * st.nb[1]);
    for (int t = 0; t < 128; t++) {
      float *g = &st.grid[(size_t(b) * 128 + t) * 4];
      R mass = g[3];
      if (mass > 0) {
        R inv = R(1) / mass;
        for (int d = 0; d < 3; d++) g[d] = std::fma(g[d], inv, incr[d]);
      }
      if (sc.sdf && mass != R(0)) {
        int i = bx * 4 + (t >> 5), j = by * 4 + ((t >> 3) & 3), k = bz * 8 + (t & 7);
        if (i > sc.res[0] || j > sc.res[1] || k > sc.res[2]) continue;
        const R *s = sc.sdf + 4 * sc.node(i, j, k);
        R phi = s[3];
        if (phi < R(-3) || R(0) < phi) continue;
        R vb[3] = {0, 0, 0}, out[3];
        friction_project(g, vb, s, sc.friction, out);
        g[0] = out[0]; g[1] = out[1]; g[2] = out[2];
      }
    }
  }
  double t3 = now_s();

  // ---- G2P (uncoloured, src/transfer.cpp:966)
  const R scale = R(-4) * sc.inv_dx * sc.dt;
#pragma omp parallel for schedule(dynamic, 4)
  for (int ob = 0; ob < nocc; ob++) {
    int b = st.block_ids[ob];
    int bz = b % st.nb[2], by = (b / st.nb[2]) % st.nb[1], bx = b / (st.nb[2] * st.nb[1]);
    alignas(64) float tile[360][4];
    std::memset(tile, 0, sizeof(tile));
    tile_io(b, tile, false);
    g_use_fast_svd = true;
    for (int32_t pi = st.block_off[ob]; pi < st.block_off[ob + 1]; pi++) {
      int64_t i = st.order[pi];
      int base[3]; R rel[3];
      base_and_rel(sc, P.x + 3 * i, base, rel);
      R w27[27];
      mls_fast_kernel(rel, w27);
      int li = base[0] - bx * 4, lj = base[1] - by * 4, lk = base[2] - bz * 8;
      R vacc[3], bmat[9];
      {
        // 4-wide SSE/FMA as the reference's LOOP macro (src/transfer.cpp:884-904):
        // v_ = fmadd(grid_vel, w, v_); w_grid_vel = w * grid_vel; b_[r] = fmadd(w_grid_vel, dpos[r], b_[r])
        __m128 v4 = _mm_setzero_ps(), b0 = v4, b1 = v4, b2 = v4;
        for (int a = 0; a < 3; a++)
          for (int bb = 0; bb < 3; bb++)
            for (int c = 0; c < 3; c++) {
              const __m128 w = _mm_set1_ps(w27[a * 9 + bb * 3 + c]);
              const __m128 g = _mm_load_ps(tile[((li + a) * 6 + (lj + bb)) * 10 + (lk + c)]);
              v4 = _mm_fmadd_ps(g, w, v4);
              const __m128 wg = _mm_mul_ps(w, g);
              b0 = _mm_fmadd_ps(wg, _mm_set1_ps(rel[0] - R(a)), b0);
              b1 = _mm_fmadd_ps(wg, _mm_set1_ps(rel[1] - R(bb)), b1);
              b2 = _mm_fmadd_ps(wg, _mm_set1_ps(rel[2] - R(c)), b2);
            }
        alignas(16) float tv[4], t0[4], t1[4], t2[4];
        _mm_store_ps(tv, v4); _mm_store_ps(t0, b0); _mm_store_ps(t1, b1); _mm_store_ps(t2, b2);
        for (int r = 0; r < 3; r++) { vacc[r] = tv[r]; at(bmat, r, 0) = t0[r]; at(bmat, r, 1) = t1[r]; at(bmat, r, 2) = t2[r]; }
      }
      std::memcpy(P.b + 9 * i, bmat, sizeof(bmat));
      for (int d = 0; d < 3; d++) P.v[3 * i + d] = vacc[d];
      R cdg[9];
      for (int c = 0; c < 3; c++)
        for (int r = 0; r < 3; r++) at(cdg, r, c) = std::fma(scale, at(bmat, r, c), r == c ? R(1) : R(0));
      const int g = P.group[i];
      plasticity(sc.mat_kind[g], sc.mat_params + g * kMatParams, cdg, P.F + 9 * i, P.ps[i]);
      for (int d = 0; d < 3; d++) P.x[3 * i + d] = std::fma(vacc[d], sc.dt, P.x[3 * i + d]);
      // clear_boundary_particles (src/mpm.cpp:583-633), fused here; the reference runs
      // it as a separate pass after G2P.
      bool bad = false;
      for (int d = 0; d < 3; d++) {
        R X = P.x[3 * i + d] * sc.inv_dx;
        if (X < R(7) || X - R(sc.res[d]) > R(-7) || !std::isfinite(X) || !std::isfinite(P.v[3 * i + d])) bad = true;
      }
      if (bad) alive[i] = 0;
    }
    g_use_fast_svd = false;
  }
  double t4 = now_s();
  st.t_sort += t1 - t0; st.t_p2g += t2 - t1; st.t_grid += t3 - t2; st.t_g2p += t4 - t3;
}

// ================================================================================
// 2D: the 88-line reference `advance(dt)` (mls-mpm88.cpp:16-69), config 1.
// Row-major 2x2 here: F = {F00,F01,F10,F11}.  polar/svd 2x2 in closed form.
// ================================================================================
template <class R> void polar2(const R *F, R *Rm, R *S) {
  R x = F[0] + F[3], y = F[2] - F[1];
  R sc = R(1) / std::sqrt(x * x + y * y);
  R c = x * sc, s = y * sc;
  Rm[0] = c; Rm[1] = -s; Rm[2] = s; Rm[3] = c;
  // S = R^T F
  S[0] = c * F[0] + s * F[2]; S[1] = c * F[1] + s * F[3];
  S[2] = -s * F[0] + c * F[2]; S[3] = -s * F[1] + c * F[3];
}
template <class R> void svd2(const R *F, R *U, R *sig, R *V) {
  // F = R S (polar), S = V diag(sig) V^T (Jacobi angle), U = R V.  Row-major 2x2.
  R Rm[4], S[4];
  polar2(F, Rm, S);
  R a = S[0], b = R(0.5) * (S[1] + S[2]), d = S[3];
  R th = R(0.5) * std::atan2(R(2) * b, a - d);
  R c = std::cos(th), s = std::sin(th);
  V[0] = c; V[1] = -s; V[2] = s; V[3] = c;
  sig[0] = c * c * a + R(2) * c * s * b + s * s * d;
  sig[1] = s * s * a - R(2) * c * s * b + c * c * d;
  U[0] = Rm[0] * V[0] + Rm[1] * V[2]; U[1] = Rm[0] * V[1] + Rm[1] * V[3];
  U[2] = Rm[2] * V[0] + Rm[3] * V[2]; U[3] = Rm[2] * V[1] + Rm[3] * V[3];
}

template <class R>
void mpm88_advance(int n, R dt, R E, R nu, R hardening, R gravity_y, int plastic, int64_t np, R *x, R *v, R *F, R *C, R *Jp,
                   R *grid /* [(n+1)^2][3] */) {
  const R dx = R(1) / n, inv_dx = R(n);
  const R particle_mass = 1, vol = 1;
  const R mu_0 = E / (2 * (1 + nu)), lambda_0 = E * nu / ((1 + nu) * (1 - 2 * nu));
  const int nn = n + 1;
  std::fill(grid, grid + size_t(nn) * nn * 3, R(0));  // mls-mpm88.cpp:17
  for (int64_t p = 0; p < np; p++) {                  // P2G, mls-mpm88.cpp:18-36
    R *px = x + 2 * p, *pv = v + 2 * p, *pF = F + 4 * p, *pC = C + 4 * p;
    int bx = int(px[0] * inv_dx - R(0.5)), by = int(px[1] * inv_dx - R(0.5));
    R fx[2] = {px[0] * inv_dx - bx, px[1] * inv_dx - by};
    R w[3][2];
    for (int d = 0; d < 2; d++) {
      w[0][d] = R(0.5) * (R(1.5) - fx[d]) * (R(1.5) - fx[d]);
      w[1][d] = R(0.75) - (fx[d] - R(1)) * (fx[d] - R(1));
      w[2][d] = R(0.5) * (fx[d] - R(0.5)) * (fx[d] - R(0.5));
    }
    R e = std::exp(hardening * (R(1) - Jp[p])), mu = mu_0 * e, lambda = lambda_0 * e;
    R J = pF[0] * pF[3] - pF[1] * pF[2];
    R r[4], s[4];
    polar2(pF, r, s);
    R D[4] = {pF[0] - r[0], pF[1] - r[1], pF[2] - r[2], pF[3] - r[3]};
    // (F-R) F^T
    R DFt[4] = {D[0] * pF[0] + D[1] * pF[1], D[0] * pF[2] + D[1] * pF[3], D[2] * pF[0] + D[3] * pF[1], D[2] * pF[2] + D[3] * pF[3]};
    R k = -4 * inv_dx * inv_dx * dt * vol;
    R stress[4] = {k * (2 * mu * DFt[0] + lambda * (J - 1) * J), k * (2 * mu * DFt[1]), k * (2 * mu * DFt[2]),
                   k * (2 * mu * DFt[3] + lambda * (J - 1) * J)};
    R affine[4];
    for (int q = 0; q < 4; q++) affine[q] = stress[q] + particle_mass * pC[q];
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) {
        R dpos[2] = {(R(i) - fx[0]) * dx, (R(j) - fx[1]) * dx};
        R wt = w[i][0] * w[j][1];
        R *g = grid + (size_t(bx + i) * nn + (by + j)) * 3;
        g[0] += wt * (pv[0] * particle_mass + affine[0] * dpos[0] + affine[1] * dpos[1]);
        g[1] += wt * (pv[1] * particle_mass + affine[2] * dpos[0] + affine[3] * dpos[1]);
        g[2] += wt * particle_mass;
      }
  }
  for (int i = 0; i <= n; i++)  // grid, mls-mpm88.cpp:37-46
    for (int j = 0; j <= n; j++) {
      R *g = grid + (size_t(i) * nn + j) * 3;
      if (g[2] > 0) {
        g[0] /= g[2]; g[1] /= g[2]; g[2] = 1;
        g[1] += dt * gravity_y;
        R boundary = R(0.05), xx = R(i) / n, yy = R(j) / n;
        if (xx < boundary || xx > 1 - boundary || yy > 1 - boundary) { g[0] = g[1] = g[2] = 0; }
        if (yy < boundary) g[1] = std::max(R(0), g[1]);
      }
    }
  for (int64_t p = 0; p < np; p++) {  // G2P, mls-mpm88.cpp:47-68
    R *px = x + 2 * p, *pv = v + 2 * p, *pF = F + 4 * p, *pC = C + 4 * p;
    int bx = int(px[0] * inv_dx - R(0.5)), by = int(px[1] * inv_dx - R(0.5));
    R fx[2] = {px[0] * inv_dx - bx, px[1] * inv_dx - by};
    R w[3][2];
    for (int d = 0; d < 2; d++) {
      w[0][d] = R(0.5) * (R(1.5) - fx[d]) * (R(1.5) - fx[d]);
      w[1][d] = R(0.75) - (fx[d] - R(1)) * (fx[d] - R(1));
      w[2][d] = R(0.5) * (fx[d] - R(0.5)) * (fx[d] - R(0.5));
    }
    pC[0] = pC[1] = pC[2] = pC[3] = 0;
    pv[0] = pv[1] = 0;
    for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++) {
        R dpos[2] = {R(i) - fx[0], R(j) - fx[1]};
        const R *g = grid + (size_t(bx + i) * nn + (by + j)) * 3;
        R wt = w[i][0] * w[j][1];
        pv[0] += wt * g[0]; pv[1] += wt * g[1];
        pC[0] += 4 * inv_dx * wt * g[0] * dpos[0]; pC[1] += 4 * inv_dx * wt * g[0] * dpos[1];
        pC[2] += 4 * inv_dx * wt * g[1] * dpos[0]; pC[3] += 4 * inv_dx * wt * g[1] * dpos[1];
      }
    px[0] += dt * pv[0]; px[1] += dt * pv[1];
    R A[4] = {1 + dt * pC[0], dt * pC[1], dt * pC[2], 1 + dt * pC[3]};
    R Fn[4] = {A[0] * pF[0] + A[1] * pF[2], A[0] * pF[1] + A[1] * pF[3], A[2] * pF[0] + A[3] * pF[2], A[2] * pF[1] + A[3] * pF[3]};
    R U[4], sig[2], V[4];
    svd2(Fn, U, sig, V);
    if (plastic)
      for (int q = 0; q < 2; q++) sig[q] = std::min(std::max(sig[q], R(1) - R(2.5e-2)), R(1) + R(7.5e-3));
    R oldJ = Fn[0] * Fn[3] - Fn[1] * Fn[2];
    // F = U sig V^T
    R US[4] = {U[0] * sig[0], U[1] * sig[1], U[2] * sig[0], U[3] * sig[1]};
    R Fo[4] = {US[0] * V[0] + US[1] * V[1], US[0] * V[2] + US[1] * V[3], US[2] * V[0] + US[3] * V[1], US[2] * V[2] + US[3] * V[3]};  // (U sig) V^T
    R newJ = Fo[0] * Fo[3] - Fo[1] * Fo[2];
    R Jp_new = std::min(std::max(Jp[p] * oldJ / newJ, R(0.6)), R(20));
    Jp[p] = Jp_new;
    for (int q = 0; q < 4; q++) pF[q] = Fo[q];
  }
}

template <class R> Scene<R> make_scene(const int *res, R dx, R dt, const R *gravity, int particle_gravity, const int32_t *mat_kind,
                                       const R *mat_params, const R *sdf, R friction) {
  Scene<R> sc;
  for (int d = 0; d < 3; d++) { sc.res[d] = res[d]; sc.gravity[d] = gravity[d]; }
  sc.dx = dx; sc.inv_dx = R(1) / dx; sc.dt = dt;
  sc.particle_gravity = particle_gravity;
  sc.mat_kind = mat_kind; sc.mat_params = mat_params; sc.sdf = sdf; sc.friction = friction;
  return sc;
}

}  // namespace

// =================================================================================
// C entry points (ctypes).  _f32 / _f64 suffixes select the precision.
// =================================================================================
#define ORACLE_API extern "C" __attribute__((visibility("default")))

#define DEFINE_FOR(R, SUF)                                                                                                     \
  ORACLE_API void oracle_quadratic_kernel_##SUF(R x, R *w, R *dw) { quadratic_kernel_axis<R>(x, w, dw); }                      \
  ORACLE_API void oracle_cubic_kernel_##SUF(R x, R *w, R *dw) { cubic_kernel_axis<R>(x, w, dw); }                              \
  ORACLE_API void oracle_mls_fast_kernel_##SUF(const R *rel, R *w27) { mls_fast_kernel<R>(rel, w27); }                         \
  ORACLE_API void oracle_svd3_##SUF(const R *A, R *U, R *s, R *V) { svd3<R>(A, U, s, V); }                                     \
  ORACLE_API void oracle_polar3_##SUF(const R *A, R *Rm, R *S) { polar3<R>(A, Rm, S); }                                        \
  ORACLE_API void oracle_calculate_force_##SUF(int kind, const R *prm, const R *F, R ps, R vol, R *out) {                      \
    calculate_force<R>(kind, prm, F, ps, vol, out);                                                                            \
  }                                                                                                                            \
  ORACLE_API void oracle_plasticity_##SUF(int kind, const R *prm, const R *cdg, R *F, R *ps) {                                 \
    plasticity<R>(kind, prm, cdg, F, *ps);                                                                                     \
  }                                                                                                                            \
  ORACLE_API void oracle_friction_project_##SUF(const R *vel, const R *base, const R *n, R friction, R *out) {                 \
    friction_project<R>(vel, base, n, friction, out);                                                                          \
  }                                                                                                                            \
  /* One full substep on a dense grid.  alive: [n] u8 in/out.  grid_rast (after P2G) and grid_vel (after update) may be */     \
  /* null; each is [(res+1)^3][4].  */                                                                                         \
  ORACLE_API void oracle_substep_##SUF(const int *res, R dx, R dt, const R *gravity, int particle_gravity, int n_groups,       \
                                       const int32_t *mat_kind, const R *mat_params, const R *sdf, R friction, int64_t n,      \
                                       R *x, R *v, R *F, R *b, const R *mass, const R *vol, R *ps, const int32_t *group,       \
                                       uint8_t *alive, R *grid_rast, R *grid_vel) {                                            \
    (void)n_groups;                                                                                                            \
    Scene<R> sc = make_scene<R>(res, dx, dt, gravity, particle_gravity, mat_kind, mat_params, sdf, friction);                  \
    Particles<R> P{n, x, v, F, b, mass, vol, ps, group};                                                                       \
    substep<R>(sc, P, alive, grid_vel, grid_rast);                                                                             \
  }                                                                                                                            \
  /* The same with rigid bodies (CPIC).  Per-body arrays have n_rigid rows (row 0 = background).  */                           \
  ORACLE_API void oracle_substep_coupled_##SUF(const int *res, R dx, R dt, const R *gravity, int particle_gravity, int n_groups, \
                                       const int32_t *mat_kind, const R *mat_params, const R *sdf, R friction, int64_t n,      \
                                       R *x, R *v, R *F, R *b, const R *mass, const R *vol, R *ps, const int32_t *group,       \
                                       uint8_t *alive, R *grid_rast, R *grid_vel, int n_rigid, const R *r_position,            \
                                       const R *r_rot, R *r_velocity, R *r_angular_velocity, const R *r_inv_mass,              \
                                       const R *r_inv_inertia, const R *r_frictions, int64_t n_samples, const R *s_offset,     \
                                       const R *s_tri, const int32_t *s_rigid, R penalty, R pushing_force, uint32_t *states,   \
                                       R *bnormal, R *bdist, uint8_t *near, uint32_t *node_state, R *node_dist) {              \
    (void)n_groups;                                                                                                            \
    Scene<R> sc = make_scene<R>(res, dx, dt, gravity, particle_gravity, mat_kind, mat_params, sdf, friction);                  \
    Particles<R> P{n, x, v, F, b, mass, vol, ps, group};                                                                       \
    Rigid<R> rg;                                                                                                               \
    rg.n_rigid = n_rigid; rg.position = r_position; rg.rot = r_rot; rg.velocity = r_velocity;                                  \
    rg.angular_velocity = r_angular_velocity; rg.inv_mass = r_inv_mass; rg.inv_inertia = r_inv_inertia;                        \
    rg.frictions = r_frictions; rg.n_samples = n_samples; rg.offset = s_offset; rg.tri = s_tri; rg.sample_rigid = s_rigid;     \
    rg.penalty = penalty; rg.pushing_force = pushing_force; rg.states = states; rg.bnormal = bnormal; rg.bdist = bdist;        \
    rg.near = near;                                                                                                            \
    substep_coupled<R>(sc, rg, P, alive, grid_vel, grid_rast, node_state, node_dist);                                          \
  }                                                                                                                            \
  ORACLE_API void oracle_mpm88_advance_##SUF(int n, R dt, R E, R nu, R hardening, R gravity_y, int plastic, int64_t np, R *x,  \
                                             R *v, R *F, R *C, R *Jp, R *grid) {                                               \
    mpm88_advance<R>(n, dt, E, nu, hardening, gravity_y, plastic, np, x, v, F, C, Jp, grid);                                   \
  }

DEFINE_FOR(float, f32)
DEFINE_FOR(double, f64)

// ---- fast fp32 OpenMP path (CPU baseline).  Opaque handle keeps sort/grid buffers.
ORACLE_API void *oracle_fast_create(const int *res) {
  FastState *st = new FastState();
  for (int d = 0; d < 3; d++) st->res[d] = res[d];
  st->nb[0] = (res[0] + 1 + 3) / 4 + 1;
  st->nb[1] = (res[1] + 1 + 3) / 4 + 1;
  st->nb[2] = (res[2] + 1 + 7) / 8 + 1;
  return st;
}
ORACLE_API void oracle_fast_destroy(void *h) { delete static_cast<FastState *>(h); }
ORACLE_API int oracle_fast_num_threads() {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}
ORACLE_API void oracle_fast_set_threads(int n) {
#ifdef _OPENMP
  omp_set_num_threads(n);
#else
  (void)n;
#endif
}
// Runs `nsub` substeps; timings[4] accumulates seconds in {sort, p2g, grid, g2p}.
ORACLE_API int64_t oracle_fast_substeps(void *h, int nsub, const int *res, float dx, float dt, const float *gravity, int particle_gravity,
                                        const int32_t *mat_kind, const float *mat_params, const float *sdf, float friction, int64_t n,
                                        float *x, float *v, float *F, float *b, const float *mass, const float *vol, float *ps,
                                        const int32_t *group, uint8_t *alive_io, double *timings) {
  FastState &st = *static_cast<FastState *>(h);
  Scene<float> sc = make_scene<float>(res, dx, dt, gravity, particle_gravity, mat_kind, mat_params, sdf, friction);
  st.t_sort = st.t_p2g = st.t_grid = st.t_g2p = 0;
  double t_io = 0;
  int64_t updates = 0;
  auto count_alive = [&](const std::vector<uint8_t> &alive) {
    int64_t na = 0;
#pragma omp parallel for reduction(+ : na) schedule(static)
    for (int64_t i = 0; i < n; i++) na += alive[i];
    return na;
  };
  if (st.reorder_interval <= 0) {
    Particles<float> P{n, x, v, F, b, mass, vol, ps, group};
    std::vector<uint8_t> alive(alive_io, alive_io + n);
    for (int s = 0; s < nsub; s++) {
      updates += count_alive(alive);
      fast_substep(st, sc, P, alive);
      st.step++;
    }
    std::memcpy(alive_io, alive.data(), n);
  } else {
    // the engine owns a re-orderable copy of the particle storage, as the reference's allocator pool;
    // the caller's arrays keep their indexing (gather on entry, scatter on exit through `origin`).
    const double tio0 = now_s();
    if (int64_t(st.origin.size()) != n) {
      st.origin.resize(n);
      for (int64_t i = 0; i < n; i++) st.origin[i] = int32_t(i);
    }
    st.sx.resize(size_t(n) * 3); st.sv.resize(size_t(n) * 3); st.sF.resize(size_t(n) * 9); st.sb.resize(size_t(n) * 9);
    st.smass.resize(n); st.svol.resize(n); st.sps.resize(n); st.sgroup.resize(n); st.salive.resize(n);
    permute_rows(st.origin, 3, x, st.sx.data()); permute_rows(st.origin, 3, v, st.sv.data());
    permute_rows(st.origin, 9, F, st.sF.data()); permute_rows(st.origin, 9, b, st.sb.data());
    permute_rows(st.origin, 1, mass, st.smass.data()); permute_rows(st.origin, 1, vol, st.svol.data());
    permute_rows(st.origin, 1, ps, st.sps.data()); permute_rows(st.origin, 1, group, st.sgroup.data());
    permute_rows(st.origin, 1, alive_io, st.salive.data());
    t_io += now_s() - tio0;
    for (int s = 0; s < nsub; s++) {
      updates += count_alive(st.salive);
      Particles<float> P{n, st.sx.data(), st.sv.data(), st.sF.data(), st.sb.data(), st.smass.data(), st.svol.data(), st.sps.data(), st.sgroup.data()};
      fast_substep(st, sc, P, st.salive, st.step % st.reorder_interval == 0);
      st.step++;
    }
    const double tio1 = now_s();
#pragma omp parallel for schedule(static)
    for (int64_t j = 0; j < n; j++) {
      const size_t o = size_t(st.origin[j]);
      for (int c = 0; c < 3; c++) { x[o * 3 + c] = st.sx[size_t(j) * 3 + c]; v[o * 3 + c] = st.sv[size_t(j) * 3 + c]; }
      for (int c = 0; c < 9; c++) { F[o * 9 + c] = st.sF[size_t(j) * 9 + c]; b[o * 9 + c] = st.sb[size_t(j) * 9 + c]; }
      ps[o] = st.sps[j];
      alive_io[o] = st.salive[j];
    }
    t_io += now_s() - tio1;
  }
  // timings[4]: copying between the caller's arrays and the re-orderable storage (a cost of this
  // harness, not of the reference's algorithm: its pool IS the storage)
  if (timings) { timings[0] = st.t_sort; timings[1] = st.t_p2g; timings[2] = st.t_grid; timings[3] = st.t_g2p; timings[4] = t_io; }
  return updates;
}
// Re-order interval of the fast path's particle storage (reference default 1000, src/mpm.cpp:45); 0 = off.
ORACLE_API void oracle_fast_set_reorder(void *h, int interval) {
  FastState &st = *static_cast<FastState *>(h);
  st.reorder_interval = interval;
  st.step = 0;
  st.origin.clear();
}
// Dense copy of the fast path's blocked grid (parity of fast vs scalar oracle).
ORACLE_API void oracle_fast_download_grid(void *h, float *dense /* [(res+1)^3][4] */) {
  FastState &st = *static_cast<FastState *>(h);
  int nx = st.res[0] + 1, ny = st.res[1] + 1, nz = st.res[2] + 1;
  for (int i = 0; i < nx; i++)
    for (int j = 0; j < ny; j++)
      for (int k = 0; k < nz; k++) {
        size_t src = fast_node_index(st, i, j, k) * 4;
        size_t dst = ((size_t(i) * ny + j) * nz + k) * 4;
        if (src + 4 <= st.grid.size()) std::memcpy(dense + dst, &st.grid[src], 16);
        else std::memset(dense + dst, 0, 16);
      }
}
