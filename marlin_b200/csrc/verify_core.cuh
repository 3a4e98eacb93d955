// The verifier's per-point and per-proof arithmetic, host and device (B2M_HD): ark-serialize point decoding, the
// Lagrange evaluation of the public input, the AHP linear-combination coefficients [reference src/ahp/mod.rs:110-221]
// (shared with the prover) and the scalars of the per-proof pairing-check combination [U ark-poly-commit marlin_pc /
// sonic_pc check_combinations].
#pragma once
#include "curve.cuh"

namespace b2m {

enum { DEC_OK = 0, DEC_BAD_FLAGS = 1, DEC_X_RANGE = 2, DEC_NOT_ON_CURVE = 3, DEC_NOT_IN_SUBGROUP = 4 };

// `CanonicalDeserialize` of a compressed short-Weierstrass affine G1 point, ark-serialize 0.3 [U ark-ec
// short_weierstrass_jacobian.rs, SWFlags]: x little-endian in sizeof(Fq)-ish bytes (48 for BLS12-381, 32 for BN254), flags in
// the top two bits of the last byte: bit 7 = y is the larger root, bit 6 = infinity, both set = error.  y = (x^3 + b)^((q+1)/4)
// (q = 3 mod 4 for both curves) must square back.  The point must lie in the prime-order subgroup ([r]P = O; BN254 G1 has
// cofactor 1).  Infinity decodes to Affine::inf() without looking at x, as ark-serialize 0.3 does.
template <class Fq, class Fr>
B2M_HD int g1_decompress(const uint8_t* bytes, Affine<Fq>* out) {
  constexpr int NB = (Fq::Params::BITS + 2 + 7) / 8;  // ark-serialize: x plus two flag bits
  *out = Affine<Fq>::inf();
  const uint8_t flags = bytes[NB - 1] & 0xc0;
  if (flags == 0xc0) return DEC_BAD_FLAGS;
  if (flags & 0x40) return DEC_OK;
  Fq x = Fq::zero();
  for (int i = 0; i < NB; i++) {
    uint8_t b = i == NB - 1 ? (uint8_t)(bytes[i] & 0x3f) : bytes[i];
    x.l[i >> 2] |= (uint32_t)b << (8 * (i & 3));
  }
  for (int i = Fq::N - 1; i >= 0; i--) {  // x < q
    if (x.l[i] != Fq::Params::mod(i)) {
      if (x.l[i] > Fq::Params::mod(i)) return DEC_X_RANGE;
      break;
    }
    if (i == 0) return DEC_X_RANGE;
  }
  x = Fq::from_canonical(x);
  const Fq rhs = x.sqr() * x + Fq::from_u64(sizeof(Fq) == 48 ? 4 : 3);
  uint32_t e[Fq::N];  // (q + 1) / 4
  uint32_t c = 1;
  for (int i = 0; i < Fq::N; i++) {
    uint64_t s = (uint64_t)Fq::Params::mod(i) + c;
    e[i] = (uint32_t)s;
    c = (uint32_t)(s >> 32);
  }
  for (int i = 0; i < Fq::N; i++) e[i] = (e[i] >> 2) | (i + 1 < Fq::N ? e[i + 1] << 30 : 0u);
  Fq y = rhs.pow_limbs(e, Fq::N);
  if (y.sqr() != rhs) return DEC_NOT_ON_CURVE;
  if (y.to_canonical().canonical_gt_half() != ((flags & 0x80) != 0)) y = y.neg();
  if (sizeof(Fq) == 48) {  // BLS12-381 G1 has cofactor h = 0x396c8c005555e1568c00aaab0000aaab
    uint32_t r[Fr::N];
    for (int i = 0; i < Fr::N; i++) r[i] = Fr::Params::mod(i);
    if (!scalar_mul<Fq>(Affine<Fq>{x, y}, r, Fr::N).is_inf()) return DEC_NOT_IN_SUBGROUP;
  }
  *out = Affine<Fq>{x, y};
  return DEC_OK;
}

// x_hat(z) = sum_i L_i(z) x_i over the multiplicative subgroup X of size n (a power of two): ark-poly
// `evaluate_all_lagrange_coefficients` dotted with the formatted public input (leading one included).
template <class Fr>
B2M_HD Fr lagrange_eval(const Fr* x, uint64_t n, const Fr& z) {
  int log_n = 0;
  while ((1ull << log_n) < n) log_n++;
  Fr w = Fr::one();
  {
    Fr root;
    for (int i = 0; i < Fr::N; i++) root.l[i] = Fr::Params::root(i);
    w = root;
    for (int i = log_n; i < Fr::Params::TWO_ADICITY; i++) w = w.sqr();
  }
  const Fr vz = z.pow_u64(n) - Fr::one();
  Fr wi = Fr::one(), acc = Fr::zero();
  if (vz.is_zero()) {  // z in X: L_i(z) = [z == w^i]
    for (uint64_t i = 0; i < n; i++, wi = wi * w)
      if (wi == z) return x[i];
    return acc;
  }
  const Fr k = vz * Fr::from_u64(n).inverse();  // L_i(z) = v_X(z) w^i / (n (z - w^i))
  for (uint64_t i = 0; i < n; i++, wi = wi * w) acc = acc + x[i] * wi * (z - wi).inverse();
  return acc * k;
}

template <class Fr>
struct Challenges {
  Fr alpha, eta_a, eta_b, eta_c, beta, gamma;
};

// Coefficients of the two sumcheck linear combinations [reference src/ahp/mod.rs:145-213], constant (`LCTerm::One`) terms
// included: outer_sumcheck = mask + za z_a + w w + h1 h_1 + outer_const, inner_sumcheck = a a_val + b b_val + c c_val +
// row row + col col + rc row_col + h2 h_2 + inner_const.  The prover uses every field but the constants.
template <class Fr>
struct LcCoeffs {
  Fr za, w, h1, outer_const;
  Fr a, b, c, row, col, rc, h2, inner_const;
};

// evals: g_1(beta), g_2(gamma), t(beta), z_b(beta) (the proof's order); h, k, n_x: |H|, |K|, |X|; x_beta: x_hat(beta).
template <class Fr>
B2M_HD LcCoeffs<Fr> lc_coefficients(const Challenges<Fr>& ch, const Fr* evals, uint64_t h, uint64_t k, uint64_t n_x, const Fr& x_beta) {
  const Fr one = Fr::one();
  const Fr &alpha = ch.alpha, &beta = ch.beta, &gamma = ch.gamma;
  const Fr &g1 = evals[0], &g2 = evals[1], &t = evals[2], &zb = evals[3];
  const Fr v_h_alpha = alpha.pow_u64(h) - one, v_h_beta = beta.pow_u64(h) - one;
  Fr r_ab = (v_h_alpha - v_h_beta) * (alpha - beta).inverse();
  if (alpha == beta) r_ab = Fr::from_u64(h) * alpha.pow_u64(h - 1);
  const Fr v_x_beta = beta.pow_u64(n_x) - one;
  const Fr vv = v_h_alpha * v_h_beta;
  const Fr v_k_gamma = gamma.pow_u64(k) - one;
  const Fr bscale = gamma * g2 + t * Fr::from_u64(k).inverse();
  LcCoeffs<Fr> c;
  c.za = r_ab * (ch.eta_a + ch.eta_c * zb);
  c.w = (t * v_x_beta).neg();
  c.h1 = v_h_beta.neg();
  c.outer_const = r_ab * ch.eta_b * zb - t * x_beta - beta * g1;
  c.a = ch.eta_a * vv;
  c.b = ch.eta_b * vv;
  c.c = ch.eta_c * vv;
  c.row = bscale * alpha;
  c.col = bscale * beta;
  c.rc = bscale.neg();
  c.h2 = v_k_gamma.neg();
  c.inner_const = (bscale * beta * alpha).neg();
  return c;
}

// ---- the per-proof combination ------------------------------------------------------------------------------------
// Each proof reduces to A (paired with h), B (with beta h) and, for SonicKZG10, C_d (with beta^-(D-d) h) per enforced bound:
//   A = sum_p rho_p (sum_l xi^(k_l) C_l - v_p g - rv_p gamma_g + z_p W_p),  B = -sum_p rho_p W_p
// over the two query points p = beta, gamma (MarlinKZG10 adds xi^(k+1) (S_l - v_l shift_power) per degree-bounded l).
// Term list (point, destination) -- the same for every proof:
enum {
  T_W = 0, T_ZA, T_ZB, T_MASK, T_T, T_G1, T_H1, T_G2, T_H2, T_SG1, T_SG2, T_WB, T_WG,  // proof points 0..12
  T_ROW, T_COL, T_AVAL, T_BVAL, T_CVAL, T_RC, T_G, T_GAMMA_G, T_SHIFT_H, T_SHIFT_K,   // verifier-key bases 13..22
  T_WB_B, T_WG_B,                                                                       // W_beta, W_gamma into B
  N_TERMS
};
constexpr int N_PROOF_POINTS = 13;

template <class Fr>
struct ProofScalars {
  Fr evals[4];      // g_1(beta), g_2(gamma), t(beta), z_b(beta)
  Fr rv[2];         // random_v at beta / gamma (zero when absent)
  Fr rho[2];        // 128-bit randomisers of the two openings
  Challenges<Fr> ch;
  Fr xi;            // opening challenge
  Fr x_beta;        // x_hat(beta)
};

// Scalars of the N_TERMS terms (Montgomery).  marlin: MarlinKZG10 (two challenges per degree-bounded polynomial) else SonicKZG10
// (one per polynomial; the bounded g_1 / g_2 terms then go to their C_d, not to A).
template <class Fr>
B2M_HD void term_scalars(const ProofScalars<Fr>& ps, bool marlin, uint64_t h, uint64_t k, uint64_t n_x, Fr* s) {
  const LcCoeffs<Fr> lc = lc_coefficients(ps.ch, ps.evals, h, k, n_x, ps.x_beta);
  const Fr xi = ps.xi, xi2 = xi * xi, xi3 = xi2 * xi, xi4 = xi3 * xi;
  const Fr rb = ps.rho[0], rg = ps.rho[1];
  // challenge of each LC at its point: beta: g_1, outer_sumcheck, t, z_b; gamma: g_2, inner_sumcheck (label order)
  const Fr c_outer = marlin ? xi2 : xi, c_t = marlin ? xi3 : xi2, c_zb = marlin ? xi4 : xi3, c_inner = marlin ? xi2 : xi;
  const Fr ob = rb * c_outer, ig = rg * c_inner;
  s[T_W] = ob * lc.w;
  s[T_ZA] = ob * lc.za;
  s[T_ZB] = rb * c_zb;
  s[T_MASK] = ob;
  s[T_T] = rb * c_t;
  s[T_G1] = rb;
  s[T_H1] = ob * lc.h1;
  s[T_G2] = rg;
  s[T_H2] = ig * lc.h2;
  s[T_SG1] = marlin ? rb * xi : Fr::zero();
  s[T_SG2] = marlin ? rg * xi : Fr::zero();
  s[T_WB] = rb * ps.ch.beta;
  s[T_WG] = rg * ps.ch.gamma;
  s[T_ROW] = ig * lc.row;
  s[T_COL] = ig * lc.col;
  s[T_AVAL] = ig * lc.a;
  s[T_BVAL] = ig * lc.b;
  s[T_CVAL] = ig * lc.c;
  s[T_RC] = ig * lc.rc;
  // combined values: sum over the point's LCs of challenge * evaluation, an LC's constant moved to the evaluation side
  const Fr vb = ps.evals[0] + c_outer * lc.outer_const.neg() + c_t * ps.evals[2] + c_zb * ps.evals[3];
  const Fr vg = ps.evals[1] + c_inner * lc.inner_const.neg();
  s[T_G] = (rb * vb + rg * vg).neg();
  s[T_GAMMA_G] = (rb * ps.rv[0] + rg * ps.rv[1]).neg();
  s[T_SHIFT_H] = marlin ? (rb * xi * ps.evals[0]).neg() : Fr::zero();
  s[T_SHIFT_K] = marlin ? (rg * xi * ps.evals[1]).neg() : Fr::zero();
  s[T_WB_B] = rb.neg();
  s[T_WG_B] = rg.neg();
}

}  // namespace b2m
