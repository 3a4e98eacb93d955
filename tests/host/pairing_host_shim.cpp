// Host build of marlin_b200/csrc/pairing.cuh and the verifier's B2M_HD pieces (verify_core.cuh) over a tiny C ABI, so
// pytest can compare the tower, the pairing and the point decoding against the Python oracle without a GPU.
// Field elements cross as Montgomery limbs (32-bit, little-endian), Fq12 as its 12 Fq coefficients in struct order
// (c0.c0.c0, c0.c0.c1, c0.c1.c0, ..., c1.c2.c1).
#include <vector>

#include "../../marlin_b200/csrc/pairing.cuh"
#include "../../marlin_b200/csrc/verify_core.cuh"
using namespace b2m;

template <class Fq>
static void tower(int op, int k, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  Fq12<Fq> x, y, z;
  memcpy(&x, a, sizeof(x));
  memcpy(&y, b, sizeof(y));
  switch (op) {
    case 0: z = x * y; break;
    case 1: z = x.sqr(); break;
    case 2: z = x.inverse(); break;
    case 3: z = x.frob(k); break;
    case 4: z = final_exponentiation(x); break;
    case 5: z = x.conj(); break;
    // sparse line products against the dense product with the same sparse element (coefficients taken from y)
    case 6: z = TowerTraits<Fq>::M_TWIST ? x.mul_by_014(y.c0.c0, y.c0.c1, y.c1.c1) : x.mul_by_034(y.c0.c0, y.c1.c0, y.c1.c1); break;
    default: z = Fq12<Fq>::one();
  }
  memcpy(out, &z, sizeof(z));
}
extern "C" void fq12_op(int curve, int op, int k, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  if (curve == 0) tower<FqBls>(op, k, a, b, out); else tower<FqBn>(op, k, a, b, out);
}

// prod_i e(p_i, q_i); g1: n affine (x, y), g2: n affine (x.c0, x.c1, y.c0, y.c1), inf: per pair (either side at infinity).
// final_exp = 0 returns the Miller-loop product only.
template <class Fq>
static void pairing(int n, const uint32_t* g1, const uint32_t* g2, const uint8_t* inf, int final_exp, uint32_t* out) {
  const int L = n_ell_coeffs<Fq>();
  std::vector<EllCoeff<Fq>> coeffs((size_t)n * L);
  std::vector<const EllCoeff<Fq>*> cp(n);
  std::vector<Fq> px(n), py(n);
  bool fl[16];
  for (int i = 0; i < n; i++) {
    G2Aff<Fq> q;
    memcpy(&q.x, g2 + (size_t)i * 4 * Fq::N, 2 * sizeof(Fq));
    memcpy(&q.y, g2 + (size_t)i * 4 * Fq::N + 2 * Fq::N, 2 * sizeof(Fq));
    q.inf = false;
    fl[i] = inf[i] != 0;
    if (!fl[i]) g2_prepare(q, coeffs.data() + (size_t)i * L);
    cp[i] = coeffs.data() + (size_t)i * L;
    memcpy(&px[i], g1 + (size_t)i * 2 * Fq::N, sizeof(Fq));
    memcpy(&py[i], g1 + (size_t)i * 2 * Fq::N + Fq::N, sizeof(Fq));
  }
  Fq12<Fq> f = miller_loop<Fq>(n, px.data(), py.data(), fl, cp.data());
  if (final_exp) f = final_exponentiation(f);
  memcpy(out, &f, sizeof(f));
}
extern "C" void pairing_product(int curve, int n, const uint32_t* g1, const uint32_t* g2, const uint8_t* inf, int final_exp, uint32_t* out) {
  if (n > 16) return;
  if (curve == 0) pairing<FqBls>(n, g1, g2, inf, final_exp, out); else pairing<FqBn>(n, g1, g2, inf, final_exp, out);
}

// ark-serialize compressed G1 decoding (verify_core.cuh g1_decompress): status per point, affine Montgomery out.
extern "C" int g1_decode(int curve, const uint8_t* bytes, uint32_t* out_xy) {
  if (curve == 0) {
    Affine<FqBls> p;
    int s = g1_decompress<FqBls, FrBls>(bytes, &p);
    memcpy(out_xy, &p, sizeof(p));
    return s;
  }
  Affine<FqBn> p;
  int s = g1_decompress<FqBn, FrBn>(bytes, &p);
  memcpy(out_xy, &p, sizeof(p));
  return s;
}

// The Marlin linear-combination coefficients (verify_core.cuh lc_coefficients) from the challenges and evaluations.
// in: alpha, eta_a, eta_b, eta_c, beta, gamma, g1(beta), g2(gamma), t(beta), z_b(beta) (Montgomery Fr, 8 limbs each);
// x: the padded public input with the leading one (n_x elements, a power of two); out: LcCoeffs in struct order.
extern "C" void lc_coeffs(int curve, const uint32_t* in, const uint32_t* x, int n_x, uint64_t h, uint64_t k, uint32_t* out) {
  auto run = [&](auto tag) {
    using Fr = decltype(tag);
    const Fr* v = reinterpret_cast<const Fr*>(in);
    Challenges<Fr> c{v[0], v[1], v[2], v[3], v[4], v[5]};
    Fr evals[4] = {v[6], v[7], v[8], v[9]};
    Fr xb = lagrange_eval(reinterpret_cast<const Fr*>(x), (uint64_t)n_x, c.beta);
    LcCoeffs<Fr> lc = lc_coefficients(c, evals, h, k, (uint64_t)n_x, xb);
    memcpy(out, &lc, sizeof(lc));
  };
  if (curve == 0) run(FrBls{}); else run(FrBn{});
}
