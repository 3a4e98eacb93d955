// Host-side G2 arithmetic for the G2 half of `KZG10::setup` [U ark-poly-commit kzg10::setup]: h, beta * h and the few
// beta^(-e) * h that SonicKZG10's verifier key keeps (`neg_powers_of_h`).  The PROVER never touches G2 (reference
// src/lib.rs:151-311 only commits and opens in G1), so this is a handful of scalar multiplications per key on the CPU with
// the same limb code as the device (field.cuh compiled for the host), written out in ark-serialize's uncompressed form so that
// an SRS file made here can be loaded by arkworks (tools/replay_rs).
//
// Fq2 (pairing.cuh) = Fq[u] / (u^2 + 1) for both supported curves; E'(Fq2): y^2 = x^3 + b' (the formulas below never need b').
#pragma once
#include <cstdint>
#include <cstring>
#include <vector>

#include "pairing.cuh"  // Fq2

namespace b2m {

template <class Fq>
struct G2Jac {  // Jacobian: (X / Z^2, Y / Z^3); infinity: Z = 0
  Fq2<Fq> X, Y, Z;
  static G2Jac inf() { return G2Jac{Fq2<Fq>::one(), Fq2<Fq>::one(), Fq2<Fq>::zero()}; }
  bool is_inf() const { return Z.is_zero(); }
  G2Jac dbl() const {  // dbl-2009-l (a = 0)
    if (is_inf()) return *this;
    const Fq2<Fq> A = X.sqr(), B = Y.sqr(), C = B.sqr();
    const Fq2<Fq> D = ((X + B).sqr() - A - C).dbl();
    const Fq2<Fq> E = A.dbl() + A, F = E.sqr();
    G2Jac r;
    r.X = F - D.dbl();
    r.Y = E * (D - r.X) - C.dbl().dbl().dbl();
    r.Z = (Y * Z).dbl();
    return r;
  }
  G2Jac add(const G2Jac& o) const {  // add-2007-bl
    if (is_inf()) return o;
    if (o.is_inf()) return *this;
    const Fq2<Fq> Z1Z1 = Z.sqr(), Z2Z2 = o.Z.sqr();
    const Fq2<Fq> U1 = X * Z2Z2, U2 = o.X * Z1Z1;
    const Fq2<Fq> S1 = Y * o.Z * Z2Z2, S2 = o.Y * Z * Z1Z1;
    if (U1 == U2) return S1 == S2 ? dbl() : inf();
    const Fq2<Fq> H = U2 - U1, I = H.dbl().sqr(), J = H * I, rr = (S2 - S1).dbl(), V = U1 * I;
    G2Jac r;
    r.X = rr.sqr() - J - V.dbl();
    r.Y = rr * (V - r.X) - (S1 * J).dbl();
    r.Z = ((Z + o.Z).sqr() - Z1Z1 - Z2Z2) * H;
    return r;
  }
  // canonical little-endian scalar of nlimbs 32-bit limbs
  G2Jac mul(const uint32_t* k, int nlimbs) const {
    G2Jac acc = inf();
    for (int i = nlimbs - 1; i >= 0; i--)
      for (int b = 31; b >= 0; b--) {
        acc = acc.dbl();
        if ((k[i] >> b) & 1u) acc = acc.add(*this);
      }
    return acc;
  }
  void to_affine(Fq2<Fq>* x, Fq2<Fq>* y) const {  // (finite points only)
    const Fq2<Fq> zi = Z.inverse(), zi2 = zi.sqr();
    *x = X * zi2;
    *y = Y * zi2 * zi;
  }
};

// `CanonicalSerialize::serialize_uncompressed` of a short-Weierstrass affine point over Fq2 [U ark-ec 0.3
// short_weierstrass_jacobian.rs + ark-ff QuadExtField]: x.c0 || x.c1 || y.c0 || y.c1, canonical little-endian, with the
// infinity flag (bit 6) in the very last byte; infinity is written as all-zero coordinates + the flag.
template <class Fq>
void g2_write_uncompressed(std::vector<uint8_t>& out, const G2Jac<Fq>& p) {
  const size_t nb = Fq::N * 4;
  if (p.is_inf()) {
    out.insert(out.end(), 4 * nb - 1, 0);
    out.push_back(1u << 6);
    return;
  }
  Fq2<Fq> x, y;
  p.to_affine(&x, &y);
  const Fq* parts[4] = {&x.c0, &x.c1, &y.c0, &y.c1};
  for (const Fq* f : parts) {
    const Fq c = f->to_canonical();
    const uint8_t* b = reinterpret_cast<const uint8_t*>(c.l);
    out.insert(out.end(), b, b + nb);
  }
}

}  // namespace b2m
