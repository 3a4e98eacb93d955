// Curve-independent interface of the batch verifier (include/b2m.h b2m_verifier / b2m_verify).
#pragma once
#include <string>
#include <vector>

#include "common.cuh"

namespace b2m {

enum { VERDICT_ACCEPT = B2M_VERDICT_ACCEPT, VERDICT_REJECT = B2M_VERDICT_REJECT, VERDICT_MALFORMED = B2M_VERDICT_MALFORMED };

struct VerifierBase {
  virtual ~VerifierBase() {}
  // `Marlin::verify` [reference src/lib.rs:315-433] for a batch of proofs of one index; verdicts[i] = VERDICT_*.
  // public_inputs[i]: n_inputs[i] Montgomery Fr (4 u64 each), without the leading one.
  virtual void verify(size_t n, const uint64_t* const* public_inputs, const size_t* n_inputs, const uint8_t* const* proofs,
                      const size_t* proof_lens, b2m_rng* rng, int* verdicts) = 0;
  std::string timings_json;  // per-stage times of the last verify (milliseconds)
};

// vk_tobytes: `IndexVerifierKey::write`; g, gamma_g: G1 and h, beta_h: G2 in ark-serialize uncompressed form; bound_points: per
// enforced bound, the MarlinKZG10 shift power powers_of_g[max_degree - bound] (G1) or the SonicKZG10 beta^-(max_degree - bound) h
// (G2), uncompressed.
VerifierBase* make_verifier_bls(Ctx& cx, int pc, const uint8_t* vk, size_t vk_len, const uint8_t* g, const uint8_t* gamma_g, const uint8_t* h,
                                const uint8_t* beta_h, size_t max_degree, size_t n_bounds, const uint64_t* bounds, const uint8_t* bound_points);
VerifierBase* make_verifier_bn(Ctx& cx, int pc, const uint8_t* vk, size_t vk_len, const uint8_t* g, const uint8_t* gamma_g, const uint8_t* h,
                               const uint8_t* beta_h, size_t max_degree, size_t n_bounds, const uint64_t* bounds, const uint8_t* bound_points);

}  // namespace b2m
