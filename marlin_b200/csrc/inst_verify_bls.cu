#include "verify_impl.cuh"
namespace b2m {
VerifierBase* make_verifier_bls(Ctx& cx, int pc, const uint8_t* vk, size_t vk_len, const uint8_t* g, const uint8_t* gamma_g, const uint8_t* h,
                                const uint8_t* beta_h, size_t max_degree, size_t n_bounds, const uint64_t* bounds, const uint8_t* bound_points) {
  return new MarlinVerifier<FrBls, FqBls>(cx, pc, vk, vk_len, g, gamma_g, h, beta_h, max_degree, n_bounds, bounds, bound_points);
}
}  // namespace b2m
