// extern "C" boundary of libb2m.so (declared in include/b2m.h).  Level 0: NTT / MSM / SRS.
// The prover-level entry points live in prover.cu.
#include "capi_types.cuh"
#include "prover.cuh"
#include "verify.cuh"
#include "comm.cuh"
#include <algorithm>
#include "g2_host.hpp"

namespace b2m {
thread_local std::string g_last_error;
}

using namespace b2m;

extern "C" {

const char* b2m_last_error(void) { return g_last_error.c_str(); }
const char* b2m_version(void) { return "b2m 0.1 (sm_100a)"; }

int b2m_ctx_create(int device, b2m_ctx** out) {
  return guard([&] {
    B2M_REQUIRE(out != nullptr, B2M_ERR_INVALID_ARG, "out is null");
    *out = new b2m_ctx(device);
  });
}

void b2m_ctx_destroy(b2m_ctx* ctx) {
  if (!ctx) return;
  if (ctx->children > 0) {  // SRSs still borrow this context: freed with the last of them
    ctx->dead = true;
    return;
  }
  b2m_release_ctx(ctx);
}

unsigned long long b2m_ctx_launches(const b2m_ctx* ctx) { return ctx ? ctx->cx.launches : 0; }

int b2m_comm_unique_id(uint8_t* id, size_t cap) {
  return guard([&] {
    B2M_REQUIRE(id && cap >= sizeof(ncclUniqueId), B2M_ERR_INVALID_ARG, "id buffer must hold %zu bytes", sizeof(ncclUniqueId));
    ncclUniqueId u;
    B2M_NCCL(NcclApi::get().GetUniqueId(&u));
    memcpy(id, &u, sizeof(u));
  });
}

int b2m_ctx_attach_comm(b2m_ctx* ctx, const uint8_t* id, size_t id_len, int rank, int world) {
  return guard([&] {
    B2M_REQUIRE(ctx && id && id_len >= sizeof(ncclUniqueId), B2M_ERR_INVALID_ARG, "bad unique id");
    B2M_REQUIRE(world >= 1 && rank >= 0 && rank < world, B2M_ERR_INVALID_ARG, "bad rank %d / world %d", rank, world);
    ctx->cx.use();
    if (world > 1) {
      ncclUniqueId u;
      memcpy(&u, id, sizeof(u));
      ncclComm_t comm;
      B2M_NCCL(NcclApi::get().CommInitRank(&comm, world, u, rank));
      ctx->cx.comm = comm;
    }
    ctx->cx.rank = rank;
    ctx->cx.world = world;
  });
}

int b2m_ctx_profile(b2m_ctx* ctx, int enable) {
  return guard([&] {
    B2M_REQUIRE(ctx != nullptr, B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    if (!enable) ctx->cx.span_report();
    ctx->cx.profiling = enable != 0;
  });
}

int b2m_ctx_profile_report(b2m_ctx* ctx, char* json, size_t cap) {
  return guard([&] {
    B2M_REQUIRE(ctx && json && cap > 0, B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    snprintf(json, cap, "%s", ctx->cx.span_report().c_str());
  });
}

int b2m_ntt(b2m_ctx* ctx, int curve, uint64_t* data, unsigned log_n, int inverse, int coset) {
  return guard([&] {
    B2M_REQUIRE(ctx && data, B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    if (curve == B2M_CURVE_BLS12_381) ctx->ntt_bls().run_host(data, log_n, inverse != 0, coset != 0);
    else if (curve == B2M_CURVE_BN254) ctx->ntt_bn().run_host(data, log_n, inverse != 0, coset != 0);
    else throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
  });
}

int b2m_srs_create(b2m_ctx* ctx, int curve, const uint64_t* powers_of_g, size_t n_g, const uint64_t* powers_of_gamma_g,
                   const uint64_t* gamma_indices, size_t n_gamma, int window_bits, b2m_srs** out) {
  return guard([&] {
    B2M_REQUIRE(ctx && powers_of_g && out, B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(curve == B2M_CURVE_BLS12_381 || curve == B2M_CURVE_BN254, B2M_ERR_INVALID_ARG, "unknown curve id");
    ctx->cx.use();
    *out = new b2m_srs(ctx, curve, powers_of_g, n_g, powers_of_gamma_g, gamma_indices, n_gamma, window_bits);
    ctx->children++;
  });
}

void b2m_srs_destroy(b2m_srs* srs) {
  if (!srs) return;
  if (srs->children > 0) {  // indexes / committer keys still borrow this SRS: freed with the last of them
    srs->dead = true;
    return;
  }
  b2m_release_srs(srs);
}

size_t b2m_srs_size(const b2m_srs* srs) { return srs ? srs->n_g : 0; }
int b2m_srs_window_bits(const b2m_srs* srs) { return srs ? srs->window_bits() : 0; }
int b2m_srs_affine_levels(const b2m_srs* srs) { return srs ? srs->affine_levels() : 0; }

int b2m_srs_msm(b2m_srs* srs, size_t base_off, const uint64_t* scalars, size_t n, uint64_t* out_xy, int* out_is_inf) {
  return guard([&] {
    B2M_REQUIRE(srs && out_xy && (scalars || n == 0), B2M_ERR_INVALID_ARG, "null argument");
    srs->ctx->cx.use();
    if (srs->curve == B2M_CURVE_BLS12_381) srs->bls->run_host(base_off, scalars, n, out_xy, out_is_inf);
    else srs->bn->run_host(base_off, scalars, n, out_xy, out_is_inf);
  });
}

}  // extern "C"
void b2m_release_ctx(b2m_ctx* ctx) {
  cudaSetDevice(ctx->cx.device);
  cudaStreamSynchronize(ctx->cx.stream);
  if (ctx->cx.comm) NcclApi::get().CommDestroy(static_cast<ncclComm_t>(ctx->cx.comm));
  delete ctx;
}
void b2m_release_srs(b2m_srs* srs) {
  b2m_ctx* ctx = srs->ctx;
  ctx->cx.use();
  cudaStreamSynchronize(ctx->cx.stream);
  delete srs;
  if (--ctx->children == 0 && ctx->dead) b2m_release_ctx(ctx);
}
extern "C" {

int b2m_msm_g1(b2m_ctx* ctx, int curve, const uint64_t* bases_xy, const uint64_t* scalars, size_t n, uint64_t* out_xy,
               int* out_is_inf) {
  b2m_srs* srs = nullptr;
  if (n == 0) {
    if (out_is_inf) *out_is_inf = 1;
    return B2M_OK;
  }
  int rc = b2m_srs_create(ctx, curve, bases_xy, n, nullptr, nullptr, 0, 0, &srs);
  if (rc != B2M_OK) return rc;
  rc = b2m_srs_msm(srs, 0, scalars, n, out_xy, out_is_inf);
  b2m_srs_destroy(srs);
  return rc;
}

int b2m_g1_powers(b2m_ctx* ctx, int curve, const uint64_t* g_xy, const uint64_t* beta, size_t n, uint64_t* out_powers_xy) {
  return guard([&] {
    B2M_REQUIRE(ctx && g_xy && beta && out_powers_xy, B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    if (curve == B2M_CURVE_BLS12_381) Msm<FrBls, FqBls>::g1_powers_host(ctx->cx, g_xy, beta, n, out_powers_xy);
    else if (curve == B2M_CURVE_BN254) Msm<FrBn, FqBn>::g1_powers_host(ctx->cx, g_xy, beta, n, out_powers_xy);
    else throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
  });
}

int b2m_fixed_base_msm(b2m_ctx* ctx, int curve, const uint64_t* g_xy, const uint64_t* scalars, size_t n, uint64_t* out_xy) {
  return guard([&] {
    B2M_REQUIRE(ctx && g_xy && (scalars || n == 0) && (out_xy || n == 0), B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    if (curve == B2M_CURVE_BLS12_381) Msm<FrBls, FqBls>::fixed_base_host(ctx->cx, g_xy, scalars, nullptr, 0, n, out_xy);
    else if (curve == B2M_CURVE_BN254) Msm<FrBn, FqBn>::fixed_base_host(ctx->cx, g_xy, scalars, nullptr, 0, n, out_xy);
    else throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
  });
}

int b2m_srs_export_g1(b2m_srs* srs, size_t first, size_t n, uint8_t* out) {
  return guard([&] {
    B2M_REQUIRE(srs && (out || n == 0), B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(first + n <= srs->n_g, B2M_ERR_INVALID_ARG, "powers [%zu, %zu) of %zu", first, first + n, srs->n_g);
    srs->ctx->cx.use();
    if (srs->curve == B2M_CURVE_BLS12_381) {
      B2M_REQUIRE(srs->bls->tab_world == 1, B2M_ERR_UNSUPPORTED, "export from a sharded key");
      Msm<FrBls, FqBls>::g1_to_bytes(srs->ctx->cx, srs->bls->tables.p + first, nullptr, n, out);
    } else {
      B2M_REQUIRE(srs->bn->tab_world == 1, B2M_ERR_UNSUPPORTED, "export from a sharded key");
      Msm<FrBn, FqBn>::g1_to_bytes(srs->ctx->cx, srs->bn->tables.p + first, nullptr, n, out);
    }
  });
}
int b2m_g1_to_uncompressed(b2m_ctx* ctx, int curve, const uint64_t* points_xy, size_t n, uint8_t* out) {
  return guard([&] {
    B2M_REQUIRE(ctx && ((points_xy && out) || n == 0), B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    if (curve == B2M_CURVE_BLS12_381) Msm<FrBls, FqBls>::g1_to_bytes(ctx->cx, nullptr, points_xy, n, out);
    else if (curve == B2M_CURVE_BN254) Msm<FrBn, FqBn>::g1_to_bytes(ctx->cx, nullptr, points_xy, n, out);
    else throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
  });
}
int b2m_g1_from_uncompressed(b2m_ctx* ctx, int curve, const uint8_t* bytes, size_t n, uint64_t* out_xy) {
  return guard([&] {
    B2M_REQUIRE(ctx && ((bytes && out_xy) || n == 0), B2M_ERR_INVALID_ARG, "null argument");
    ctx->cx.use();
    if (curve == B2M_CURVE_BLS12_381) Msm<FrBls, FqBls>::g1_from_bytes(ctx->cx, bytes, n, out_xy);
    else if (curve == B2M_CURVE_BN254) Msm<FrBn, FqBn>::g1_from_bytes(ctx->cx, bytes, n, out_xy);
    else throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
  });
}

}  // extern "C"
// standard G2 generators (canonical x.c0, x.c1, y.c0, y.c1; big-endian hex), checked on-curve / order r in tests/test_srs_files.py
static const char* const G2_GEN_BLS[4] = {
    "024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8",
    "13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e",
    "0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801",
    "0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be"};
static const char* const G2_GEN_BN[4] = {
    "1800deef121f1e76426a00665e5c4479674322d4f75edadd46debd5cd992f6ed", "198e9393920d483a7260bfb731fb5d25f1aa493335a9e71297e485b7aef312c2",
    "12c85ea5db8c6deb4aab71808dcb408fe3d1e7690c43d37b4ce6cc0166fa7daa", "090689d0585ff075ec9e99ad690c3395bc4b313370b38ef355acdadcd122975b"};

template <class Fq>
static Fq fq_from_hex(const char* hex) {
  Fq c = Fq::zero();
  const size_t len = strlen(hex);
  for (size_t i = 0; i < len; i++) {
    const char ch = hex[len - 1 - i];
    const uint32_t v = ch >= 'a' ? ch - 'a' + 10 : ch - '0';
    c.l[i / 8] |= v << (4 * (i % 8));
  }
  return Fq::from_canonical(c);
}
template <class Fq>
static void g2_scalar_muls_impl(const char* const gen[4], const uint8_t* h_bytes, const uint64_t* scalars, size_t n, uint8_t* out) {
  G2Jac<Fq> h;
  if (h_bytes) {
    Fq parts[4];
    for (int k = 0; k < 4; k++) {
      Fq c;
      memcpy(c.l, h_bytes + (size_t)k * Fq::N * 4, Fq::N * 4);
      if (k == 3) {
        B2M_REQUIRE(!((c.l[Fq::N - 1] >> 30) & 1u), B2M_ERR_INVALID_ARG, "the G2 base is the point at infinity");
        c.l[Fq::N - 1] &= 0x3fffffffu;
      }
      parts[k] = Fq::from_canonical(c);
    }
    h = G2Jac<Fq>{Fq2<Fq>{parts[0], parts[1]}, Fq2<Fq>{parts[2], parts[3]}, Fq2<Fq>::one()};
  } else {
    h = G2Jac<Fq>{Fq2<Fq>{fq_from_hex<Fq>(gen[0]), fq_from_hex<Fq>(gen[1])}, Fq2<Fq>{fq_from_hex<Fq>(gen[2]), fq_from_hex<Fq>(gen[3])}, Fq2<Fq>::one()};
  }
  std::vector<uint8_t> bytes;
  for (size_t i = 0; i < n; i++) g2_write_uncompressed<Fq>(bytes, h.mul(reinterpret_cast<const uint32_t*>(scalars + 4 * i), 8));
  memcpy(out, bytes.data(), bytes.size());
}
extern "C" {
int b2m_g2_scalar_muls(int curve, const uint8_t* h_uncompressed, const uint64_t* scalars, size_t n, uint8_t* out) {
  return guard([&] {
    B2M_REQUIRE((scalars && out) || n == 0, B2M_ERR_INVALID_ARG, "null argument");
    if (curve == B2M_CURVE_BLS12_381) g2_scalar_muls_impl<FqBls>(G2_GEN_BLS, h_uncompressed, scalars, n, out);
    else if (curve == B2M_CURVE_BN254) g2_scalar_muls_impl<FqBn>(G2_GEN_BN, h_uncompressed, scalars, n, out);
    else throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
  });
}

// ---- Level 1 ----------------------------------------------------------------------------------
int b2m_pc_commit(b2m_srs* srs, int pc_variant, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs,
                  const int64_t* degree_bounds, const int64_t* hiding_bounds, b2m_rng* rng, uint64_t* out_comm_xy,
                  uint64_t* out_shifted_xy, uint64_t* out_rand, uint64_t* out_shifted_rand, size_t rand_stride) {
  return guard([&] {
    B2M_REQUIRE(srs && coeffs && n_coeffs && degree_bounds && hiding_bounds && out_comm_xy && out_rand, B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(pc_variant == B2M_PC_MARLIN_KZG10 || pc_variant == B2M_PC_SONIC_KZG10, B2M_ERR_INVALID_ARG, "unknown PC variant");
    B2M_REQUIRE(pc_variant != B2M_PC_MARLIN_KZG10 || (out_shifted_xy && out_shifted_rand), B2M_ERR_INVALID_ARG,
                "MarlinKZG10 needs the shifted output buffers");
    B2M_REQUIRE(rng == nullptr || rng->kind == B2M_RNG_CHACHA8 || rng->kind == B2M_RNG_CHACHA12 || rng->kind == B2M_RNG_CHACHA20 ||
                    (rng->kind == B2M_RNG_CALLBACK && rng->next_u64 != nullptr),
                B2M_ERR_MISSING_RNG, "unsupported rng kind");
    srs->ctx->cx.use();
    if (srs->curve == B2M_CURVE_BLS12_381)
      pc_commit_bls(srs, pc_variant, n_polys, coeffs, n_coeffs, degree_bounds, hiding_bounds, rng, out_comm_xy, out_shifted_xy, out_rand,
                    out_shifted_rand, rand_stride);
    else
      pc_commit_bn(srs, pc_variant, n_polys, coeffs, n_coeffs, degree_bounds, hiding_bounds, rng, out_comm_xy, out_shifted_xy, out_rand,
                   out_shifted_rand, rand_stride);
  });
}

int b2m_pc_open(b2m_srs* srs, int pc_variant, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs,
                const int64_t* degree_bounds, const uint64_t* rands, const uint64_t* shifted_rands, size_t rand_stride,
                int64_t max_degree_bound, const uint64_t* point, const uint64_t* opening_challenge, uint64_t* out_w_xy,
                int* out_has_random_v, uint64_t* out_random_v) {
  return guard([&] {
    B2M_REQUIRE(srs && coeffs && n_coeffs && degree_bounds && point && opening_challenge && out_w_xy && out_has_random_v && out_random_v,
                B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(pc_variant == B2M_PC_MARLIN_KZG10 || pc_variant == B2M_PC_SONIC_KZG10, B2M_ERR_INVALID_ARG, "unknown PC variant");
    B2M_REQUIRE(n_polys >= 1, B2M_ERR_INVALID_ARG, "no polynomials");
    srs->ctx->cx.use();
    if (srs->curve == B2M_CURVE_BLS12_381)
      pc_open_bls(srs, pc_variant, n_polys, coeffs, n_coeffs, degree_bounds, rands, shifted_rands, rand_stride, max_degree_bound, point,
                  opening_challenge, out_w_xy, out_has_random_v, out_random_v);
    else
      pc_open_bn(srs, pc_variant, n_polys, coeffs, n_coeffs, degree_bounds, rands, shifted_rands, rand_stride, max_degree_bound, point,
                 opening_challenge, out_w_xy, out_has_random_v, out_random_v);
  });
}

int b2m_trim(b2m_srs* srs, int pc_variant, size_t supported_degree, size_t supported_hiding_bound, const uint64_t* enforced_degree_bounds,
             size_t n_bounds, b2m_ck** out) {
  return guard([&] {
    B2M_REQUIRE(srs && out && (enforced_degree_bounds || n_bounds == 0), B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(pc_variant == B2M_PC_MARLIN_KZG10 || pc_variant == B2M_PC_SONIC_KZG10, B2M_ERR_INVALID_ARG, "unknown PC variant");
    const size_t D = srs->n_g - 1;
    B2M_REQUIRE(supported_degree >= 1 && supported_degree <= D, B2M_ERR_DEGREE_TOO_LARGE, "supported degree %zu out of range (max degree %zu)",
                supported_degree, D);  // TrimmingDegreeTooLarge / DegreeIsZero
    std::unique_ptr<b2m_ck> ck(new b2m_ck{srs, pc_variant, supported_degree, supported_hiding_bound, {}});
    for (size_t k = 0; k < n_bounds; k++) {
      B2M_REQUIRE(enforced_degree_bounds[k] <= supported_degree, B2M_ERR_DEGREE_TOO_LARGE, "enforced degree bound %llu exceeds the supported degree %zu",
                  (unsigned long long)enforced_degree_bounds[k], supported_degree);
      ck->bounds.push_back(enforced_degree_bounds[k]);
    }
    std::sort(ck->bounds.begin(), ck->bounds.end());
    ck->bounds.erase(std::unique(ck->bounds.begin(), ck->bounds.end()), ck->bounds.end());
    // the hiding powers this key will be asked for must be resident (throws B2M_ERR_INVALID_ARG naming the missing power)
    for (size_t i = 0; i <= supported_hiding_bound + 1; i++) srs->gamma_slot(i);
    if (pc_variant == B2M_PC_SONIC_KZG10)
      for (uint64_t b : ck->bounds)
        for (size_t i = 0; i <= supported_hiding_bound + 1; i++) srs->gamma_slot(D - b + i);
    *out = ck.release();
    srs->children++;
  });
}

void b2m_ck_destroy(b2m_ck* ck) {
  if (!ck) return;
  b2m_srs* srs = ck->srs;
  delete ck;
  if (--srs->children == 0 && srs->dead) b2m_release_srs(srs);
}

size_t b2m_ck_supported_degree(const b2m_ck* ck) { return ck ? ck->supported_degree : 0; }

int b2m_ck_shift_power(const b2m_ck* ck, uint64_t bound, uint64_t* out_xy) {
  return guard([&] {
    B2M_REQUIRE(ck && out_xy, B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(ck->enforced(bound), B2M_ERR_INVALID_ARG, "degree bound %llu is not enforced by this committer key", (unsigned long long)bound);
    b2m_srs* srs = ck->srs;
    srs->ctx->cx.use();
    const size_t slot = srs->n_g - 1 - bound;
    if (srs->curve == B2M_CURVE_BLS12_381) srs->bls->read_power(slot, out_xy);
    else srs->bn->read_power(slot, out_xy);
  });
}

static void ck_check_polys(const b2m_ck* ck, size_t n_polys, const size_t* n_coeffs, const int64_t* degree_bounds, const int64_t* hiding_bounds) {
  for (size_t i = 0; i < n_polys; i++) {
    B2M_REQUIRE(n_coeffs[i] <= ck->supported_degree + 1, B2M_ERR_DEGREE_TOO_LARGE, "polynomial %zu has degree %zu, the committer key supports %zu", i,
                n_coeffs[i] ? n_coeffs[i] - 1 : 0, ck->supported_degree);  // TooManyCoefficients
    if (degree_bounds[i] >= 0)
      B2M_REQUIRE(ck->enforced((uint64_t)degree_bounds[i]), B2M_ERR_INVALID_ARG, "polynomial %zu: degree bound %lld is not enforced by this committer key", i,
                  (long long)degree_bounds[i]);  // UnsupportedDegreeBound
    if (hiding_bounds && hiding_bounds[i] >= 0)
      B2M_REQUIRE((size_t)hiding_bounds[i] <= ck->hiding_bound, B2M_ERR_INVALID_ARG, "polynomial %zu: hiding bound %lld above the supported %zu", i,
                  (long long)hiding_bounds[i], ck->hiding_bound);  // HidingBoundToolarge
  }
}

int b2m_ck_commit(b2m_ck* ck, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs, const int64_t* degree_bounds,
                  const int64_t* hiding_bounds, b2m_rng* rng, uint64_t* out_comm_xy, uint64_t* out_shifted_xy, uint64_t* out_rand,
                  uint64_t* out_shifted_rand, size_t rand_stride) {
  int rc = guard([&] {
    B2M_REQUIRE(ck && n_coeffs && degree_bounds && hiding_bounds, B2M_ERR_INVALID_ARG, "null argument");
    ck_check_polys(ck, n_polys, n_coeffs, degree_bounds, hiding_bounds);
  });
  if (rc != B2M_OK) return rc;
  return b2m_pc_commit(ck->srs, ck->pc, n_polys, coeffs, n_coeffs, degree_bounds, hiding_bounds, rng, out_comm_xy, out_shifted_xy, out_rand,
                       out_shifted_rand, rand_stride);
}

int b2m_ck_open_combinations(b2m_ck* ck, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs, const int64_t* degree_bounds,
                             const int* hiding, const uint64_t* rands, const uint64_t* shifted_rands, size_t rand_stride, size_t n_lcs,
                             const size_t* lc_term_off, const int64_t* lc_poly, const uint64_t* lc_coeff, size_t n_queries, const size_t* query_lc,
                             const size_t* query_point, size_t n_points, const uint64_t* points, const uint64_t* opening_challenge,
                             uint64_t* out_w_xy, int* out_has_random_v, uint64_t* out_random_v) {
  return guard([&] {
    B2M_REQUIRE(ck && coeffs && n_coeffs && degree_bounds && hiding && rands && lc_term_off && lc_poly && lc_coeff && query_lc && query_point &&
                    points && opening_challenge && out_w_xy && out_has_random_v && out_random_v,
                B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(n_polys >= 1 && n_lcs >= 1 && n_points >= 1 && n_queries >= 1, B2M_ERR_INVALID_ARG, "empty opening");
    B2M_REQUIRE(ck->pc != B2M_PC_MARLIN_KZG10 || shifted_rands, B2M_ERR_INVALID_ARG, "MarlinKZG10 needs the shifted randomness");
    ck_check_polys(ck, n_polys, n_coeffs, degree_bounds, nullptr);
    for (size_t q = 0; q < n_queries; q++) B2M_REQUIRE(query_point[q] < n_points, B2M_ERR_INVALID_ARG, "query %zu names point %zu of %zu", q, query_point[q], n_points);
    b2m_srs* srs = ck->srs;
    srs->ctx->cx.use();
    if (srs->curve == B2M_CURVE_BLS12_381)
      pc_open_combinations_bls(srs, ck->pc, ck->max_bound(), n_polys, coeffs, n_coeffs, degree_bounds, hiding, rands, shifted_rands, rand_stride, n_lcs,
                               lc_term_off, lc_poly, lc_coeff, n_queries, query_lc, query_point, n_points, points, opening_challenge, out_w_xy,
                               out_has_random_v, out_random_v);
    else
      pc_open_combinations_bn(srs, ck->pc, ck->max_bound(), n_polys, coeffs, n_coeffs, degree_bounds, hiding, rands, shifted_rands, rand_stride, n_lcs,
                              lc_term_off, lc_poly, lc_coeff, n_queries, query_lc, query_point, n_points, points, opening_challenge, out_w_xy,
                              out_has_random_v, out_random_v);
  });
}

// ---- Level 2 ----------------------------------------------------------------------------------
struct b2m_index {
  b2m_srs* srs;
  std::unique_ptr<IndexBase> impl;
};

int b2m_index_create(b2m_srs* srs, int pc_variant, size_t num_constraints, size_t num_variables, size_t num_instance_variables,
                     const b2m_matrix* a, const b2m_matrix* b, const b2m_matrix* c, b2m_index** out) {
  return guard([&] {
    B2M_REQUIRE(srs && a && b && c && out, B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(pc_variant == B2M_PC_MARLIN_KZG10 || pc_variant == B2M_PC_SONIC_KZG10, B2M_ERR_INVALID_ARG, "unknown PC variant");
    srs->ctx->cx.use();
    std::unique_ptr<b2m_index> idx(new b2m_index);
    idx->srs = srs;
    if (srs->curve == B2M_CURVE_BLS12_381)
      idx->impl.reset(make_index_bls(srs, pc_variant, num_constraints, num_variables, num_instance_variables, a, b, c));
    else
      idx->impl.reset(make_index_bn(srs, pc_variant, num_constraints, num_variables, num_instance_variables, a, b, c));
    *out = idx.release();
    srs->children++;
  });
}

void b2m_index_destroy(b2m_index* idx) {
  if (!idx) return;
  b2m_srs* srs = idx->srs;
  srs->ctx->cx.use();
  cudaStreamSynchronize(srs->ctx->cx.stream);
  delete idx;
  if (--srs->children == 0 && srs->dead) b2m_release_srs(srs);
}

int b2m_index_vk_bytes(const b2m_index* idx, uint8_t* out, size_t cap, size_t* len) {
  return guard([&] {
    B2M_REQUIRE(idx && len, B2M_ERR_INVALID_ARG, "null argument");
    *len = idx->impl->vk_bytes.size();
    if (out) {
      B2M_REQUIRE(cap >= *len, B2M_ERR_INVALID_ARG, "buffer too small (%zu < %zu)", cap, *len);
      memcpy(out, idx->impl->vk_bytes.data(), *len);
    }
  });
}

int b2m_index_comms(const b2m_index* idx, uint64_t* out_xy) {
  return guard([&] {
    B2M_REQUIRE(idx && out_xy, B2M_ERR_INVALID_ARG, "null argument");
    memcpy(out_xy, idx->impl->comms_xy.data(), idx->impl->comms_xy.size() * sizeof(uint64_t));
  });
}

int b2m_prove(b2m_index* idx, const uint64_t* formatted_input, size_t n_input, const uint64_t* witness, size_t n_witness,
              b2m_rng* zk_rng, uint8_t* proof, size_t cap, size_t* proof_len) {
  return guard([&] {
    B2M_REQUIRE(idx && proof && proof_len, B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(formatted_input == nullptr || witness || n_witness == 0, B2M_ERR_INVALID_ARG, "null witness");
    B2M_REQUIRE(zk_rng != nullptr, B2M_ERR_MISSING_RNG, "zk_rng is required (hiding commitments)");
    idx->srs->ctx->cx.use();
    std::vector<uint8_t> bytes;
    idx->impl->prove(formatted_input, n_input, witness, n_witness, zk_rng, bytes);
    *proof_len = bytes.size();
    B2M_REQUIRE(cap >= bytes.size(), B2M_ERR_INVALID_ARG, "proof buffer too small (%zu < %zu)", cap, bytes.size());
    memcpy(proof, bytes.data(), bytes.size());
  });
}

int b2m_index_stage(b2m_index* idx, const uint64_t* formatted_input, size_t n_input, const uint64_t* witness, size_t n_witness) {
  return guard([&] {
    B2M_REQUIRE(idx && formatted_input && (witness || n_witness == 0), B2M_ERR_INVALID_ARG, "null argument");
    idx->srs->ctx->cx.use();
    idx->impl->stage(formatted_input, n_input, witness, n_witness);
  });
}

int b2m_prove_timings(const b2m_index* idx, char* json, size_t cap) {
  return guard([&] {
    B2M_REQUIRE(idx && json && cap > 0, B2M_ERR_INVALID_ARG, "null argument");
    snprintf(json, cap, "%s", idx->impl->timings_json.c_str());
  });
}

// ---- Level 3 ----------------------------------------------------------------------------------
struct b2m_verifier {
  b2m_ctx* ctx;
  std::unique_ptr<VerifierBase> impl;
};

int b2m_verifier_create(b2m_ctx* ctx, int curve, int pc_variant, const uint8_t* vk_tobytes, size_t vk_len, const uint8_t* g,
                        const uint8_t* gamma_g, const uint8_t* h, const uint8_t* beta_h, size_t max_degree, size_t n_bounds,
                        const uint64_t* bounds, const uint8_t* bound_points, b2m_verifier** out) {
  return guard([&] {
    B2M_REQUIRE(ctx && vk_tobytes && g && gamma_g && h && beta_h && out && (n_bounds == 0 || (bounds && bound_points)), B2M_ERR_INVALID_ARG,
                "null argument");
    B2M_REQUIRE(pc_variant == B2M_PC_MARLIN_KZG10 || pc_variant == B2M_PC_SONIC_KZG10, B2M_ERR_INVALID_ARG, "unknown PC variant");
    ctx->cx.use();
    std::unique_ptr<b2m_verifier> v(new b2m_verifier);
    v->ctx = ctx;
    if (curve == B2M_CURVE_BLS12_381)
      v->impl.reset(make_verifier_bls(ctx->cx, pc_variant, vk_tobytes, vk_len, g, gamma_g, h, beta_h, max_degree, n_bounds, bounds, bound_points));
    else if (curve == B2M_CURVE_BN254)
      v->impl.reset(make_verifier_bn(ctx->cx, pc_variant, vk_tobytes, vk_len, g, gamma_g, h, beta_h, max_degree, n_bounds, bounds, bound_points));
    else
      throw Error(B2M_ERR_INVALID_ARG, "unknown curve id");
    *out = v.release();
    ctx->children++;
  });
}

void b2m_verifier_destroy(b2m_verifier* ver) {
  if (!ver) return;
  b2m_ctx* ctx = ver->ctx;
  ctx->cx.use();
  cudaStreamSynchronize(ctx->cx.stream);
  delete ver;
  if (--ctx->children == 0 && ctx->dead) b2m_release_ctx(ctx);
}

int b2m_verify(b2m_verifier* ver, size_t n_proofs, const uint64_t* const* public_inputs, const size_t* n_inputs, const uint8_t* const* proofs,
               const size_t* proof_lens, b2m_rng* rng, int* verdicts) {
  return guard([&] {
    B2M_REQUIRE(ver, B2M_ERR_INVALID_ARG, "null verifier");
    ver->ctx->cx.use();
    ver->impl->verify(n_proofs, public_inputs, n_inputs, proofs, proof_lens, rng, verdicts);
  });
}

int b2m_verify_timings(const b2m_verifier* ver, char* json, size_t cap) {
  return guard([&] {
    B2M_REQUIRE(ver && json && cap > 0, B2M_ERR_INVALID_ARG, "null argument");
    snprintf(json, cap, "%s", ver->impl->timings_json.c_str());
  });
}

}  // extern "C"
