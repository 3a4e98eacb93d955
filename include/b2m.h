/* b2m.h -- C ABI of the B200-native Marlin prover hot path.
 *
 * The reference (arkworks-rs/marlin) has no FFI; its seam is the generic parameter
 * `PC: PolynomialCommitment<F, DensePolynomial<F>>` of `Marlin<F, PC, FS>`
 * (reference src/lib.rs:64-71) and, one level down, the two upstream free functions every
 * commit/open and every AHP round bottoms out in.  Each entry point below names the
 * reference interface it replaces.  A Rust shim binding these (see INTEGRATION.md) turns the
 * library into a drop-in `PC` / prover backend.
 *
 * Conventions
 *   - Field elements cross the boundary exactly as ark-ff 0.3 stores them: little-endian
 *     u64 limbs in MONTGOMERY form (Fr: 4 limbs; Fq: 6 limbs for BLS12-381, 4 for BN254),
 *     except MSM scalars, which are canonical integers (`into_repr()`), as in
 *     `VariableBaseMSM::multi_scalar_mul(&[G::Affine], &[BigInt])`.
 *   - A G1 affine point is x||y (2*LQ u64 limbs, Montgomery); the point at infinity is
 *     encoded as x = y = 0 (never a curve point since b != 0).
 *   - Every function returns B2M_OK or an error code; b2m_last_error() gives the message.
 *     The library never aborts the host process and never falls back to the CPU.
 *   - A b2m_ctx owns one device and one stream; it is not thread-safe, distinct contexts
 *     are independent.  All calls are synchronous at return.
 */
#ifndef B2M_H
#define B2M_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  B2M_OK = 0,
  B2M_ERR_INVALID_ARG = 1,
  B2M_ERR_INDEX_TOO_LARGE = 2,          /* reference src/error.rs:7  Error::IndexTooLarge */
  B2M_ERR_INSTANCE_MISMATCH = 3,        /* reference src/ahp/mod.rs:276 InstanceDoesNotMatchIndex */
  B2M_ERR_INVALID_PUBLIC_INPUT_LEN = 4, /* reference src/ahp/mod.rs:274 InvalidPublicInputLength */
  B2M_ERR_NON_SQUARE = 5,               /* reference src/ahp/mod.rs:278 NonSquareMatrix */
  B2M_ERR_DEGREE_TOO_LARGE = 6,         /* SynthesisError::PolynomialDegreeTooLarge / PC degree errors */
  B2M_ERR_MISSING_RNG = 7,              /* [U ark-poly-commit Error::MissingRng] */
  B2M_ERR_CUDA = 8,
  B2M_ERR_NCCL = 9,
  B2M_ERR_UNSUPPORTED = 10
};

enum { B2M_CURVE_BLS12_381 = 0, B2M_CURVE_BN254 = 1 };
enum { B2M_PC_MARLIN_KZG10 = 0, B2M_PC_SONIC_KZG10 = 1 };
/* stream ciphers behind `RngCore`: rand 0.8 StdRng (= ChaCha12, `ark_std::test_rng`) and
 * rand_chacha::ChaChaRng (= ChaCha20). */
enum { B2M_RNG_CHACHA12 = 12, B2M_RNG_CHACHA20 = 20, B2M_RNG_CHACHA8 = 8,
       /* any other `RngCore`: the library pulls every random u64 through a host callback (b2m_rng::next_u64) */
       B2M_RNG_CALLBACK = 1 };

typedef struct b2m_ctx b2m_ctx;
typedef struct b2m_srs b2m_srs;
typedef struct b2m_ck b2m_ck;
typedef struct b2m_index b2m_index;

const char* b2m_last_error(void);
const char* b2m_version(void);

/* One context per GPU. */
int b2m_ctx_create(int device, b2m_ctx** out);
void b2m_ctx_destroy(b2m_ctx* ctx);
/* Number of kernel launches issued through this context so far. */
unsigned long long b2m_ctx_launches(const b2m_ctx* ctx);
/* Multi-GPU MSM (one process per GPU of one node): rank 0 obtains an NCCL unique id (128 bytes), the
 * caller broadcasts it, every rank attaches its context.  From then on every MSM issued through the
 * context is sharded by (base, scalar) chunk across the ranks and the partial sums are exchanged with one
 * all-gather; all ranks must issue the same sequence of calls. */
int b2m_comm_unique_id(uint8_t* id, size_t cap);
int b2m_ctx_attach_comm(b2m_ctx* ctx, const uint8_t* id, size_t id_len, int rank, int world);

/* Per-kernel device timing (CUDA events on the context's stream) for the dominant kernels: enable,
 * run, then read {"kernel": {"launches", "ms", "units"}} -- units are (base, scalar) pairs for the MSM
 * kernels and points for the NTT.  Reading the report clears it. */
int b2m_ctx_profile(b2m_ctx* ctx, int enable);
int b2m_ctx_profile_report(b2m_ctx* ctx, char* json, size_t cap);

/* ---- Level 0: kernel ABI ------------------------------------------------------------- */

/* Replaces `Radix2EvaluationDomain::{fft,ifft,coset_fft,coset_ifft}_in_place(&mut Vec<F>)`
 * [U ark-poly 0.3 domain/radix2]; call sites reference src/ahp/prover.rs:321-326,350-353,
 * 359,365,427,467,488,532-545,655,681,685.  `data` is a HOST buffer of 2^log_n Fr elements
 * (natural order in and out); inverse != 0 also scales by n^-1; coset != 0 uses the coset
 * g*H with g = F::multiplicative_generator(). */
int b2m_ntt(b2m_ctx* ctx, int curve, uint64_t* data, unsigned log_n, int inverse, int coset);

/* Replaces `VariableBaseMSM::multi_scalar_mul(bases, scalars)` [U ark-ec 0.3 msm/variable_base.rs].
 * One-shot form: uploads `bases`, builds the window tables, runs the MSM, frees everything.
 * out_xy receives the affine result (Montgomery), *out_is_inf is set for the identity. */
int b2m_msm_g1(b2m_ctx* ctx, int curve, const uint64_t* bases_xy, const uint64_t* scalars, size_t n,
               uint64_t* out_xy, int* out_is_inf);

/* Device-resident committer key: the G1 powers of `PC::UniversalParams` (what `PC::trim`,
 * reference src/lib.rs:115-121, slices).  powers_of_g: n_g affine points (beta^i G);
 * powers_of_gamma_g: n_gamma affine points beta^(gamma_indices[k]) gamma G used for hiding
 * (`UniversalParams::powers_of_gamma_g` is a BTreeMap<usize, G1Affine> upstream; Marlin's PC needs
 * indices 0..=2, Sonic's additionally max_degree - bound + 0..=2 per enforced bound);
 * gamma_indices == NULL means 0..n_gamma-1.  window_bits = 0 picks the window from n_g.  The library precomputes 2^(c*w) multiples of
 * every power (HBM for doublings) so every later MSM over any contiguous slice is one
 * bucket pass. */
int b2m_srs_create(b2m_ctx* ctx, int curve, const uint64_t* powers_of_g, size_t n_g,
                   const uint64_t* powers_of_gamma_g, const uint64_t* gamma_indices, size_t n_gamma,
                   int window_bits, b2m_srs** out);
void b2m_srs_destroy(b2m_srs* srs);
size_t b2m_srs_size(const b2m_srs* srs);
int b2m_srs_window_bits(const b2m_srs* srs);
/* Batched-affine levels the MSMs of this key run before the XYZZ bucket pass (0: none; MSMs with few bucket
 * references skip them regardless).  Diagnostic, like b2m_srs_window_bits. */
int b2m_srs_affine_levels(const b2m_srs* srs);
/* MSM over the slice powers_of_g[base_off .. base_off+n) with canonical host scalars. */
int b2m_srs_msm(b2m_srs* srs, size_t base_off, const uint64_t* scalars, size_t n, uint64_t* out_xy,
                int* out_is_inf);
/* SRS generation, the G1 half of `KZG10::setup` (reference src/lib.rs:79-96 -> [U ark-poly-commit kzg10::setup]):
 * b2m_g1_powers fills powers_of_g[i] = beta^i * g for i < n; b2m_fixed_base_msm is the general
 * `FixedBaseMSM::multi_scalar_mul(.., g, scalars)` [U ark-ec msm/fixed_base.rs] (out[i] = scalars[i] * g, e.g. the
 * powers_of_gamma_g at arbitrary exponents).  Both: one 8-bit window table of g, <= 32 mixed additions per scalar, batch
 * normalisation to affine.  beta and scalars are canonical Fr. */
int b2m_g1_powers(b2m_ctx* ctx, int curve, const uint64_t* g_xy, const uint64_t* beta, size_t n,
                  uint64_t* out_powers_xy);
int b2m_fixed_base_msm(b2m_ctx* ctx, int curve, const uint64_t* g_xy, const uint64_t* scalars, size_t n,
                       uint64_t* out_xy);

/* G2 half of `KZG10::setup` [U ark-poly-commit kzg10::setup: h, beta_h, neg_powers_of_h]: out[i] = scalars[i] * h, written as
 * ark-serialize `serialize_uncompressed` bytes (4 * sizeof(Fq) per point, infinity flag in the last byte).  h_uncompressed:
 * the G2 base in the same byte form, or NULL for the curve's standard G2 generator.  Host-side (the prover never touches G2;
 * a key needs 2 + #degree-bounds of these), no b2m_ctx needed. */
int b2m_g2_scalar_muls(int curve, const uint8_t* h_uncompressed, const uint64_t* scalars, size_t n, uint8_t* out);

/* G1 points between the device and ark-serialize files: powers_of_g[first .. first + n) of a resident SRS as
 * `serialize_uncompressed` bytes (2 * sizeof(Fq) per point: canonical little-endian x || y, infinity flag = bit 6 of the last
 * byte), and the inverse conversion of such bytes to the affine Montgomery limbs b2m_srs_create takes (no curve / subgroup
 * check: like `deserialize_unchecked`).  Conversions run on the GPU. */
int b2m_srs_export_g1(b2m_srs* srs, size_t first, size_t n, uint8_t* out);
int b2m_g1_from_uncompressed(b2m_ctx* ctx, int curve, const uint8_t* bytes, size_t n, uint64_t* out_xy);
int b2m_g1_to_uncompressed(b2m_ctx* ctx, int curve, const uint64_t* points_xy, size_t n, uint8_t* out);

/* The caller's `zk_rng: &mut R` / `rng: Option<&mut dyn RngCore>` (reference src/lib.rs:154,125).  Two forms:
 *  - kind = B2M_RNG_CHACHA8/12/20, the fast path for the generators the reference's tests and benches use
 *    (`ark_std::test_rng()` = ChaCha12, `rand_chacha::ChaChaRng` = ChaCha20): the stream is described by its key and
 *    word position, so the mask polynomial (3|H| draws, src/ahp/prover.rs:371) is sampled on the device bit-exactly;
 *    word_pos is updated to the position after the call.
 *  - kind = B2M_RNG_CALLBACK, any other generator: every `next_u64()` the reference would issue is pulled, in the
 *    reference's order, through `next_u64(state)` on the calling thread (a Rust shim passes a trampoline over
 *    `&mut dyn RngCore`); the mask polynomial is then drawn on the host and uploaded once.  key / word_pos are unused.
 * Draw order and counts are those of ark-ff 0.3 `F::rand` (4 u64 limbs per attempt, low limb first, rejection sampling). */
typedef struct {
  int kind;          /* B2M_RNG_CHACHA* or B2M_RNG_CALLBACK */
  uint8_t key[32];
  uint64_t word_pos; /* number of 32-bit words already consumed from the stream */
  uint64_t (*next_u64)(void* state); /* B2M_RNG_CALLBACK only */
  void* state;
} b2m_rng;

/* ---- Level 1: polynomial-commitment ABI --------------------------------------------------------- */

/* Replaces `PC::commit(ck, polynomials, rng)` for PC = MarlinKZG10 / SonicKZG10 [U ark-poly-commit 0.3
 * marlin_pc/mod.rs, sonic_pc/mod.rs commit -> kzg10::KZG10::commit]; call sites reference
 * src/lib.rs:125,172,193,213.  Polynomials are host coefficient arrays (Montgomery Fr, low degree first)
 * committed in order with the blinding polynomials drawn from `rng` exactly as the reference does
 * (hiding_bound h draws h + 2 coefficients; MarlinKZG10 draws a second set for the shifted commitment).
 *   degree_bounds[i] / hiding_bounds[i] : -1 for None.
 *   out_comm_xy[i]      affine commitment; out_shifted_xy[i]: MarlinKZG10 shifted commitment of a bounded
 *                        polynomial (all-zero when absent; unused for SonicKZG10).
 *   out_rand / out_shifted_rand : blinding polynomial coefficients, rand_stride Fr per polynomial (zero padded).
 * rng may be NULL when no polynomial is hiding (B2M_ERR_MISSING_RNG otherwise). */
int b2m_pc_commit(b2m_srs* srs, int pc_variant, size_t n_polys, const uint64_t* const* coeffs,
                  const size_t* n_coeffs, const int64_t* degree_bounds, const int64_t* hiding_bounds,
                  b2m_rng* rng, uint64_t* out_comm_xy, uint64_t* out_shifted_xy, uint64_t* out_rand,
                  uint64_t* out_shifted_rand, size_t rand_stride);

/* Replaces `PC::open_individual_opening_challenges(ck, polynomials, commitments, point, challenges, rands)`
 * for one point [U ark-poly-commit 0.3 marlin_pc/mod.rs, sonic_pc/mod.rs -> kzg10::KZG10::open], the call the
 * generic `open_combinations` / `batch_open` code ends in (reference src/lib.rs:292-302).  Polynomials and their
 * commitment randomness are given in query order; challenge k is opening_challenge^k starting at k = 0
 * (MarlinKZG10 spends a second challenge on every degree-bounded polynomial).  max_degree_bound: the largest
 * enforced bound of the committer key (MarlinKZG10 shifted powers), -1 if none.
 * Output: the `kzg10::Proof { w, random_v }`. */
int b2m_pc_open(b2m_srs* srs, int pc_variant, size_t n_polys, const uint64_t* const* coeffs,
                const size_t* n_coeffs, const int64_t* degree_bounds, const uint64_t* rands,
                const uint64_t* shifted_rands, size_t rand_stride, int64_t max_degree_bound,
                const uint64_t* point, const uint64_t* opening_challenge, uint64_t* out_w_xy,
                int* out_has_random_v, uint64_t* out_random_v);

/* Replaces `PC::trim(pp, supported_degree, supported_hiding_bound, enforced_degree_bounds)` (reference src/lib.rs:112-121)
 * for PC = MarlinKZG10 / SonicKZG10 [U ark-poly-commit 0.3 marlin_pc/mod.rs, sonic_pc/mod.rs trim].  The device-resident
 * SRS already holds every power, so trimming selects and validates: supported_degree <= max_degree, the hiding bound needs
 * powers 0..=supported_hiding_bound+1 of gamma*G (SonicKZG10 additionally max_degree - bound + 0..=hiding_bound+1 per enforced
 * bound), every enforced bound <= supported_degree.  The committer key borrows the SRS (destroy the key first).
 * Errors: B2M_ERR_DEGREE_TOO_LARGE (TrimmingDegreeTooLarge / bound above the supported degree), B2M_ERR_INVALID_ARG. */
int b2m_trim(b2m_srs* srs, int pc_variant, size_t supported_degree, size_t supported_hiding_bound,
             const uint64_t* enforced_degree_bounds, size_t n_bounds, b2m_ck** out);
void b2m_ck_destroy(b2m_ck* ck);
size_t b2m_ck_supported_degree(const b2m_ck* ck);
/* `vk.degree_bounds_and_shift_powers` of MarlinKZG10's verifier key: shift power for an enforced bound =
 * powers_of_g[max_degree - bound] (affine x||y Montgomery).  B2M_ERR_INVALID_ARG if the bound is not enforced. */
int b2m_ck_shift_power(const b2m_ck* ck, uint64_t bound, uint64_t* out_xy);
/* `PC::commit(ck, ..)` with the committer key's checks [U ark-poly-commit check_degrees_and_bounds]: a polynomial longer than
 * supported_degree + 1 coefficients, a degree bound that is not one of the enforced bounds (or below the polynomial's degree)
 * or a hiding bound above the supported one fail with B2M_ERR_DEGREE_TOO_LARGE / B2M_ERR_INVALID_ARG.  Otherwise identical
 * to b2m_pc_commit. */
int b2m_ck_commit(b2m_ck* ck, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs,
                  const int64_t* degree_bounds, const int64_t* hiding_bounds, b2m_rng* rng, uint64_t* out_comm_xy,
                  uint64_t* out_shifted_xy, uint64_t* out_rand, uint64_t* out_shifted_rand, size_t rand_stride);

/* Replaces `PC::open_combinations(ck, lc_s, polynomials, commitments, query_set, opening_challenge, rands, rng)`
 * (reference src/lib.rs:292-302) [U ark-poly-commit 0.3 marlin_pc / sonic_pc open_combinations_individual_opening_challenges].
 *   polynomials / rands       : as for b2m_pc_commit / b2m_pc_open (hiding[i] != 0 iff polynomial i was committed hiding).
 *   linear combinations       : LC l has the terms [lc_term_off[l], lc_term_off[l+1]); term t is lc_coeff[t] (Montgomery Fr)
 *                               times polynomial lc_poly[t], or the constant `LCTerm::One` when lc_poly[t] < 0 (which only
 *                               shifts the evaluation and is skipped, as upstream does).  The caller passes the LCs in the
 *                               order of their labels (upstream sorts them, reference src/ahp/mod.rs:219).  An LC may carry a
 *                               degree bound only if it is a single polynomial with coefficient one
 *                               (else B2M_ERR_INVALID_ARG: EquationHasDegreeBounds).
 *   query set                 : pairs (query_lc[q], query_point[q]); points[] are the distinct evaluation points in the order
 *                               of their point labels (upstream iterates a BTreeMap keyed by the label: "beta" < "gamma").
 *   opening challenge         : xi; challenge k is xi^k, restarting at k = 0 for every point.
 * Output: one `kzg10::Proof {w, random_v}` per point -- `BatchLCProof.proof` (its `evals` field is None upstream). */
int b2m_ck_open_combinations(b2m_ck* ck, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs,
                             const int64_t* degree_bounds, const int* hiding, const uint64_t* rands,
                             const uint64_t* shifted_rands, size_t rand_stride, size_t n_lcs, const size_t* lc_term_off,
                             const int64_t* lc_poly, const uint64_t* lc_coeff, size_t n_queries, const size_t* query_lc,
                             const size_t* query_point, size_t n_points, const uint64_t* points,
                             const uint64_t* opening_challenge, uint64_t* out_w_xy, int* out_has_random_v,
                             uint64_t* out_random_v);

/* ---- Level 2: prover ABI ---------------------------------------------------------------- */

/* R1CS matrix in CSR form, as `ConstraintSystem::to_matrices()` yields it
 * (reference src/ahp/indexer.rs:81 `Matrix<F> = Vec<Vec<(F, usize)>>`): row r holds entries
 * [row_ptr[r], row_ptr[r+1]); coeff is Montgomery Fr (4 u64 each). */
typedef struct {
  const uint64_t* row_ptr; /* num_constraints + 1 */
  const uint64_t* col;     /* nnz column (variable) indices */
  const uint64_t* coeff;   /* nnz * 4 limbs */
} b2m_matrix;

/* Replaces `Marlin::index` (reference src/lib.rs:100-148): AHP indexer
 * (src/ahp/indexer.rs:151-234, src/ahp/constraint_systems.rs:125-262) + `PC::trim` +
 * commitment to the six index polynomials.  The matrices must already be padded/squared
 * (num_constraints == num_variables) as `make_matrices_square_for_indexer` leaves them.
 * vk_bytes receives `IndexVerifierKey::write` (ToBytes) output: index_info || index_comms. */
int b2m_index_create(b2m_srs* srs, int pc_variant, size_t num_constraints, size_t num_variables,
                     size_t num_instance_variables, const b2m_matrix* a, const b2m_matrix* b,
                     const b2m_matrix* c, b2m_index** out);
void b2m_index_destroy(b2m_index* idx);
/* Serialized `index_vk` as the transcript sees it (ToBytes, reference src/data_structures.rs:36-43). */
int b2m_index_vk_bytes(const b2m_index* idx, uint8_t* out, size_t cap, size_t* len);
/* Commitments to the index polynomials (affine x||y Montgomery, 6 points). */
int b2m_index_comms(const b2m_index* idx, uint64_t* out_xy);


/* Replaces `Marlin::prove` (reference src/lib.rs:151-311).  formatted_input: the instance
 * assignment including the leading one (|X| elements); witness: the witness assignment
 * (num_variables - |X| elements), both Montgomery Fr.  proof receives the
 * `CanonicalSerialize` bytes of `Proof<F, PC>` (reference src/data_structures.rs:100-110). */
int b2m_prove(b2m_index* idx, const uint64_t* formatted_input, size_t n_input,
              const uint64_t* witness, size_t n_witness, b2m_rng* zk_rng, uint8_t* proof,
              size_t cap, size_t* proof_len);

/* Copy an instance into HBM ahead of time.  A later b2m_prove(idx, NULL, 0, NULL, 0, ...) proves the
 * staged instance without any host-to-device input traffic (bench.py's device-resident timing). */
int b2m_index_stage(b2m_index* idx, const uint64_t* formatted_input, size_t n_input,
                    const uint64_t* witness, size_t n_witness);

/* Per-phase device timings of the last b2m_prove on this index (milliseconds), labelled
 * with the reference's own timer names (ark_std start_timer! labels, SURVEY.md section 5). */
int b2m_prove_timings(const b2m_index* idx, char* json, size_t cap);

/* ---- Level 3: verifier ABI -------------------------------------------------------------- */

/* Per-proof outcome of b2m_verify. */
enum { B2M_VERDICT_ACCEPT = 0, B2M_VERDICT_REJECT = 1, B2M_VERDICT_MALFORMED = 2 };

typedef struct b2m_verifier b2m_verifier;

/* The verifier key of `Marlin::verify` (reference src/lib.rs:315-433), device resident: the index_vk ToBytes image (what
 * b2m_index_vk_bytes returns; absorbed verbatim by the transcript) plus the PC verifier key [U ark-poly-commit marlin_pc /
 * sonic_pc VerifierKey]: g, gamma_g (G1) and h, beta_h (G2) as ark-serialize `serialize_uncompressed` bytes, the SRS's
 * max_degree and the enforced degree bounds with, per bound, the MarlinKZG10 shift power powers_of_g[max_degree - bound] (G1,
 * 2 * sizeof(Fq) bytes) or the SonicKZG10 beta^-(max_degree - bound) h (G2, 4 * sizeof(Fq) bytes), uncompressed, concatenated.
 * h and beta_h are prepared once (Miller-loop line coefficients).  Errors: B2M_ERR_NON_SQUARE, B2M_ERR_DEGREE_TOO_LARGE
 * (the index needs a larger supported degree), B2M_ERR_INVALID_ARG (a degree bound the index needs is not enforced --
 * EquationHasDegreeBounds --, malformed bytes).  The verifier borrows the context. */
int b2m_verifier_create(b2m_ctx* ctx, int curve, int pc_variant, const uint8_t* vk_tobytes, size_t vk_len, const uint8_t* g,
                        const uint8_t* gamma_g, const uint8_t* h, const uint8_t* beta_h, size_t max_degree, size_t n_bounds,
                        const uint64_t* bounds, const uint8_t* bound_points, b2m_verifier** out);
void b2m_verifier_destroy(b2m_verifier* ver);

/* `Marlin::verify` for n_proofs proofs of the verifier's index.  public_inputs[i]: n_inputs[i] Montgomery Fr (4 u64 each),
 * without the leading one (as `R1CS.public_input()`); proofs[i]: `CanonicalSerialize` bytes of `Proof<F, PC>`.  rng supplies
 * the 128-bit randomisers of the batched check [U ark-poly-commit check_combinations(.., rng)]: two per proof, then one per
 * proof for the batch fold.  verdicts[i] = B2M_VERDICT_ACCEPT / REJECT / MALFORMED (unparsable bytes, a point off the curve or
 * outside the prime-order subgroup, an evaluation >= r); a proof never affects another's verdict.  The return code is not
 * B2M_OK only for misuse (null arguments, an unreduced public input) or CUDA errors. */
int b2m_verify(b2m_verifier* ver, size_t n_proofs, const uint64_t* const* public_inputs, const size_t* n_inputs,
               const uint8_t* const* proofs, const size_t* proof_lens, b2m_rng* rng, int* verdicts);
/* Per-stage times of the last b2m_verify (milliseconds; device stages from CUDA events, "transcript" on the host). */
int b2m_verify_timings(const b2m_verifier* ver, char* json, size_t cap);

#ifdef __cplusplus
}
#endif
#endif /* B2M_H */
