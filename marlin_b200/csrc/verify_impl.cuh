// Batch verifier: `Marlin::verify` [reference src/lib.rs:315-433, src/ahp/verifier.rs, src/ahp/mod.rs:110-221] for many proofs of
// one index, with every per-proof step after the transcript on the device and one pairing product for the whole batch.
//
// Stages of verify() (timings_json reports each):
//   decode      one thread per compressed G1 point of every proof (verify_core.cuh g1_decompress)
//   transcript  Fiat-Shamir replay per proof on a pool of host threads (hostutil.hpp, the prover's ToBytes serialisation)
//   scalars     one thread per proof: x_hat(beta), the LC coefficients and the N_TERMS combination scalars (verify_core.cuh)
//   combine     one thread per (proof, term) scalar multiplication, then one per (proof, slot) sum: the per-proof points
//               A_i (paired with h), B_i (with beta h) and, SonicKZG10, C_i,d (with beta^-(D-d) h)
//   fold        sum_i r_i A_i, sum_i r_i B_i, sum_i r_i C_i,d with fresh 128-bit r_i
//   pairing     one multi-pairing of the folded points against the prepared G2 bases; only if it is not 1, the same kernel runs
//               once more with one product per proof for exact verdicts
// The caller's rng supplies, in this order, rho_beta and rho_gamma of every proof (two u64 each), then r_i of every proof.
#pragma once
#include <chrono>
#include <thread>

#include "pairing.cuh"
#include "prover_impl.cuh"
#include "verify.cuh"
#include "verify_core.cuh"

namespace b2m {

constexpr int VER_MAX_SLOTS = 4;   // A, B and at most two SonicKZG10 bounds (|H| - 2, |K| - 2)
constexpr int VER_FOLD_THREADS = 64;

struct DestMap {
  int8_t d[N_TERMS];
};

template <class Fq, class Fr>
__global__ void ver_decode_kernel(const uint8_t* bytes, const uint8_t* present, size_t n, Affine<Fq>* out, uint8_t* status) {
  constexpr int NB = (Fq::Params::BITS + 2 + 7) / 8;
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Affine<Fq> p = Affine<Fq>::inf();
  int s = DEC_OK;
  if (present[i]) s = g1_decompress<Fq, Fr>(bytes + i * NB, &p);
  out[i] = p;
  status[i] = (uint8_t)s;
}

template <class Fr>
__global__ void ver_scalars_kernel(const ProofScalars<Fr>* ps, const Fr* formatted, const uint32_t* n_x, size_t stride, const uint8_t* live,
                                   size_t n, bool marlin, uint64_t h, uint64_t k, Fr* out) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr s[N_TERMS];
  if (live[i]) {
    ProofScalars<Fr> p = ps[i];
    p.x_beta = lagrange_eval(formatted + i * stride, n_x[i], p.ch.beta);
    term_scalars(p, marlin, h, k, n_x[i], s);
    for (int t = 0; t < N_TERMS; t++) s[t] = s[t].to_canonical();
  } else {
    for (int t = 0; t < N_TERMS; t++) s[t] = Fr::zero();
  }
  for (int t = 0; t < N_TERMS; t++) out[i * N_TERMS + t] = s[t];
}

template <class Fq, class Fr>
__global__ void ver_term_kernel(const Affine<Fq>* pts, const Affine<Fq>* bases, const Fr* sc, size_t n, XYZZ<Fq>* out) {
  const size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (g >= n * N_TERMS) return;
  const size_t i = g / N_TERMS;
  const int t = (int)(g % N_TERMS);
  const Affine<Fq> b = t < N_PROOF_POINTS ? pts[i * N_PROOF_POINTS + t]
                       : t < T_WB_B      ? bases[t - N_PROOF_POINTS]
                                         : pts[i * N_PROOF_POINTS + (t == T_WB_B ? T_WB : T_WG)];
  out[g] = scalar_mul<Fq>(b, sc[g].l, Fr::N);
}

template <class Fq>
__global__ void ver_sum_kernel(const XYZZ<Fq>* terms, DestMap dest, int ns, size_t n, Affine<Fq>* out) {
  const size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (g >= n * ns) return;
  const size_t i = g / ns;
  const int s = (int)(g % ns);
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  for (int t = 0; t < N_TERMS; t++)
    if (dest.d[t] == s) acc.add(terms[i * N_TERMS + t]);
  out[g] = acc.to_affine();
}

template <class Fq>
__global__ void ver_fold_scale_kernel(const Affine<Fq>* pts, const uint32_t* r, int ns, size_t n, XYZZ<Fq>* out) {
  const size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (g >= n * ns) return;
  out[g] = scalar_mul<Fq>(pts[g], r + 4 * (g / ns), 4);
}

// one block per slot
template <class Fq>
__global__ void ver_fold_reduce_kernel(const XYZZ<Fq>* in, int ns, size_t n, Affine<Fq>* out) {
  __shared__ XYZZ<Fq> sh[VER_FOLD_THREADS];
  const int s = blockIdx.x;
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  for (size_t i = threadIdx.x; i < n; i += blockDim.x) acc.add(in[i * ns + s]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int w = VER_FOLD_THREADS / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) {
      XYZZ<Fq> a = sh[threadIdx.x];
      a.add(sh[threadIdx.x + w]);
      sh[threadIdx.x] = a;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) out[s] = sh[0].to_affine();
}

// one thread per product prod_s e(pts[j * ns + s], Q_s) against the prepared Q_s
template <class Fq>
__global__ void ver_pairing_kernel(const Affine<Fq>* pts, const EllCoeff<Fq>* coeffs, int ns, size_t n_prod, uint8_t* is_one) {
  const size_t j = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (j >= n_prod) return;
  Fq px[VER_MAX_SLOTS], py[VER_MAX_SLOTS];
  bool inf[VER_MAX_SLOTS];
  const EllCoeff<Fq>* cp[VER_MAX_SLOTS];
  for (int s = 0; s < ns; s++) {
    const Affine<Fq> p = pts[j * ns + s];
    inf[s] = p.is_inf();
    px[s] = p.x;
    py[s] = p.y;
    cp[s] = coeffs + (size_t)s * n_ell_coeffs<Fq>();
  }
  is_one[j] = final_exponentiation(miller_loop<Fq>(ns, px, py, inf, cp)).is_one() ? 1 : 0;
}

template <class Fr, class Fq>
struct MarlinVerifier : VerifierBase {
  using Pt = Affine<Fq>;
  using M = MarlinIndex<Fr, Fq>;
  static constexpr int NB = (Fq::Params::BITS + 2 + 7) / 8;  // compressed G1
  static constexpr int FQ_BYTES = Fq::N * 4;
  static constexpr int FR_BYTES = Fr::N * 4;
  static constexpr int L = n_ell_coeffs<Fq>();

  Ctx& cx;
  int pc;
  bool marlin;
  std::vector<uint8_t> vk_bytes;
  uint64_t H = 0, K = 0;
  int ns = 2;
  DestMap dest;
  DBuf<Pt> bases;                // index comms (row, col, a_val, b_val, c_val, row_col), g, gamma_g, shift(|H|-2), shift(|K|-2)
  DBuf<EllCoeff<Fq>> prepared;   // ns x L: h, beta_h, SonicKZG10 beta^-(D-d) h

  // ---- ark-serialize helpers ------------------------------------------------------------------------------------
  template <class F>
  static bool canon_from_le(const uint8_t* b, int nbytes, F* out) {  // canonical < modulus -> Montgomery
    F c = F::zero();
    for (int i = 0; i < nbytes; i++) c.l[i >> 2] |= (uint32_t)b[i] << (8 * (i & 3));
    for (int i = F::N - 1; i >= 0; i--) {
      if (c.l[i] != F::Params::mod(i)) {
        if (c.l[i] > F::Params::mod(i)) return false;
        break;
      }
      if (i == 0) return false;
    }
    *out = F::from_canonical(c);
    return true;
  }
  static Pt g1_uncompressed(const uint8_t* b, const char* what) {  // x || y, infinity flag = bit 6 of the last byte
    if (b[2 * FQ_BYTES - 1] & 0x40) return Pt::inf();
    uint8_t y[FQ_BYTES];
    memcpy(y, b + FQ_BYTES, FQ_BYTES);
    y[FQ_BYTES - 1] &= 0x3f;
    Pt p;
    B2M_REQUIRE(canon_from_le(b, FQ_BYTES, &p.x) && canon_from_le(y, FQ_BYTES, &p.y), B2M_ERR_INVALID_ARG, "%s: coordinate out of range", what);
    B2M_REQUIRE(p.y.sqr() == p.x.sqr() * p.x + Fq::from_u64(FQ_BYTES == 48 ? 4 : 3), B2M_ERR_INVALID_ARG, "%s is not on the curve", what);
    return p;
  }
  static G2Aff<Fq> g2_uncompressed(const uint8_t* b, const char* what) {  // x.c0 || x.c1 || y.c0 || y.c1
    B2M_REQUIRE(!(b[4 * FQ_BYTES - 1] & 0x40), B2M_ERR_INVALID_ARG, "%s is the point at infinity", what);
    uint8_t last[FQ_BYTES];
    memcpy(last, b + 3 * FQ_BYTES, FQ_BYTES);
    last[FQ_BYTES - 1] &= 0x3f;
    G2Aff<Fq> q;
    q.inf = false;
    B2M_REQUIRE(canon_from_le(b, FQ_BYTES, &q.x.c0) && canon_from_le(b + FQ_BYTES, FQ_BYTES, &q.x.c1) &&
                    canon_from_le(b + 2 * FQ_BYTES, FQ_BYTES, &q.y.c0) && canon_from_le(last, FQ_BYTES, &q.y.c1),
                B2M_ERR_INVALID_ARG, "%s: coordinate out of range", what);
    B2M_REQUIRE(q.y.sqr() == q.x.sqr() * q.x + twist_b<Fq>(), B2M_ERR_INVALID_ARG, "%s is not on the twist", what);
    return q;
  }
  static uint64_t pow2_at_least(uint64_t n) {
    uint64_t s = 1;
    while (s < n) s <<= 1;
    return s;
  }

  MarlinVerifier(Ctx& c, int pc_, const uint8_t* vk, size_t vk_len, const uint8_t* g, const uint8_t* gamma_g, const uint8_t* h,
                 const uint8_t* beta_h, size_t max_degree, size_t n_bounds, const uint64_t* bounds, const uint8_t* bound_points)
      : cx(c), pc(pc_), marlin(pc_ == B2M_PC_MARLIN_KZG10) {
    const size_t comm_len = marlin ? 2 * (2 * FQ_BYTES + 1) + 1 : 2 * FQ_BYTES + 1;
    B2M_REQUIRE(vk && vk_len == 24 + 6 * comm_len, B2M_ERR_INVALID_ARG, "index_vk is %zu bytes, expected %zu", vk_len, 24 + 6 * comm_len);
    vk_bytes.assign(vk, vk + vk_len);
    uint64_t info[3];
    memcpy(info, vk, 24);
    const uint64_t nv = info[0], nc = info[1], nnz = info[2];
    B2M_REQUIRE(nc == nv, B2M_ERR_NON_SQUARE, "index_vk: %llu constraints, %llu variables", (unsigned long long)nc, (unsigned long long)nv);
    H = pow2_at_least(nc);
    K = pow2_at_least(nnz);
    B2M_REQUIRE(H >= 2 && K >= 2 && H <= (1ull << Fr::Params::TWO_ADICITY) && K <= (1ull << Fr::Params::TWO_ADICITY), B2M_ERR_INVALID_ARG,
                "index_vk: unsupported domain sizes");
    const uint64_t supported = std::max(std::max(2 * H - 1, 3 * H - 1), K - 1);  // AHPForR1CS::max_degree
    B2M_REQUIRE(supported <= max_degree, B2M_ERR_DEGREE_TOO_LARGE, "the index needs degree %llu, the key supports %zu",
                (unsigned long long)supported, max_degree);
    int bi_h = -1, bi_k = -1;
    for (size_t i = 0; i < n_bounds; i++) {
      B2M_REQUIRE(bounds[i] <= max_degree, B2M_ERR_DEGREE_TOO_LARGE, "degree bound %llu above the maximum degree", (unsigned long long)bounds[i]);
      if (bounds[i] == H - 2) bi_h = (int)i;
      if (bounds[i] == K - 2) bi_k = (int)i;
    }
    B2M_REQUIRE(bi_h >= 0 && bi_k >= 0, B2M_ERR_INVALID_ARG, "the key does not enforce the degree bounds %llu and %llu the index needs",
                (unsigned long long)(H - 2), (unsigned long long)(K - 2));
    std::vector<Pt> b(10, Pt::inf());
    for (int i = 0; i < 6; i++) {
      const uint8_t* p = vk + 24 + i * comm_len;
      const uint8_t inf = p[2 * FQ_BYTES];
      if (!inf) {
        B2M_REQUIRE(canon_from_le(p, FQ_BYTES, &b[i].x) && canon_from_le(p + FQ_BYTES, FQ_BYTES, &b[i].y), B2M_ERR_INVALID_ARG,
                    "index commitment %d out of range", i);
      }
    }
    b[6] = g1_uncompressed(g, "g");
    b[7] = g1_uncompressed(gamma_g, "gamma_g");
    std::vector<G2Aff<Fq>> q = {g2_uncompressed(h, "h"), g2_uncompressed(beta_h, "beta_h")};
    for (int t = 0; t < N_TERMS; t++) dest.d[t] = 0;
    dest.d[T_WB_B] = dest.d[T_WG_B] = 1;
    if (marlin) {
      b[8] = g1_uncompressed(bound_points + (size_t)bi_h * 2 * FQ_BYTES, "shift power");
      b[9] = g1_uncompressed(bound_points + (size_t)bi_k * 2 * FQ_BYTES, "shift power");
    } else {
      q.push_back(g2_uncompressed(bound_points + (size_t)bi_h * 4 * FQ_BYTES, "neg power of h"));
      dest.d[T_G1] = 2;
      if (bi_k != bi_h) q.push_back(g2_uncompressed(bound_points + (size_t)bi_k * 4 * FQ_BYTES, "neg power of h"));
      dest.d[T_G2] = bi_k != bi_h ? 3 : 2;
    }
    ns = (int)q.size();
    std::vector<EllCoeff<Fq>> coeffs((size_t)ns * L);
    for (int s = 0; s < ns; s++) g2_prepare(q[s], coeffs.data() + (size_t)s * L);
    bases = DBuf<Pt>(cx, 10);
    bases.upload(b.data(), 10);
    prepared = DBuf<EllCoeff<Fq>>(cx, coeffs.size());
    prepared.upload(coeffs.data(), coeffs.size());
    cx.sync();
  }

  // ---- proof layout (`Proof::deserialize`, the inverse of MarlinIndex::prove's tail) ----------------------------
  struct Parsed {
    bool ok = false;
    uint8_t comp[N_PROOF_POINTS][NB];
    uint8_t present[N_PROOF_POINTS];
    Fr evals[4];
    const uint8_t* eval_bytes = nullptr;
    Fr rv[2];
  };
  struct Cursor {
    const uint8_t* p;
    size_t left;
    bool take(size_t n, const uint8_t** out) {
      if (left < n) return false;
      *out = p;
      p += n;
      left -= n;
      return true;
    }
    bool u64(uint64_t* v) {
      const uint8_t* b;
      if (!take(8, &b)) return false;
      memcpy(v, b, 8);
      return true;
    }
    bool byte(uint8_t* v) {
      const uint8_t* b;
      if (!take(1, &b)) return false;
      *v = *b;
      return true;
    }
  };
  bool parse(const uint8_t* bytes, size_t len, Parsed& out) const {
    if (!bytes) return false;
    Cursor c{bytes, len};
    uint64_t v;
    uint8_t flag;
    const uint8_t* b;
    memset(out.present, 0, sizeof(out.present));
    // round r's commitments land in these slots; the bounded ones (g_1, g_2) carry MarlinKZG10's shifted commitment
    static const int slots[3][4] = {{T_W, T_ZA, T_ZB, T_MASK}, {T_T, T_G1, T_H1, -1}, {T_G2, T_H2, -1, -1}};
    static const int counts[3] = {4, 3, 2};
    if (!c.u64(&v) || v != 3) return false;
    for (int r = 0; r < 3; r++) {
      if (!c.u64(&v) || v != (uint64_t)counts[r]) return false;
      for (int k = 0; k < counts[r]; k++) {
        const int s = slots[r][k];
        if (!c.take(NB, &b)) return false;
        memcpy(out.comp[s], b, NB);
        out.present[s] = 1;
        if (marlin) {
          const bool bounded = s == T_G1 || s == T_G2;
          if (!c.byte(&flag) || flag != (bounded ? 1 : 0)) return false;
          if (bounded) {
            const int sh = s == T_G1 ? T_SG1 : T_SG2;
            if (!c.take(NB, &b)) return false;
            memcpy(out.comp[sh], b, NB);
            out.present[sh] = 1;
          }
        }
      }
    }
    if (!c.u64(&v) || v != 4) return false;
    if (!c.take(4 * FR_BYTES, &out.eval_bytes)) return false;
    for (int i = 0; i < 4; i++)
      if (!canon_from_le(out.eval_bytes + i * FR_BYTES, FR_BYTES, &out.evals[i])) return false;
    if (!c.u64(&v) || v != 3) return false;
    for (int i = 0; i < 3; i++)
      if (!c.byte(&flag) || flag != 0) return false;  // ProverMsg::EmptyMessage
    if (!c.u64(&v) || v != 2) return false;
    for (int p = 0; p < 2; p++) {
      const int s = p == 0 ? T_WB : T_WG;
      if (!c.take(NB, &b)) return false;
      memcpy(out.comp[s], b, NB);
      out.present[s] = 1;
      out.rv[p] = Fr::zero();
      if (!c.byte(&flag) || flag > 1) return false;
      if (flag) {
        if (!c.take(FR_BYTES, &b) || !canon_from_le(b, FR_BYTES, &out.rv[p])) return false;
      }
    }
    if (!c.byte(&flag) || flag != 0) return false;  // BatchLCProof.evals = None
    out.ok = c.left == 0;
    return out.ok;
  }

  // ---- transcript --------------------------------------------------------------------------------------------
  Fr sample_outside_h(FiatShamir& fs) const {
    for (;;) {
      Fr t = field_rand<Fr>(fs);
      if (t.pow_u64(H) != Fr::one()) return t;
    }
  }
  void put_comm(std::vector<uint8_t>& out, const Pt* pts, int slot) const {
    M::put_affine_tobytes(out, pts[slot]);
    if (!marlin) return;
    const int sh = slot == T_G1 ? T_SG1 : slot == T_G2 ? T_SG2 : -1;
    out.push_back(sh >= 0 ? 1 : 0);
    M::put_affine_tobytes(out, sh >= 0 ? pts[sh] : Pt::inf());
  }
  void transcript(const Fr* formatted, uint64_t n_x, const Pt* pts, const Parsed& pr, ProofScalars<Fr>& ps) const {
    static const char name[] = "MARLIN-2019";
    std::vector<uint8_t> init(name, name + sizeof(name) - 1);
    init.insert(init.end(), vk_bytes.begin(), vk_bytes.end());
    for (uint64_t i = 1; i < n_x; i++) M::put_fr_canonical(init, formatted[i]);
    FiatShamir fs(init);
    std::vector<uint8_t> bytes;
    for (int s : {T_W, T_ZA, T_ZB, T_MASK}) put_comm(bytes, pts, s);
    fs.absorb(bytes);
    ps.ch.alpha = sample_outside_h(fs);
    ps.ch.eta_a = field_rand<Fr>(fs);
    ps.ch.eta_b = field_rand<Fr>(fs);
    ps.ch.eta_c = field_rand<Fr>(fs);
    bytes.clear();
    for (int s : {T_T, T_G1, T_H1}) put_comm(bytes, pts, s);
    fs.absorb(bytes);
    ps.ch.beta = sample_outside_h(fs);
    bytes.clear();
    for (int s : {T_G2, T_H2}) put_comm(bytes, pts, s);
    fs.absorb(bytes);
    ps.ch.gamma = field_rand<Fr>(fs);
    fs.absorb(std::vector<uint8_t>(pr.eval_bytes, pr.eval_bytes + 4 * FR_BYTES));
    const uint64_t lo = fs.next_u64(), hi = fs.next_u64();  // F::from(u128::rand(fs_rng))
    Fr c = Fr::zero();
    c.l[0] = (uint32_t)lo; c.l[1] = (uint32_t)(lo >> 32); c.l[2] = (uint32_t)hi; c.l[3] = (uint32_t)(hi >> 32);
    ps.xi = Fr::from_canonical(c);
    for (int i = 0; i < 4; i++) ps.evals[i] = pr.evals[i];
    ps.rv[0] = pr.rv[0];
    ps.rv[1] = pr.rv[1];
  }

  struct Events {
    Ctx& cx;
    std::vector<std::pair<const char*, std::pair<cudaEvent_t, cudaEvent_t>>> ev;
    explicit Events(Ctx& c) : cx(c) {}
    ~Events() {
      for (auto& e : ev) { cudaEventDestroy(e.second.first); cudaEventDestroy(e.second.second); }
    }
    size_t begin(const char* name) {
      cudaEvent_t a, b;
      B2M_CUDA(cudaEventCreate(&a));
      B2M_CUDA(cudaEventCreate(&b));
      B2M_CUDA(cudaEventRecord(a, cx.stream));
      ev.push_back({name, {a, b}});
      return ev.size() - 1;
    }
    void end(size_t i) { B2M_CUDA(cudaEventRecord(ev[i].second.second, cx.stream)); }
    double ms(const char* name) {
      double t = 0;
      for (auto& e : ev)
        if (!strcmp(e.first, name)) {
          float m = 0;
          cudaEventElapsedTime(&m, e.second.first, e.second.second);
          t += m;
        }
      return t;
    }
  };

  void run_pairing(const DBuf<Pt>& pts, size_t n_prod, DBuf<uint8_t>& ok) {
    size_t sp = cx.span_begin("verify_pairing", (double)n_prod);
    ver_pairing_kernel<Fq><<<div_up(n_prod, 32), 32, 0, cx.stream>>>(pts.p, prepared.p, ns, n_prod, ok.p);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    cx.span_end(sp);
  }

  void verify(size_t n, const uint64_t* const* public_inputs, const size_t* n_inputs, const uint8_t* const* proofs, const size_t* proof_lens,
              b2m_rng* rng, int* verdicts) override {
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();
    timings_json = "{}";
    if (n == 0) return;
    B2M_REQUIRE(public_inputs && n_inputs && proofs && proof_lens && verdicts, B2M_ERR_INVALID_ARG, "null argument");
    B2M_REQUIRE(rng != nullptr, B2M_ERR_MISSING_RNG, "the batch verifier needs an rng for its randomisers");
    // formatted public inputs: leading one, padded to |X| = next power of two of (#inputs + 1)
    size_t stride = 1;
    std::vector<uint32_t> n_x(n);
    for (size_t i = 0; i < n; i++) {
      B2M_REQUIRE(public_inputs[i] || n_inputs[i] == 0, B2M_ERR_INVALID_ARG, "null public input %zu", i);
      n_x[i] = (uint32_t)pow2_at_least(n_inputs[i] + 1);
      stride = std::max(stride, (size_t)n_x[i]);
    }
    std::vector<Fr> formatted(n * stride, Fr::zero());
    for (size_t i = 0; i < n; i++) {
      formatted[i * stride] = Fr::one();
      for (size_t j = 0; j < n_inputs[i]; j++) {
        Fr v;  // Montgomery limbs: only the range (< r) is checked here
        B2M_REQUIRE(canon_from_le(reinterpret_cast<const uint8_t*>(public_inputs[i] + 4 * j), FR_BYTES, &v), B2M_ERR_INVALID_ARG,
                    "public input %zu[%zu] is not a reduced field element", i, j);
        memcpy(formatted[i * stride + 1 + j].l, public_inputs[i] + 4 * j, FR_BYTES);
      }
    }
    // parse
    std::vector<Parsed> parsed(n);
    std::vector<uint8_t> comp(n * N_PROOF_POINTS * NB, 0), present(n * N_PROOF_POINTS, 0);
    for (size_t i = 0; i < n; i++) {
      if (parse(proofs[i], proof_lens[i], parsed[i])) {
        memcpy(&comp[i * N_PROOF_POINTS * NB], parsed[i].comp, sizeof(parsed[i].comp));
        memcpy(&present[i * N_PROOF_POINTS], parsed[i].present, N_PROOF_POINTS);
      }
    }
    const auto t_parse = clk::now();
    Events ev(cx);
    // decode
    const size_t np = n * N_PROOF_POINTS;
    DBuf<uint8_t> d_comp(cx, comp.size()), d_present(cx, np), d_status(cx, np);
    DBuf<Pt> d_pts(cx, np);
    d_comp.upload(comp.data(), comp.size());
    d_present.upload(present.data(), np);
    size_t e = ev.begin("decode");
    ver_decode_kernel<Fq, Fr><<<div_up(np, 128), 128, 0, cx.stream>>>(d_comp.p, d_present.p, np, d_pts.p, d_status.p);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    ev.end(e);
    std::vector<Pt> pts(np);
    std::vector<uint8_t> status(np);
    d_status.download(status.data(), np);
    d_pts.download(pts.data(), np);
    std::vector<uint8_t> live(n);
    for (size_t i = 0; i < n; i++) {
      bool ok = parsed[i].ok;
      for (int s = 0; ok && s < N_PROOF_POINTS; s++) ok = status[i * N_PROOF_POINTS + s] == DEC_OK;
      live[i] = ok ? 1 : 0;
      verdicts[i] = ok ? VERDICT_ACCEPT : VERDICT_MALFORMED;
    }
    // randomisers (drawn for every proof, in a fixed order, so that verdicts never depend on which proofs are malformed)
    ZkSource<b2m_rng> zs(rng);
    std::vector<ProofScalars<Fr>> ps(n);
    auto rand128 = [&](uint32_t* limbs) {
      const uint64_t lo = zs.next_u64(), hi = zs.next_u64();
      limbs[0] = (uint32_t)lo; limbs[1] = (uint32_t)(lo >> 32); limbs[2] = (uint32_t)hi; limbs[3] = (uint32_t)(hi >> 32);
    };
    for (size_t i = 0; i < n; i++)
      for (int p = 0; p < 2; p++) {
        Fr c = Fr::zero();
        rand128(c.l);
        ps[i].rho[p] = Fr::from_canonical(c);
      }
    std::vector<uint32_t> fold_r(4 * n);
    for (size_t i = 0; i < n; i++) {
      rand128(&fold_r[4 * i]);
      if (!live[i]) memset(&fold_r[4 * i], 0, 16);
    }
    zs.commit_position();
    // transcripts on a pool of host threads
    const auto t_tr0 = clk::now();
    {
      const unsigned nt = std::max(1u, std::min<unsigned>(std::thread::hardware_concurrency(), (unsigned)((n + 15) / 16)));
      std::vector<std::thread> pool;
      for (unsigned t = 0; t < nt; t++)
        pool.emplace_back([&, t] {
          for (size_t i = t; i < n; i += nt)
            if (live[i]) transcript(&formatted[i * stride], n_x[i], &pts[i * N_PROOF_POINTS], parsed[i], ps[i]);
        });
      for (auto& th : pool) th.join();
    }
    const auto t_tr1 = clk::now();
    size_t n_live = 0;
    for (size_t i = 0; i < n; i++) n_live += live[i];
    if (n_live > 0) {
      // scalars
      DBuf<ProofScalars<Fr>> d_ps(cx, n);
      DBuf<Fr> d_fmt(cx, formatted.size()), d_sc(cx, n * N_TERMS);
      DBuf<uint32_t> d_nx(cx, n), d_r(cx, 4 * n);
      DBuf<uint8_t> d_live(cx, n);
      d_ps.upload(ps.data(), n);
      d_fmt.upload(formatted.data(), formatted.size());
      d_nx.upload(n_x.data(), n);
      d_r.upload(fold_r.data(), 4 * n);
      d_live.upload(live.data(), n);
      e = ev.begin("scalars");
      ver_scalars_kernel<Fr><<<div_up(n, 64), 64, 0, cx.stream>>>(d_ps.p, d_fmt.p, d_nx.p, stride, d_live.p, n, marlin, H, K, d_sc.p);
      B2M_CHECK_LAUNCH();
      cx.launches++;
      ev.end(e);
      // per-proof combination
      DBuf<XYZZ<Fq>> d_terms(cx, n * N_TERMS);
      DBuf<Pt> d_proof_pts(cx, n * ns);
      e = ev.begin("combine");
      ver_term_kernel<Fq, Fr><<<div_up(n * N_TERMS, 128), 128, 0, cx.stream>>>(d_pts.p, bases.p, d_sc.p, n, d_terms.p);
      B2M_CHECK_LAUNCH();
      ver_sum_kernel<Fq><<<div_up(n * ns, 128), 128, 0, cx.stream>>>(d_terms.p, dest, ns, n, d_proof_pts.p);
      B2M_CHECK_LAUNCH();
      cx.launches += 2;
      ev.end(e);
      // fold
      DBuf<XYZZ<Fq>> d_scaled(cx, n * ns);
      DBuf<Pt> d_folded(cx, ns);
      e = ev.begin("fold");
      ver_fold_scale_kernel<Fq><<<div_up(n * ns, 128), 128, 0, cx.stream>>>(d_proof_pts.p, d_r.p, ns, n, d_scaled.p);
      B2M_CHECK_LAUNCH();
      ver_fold_reduce_kernel<Fq><<<ns, VER_FOLD_THREADS, 0, cx.stream>>>(d_scaled.p, ns, n, d_folded.p);
      B2M_CHECK_LAUNCH();
      cx.launches += 2;
      ev.end(e);
      // one multi-pairing for the batch
      DBuf<uint8_t> d_ok(cx, n);
      e = ev.begin("pairing");
      run_pairing(d_folded, 1, d_ok);
      ev.end(e);
      uint8_t all_ok = 0;
      d_ok.download(&all_ok, 1);
      if (!all_ok) {  // exact per-proof verdicts from the per-proof points already computed
        e = ev.begin("pairing");
        run_pairing(d_proof_pts, n, d_ok);
        ev.end(e);
        std::vector<uint8_t> ok(n);
        d_ok.download(ok.data(), n);
        for (size_t i = 0; i < n; i++)
          if (live[i] && !ok[i]) verdicts[i] = VERDICT_REJECT;
      }
    }
    cx.sync();
    auto host_ms = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    timings_json = fmt("{\"parse\": %.4f, \"decode\": %.4f, \"transcript\": %.4f, \"scalars\": %.4f, \"combine\": %.4f, \"fold\": %.4f, "
                       "\"pairing\": %.4f, \"total\": %.4f}",
                       host_ms(t0, t_parse), ev.ms("decode"), host_ms(t_tr0, t_tr1), ev.ms("scalars"), ev.ms("combine"), ev.ms("fold"),
                       ev.ms("pairing"), host_ms(t0, clk::now()));
  }
};

}  // namespace b2m
