// Device-resident Marlin index and prover: `Marlin::index` and `Marlin::prove`
// [reference src/lib.rs:100-311] driving the AHP rounds of src/ahp/prover.rs with every polynomial,
// the index and the SRS resident in HBM.  The host runs only the Fiat-Shamir transcript
// (src/rng.rs), the O(1) scalar bookkeeping of src/ahp/mod.rs:110-221 and the three-coefficient
// blinding polynomials of KZG10; per round it reads back 2-4 commitments and sends 1-4 challenges.
//
// Differences from the reference that do not change any output (all arithmetic is exact):
//  * eta_c*z_a*z_b + eta_a*z_a + eta_b*z_b is formed directly in evaluation form on the 4|H| domain
//    (the reference interpolates z_c, sums coefficients, and evaluates again: prover.rs:467-480,533);
//  * h_2 = -(b*f)[|K|..) : the quotient of (a - b*f) by v_K only sees the high half of b*f, and the
//    K-sized a(X) is never materialised (prover.rs:625-640, 685-688);
//  * LC commitments inside open_combinations are not computed (they do not enter the proof);
//  * the two zero-valued sumcheck LCs are not evaluated (lib.rs:279 discards them).
#pragma once
#include <algorithm>
#include <chrono>
#include <cstring>

#include "capi_types.cuh"
#include "hostutil.hpp"
#include "poly_impl.cuh"
#include "prover.cuh"
#include "comm.cuh"
#include "scan.cuh"
#include "verify_core.cuh"

namespace b2m {

template <class Fr>
struct LcTerms {  // out[i] = sum_t coef[t] * (i < len[t] ? src[t][i] : 0)
  static constexpr int MAX = 8;
  const Fr* src[MAX];
  size_t len[MAX];
  Fr coef[MAX];
  int n = 0;
  void add(const Fr* p, size_t l, const Fr& c) {
    src[n] = p; len[n] = l; coef[n] = c; n++;
  }
};
template <class Fr>
__global__ void lincomb_kernel(LcTerms<Fr> t, size_t n, Fr* out) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr acc = Fr::zero();
  for (int k = 0; k < t.n; k++)
    if (i < t.len[k]) acc = acc + t.coef[k] * ld_fr(t.src[k] + i);
  st_fr(out + i, acc);
}

template <class Fr, class Fq>
struct MarlinIndex : IndexBase {
  using Pt = Affine<Fq>;
  using Xy = XYZZ<Fq>;
  static constexpr int LQ = Fq::N / 2;  // u64 limbs of Fq
  static constexpr int FQ_BYTES = Fq::N * 4;

  b2m_srs* srs;
  Ctx& cx;
  Ntt<Fr>& ntt;
  Msm<Fr, Fq>& msm;
  int pc;
  size_t nc, nv, ni, nnz;  // constraints, variables, |X| (formatted input), joint non-zeros
  size_t H, K, X, D;       // domain sizes and the SRS max degree
  int log_h, log_k, log_x;

  DBuf<uint32_t> a_rowptr, a_col, b_rowptr, b_col;
  DBuf<Fr> a_coeff, b_coeff;
  DBuf<uint32_t> t_colptr, t_row;
  DBuf<uint8_t> t_mat;
  DBuf<Fr> t_coeff;
  size_t t_entries = 0;
  DBuf<Fr> ipoly[6], ieval[6];  // row, col, a_val, b_val, c_val, row_col (coefficients / evaluations on K)
  Pt index_comms[6];

  struct Timer {
    Ctx& cx;
    std::vector<std::pair<std::string, std::pair<cudaEvent_t, cudaEvent_t>>> spans;
    explicit Timer(Ctx& c) : cx(c) {}
    size_t begin(const char* label) {
      cudaEvent_t a, b;
      cudaEventCreate(&a); cudaEventCreate(&b);
      cudaEventRecord(a, cx.stream);
      spans.push_back({label, {a, b}});
      return spans.size() - 1;
    }
    void end(size_t id) { cudaEventRecord(spans[id].second.second, cx.stream); }
    std::string json() {
      cudaStreamSynchronize(cx.stream);
      std::string s = "{";
      for (size_t i = 0; i < spans.size(); i++) {
        float ms = 0;
        cudaEventElapsedTime(&ms, spans[i].second.first, spans[i].second.second);
        s += fmt("%s\"%s\": %.4f", i ? ", " : "", spans[i].first.c_str(), ms);
        cudaEventDestroy(spans[i].second.first);
        cudaEventDestroy(spans[i].second.second);
      }
      return s + "}";
    }
  };

  static int log2_ceil(size_t n) {
    int l = 0;
    while (((size_t)1 << l) < n) l++;
    return l;
  }
  // [U ark-poly reindex_by_subdomain]
  size_t reindex(size_t i) const {
    size_t period = H / X;
    if (i < X) return i * period;
    size_t j = i - X, x = period - 1;
    return j + j / x + 1;
  }
  static Fr fr_from_limbs(const uint64_t* p) {
    Fr r;
    memcpy(r.l, p, sizeof(r.l));
    return r;
  }
  static bool is_pow2(size_t v) { return v && !(v & (v - 1)); }

  // shifted_powers(bound) start at powers_of_g[D - bound]   [U marlin_pc / sonic_pc CommitterKey]
  size_t shifted_off(size_t bound) const { return D - bound; }

  // ---------------------------------------------------------------------------------------------
  // `Marlin::index`: AHPForR1CS::index + trim + commit
  // ---------------------------------------------------------------------------------------------
  MarlinIndex(b2m_srs* s, Ntt<Fr>& ntt_, Msm<Fr, Fq>& msm_, int pc_, size_t nc_, size_t nv_, size_t ni_)
      : srs(s), cx(s->ctx->cx), ntt(ntt_), msm(msm_), pc(pc_), nc(nc_), nv(nv_), ni(ni_) {}

  // (extended device lambdas may not live in a constructor, hence a separate build step)
  void build(const b2m_matrix* a, const b2m_matrix* b, const b2m_matrix* c) {
    B2M_REQUIRE(nc == nv, B2M_ERR_NON_SQUARE, "matrices are not square: %zu constraints, %zu variables", nc, nv);
    B2M_REQUIRE(is_pow2(ni), B2M_ERR_INVALID_PUBLIC_INPUT_LEN, "formatted public input length %zu is not a power of two", ni);
    B2M_REQUIRE(nc >= 1 && ni <= nv, B2M_ERR_INVALID_ARG, "bad dimensions");
    const int S = Fr::Params::TWO_ADICITY;
    log_h = log2_ceil(nc); log_x = log2_ceil(ni);
    H = (size_t)1 << log_h; X = ni;
    B2M_REQUIRE(X < H, B2M_ERR_INVALID_ARG, "|X| must be smaller than |H|");

    // joint matrix (sorted union of the column sets per row) [reference indexer.rs:83-102]
    std::vector<uint32_t> jr, jc;
    std::vector<Fr> va, vb, vc;
    std::vector<uint64_t> cols;
    const b2m_matrix* ms[3] = {a, b, c};
    for (size_t r = 0; r < nc; r++) {
      cols.clear();
      for (int m = 0; m < 3; m++)
        for (uint64_t e = ms[m]->row_ptr[r]; e < ms[m]->row_ptr[r + 1]; e++) {
          B2M_REQUIRE(ms[m]->col[e] < nv, B2M_ERR_INVALID_ARG, "column index %llu out of range", (unsigned long long)ms[m]->col[e]);
          cols.push_back(ms[m]->col[e]);
        }
      std::sort(cols.begin(), cols.end());
      cols.erase(std::unique(cols.begin(), cols.end()), cols.end());
      for (uint64_t col : cols) {
        jr.push_back((uint32_t)r);
        jc.push_back((uint32_t)reindex(col));
        Fr v[3];
        for (int m = 0; m < 3; m++) {
          v[m] = Fr::zero();
          for (uint64_t e = ms[m]->row_ptr[r]; e < ms[m]->row_ptr[r + 1]; e++)
            if (ms[m]->col[e] == col) v[m] = fr_from_limbs(ms[m]->coeff + 4 * e);  // BTreeMap collect: last wins
        }
        va.push_back(v[0]); vb.push_back(v[1]); vc.push_back(v[2]);
      }
    }
    nnz = jr.size();
    B2M_REQUIRE(nnz >= 1, B2M_ERR_INVALID_ARG, "empty constraint matrices");
    log_k = log2_ceil(nnz);
    K = (size_t)1 << log_k;
    B2M_REQUIRE(log_k + 1 <= S && log_h + 2 <= S, B2M_ERR_DEGREE_TOO_LARGE, "domains exceed the field's 2-adicity");
    D = srs->n_g - 1;
    size_t md = std::max(std::max(2 * H - 1, 3 * H - 1), K - 1);  // reference src/ahp/mod.rs:83-92 with zk_bound = 1
    B2M_REQUIRE(D >= md, B2M_ERR_INDEX_TOO_LARGE, "SRS max degree %zu < index max degree %zu", D, md);
    B2M_REQUIRE(D >= K - 2 && D >= H - 2, B2M_ERR_INDEX_TOO_LARGE, "SRS too small for the degree bounds");

    // CSR copies of A and B for z_A = A z, z_B = B z  [reference prover.rs:256-276]
    auto upload_csr = [&](const b2m_matrix* m, DBuf<uint32_t>& rp, DBuf<uint32_t>& cl, DBuf<Fr>& cf) {
      size_t ne = m->row_ptr[nc];
      std::vector<uint32_t> hrp(nc + 1), hcl(ne ? ne : 1);
      for (size_t r = 0; r <= nc; r++) hrp[r] = (uint32_t)m->row_ptr[r];
      for (size_t e = 0; e < ne; e++) hcl[e] = (uint32_t)m->col[e];
      rp = DBuf<uint32_t>(cx, nc + 1); cl = DBuf<uint32_t>(cx, ne ? ne : 1); cf = DBuf<Fr>(cx, ne ? ne : 1);
      rp.upload(hrp.data(), nc + 1);
      if (ne) { cl.upload(hcl.data(), ne); cf.upload(reinterpret_cast<const Fr*>(m->coeff), ne); }
      cx.sync();
    };
    upload_csr(a, a_rowptr, a_col, a_coeff);
    upload_csr(b, b_rowptr, b_col, b_coeff);

    // entries of A, B, C bucketed by reindexed column for t(X)  [reference prover.rs:411-428]
    {
      std::vector<uint32_t> cnt(H + 1, 0);
      for (int m = 0; m < 3; m++)
        for (uint64_t e = 0; e < ms[m]->row_ptr[nc]; e++) cnt[reindex(ms[m]->col[e]) + 1]++;
      for (size_t i = 0; i < H; i++) cnt[i + 1] += cnt[i];
      t_entries = cnt[H];
      std::vector<uint32_t> pos(cnt.begin(), cnt.end() - 1), hrow(t_entries ? t_entries : 1);
      std::vector<uint8_t> hmat(t_entries ? t_entries : 1);
      std::vector<Fr> hco(t_entries ? t_entries : 1);
      for (int m = 0; m < 3; m++)
        for (size_t r = 0; r < nc; r++)
          for (uint64_t e = ms[m]->row_ptr[r]; e < ms[m]->row_ptr[r + 1]; e++) {
            uint32_t p = pos[reindex(ms[m]->col[e])]++;
            hrow[p] = (uint32_t)r; hmat[p] = (uint8_t)m; hco[p] = fr_from_limbs(ms[m]->coeff + 4 * e);
          }
      t_colptr = DBuf<uint32_t>(cx, H + 1); t_row = DBuf<uint32_t>(cx, hrow.size());
      t_mat = DBuf<uint8_t>(cx, hmat.size()); t_coeff = DBuf<Fr>(cx, hco.size());
      t_colptr.upload(cnt.data(), H + 1); t_row.upload(hrow.data(), hrow.size());
      t_mat.upload(hmat.data(), hmat.size()); t_coeff.upload(hco.data(), hco.size());
      cx.sync();
    }

    // arithmetization of M* on the device [reference constraint_systems.rs:125-262]
    ntt.ensure_table(std::max(log_k + 1, log_h + 2));
    const Fr* tw = ntt.table.tw;
    const int ml = ntt.table.max_log, lh = log_h;
    {
      DBuf<uint32_t> djr(cx, nnz), djc(cx, nnz);
      DBuf<Fr> dva(cx, nnz), dvb(cx, nnz), dvc(cx, nnz);
      djr.upload(jr.data(), nnz); djc.upload(jc.data(), nnz);
      dva.upload(va.data(), nnz); dvb.upload(vb.data(), nnz); dvc.upload(vc.data(), nnz);
      for (int i = 0; i < 6; i++) { ieval[i] = DBuf<Fr>(cx, K); ipoly[i] = DBuf<Fr>(cx, K); }
      Fr* e_row = ieval[0].p; Fr* e_col = ieval[1].p; Fr* e_a = ieval[2].p; Fr* e_b = ieval[3].p; Fr* e_c = ieval[4].p;
      Fr* e_rc = ieval[5].p;
      const uint32_t* pjr = djr.p; const uint32_t* pjc = djc.p;
      const Fr* pva = dva.p; const Fr* pvb = dvb.p; const Fr* pvc = dvc.p;
      Fr h_inv = Fr::from_u64(H).inverse();
      size_t nz = nnz;
      ew(cx, K, [=] __device__(size_t k) {
        if (k < nz) {
          Fr colv = domain_element(tw, ml, lh, pjc[k]);  // elems[reindex(i)]
          Fr rowv = domain_element(tw, ml, lh, pjr[k]);  // elems[r]
          Fr sc = colv * h_inv;                          // 1 / u_H(col_val, col_val)
          st_fr(e_row + k, colv);                        // transposed: "row" holds the column element
          st_fr(e_col + k, rowv);
          st_fr(e_a + k, ld_fr(pva + k) * sc);
          st_fr(e_b + k, ld_fr(pvb + k) * sc);
          st_fr(e_c + k, ld_fr(pvc + k) * sc);
          st_fr(e_rc + k, colv * rowv);
        } else {
          st_fr(e_row + k, Fr::one()); st_fr(e_col + k, Fr::one()); st_fr(e_rc + k, Fr::one());
          st_fr(e_a + k, Fr::zero()); st_fr(e_b + k, Fr::zero()); st_fr(e_c + k, Fr::zero());
        }
      });
      DBuf<Fr> work(cx, K);
      for (int i = 0; i < 6; i++) {
        B2M_CUDA(cudaMemcpyAsync(work.p, ieval[i].p, K * sizeof(Fr), cudaMemcpyDeviceToDevice, cx.stream));
        ntt.run(work.p, ipoly[i].p, log_k, true);
      }
      cx.sync();
    }
    // commit to the index polynomials, rng = None [reference lib.rs:124-125]
    {
      DBuf<Pt> out(cx, 6);
      MsmJob<Fr, Fq> jobs[6];
      for (int i = 0; i < 6; i++) jobs[i] = MsmJob<Fr, Fq>{ipoly[i].p, true, K, 0, nullptr, 0, 0, nullptr, 0, nullptr, out.p + i};
      msm.run_batch(jobs, 6);
      out.download(index_comms, 6);
    }
    comms_xy.resize(6 * 2 * LQ);
    memcpy(comms_xy.data(), index_comms, sizeof(index_comms));
    // IndexVerifierKey::write: index_info (3 x u64) || index_comms  [reference data_structures.rs:36-43, indexer.rs:63-69]
    put_u64(vk_bytes, nv); put_u64(vk_bytes, nc); put_u64(vk_bytes, nnz);
    for (int i = 0; i < 6; i++) write_commitment(vk_bytes, index_comms[i], false, Pt::inf());
  }

  // ---- ToBytes / CanonicalSerialize of group and field elements (SURVEY.md A.2 / A.3) ------------
  static void put_fq_canonical(std::vector<uint8_t>& out, const Fq& mont) {
    Fq c = mont.to_canonical();
    const uint8_t* p = reinterpret_cast<const uint8_t*>(c.l);
    out.insert(out.end(), p, p + FQ_BYTES);
  }
  static void put_fr_canonical(std::vector<uint8_t>& out, const Fr& mont) {
    Fr c = mont.to_canonical();
    const uint8_t* p = reinterpret_cast<const uint8_t*>(c.l);
    out.insert(out.end(), p, p + Fr::N * 4);
  }
  static void put_affine_tobytes(std::vector<uint8_t>& out, const Pt& P) {  // x || y || infinity
    if (P.is_inf()) {
      out.insert(out.end(), FQ_BYTES, 0);
      out.push_back(1);
      out.insert(out.end(), FQ_BYTES - 1, 0);
      out.push_back(1);
    } else {
      put_fq_canonical(out, P.x);
      put_fq_canonical(out, P.y);
      out.push_back(0);
    }
  }
  void write_commitment(std::vector<uint8_t>& out, const Pt& comm, bool has_shifted, const Pt& shifted) const {
    put_affine_tobytes(out, comm);
    if (pc == B2M_PC_MARLIN_KZG10) {  // comm || bool || (shifted or identity)
      out.push_back(has_shifted ? 1 : 0);
      put_affine_tobytes(out, has_shifted ? shifted : Pt::inf());
    }
  }
  static void put_compressed(std::vector<uint8_t>& out, const Pt& P) {
    if (P.is_inf()) {
      out.insert(out.end(), FQ_BYTES - 1, 0);
      out.push_back(1 << 6);
      return;
    }
    Fq x = P.x.to_canonical(), y = P.y.to_canonical();
    size_t at = out.size();
    const uint8_t* p = reinterpret_cast<const uint8_t*>(x.l);
    out.insert(out.end(), p, p + FQ_BYTES);
    if (y.canonical_gt_half()) out[at + FQ_BYTES - 1] |= 1 << 7;
  }

  // ---- small host-side polynomials (the 3-coefficient KZG blinding polynomials) -------------------
  typedef std::vector<Fr> HPoly;
  static void hp_axpy(HPoly& acc, const Fr& k, const HPoly& p) {
    if (acc.size() < p.size()) acc.resize(p.size(), Fr::zero());
    for (size_t i = 0; i < p.size(); i++) acc[i] = acc[i] + k * p[i];
  }
  static Fr hp_eval(const HPoly& p, const Fr& z) {
    Fr acc = Fr::zero();
    for (size_t i = p.size(); i-- > 0;) acc = acc * z + p[i];
    return acc;
  }
  static HPoly hp_div_linear(const HPoly& p, const Fr& z) {  // quotient of p / (X - z)
    if (p.size() <= 1) return HPoly();
    HPoly q(p.size() - 1);
    Fr acc = Fr::zero();
    for (size_t i = p.size() - 1; i >= 1; i--) {
      acc = p[i] + acc * z;
      q[i - 1] = acc;
    }
    return q;
  }
  static bool hp_is_zero(const HPoly& p) {
    for (auto& c : p)
      if (!c.is_zero()) return false;
    return true;
  }

  // ---- device helpers -----------------------------------------------------------------------------
  // c (|H| + 1 coefficients, c[|H|] not yet written) += rho * v_H    [reference prover.rs:350-366]
  void blind(Fr* c, Fr rho) {
    const size_t Hh = H;
    ew(cx, 2, [=] __device__(size_t i) {
      if (i == 0) st_fr(c, ld_fr(c) - rho);
      else st_fr(c + Hh, rho);
    });
  }
  void lincomb(const LcTerms<Fr>& t, size_t n, Fr* out) {
    lincomb_kernel<Fr><<<div_up(n, 256), 256, 0, cx.stream>>>(t, n, out);
    B2M_CHECK_LAUNCH();
    cx.launches++;
  }
  // forward NTT of `len` coefficients zero-extended to 2^log_n, result in `out` (2^log_n elements)
  void fft_padded(const Fr* coeffs, size_t len, int log_n, Fr* out) {
    size_t n = (size_t)1 << log_n;
    DBuf<Fr> work(cx, n);
    B2M_CUDA(cudaMemcpyAsync(work.p, coeffs, len * sizeof(Fr), cudaMemcpyDeviceToDevice, cx.stream));
    if (n > len) B2M_CUDA(cudaMemsetAsync(work.p + len, 0, (n - len) * sizeof(Fr), cx.stream));
    ntt.run(work.p, out, log_n, false);
  }
  // A group of INDEPENDENT transforms of one round.  One GPU: run them in order.  Several GPUs (the prover is replicated, so
  // every rank holds every input): transform j is computed by rank j mod world only and its result broadcast over NVLink --
  // north_star keeps a single NTT on one GPU, but a round's independent transforms need not all run on the same one.  Worth it
  // for large transforms only (>= 2^24 points: at 2^24 constraints on 8 GPUs the NTTs are the largest term of the proof and
  // sharing cut them from 319 to 182 + 58 ms of broadcasts); results are bit-identical either way.
  struct NttJob {
    const Fr* coeffs;  // padded form: `len` coefficients zero-extended to 2^log_n (work == nullptr)
    size_t len;
    Fr* work;          // direct form: 2^log_n values, overwritten
    Fr* out;
    int log_n;
    bool inverse;
  };
  int ntt_share_min_log = 24;  // measured (profiles/r02_scaling_notes.md): sharing 2^22-point transforms across 8 GPUs costs more in rank skew than it saves
  void run_ntt_group(const std::vector<NttJob>& jobs) {
    const bool share = cx.world > 1 && cx.comm != nullptr && jobs.size() > 1 && jobs[0].log_n >= ntt_share_min_log;
    for (size_t j = 0; j < jobs.size(); j++) {
      if (share && (int)(j % (size_t)cx.world) != cx.rank) continue;
      const NttJob& q = jobs[j];
      if (q.work) ntt.run(q.work, q.out, q.log_n, q.inverse);
      else fft_padded(q.coeffs, q.len, q.log_n, q.out);
    }
    if (!share) return;
    size_t sp = cx.span_begin("ntt_broadcast", 0.0);
    for (size_t j = 0; j < jobs.size(); j++) broadcast_bytes(cx, jobs[j].out, sizeof(Fr) << jobs[j].log_n, (int)(j % (size_t)cx.world));
    cx.span_end(sp);
  }
  Fr download_fr(const Fr* p) {
    Fr h;
    B2M_CUDA(cudaMemcpyAsync(&h, p, sizeof(Fr), cudaMemcpyDeviceToHost, cx.stream));
    cx.sync();
    return h;
  }

  // One KZG10::commit as an MSM job: powers_of_g[off..off+len) against the coefficients, and the blinding
  // polynomial against the gamma powers starting at gamma slot `gslot` -- all in the same bucket pass.
  MsmJob<Fr, Fq> kzg_commit_job(const Fr* coeffs, size_t len, size_t off, const HPoly& blinding, size_t gslot, Pt* out_dev,
                                std::vector<DBuf<Fr>>& keep_sc) {
    const Fr* s2 = nullptr;
    if (!blinding.empty()) {
      keep_sc.emplace_back(cx, blinding.size());
      keep_sc.back().upload(blinding.data(), blinding.size());
      s2 = keep_sc.back().p;
    }
    return MsmJob<Fr, Fq>{coeffs, true, len, off, s2, blinding.size(), gslot, nullptr, 0, nullptr, out_dev};
  }

  struct Oracle {       // a labelled polynomial living in HBM
    const Fr* p = nullptr;
    size_t len = 0;
    bool bounded = false;
    size_t bound = 0;
    bool hiding = false;
    HPoly rand, shifted_rand;  // kzg10::Randomness blinding polynomials (host)
    Pt comm, shifted_comm;
  };

  // `PC::commit` over a round's oracles, drawing blinding polynomials from zk in the reference's order.
  void commit_round(std::vector<Oracle*>& polys, ZkSource<b2m_rng>& zk) {
    std::vector<DBuf<Fr>> keep_sc;
    DBuf<Pt> out(cx, 2 * polys.size());
    out.zero();  // the shifted slot of an unbounded polynomial is never written
    std::vector<MsmJob<Fr, Fq>> jobs;
    for (size_t i = 0; i < polys.size(); i++) {
      Oracle& o = *polys[i];
      auto draw = [&]() {
        HPoly r;
        if (o.hiding)
          for (int k = 0; k < 3; k++) r.push_back(field_rand<Fr>(zk));  // degree hiding_bound + 1 = 2
        return r;
      };
      if (pc == B2M_PC_MARLIN_KZG10) {
        o.rand = draw();
        jobs.push_back(kzg_commit_job(o.p, o.len, 0, o.rand, srs->gamma_slot(0), out.p + 2 * i, keep_sc));
        if (o.bounded) {
          o.shifted_rand = draw();
          jobs.push_back(kzg_commit_job(o.p, o.len, shifted_off(o.bound), o.shifted_rand, srs->gamma_slot(0), out.p + 2 * i + 1, keep_sc));
        }
      } else {
        o.rand = draw();
        if (o.bounded)
          jobs.push_back(kzg_commit_job(o.p, o.len, shifted_off(o.bound), o.rand, o.hiding ? sonic_gamma_slot(o.bound) : 0,
                                        out.p + 2 * i, keep_sc));
        else
          jobs.push_back(kzg_commit_job(o.p, o.len, 0, o.rand, o.hiding ? srs->gamma_slot(0) : 0, out.p + 2 * i, keep_sc));
      }
    }
    msm.run_batch(jobs.data(), (int)jobs.size());
    std::vector<Pt> h(2 * polys.size());
    out.download(h.data(), h.size());
    for (size_t i = 0; i < polys.size(); i++) {
      polys[i]->comm = h[2 * i];
      polys[i]->shifted_comm = h[2 * i + 1];
    }
  }
  // sonic_pc shifted_powers_of_gamma_g[bound]: powers max_degree - bound + {0, 1, 2} in consecutive slots
  size_t sonic_gamma_slot(size_t bound) const {
    size_t s0 = srs->gamma_slot(D - bound);
    for (size_t i = 1; i < 3; i++)
      B2M_REQUIRE(srs->gamma_slot(D - bound + i) == s0 + i, B2M_ERR_INVALID_ARG, "gamma powers for bound %zu are not consecutive", bound);
    return s0;
  }
  void absorb_comms(FiatShamir& fs, std::vector<Oracle*>& polys) {
    std::vector<uint8_t> bytes;
    for (auto* o : polys) write_commitment(bytes, o->comm, o->bounded && pc == B2M_PC_MARLIN_KZG10, o->shifted_comm);
    fs.absorb(bytes);
  }
  Fr sample_outside_h(FiatShamir& fs) {  // sample_element_outside_domain
    for (;;) {
      Fr t = field_rand<Fr>(fs);
      if (t.pow_u64(H) != Fr::one()) return t;
    }
  }

  // ---------------------------------------------------------------------------------------------
  // `Marlin::prove`
  // ---------------------------------------------------------------------------------------------
  DBuf<Fr> staged_z;
  std::vector<uint64_t> staged_input;

  void check_instance(size_t n_input, size_t n_witness) const {
    B2M_REQUIRE(n_input + n_witness == nv, B2M_ERR_INSTANCE_MISMATCH, "instance (%zu + %zu variables) does not match the index (%zu)",
                n_input, n_witness, nv);
    B2M_REQUIRE(n_input == ni && is_pow2(n_input), B2M_ERR_INVALID_PUBLIC_INPUT_LEN, "formatted public input length %zu (index: %zu)",
                n_input, ni);
  }
  void stage(const uint64_t* formatted_input, size_t n_input, const uint64_t* witness, size_t n_witness) override {
    check_instance(n_input, n_witness);
    staged_z = DBuf<Fr>(cx, nv);
    staged_z.upload(reinterpret_cast<const Fr*>(formatted_input), ni);
    if (n_witness) B2M_CUDA(cudaMemcpyAsync(staged_z.p + ni, witness, n_witness * sizeof(Fr), cudaMemcpyHostToDevice, cx.stream));
    staged_input.assign(formatted_input, formatted_input + 4 * ni);
    cx.sync();
  }

  void prove(const uint64_t* formatted_input, size_t n_input, const uint64_t* witness, size_t n_witness, b2m_rng* rng,
             std::vector<uint8_t>& proof) override {
    const bool use_staged = formatted_input == nullptr;
    if (use_staged) {
      B2M_REQUIRE(staged_z.p != nullptr, B2M_ERR_INVALID_ARG, "no staged instance: call b2m_index_stage first");
      formatted_input = staged_input.data();
      n_input = ni;
      n_witness = nv - ni;
    }
    B2M_REQUIRE(n_input + n_witness == nv, B2M_ERR_INSTANCE_MISMATCH, "instance (%zu + %zu variables) does not match the index (%zu)",
                n_input, n_witness, nv);
    B2M_REQUIRE(n_input == ni && is_pow2(n_input), B2M_ERR_INVALID_PUBLIC_INPUT_LEN, "formatted public input length %zu (index: %zu)",
                n_input, ni);
    B2M_REQUIRE(rng->kind == B2M_RNG_CHACHA8 || rng->kind == B2M_RNG_CHACHA12 || rng->kind == B2M_RNG_CHACHA20 ||
                    (rng->kind == B2M_RNG_CALLBACK && rng->next_u64 != nullptr),
                B2M_ERR_MISSING_RNG, "unsupported rng kind %d", rng->kind);
    if (const char* e = getenv("B2M_NTT_SHARE_MIN_LOG")) ntt_share_min_log = atoi(e);
    Timer tm(cx);
    size_t t_all = tm.begin("Marlin::Prover");
    ZkSource<b2m_rng> zk(rng);
    const Fr* tw = ntt.table.tw;
    const int ml = ntt.table.max_log, lh = log_h;
    const size_t Hh = H, Xx = X, Kk = K;
    const Fr one = Fr::one();

    // ---- prover_init [reference prover.rs:211-306] --------------------------------------------------
    size_t t_init = tm.begin("AHP::Prover::Init");
    DBuf<Fr> z(cx, nv), z_a(cx, H), z_b(cx, H);
    if (use_staged) {
      B2M_CUDA(cudaMemcpyAsync(z.p, staged_z.p, nv * sizeof(Fr), cudaMemcpyDeviceToDevice, cx.stream));
    } else {
      z.upload(reinterpret_cast<const Fr*>(formatted_input), ni);
      if (n_witness) B2M_CUDA(cudaMemcpyAsync(z.p + ni, witness, n_witness * sizeof(Fr), cudaMemcpyHostToDevice, cx.stream));
    }
    z_a.zero(); z_b.zero();
    spmv_kernel<Fr><<<div_up(nc, 256), 256, 0, cx.stream>>>(a_rowptr.p, a_col.p, a_coeff.p, z.p, nc, z_a.p);
    spmv_kernel<Fr><<<div_up(nc, 256), 256, 0, cx.stream>>>(b_rowptr.p, b_col.p, b_coeff.p, z.p, nc, z_b.p);
    B2M_CHECK_LAUNCH();
    cx.launches += 2;
    tm.end(t_init);

    // transcript: FS::initialize(to_bytes![PROTOCOL_NAME, index_vk, public_input]) [reference lib.rs:161-163]
    std::vector<uint8_t> init_bytes;
    const char* proto = "MARLIN-2019";
    init_bytes.insert(init_bytes.end(), proto, proto + 11);
    init_bytes.insert(init_bytes.end(), vk_bytes.begin(), vk_bytes.end());
    for (size_t i = 1; i < ni; i++) put_fr_canonical(init_bytes, fr_from_limbs(formatted_input + 4 * i));
    FiatShamir fs(init_bytes);

    // ---- first round [reference prover.rs:309-409] ---------------------------------------------------
    size_t t_r1 = tm.begin("AHP::Prover::FirstRound");
    DBuf<Fr> x_poly(cx, X);
    {
      DBuf<Fr> xw(cx, X);
      B2M_CUDA(cudaMemcpyAsync(xw.p, z.p, X * sizeof(Fr), cudaMemcpyDeviceToDevice, cx.stream));
      ntt.run(xw.p, x_poly.p, log_x, true);
    }
    DBuf<Fr> wt(cx, H + 1);  // (iFFT_H(w - x) + rho v_H); w_poly = its suffix sums shifted by |X|
    DBuf<Fr> za_poly(cx, H + 1), zb_poly(cx, H + 1);
    {
      DBuf<Fr> x_evals(cx, H), w_evals(cx, H);
      fft_padded(x_poly.p, X, log_h, x_evals.p);
      const size_t ratio = H / X, nw = n_witness;
      const Fr* pw = z.p + ni; const Fr* pxe = x_evals.p; Fr* pwe = w_evals.p;
      ew(cx, H, [=] __device__(size_t k) {
        Fr v = Fr::zero();
        if (k % ratio != 0) {
          size_t j = k - k / ratio - 1;
          Fr wv = j < nw ? ld_fr(pw + j) : Fr::zero();
          v = wv - ld_fr(pxe + k);
        }
        st_fr(pwe + k, v);
      });
      run_ntt_group({NttJob{nullptr, 0, w_evals.p, wt.p, log_h, true}, NttJob{nullptr, 0, z_a.p, za_poly.p, log_h, true},
                     NttJob{nullptr, 0, z_b.p, zb_poly.p, log_h, true}});
    }
    Fr rho_w = field_rand<Fr>(zk), rho_a = field_rand<Fr>(zk), rho_b = field_rand<Fr>(zk);
    blind(wt.p, rho_w);
    rec_suffix<Fr>(cx, wt.p, wt.p, H + 1, X, one, false);  // divide by v_X: q[i] = S[i + |X|]
    Oracle o_w; o_w.p = wt.p + X; o_w.len = H + 1 - X; o_w.hiding = true;
    blind(za_poly.p, rho_a);
    blind(zb_poly.p, rho_b);
    Oracle o_za; o_za.p = za_poly.p; o_za.len = H + 1; o_za.hiding = true;
    Oracle o_zb; o_zb.p = zb_poly.p; o_zb.len = H + 1; o_zb.hiding = true;
    // mask polynomial: 3|H| rejection-sampled coefficients straight from the ChaCha stream
    DBuf<Fr> mask(cx, 3 * H);
    sample_mask(zk, mask.p, 3 * H);
    {
      Fr* pm = mask.p;
      ew(cx, 1, [=] __device__(size_t) { st_fr(pm, (ld_fr(pm + Hh) + ld_fr(pm + 2 * Hh)).neg()); });  // mask[0] -= sum_i mask[i|H|]
    }
    Oracle o_mask; o_mask.p = mask.p; o_mask.len = 3 * H;
    tm.end(t_r1);
    size_t t_c1 = tm.begin("Committing to first round polys");
    std::vector<Oracle*> first = {&o_w, &o_za, &o_zb, &o_mask};
    commit_round(first, zk);
    tm.end(t_c1);
    absorb_comms(fs, first);
    // verifier_first_round [reference verifier.rs:44-79]
    Fr alpha = sample_outside_h(fs);
    Fr eta_a = field_rand<Fr>(fs), eta_b = field_rand<Fr>(fs), eta_c = field_rand<Fr>(fs);

    // ---- second round [reference prover.rs:443-570] --------------------------------------------------
    size_t t_r2 = tm.begin("AHP::Prover::SecondRound");
    const int log_m = log_h + 2;  // mul_domain = 4|H|
    const size_t M = (size_t)1 << log_m;
    DBuf<Fr> summed_ev(cx, M);  // evaluations of eta_c z_a z_b + eta_a z_a + eta_b z_b on 4|H|
    {
      DBuf<Fr> ea(cx, M), eb(cx, M);
      run_ntt_group({NttJob{za_poly.p, H + 1, nullptr, ea.p, log_m, false}, NttJob{zb_poly.p, H + 1, nullptr, eb.p, log_m, false}});
      const Fr* pa = ea.p; const Fr* pb = eb.p; Fr* ps = summed_ev.p;
      ew(cx, M, [=] __device__(size_t i) {
        Fr x = ld_fr(pa + i), y = ld_fr(pb + i);
        st_fr(ps + i, eta_c * x * y + eta_a * x + eta_b * y);
      });
    }
    // r(alpha, X) on H: v_H(alpha) / (alpha - w^i)   [reference mod.rs:311-318]
    Fr v_h_alpha = alpha.pow_u64(H) - one;
    DBuf<Fr> r_alpha_ev(cx, H), r_alpha_poly(cx, H), t_poly(cx, H);
    {
      Fr* pr = r_alpha_ev.p;
      ew(cx, H, [=] __device__(size_t i) { st_fr(pr + i, alpha - domain_element(tw, ml, lh, i)); });
      batch_inverse<Fr>(cx, r_alpha_ev.p, H);
      ew(cx, H, [=] __device__(size_t i) { st_fr(pr + i, ld_fr(pr + i) * v_h_alpha); });
    }
    // t(X): segmented sums of eta_M * M[r][c] * r(alpha, w^r) by reindexed column  [reference prover.rs:411-428]
    {
      DBuf<Fr> prod(cx, t_entries + 1), t_ev(cx, H);
      const uint32_t* prow = t_row.p; const uint8_t* pmat = t_mat.p; const Fr* pco = t_coeff.p; const Fr* pr = r_alpha_ev.p;
      Fr* pp = prod.p;
      const size_t ne = t_entries;
      ew(cx, ne + 1, [=] __device__(size_t e) {
        if (e == ne) { st_fr(pp + e, Fr::zero()); return; }
        uint8_t m = pmat[e];
        Fr eta = m == 0 ? eta_a : (m == 1 ? eta_b : eta_c);
        st_fr(pp + e, eta * ldg_fr(pco + e) * ld_fr(pr + prow[e]));
      });
      rec_suffix<Fr>(cx, prod.p, prod.p, ne + 1, 1, one, false);  // suffix sums
      const uint32_t* pcp = t_colptr.p; Fr* pt = t_ev.p;
      ew(cx, H, [=] __device__(size_t j) { st_fr(pt + j, ld_fr(pp + pcp[j]) - ld_fr(pp + pcp[j + 1])); });
      // r(alpha, X) and t(X) by interpolation on H: two independent transforms (r_alpha_ev is not read again)
      run_ntt_group({NttJob{nullptr, 0, r_alpha_ev.p, r_alpha_poly.p, log_h, true}, NttJob{nullptr, 0, t_ev.p, t_poly.p, log_h, true}});
    }
    // z(X) = w(X) v_X(X) + x(X)    [reference prover.rs:501-518]
    DBuf<Fr> z_poly(cx, H + 1);
    {
      const Fr* pw = o_w.p; const size_t lw = o_w.len; const Fr* px = x_poly.p; Fr* pz = z_poly.p;
      ew(cx, H + 1, [=] __device__(size_t i) {
        Fr v = Fr::zero();
        if (i >= Xx) v = ld_fr(pw + (i - Xx));
        if (i < lw) v = v - ld_fr(pw + i);
        if (i < Xx) v = v + ld_fr(px + i);
        st_fr(pz + i, v);
      });
    }
    // q_1 = mask + r_alpha * summed - z * t on 4|H|; (h_1, X g_1) = q_1 / v_H   [reference prover.rs:520-552]
    DBuf<Fr> g1(cx, H), h1(cx, 2 * H);
    {
      DBuf<Fr> er(cx, M), ez(cx, M), et(cx, M), rhs(cx, M);
      run_ntt_group({NttJob{r_alpha_poly.p, H, nullptr, er.p, log_m, false}, NttJob{z_poly.p, H + 1, nullptr, ez.p, log_m, false},
                     NttJob{t_poly.p, H, nullptr, et.p, log_m, false}});
      Fr* pr = er.p; const Fr* ps = summed_ev.p; const Fr* pz = ez.p; const Fr* pt = et.p;
      ew(cx, M, [=] __device__(size_t i) { st_fr(pr + i, ld_fr(pr + i) * ld_fr(ps + i) - ld_fr(pz + i) * ld_fr(pt + i)); });
      ntt.run(er.p, rhs.p, log_m, true);
      // q_1 has 3|H| coefficients: blocks B0 | B1 | B2.  h_1 = [B1 + B2 | B2], X g_1 = B0 + B1 + B2.
      const Fr* pm = mask.p; const Fr* pq = rhs.p; Fr* pg = g1.p; Fr* ph = h1.p;
      ew(cx, H, [=] __device__(size_t i) {
        Fr b0 = ld_fr(pm + i) + ld_fr(pq + i);
        Fr b1 = ld_fr(pm + Hh + i) + ld_fr(pq + Hh + i);
        Fr b2 = ld_fr(pm + 2 * Hh + i) + ld_fr(pq + 2 * Hh + i);
        Fr hi = b1 + b2;
        st_fr(ph + i, hi);
        st_fr(ph + Hh + i, b2);
        if (i >= 1) st_fr(pg + i - 1, b0 + hi);  // g_1 = (X g_1) / X; coefficient 0 of X g_1 is zero
      });
    }
    Oracle o_t; o_t.p = t_poly.p; o_t.len = H;
    Oracle o_g1; o_g1.p = g1.p; o_g1.len = H - 1; o_g1.bounded = true; o_g1.bound = H - 2; o_g1.hiding = true;
    Oracle o_h1; o_h1.p = h1.p; o_h1.len = 2 * H;
    tm.end(t_r2);
    size_t t_c2 = tm.begin("Committing to second round polys");
    std::vector<Oracle*> second = {&o_t, &o_g1, &o_h1};
    commit_round(second, zk);
    tm.end(t_c2);
    absorb_comms(fs, second);
    Fr beta = sample_outside_h(fs);  // verifier_second_round

    // ---- third round [reference prover.rs:588-706] ----------------------------------------------------
    size_t t_r3 = tm.begin("AHP::Prover::ThirdRound");
    Fr v_h_beta = beta.pow_u64(H) - one;
    Fr vv = v_h_alpha * v_h_beta;
    Fr ea_v = eta_a * vv, eb_v = eta_b * vv, ec_v = eta_c * vv;
    DBuf<Fr> f_poly(cx, K), h2(cx, K);
    {
      DBuf<Fr> b_ev(cx, K), f_ev(cx, K), b_poly(cx, K);
      const Fr* prow = ieval[0].p; const Fr* pcol = ieval[1].p; const Fr* pva = ieval[2].p; const Fr* pvb = ieval[3].p;
      const Fr* pvc = ieval[4].p;
      Fr* pb = b_ev.p; Fr* pf = f_ev.p;
      // b|_K = alpha beta - alpha row - beta col + row_col = (beta - row)(alpha - col)
      ew(cx, K, [=] __device__(size_t i) {
        Fr d = (beta - ld_fr(prow + i)) * (alpha - ld_fr(pcol + i));
        st_fr(pb + i, d);
        st_fr(pf + i, d);
      });
      batch_inverse<Fr>(cx, f_ev.p, K);
      ew(cx, K, [=] __device__(size_t i) {
        st_fr(pf + i, ld_fr(pf + i) * (ea_v * ld_fr(pva + i) + eb_v * ld_fr(pvb + i) + ec_v * ld_fr(pvc + i)));
      });
      run_ntt_group({NttJob{nullptr, 0, b_ev.p, b_poly.p, log_k, true}, NttJob{nullptr, 0, f_ev.p, f_poly.p, log_k, true}});
      // b * f on 2|K|; h_2 = (a - b f) / v_K = -(b f)[|K| ..]
      DBuf<Fr> eb2(cx, 2 * K), ef2(cx, 2 * K), bf(cx, 2 * K);
      run_ntt_group({NttJob{b_poly.p, K, nullptr, eb2.p, log_k + 1, false}, NttJob{f_poly.p, K, nullptr, ef2.p, log_k + 1, false}});
      Fr* p1 = eb2.p; const Fr* p2 = ef2.p;
      ew(cx, 2 * K, [=] __device__(size_t i) { st_fr(p1 + i, ld_fr(p1 + i) * ld_fr(p2 + i)); });
      ntt.run(eb2.p, bf.p, log_k + 1, true);
      const Fr* pbf = bf.p; Fr* ph = h2.p;
      ew(cx, K, [=] __device__(size_t i) { st_fr(ph + i, ld_fr(pbf + Kk + i).neg()); });
    }
    Oracle o_g2; o_g2.p = f_poly.p + 1; o_g2.len = K - 1; o_g2.bounded = true; o_g2.bound = K - 2;
    Oracle o_h2; o_h2.p = h2.p; o_h2.len = K - 1;
    tm.end(t_r3);
    size_t t_c3 = tm.begin("Committing to third round polys");
    std::vector<Oracle*> third = {&o_g2, &o_h2};
    commit_round(third, zk);
    tm.end(t_c3);
    absorb_comms(fs, third);
    Fr gamma = field_rand<Fr>(fs);  // verifier_third_round

    // ---- evaluations [reference lib.rs:264-289, mod.rs:110-221] -----------------------------------------
    size_t t_ev = tm.begin("Evaluating linear combinations over query set");
    // S(p, z)[j] = sum_{m >= j} p_m z^(m-j): S[0] = p(z), S[1..] = quotient of p / (X - z)
    DBuf<Fr> s_g1(cx, o_g1.len), s_g2(cx, o_g2.len), s_tmp(cx, H + 1);
    rec_suffix<Fr>(cx, o_g1.p, s_g1.p, o_g1.len, 1, beta, true);
    rec_suffix<Fr>(cx, o_g2.p, s_g2.p, o_g2.len, 1, gamma, true);
    Fr g1_at_beta = download_fr(s_g1.p), g2_at_gamma = download_fr(s_g2.p);
    rec_suffix<Fr>(cx, o_zb.p, s_tmp.p, o_zb.len, 1, beta, true);
    Fr zb_at_beta = download_fr(s_tmp.p);
    rec_suffix<Fr>(cx, o_t.p, s_tmp.p, o_t.len, 1, beta, true);
    Fr t_at_beta = download_fr(s_tmp.p);
    Fr evals[4] = {g1_at_beta, g2_at_gamma, t_at_beta, zb_at_beta};  // sorted by label: g_1, g_2, t, z_b
    {
      std::vector<uint8_t> eb;
      for (auto& e : evals) put_fr_canonical(eb, e);
      fs.absorb(eb);
    }
    // opening_challenge: F::from(u128::rand(fs_rng))  [reference lib.rs:290]
    Fr xi;
    {
      uint64_t lo = fs.next_u64(), hi = fs.next_u64();
      Fr c = Fr::zero();
      c.l[0] = (uint32_t)lo; c.l[1] = (uint32_t)(lo >> 32); c.l[2] = (uint32_t)hi; c.l[3] = (uint32_t)(hi >> 32);
      xi = Fr::from_canonical(c);
    }
    // linear-combination coefficients [reference mod.rs:145-213], shared with the verifier (verify_core.cuh); the prover skips the
    // constant terms, so x_hat(beta) is not needed here
    const LcCoeffs<Fr> lc = lc_coefficients(Challenges<Fr>{alpha, eta_a, eta_b, eta_c, beta, gamma}, evals, H, K, X, Fr::zero());
    const Fr c_za = lc.za, c_w = lc.w, c_h1 = lc.h1;
    const Fr ci_a = lc.a, ci_b = lc.b, ci_c = lc.c, ci_row = lc.row, ci_col = lc.col, ci_rc = lc.rc, ci_h2 = lc.h2;
    tm.end(t_ev);

    // ---- open_combinations [U ark-poly-commit marlin_pc / sonic_pc; SURVEY.md App. B] ---------------------
    size_t t_op = tm.begin("PC::open_combinations");
    Fr xp[6];
    xp[0] = one;
    for (int i = 1; i < 6; i++) xp[i] = xp[i - 1] * xi;
    const bool marlin = pc == B2M_PC_MARLIN_KZG10;
    // challenge indices: Marlin PC burns two per degree-bounded polynomial, Sonic one per polynomial
    const Fr ch_outer = marlin ? xp[2] : xp[1], ch_t = marlin ? xp[3] : xp[2], ch_zb = marlin ? xp[4] : xp[3];
    const Fr ch_inner = marlin ? xp[2] : xp[1];
    DBuf<Pt> w_out(cx, 2);
    std::vector<MsmJob<Fr, Fq>> shifted_jobs, final_jobs;
    HPoly r_beta;       // combined hiding randomness at beta
    HPoly sr_beta;      // shifted randomness (Marlin PC): xi * shifted_rand(g_1)
    std::vector<DBuf<Fr>> keep_sc;
    std::vector<DBuf<Xy>> keep_pt;
    {
      // point beta: labels g_1, outer_sumcheck, t, z_b
      DBuf<Fr> pbeta(cx, 3 * H), sbeta(cx, 3 * H);
      LcTerms<Fr> lt;
      lt.add(o_g1.p, o_g1.len, one);
      lt.add(o_mask.p, o_mask.len, ch_outer);
      lt.add(o_za.p, o_za.len, ch_outer * c_za);
      lt.add(o_w.p, o_w.len, ch_outer * c_w);
      lt.add(o_h1.p, o_h1.len, ch_outer * c_h1);
      lt.add(o_t.p, o_t.len, ch_t);
      lt.add(o_zb.p, o_zb.len, ch_zb);
      lincomb(lt, 3 * H, pbeta.p);
      rec_suffix<Fr>(cx, pbeta.p, sbeta.p, 3 * H, 1, beta, true);
      hp_axpy(r_beta, one, o_g1.rand);
      HPoly r_outer;
      hp_axpy(r_outer, c_za, o_za.rand);
      hp_axpy(r_outer, c_w, o_w.rand);
      hp_axpy(r_beta, ch_outer, r_outer);
      hp_axpy(r_beta, ch_zb, o_zb.rand);
      HPoly hw = hp_is_zero(r_beta) ? HPoly() : hp_div_linear(r_beta, beta);  // hiding witness r / (X - beta)
      DBuf<Xy> ex(cx, 2);
      int n_extra = 0;
      if (marlin) {
        hp_axpy(sr_beta, xp[1], o_g1.shifted_rand);
        if (!hp_is_zero(o_g1.shifted_rand)) hp_axpy(hw, xp[1], hp_div_linear(o_g1.shifted_rand, beta));
        // shifted witness: xi * (g_1 / (X - beta)) against powers_of_g[D - (|H| - 2) ..]
        DBuf<Fr> sw(cx, o_g1.len);
        const Fr* ps = s_g1.p + 1; Fr* pd = sw.p; const Fr x1 = xp[1];
        ew(cx, o_g1.len - 1, [=] __device__(size_t i) { st_fr(pd + i, ld_fr(ps + i) * x1); });
        shifted_jobs.push_back(MsmJob<Fr, Fq>{sw.p, true, o_g1.len - 1, shifted_off(o_g1.bound), nullptr, 0, 0, nullptr, 0, ex.p + n_extra,
                                              nullptr});
        n_extra++;
        keep_sc.push_back(std::move(sw));
      }
      const Fr* hw_dev = nullptr;
      if (!hw.empty()) {
        keep_sc.emplace_back(cx, hw.size());
        keep_sc.back().upload(hw.data(), hw.size());
        hw_dev = keep_sc.back().p;
      }
      final_jobs.push_back(MsmJob<Fr, Fq>{sbeta.p + 1, true, 3 * H - 1, 0, hw_dev, hw.size(), srs->gamma_slot(0), ex.p, n_extra, nullptr,
                                          w_out.p});
      keep_pt.push_back(std::move(ex));
      keep_sc.push_back(std::move(pbeta));
      keep_sc.push_back(std::move(sbeta));
    }
    {
      // point gamma: labels g_2, inner_sumcheck (nothing hiding)
      DBuf<Fr> pg(cx, K), sg(cx, K);
      LcTerms<Fr> lt;
      lt.add(o_g2.p, o_g2.len, one);
      lt.add(ipoly[2].p, K, ch_inner * ci_a);
      lt.add(ipoly[3].p, K, ch_inner * ci_b);
      lt.add(ipoly[4].p, K, ch_inner * ci_c);
      lt.add(ipoly[0].p, K, ch_inner * ci_row);
      lt.add(ipoly[1].p, K, ch_inner * ci_col);
      lt.add(ipoly[5].p, K, ch_inner * ci_rc);
      lt.add(o_h2.p, o_h2.len, ch_inner * ci_h2);
      lincomb(lt, K, pg.p);
      rec_suffix<Fr>(cx, pg.p, sg.p, K, 1, gamma, true);
      DBuf<Xy> ex(cx, 1);
      int n_extra = 0;
      if (marlin) {
        DBuf<Fr> sw(cx, o_g2.len);
        const Fr* ps = s_g2.p + 1; Fr* pd = sw.p; const Fr x1 = xp[1];
        ew(cx, o_g2.len - 1, [=] __device__(size_t i) { st_fr(pd + i, ld_fr(ps + i) * x1); });
        shifted_jobs.push_back(MsmJob<Fr, Fq>{sw.p, true, o_g2.len - 1, shifted_off(o_g2.bound), nullptr, 0, 0, nullptr, 0, ex.p, nullptr});
        n_extra = 1;
        keep_sc.push_back(std::move(sw));
      }
      final_jobs.push_back(MsmJob<Fr, Fq>{sg.p + 1, true, K - 1, 0, nullptr, 0, 0, ex.p, n_extra, nullptr, w_out.p + 1});
      keep_pt.push_back(std::move(ex));
      keep_sc.push_back(std::move(pg));
      keep_sc.push_back(std::move(sg));
    }
    // the shifted parts feed the final points as `extra` terms, so they form their own (earlier) batch
    if (!shifted_jobs.empty()) msm.run_batch(shifted_jobs.data(), (int)shifted_jobs.size());
    msm.run_batch(final_jobs.data(), (int)final_jobs.size());
    Pt w_pts[2];
    w_out.download(w_pts, 2);
    tm.end(t_op);

    // ---- Proof::new + CanonicalSerialize [reference data_structures.rs:100-126; SURVEY.md A.3] -----------
    proof.clear();
    put_u64(proof, 3);
    std::vector<Oracle*>* rounds[3] = {&first, &second, &third};
    for (auto* rd : rounds) {
      put_u64(proof, rd->size());
      for (auto* o : *rd) {
        put_compressed(proof, o->comm);
        if (marlin) {
          if (o->bounded) { proof.push_back(1); put_compressed(proof, o->shifted_comm); }
          else proof.push_back(0);
        }
      }
    }
    put_u64(proof, 4);
    for (auto& e : evals) put_fr_canonical(proof, e);
    put_u64(proof, 3);
    proof.push_back(0); proof.push_back(0); proof.push_back(0);  // three ProverMsg::EmptyMessage
    put_u64(proof, 2);
    put_compressed(proof, w_pts[0]);
    {
      // random_v at beta: r(beta) (+ shifted_r(beta) for Marlin PC); Some iff the combined randomness is hiding
      bool hiding = !hp_is_zero(r_beta);
      if (hiding) {
        Fr rv = hp_eval(r_beta, beta);
        if (marlin) rv = rv + hp_eval(sr_beta, beta);
        proof.push_back(1);
        put_fr_canonical(proof, rv);
      } else {
        proof.push_back(0);
      }
    }
    put_compressed(proof, w_pts[1]);
    proof.push_back(0);  // gamma: no hiding polynomial is opened there
    proof.push_back(0);  // BatchLCProof.evals = None
    zk.commit_position();
    tm.end(t_all);
    timings_json = tm.json();
  }

  // DensePolynomial::rand(3|H| - 1, zk_rng): on the device when the rng is a ChaCha stream position (attempts are 8-word
  // slices of the stream), on the host through the caller's callback otherwise (one upload).
  void sample_mask(ZkSource<b2m_rng>& zks, Fr* out, size_t need) {
    if (zks.callback) {
      std::vector<Fr> h(need);
      for (size_t i = 0; i < need; i++) h[i] = field_rand<Fr>(zks);
      B2M_CUDA(cudaMemcpyAsync(out, h.data(), need * sizeof(Fr), cudaMemcpyHostToDevice, cx.stream));
      cx.sync();
      return;
    }
    ChaChaHost& zk = zks.cc;
    ChaChaKey key;
    memcpy(key.k, zk.key, 32);
    size_t have = 0;
    while (have < need) {
      size_t want = need - have;
      size_t na = want + want / 8 + 1024;  // acceptance probability ~0.906 for BLS12-381, 0.76 for BN254 (loops if short)
      DBuf<Fr> cand(cx, na);
      DBuf<uint32_t> acc(cx, na), rank(cx, na);
      DBuf<unsigned long long> last(cx, 1);
      B2M_CUDA(cudaMemsetAsync(last.p, 0xff, sizeof(unsigned long long), cx.stream));
      sample_attempts_kernel<Fr><<<div_up(na, 128), 128, 0, cx.stream>>>(key, zk.rounds, zk.word_pos, na, cand.p, acc.p);
      B2M_CHECK_LAUNCH();
      cx.launches++;
      exclusive_scan_u32(cx, acc.p, rank.p, na);
      sample_compact_kernel<Fr><<<div_up(na, 256), 256, 0, cx.stream>>>(cand.p, acc.p, rank.p, na, have, need, out, last.p);
      B2M_CHECK_LAUNCH();
      cx.launches++;
      unsigned long long h_last;
      uint32_t tail[2];
      last.download(&h_last, 1);
      B2M_CUDA(cudaMemcpyAsync(&tail[0], rank.p + na - 1, 4, cudaMemcpyDeviceToHost, cx.stream));
      B2M_CUDA(cudaMemcpyAsync(&tail[1], acc.p + na - 1, 4, cudaMemcpyDeviceToHost, cx.stream));
      cx.sync();
      size_t accepted = (size_t)tail[0] + tail[1];
      if (h_last != ~0ull) {  // reached `need`: the stream position is right after that attempt
        zk.word_pos += 8ull * (h_last + 1);
        have = need;
      } else {
        zk.word_pos += 8ull * na;
        have += accepted;
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------------
// Level 1: `PC::commit` over host polynomials [U ark-poly-commit marlin_pc / sonic_pc commit]
// ---------------------------------------------------------------------------------------------------
template <class Fr, class Fq>
void pc_commit_impl(b2m_srs* srs, Msm<Fr, Fq>& msm, int pc, size_t n_polys, const uint64_t* const* coeffs, const size_t* n_coeffs,
                    const int64_t* degree_bounds, const int64_t* hiding_bounds, b2m_rng* rng, uint64_t* out_comm_xy,
                    uint64_t* out_shifted_xy, uint64_t* out_rand, uint64_t* out_shifted_rand, size_t rand_stride) {
  using Pt = Affine<Fq>;
  Ctx& cx = srs->ctx->cx;
  const size_t D = srs->n_g - 1;
  const bool marlin = pc == B2M_PC_MARLIN_KZG10;
  bool any_hiding = false;
  for (size_t i = 0; i < n_polys; i++) any_hiding = any_hiding || hiding_bounds[i] >= 0;
  B2M_REQUIRE(!any_hiding || rng != nullptr, B2M_ERR_MISSING_RNG, "a hiding bound was requested but rng is null");
  ZkSource<b2m_rng> zk(rng);
  std::vector<DBuf<Fr>> polys, blind;
  std::vector<MsmJob<Fr, Fq>> jobs;
  DBuf<Pt> out(cx, 2 * n_polys);
  B2M_CUDA(cudaMemsetAsync(out.p, 0, 2 * n_polys * sizeof(Pt), cx.stream));
  memset(out_rand, 0, n_polys * rand_stride * sizeof(Fr));
  if (out_shifted_rand) memset(out_shifted_rand, 0, n_polys * rand_stride * sizeof(Fr));
  auto draw = [&](int64_t hb, uint64_t* dst) -> std::vector<Fr> {
    std::vector<Fr> r;
    if (hb < 0) return r;
    B2M_REQUIRE((size_t)hb + 2 <= rand_stride, B2M_ERR_INVALID_ARG, "rand_stride %zu < hiding bound %lld + 2", rand_stride, (long long)hb);
    for (int64_t k = 0; k < hb + 2; k++) r.push_back(field_rand<Fr>(zk));  // Randomness::rand: degree hiding_bound + 1
    memcpy(dst, r.data(), r.size() * sizeof(Fr));
    return r;
  };
  auto job = [&](const Fr* dev, size_t len, size_t off, const std::vector<Fr>& b, size_t gslot, Pt* dst) {
    const Fr* s2 = nullptr;
    if (!b.empty()) {
      blind.emplace_back(cx, b.size());
      blind.back().upload(b.data(), b.size());
      s2 = blind.back().p;
      for (size_t k = 1; k < b.size(); k++)
        B2M_REQUIRE(srs->gamma_slot(srs->gamma_idx[gslot] + k) == gslot + k, B2M_ERR_INVALID_ARG, "gamma powers are not consecutive");
    }
    jobs.push_back(MsmJob<Fr, Fq>{dev, true, len, off, s2, b.size(), gslot, nullptr, 0, nullptr, dst});
  };
  for (size_t i = 0; i < n_polys; i++) {
    const size_t len = n_coeffs[i];
    B2M_REQUIRE(len <= srs->n_g, B2M_ERR_DEGREE_TOO_LARGE, "polynomial %zu has %zu coefficients, the SRS %zu powers", i, len, srs->n_g);
    polys.emplace_back(cx, len ? len : 1);
    if (len) polys.back().upload(reinterpret_cast<const Fr*>(coeffs[i]), len);
    const int64_t d = degree_bounds[i], hb = hiding_bounds[i];
    if (d >= 0) {
      B2M_REQUIRE((size_t)d <= D && len <= (size_t)d + 1, B2M_ERR_DEGREE_TOO_LARGE, "polynomial %zu exceeds its degree bound %lld", i, (long long)d);
    }
    if (marlin) {
      job(polys.back().p, len, 0, draw(hb, out_rand + 4 * rand_stride * i), hb >= 0 ? srs->gamma_slot(0) : 0, out.p + 2 * i);
      if (d >= 0)
        job(polys.back().p, len, D - (size_t)d, draw(hb, out_shifted_rand + 4 * rand_stride * i), hb >= 0 ? srs->gamma_slot(0) : 0,
            out.p + 2 * i + 1);
    } else {
      if (d >= 0) job(polys.back().p, len, D - (size_t)d, draw(hb, out_rand + 4 * rand_stride * i), hb >= 0 ? srs->gamma_slot(D - (size_t)d) : 0, out.p + 2 * i);
      else job(polys.back().p, len, 0, draw(hb, out_rand + 4 * rand_stride * i), hb >= 0 ? srs->gamma_slot(0) : 0, out.p + 2 * i);
    }
  }
  for (size_t at = 0; at < jobs.size(); at += MSM_MAX_BATCH)
    msm.run_batch(jobs.data() + at, (int)std::min<size_t>(MSM_MAX_BATCH, jobs.size() - at));
  std::vector<Pt> h(2 * n_polys);
  out.download(h.data(), h.size());
  for (size_t i = 0; i < n_polys; i++) {
    memcpy(out_comm_xy + i * (2 * Fq::N / 2), &h[2 * i], sizeof(Pt));
    if (out_shifted_xy) memcpy(out_shifted_xy + i * (2 * Fq::N / 2), &h[2 * i + 1], sizeof(Pt));
  }
  zk.commit_position();
}

// ---------------------------------------------------------------------------------------------------
// Level 1: `PC::open_individual_opening_challenges` at one point [U ark-poly-commit marlin_pc / sonic_pc open]
// ---------------------------------------------------------------------------------------------------
template <class Fr>
struct OpenItem {  // one labelled polynomial resident in HBM, with its commitment randomness
  const Fr* dev;
  size_t len;
  int64_t bound;  // degree bound or -1
  std::vector<Fr> rand, srand;  // blinding polynomials (trailing zeros stripped; empty = not hiding)
};

template <class Fr, class Fq>
void pc_open_point_dev(b2m_srs* srs, Msm<Fr, Fq>& msm, int pc, const std::vector<OpenItem<Fr>>& items, int64_t max_degree_bound, const Fr& z,
                       const Fr& xi, uint64_t* out_w_xy, int* out_has_random_v, uint64_t* out_random_v) {
  using Pt = Affine<Fq>;
  using Xy = XYZZ<Fq>;
  using M = MarlinIndex<Fr, Fq>;
  typedef typename M::HPoly HPoly;
  Ctx& cx = srs->ctx->cx;
  const size_t D = srs->n_g - 1;
  const bool marlin = pc == B2M_PC_MARLIN_KZG10;
  const Fr one = Fr::one();
  size_t max_len = 1;
  for (auto& it : items) max_len = std::max(max_len, it.len);
  std::vector<DBuf<Fr>> keep;
  DBuf<Fr> comb(cx, max_len), tmp(cx, max_len);
  comb.zero();
  std::vector<MsmJob<Fr, Fq>> shifted_jobs;
  DBuf<Xy> ex(cx, items.size() + 1);
  int n_extra = 0;
  HPoly r, sr, srw;
  Fr ch = one;
  bool enforce = false;
  for (auto& it : items) {
    const size_t len = it.len;
    B2M_REQUIRE(len <= srs->n_g, B2M_ERR_DEGREE_TOO_LARGE, "a polynomial has %zu coefficients, the SRS %zu powers", len, srs->n_g);
    // comb += ch * p_i
    LcTerms<Fr> lt;
    lt.add(comb.p, max_len, one);
    lt.add(it.dev, len, ch);
    lincomb_kernel<Fr><<<div_up(max_len, 256), 256, 0, cx.stream>>>(lt, max_len, tmp.p);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    std::swap(comb, tmp);
    M::hp_axpy(r, ch, it.rand);
    ch = ch * xi;
    if (marlin && it.bound >= 0) {
      B2M_REQUIRE(max_degree_bound >= it.bound && (size_t)max_degree_bound <= D, B2M_ERR_DEGREE_TOO_LARGE, "bad degree bounds");
      enforce = true;
      if (len > 1) {
        // shifted witness ch1 * (p_i / (X - z)) against shifted_powers: powers_of_g[D - bound ..]
        keep.emplace_back(cx, len);
        DBuf<Fr>& sfx_i = keep.back();
        rec_suffix<Fr>(cx, it.dev, sfx_i.p, len, 1, z, true);
        Fr* ps = sfx_i.p;
        const Fr c1 = ch;
        ew(cx, len - 1, [=] __device__(size_t k) { st_fr(ps + 1 + k, ld_fr(ps + 1 + k) * c1); });
        shifted_jobs.push_back(MsmJob<Fr, Fq>{sfx_i.p + 1, true, len - 1, D - (size_t)it.bound, nullptr, 0, 0, nullptr, 0, ex.p + n_extra, nullptr});
        n_extra++;
      }
      M::hp_axpy(sr, ch, it.srand);
      if (!M::hp_is_zero(it.srand)) M::hp_axpy(srw, ch, M::hp_div_linear(it.srand, z));
      ch = ch * xi;
    }
  }
  // witness of the combination and its hiding part
  DBuf<Fr> sfx(cx, max_len);
  rec_suffix<Fr>(cx, comb.p, sfx.p, max_len, 1, z, true);
  const bool hiding = !M::hp_is_zero(r);
  HPoly hw = hiding ? M::hp_div_linear(r, z) : HPoly();
  if (marlin && enforce) M::hp_axpy(hw, one, srw);
  const Fr* hw_dev = nullptr;
  if (!hw.empty()) {
    keep.emplace_back(cx, hw.size());
    keep.back().upload(hw.data(), hw.size());
    hw_dev = keep.back().p;
  }
  for (size_t at = 0; at < shifted_jobs.size(); at += MSM_MAX_BATCH)
    msm.run_batch(shifted_jobs.data() + at, (int)std::min<size_t>(MSM_MAX_BATCH, shifted_jobs.size() - at));
  DBuf<Pt> w(cx, 1);
  MsmJob<Fr, Fq> fin{sfx.p + 1, true, max_len - 1, 0, hw_dev, hw.size(), hw.empty() ? 0 : srs->gamma_slot(0), ex.p, n_extra, nullptr, w.p};
  msm.run_batch(&fin, 1);
  Pt hwp;
  w.download(&hwp, 1);
  memcpy(out_w_xy, &hwp, sizeof(hwp));
  *out_has_random_v = hiding ? 1 : 0;
  Fr rv = Fr::zero();
  if (hiding) {
    rv = M::hp_eval(r, z);
    if (marlin && enforce) rv = rv + M::hp_eval(sr, z);
  }
  memcpy(out_random_v, rv.l, sizeof(rv.l));
}

template <class Fr>
static std::vector<Fr> host_rand_poly(const uint64_t* base, size_t rand_stride, size_t i) {
  std::vector<Fr> h;
  if (!base) return h;
  for (size_t k = 0; k < rand_stride; k++) {
    Fr c;
    memcpy(c.l, base + 4 * (rand_stride * i + k), sizeof(c.l));
    h.push_back(c);
  }
  while (!h.empty() && h.back().is_zero()) h.pop_back();
  return h;
}

template <class Fr, class Fq>
void pc_open_impl(b2m_srs* srs, Ntt<Fr>& ntt, Msm<Fr, Fq>& msm, int pc, size_t n_polys, const uint64_t* const* coeffs,
                  const size_t* n_coeffs, const int64_t* degree_bounds, const uint64_t* rands, const uint64_t* shifted_rands,
                  size_t rand_stride, int64_t max_degree_bound, const uint64_t* point, const uint64_t* opening_challenge,
                  uint64_t* out_w_xy, int* out_has_random_v, uint64_t* out_random_v) {
  (void)ntt;
  Ctx& cx = srs->ctx->cx;
  Fr z, xi;
  memcpy(z.l, point, sizeof(z.l));
  memcpy(xi.l, opening_challenge, sizeof(xi.l));
  std::vector<DBuf<Fr>> dev;
  std::vector<OpenItem<Fr>> items;
  for (size_t i = 0; i < n_polys; i++) {
    const size_t len = n_coeffs[i];
    B2M_REQUIRE(len <= srs->n_g, B2M_ERR_DEGREE_TOO_LARGE, "polynomial %zu has %zu coefficients, the SRS %zu powers", i, len, srs->n_g);
    dev.emplace_back(cx, len ? len : 1);
    if (len) dev.back().upload(reinterpret_cast<const Fr*>(coeffs[i]), len);
    items.push_back(OpenItem<Fr>{dev.back().p, len, degree_bounds[i], host_rand_poly<Fr>(rands, rand_stride, i),
                                 host_rand_poly<Fr>(shifted_rands, rand_stride, i)});
  }
  pc_open_point_dev<Fr, Fq>(srs, msm, pc, items, max_degree_bound, z, xi, out_w_xy, out_has_random_v, out_random_v);
}

// ---------------------------------------------------------------------------------------------------
// Level 1: `PC::open_combinations` [U ark-poly-commit marlin_pc / sonic_pc open_combinations_individual_opening_challenges]
// ---------------------------------------------------------------------------------------------------
template <class Fr, class Fq>
void pc_open_combinations_impl(b2m_srs* srs, Msm<Fr, Fq>& msm, int pc, int64_t max_degree_bound, size_t n_polys, const uint64_t* const* coeffs,
                               const size_t* n_coeffs, const int64_t* degree_bounds, const int* hiding, const uint64_t* rands,
                               const uint64_t* shifted_rands, size_t rand_stride, size_t n_lcs, const size_t* lc_term_off, const int64_t* lc_poly,
                               const uint64_t* lc_coeff, size_t n_queries, const size_t* query_lc, const size_t* query_point, size_t n_points,
                               const uint64_t* points, const uint64_t* opening_challenge, uint64_t* out_w_xy, int* out_has_random_v,
                               uint64_t* out_random_v) {
  using M = MarlinIndex<Fr, Fq>;
  Ctx& cx = srs->ctx->cx;
  const bool marlin = pc == B2M_PC_MARLIN_KZG10;
  Fr xi;
  memcpy(xi.l, opening_challenge, sizeof(xi.l));
  const Fr one = Fr::one();
  std::vector<DBuf<Fr>> dev;
  for (size_t i = 0; i < n_polys; i++) {
    const size_t len = n_coeffs[i];
    B2M_REQUIRE(len <= srs->n_g, B2M_ERR_DEGREE_TOO_LARGE, "polynomial %zu has %zu coefficients, the SRS %zu powers", i, len, srs->n_g);
    dev.emplace_back(cx, len ? len : 1);
    if (len) dev.back().upload(reinterpret_cast<const Fr*>(coeffs[i]), len);
  }
  // the linear-combination polynomials, their randomness and degree bound
  std::vector<DBuf<Fr>> lc_dev;
  std::vector<OpenItem<Fr>> lcs;
  for (size_t l = 0; l < n_lcs; l++) {
    const size_t t0 = lc_term_off[l], t1 = lc_term_off[l + 1];
    size_t len = 1;
    for (size_t t = t0; t < t1; t++)
      if (lc_poly[t] >= 0) {
        B2M_REQUIRE((size_t)lc_poly[t] < n_polys, B2M_ERR_INVALID_ARG, "linear combination %zu names polynomial %lld of %zu", l, (long long)lc_poly[t], n_polys);
        len = std::max(len, n_coeffs[lc_poly[t]]);
      }
    lc_dev.emplace_back(cx, len);
    lc_dev.back().zero();
    DBuf<Fr> tmp(cx, len);
    OpenItem<Fr> item{nullptr, len, -1, {}, {}};
    const size_t num_terms = t1 - t0;
    for (size_t t = t0; t < t1; t++) {
      if (lc_poly[t] < 0) continue;  // LCTerm::One: affects the evaluation only
      const size_t i = (size_t)lc_poly[t];
      Fr c;
      memcpy(c.l, lc_coeff + 4 * t, sizeof(c.l));
      if (degree_bounds[i] >= 0) {
        B2M_REQUIRE(num_terms == 1 && c == one, B2M_ERR_INVALID_ARG,
                    "linear combination %zu: a degree-bounded polynomial may only appear alone with coefficient one", l);
        item.bound = degree_bounds[i];
      }
      LcTerms<Fr> lt;
      lt.add(lc_dev.back().p, len, one);
      lt.add(dev[i].p, n_coeffs[i], c);
      lincomb_kernel<Fr><<<div_up(len, 256), 256, 0, cx.stream>>>(lt, len, tmp.p);
      B2M_CHECK_LAUNCH();
      cx.launches++;
      std::swap(lc_dev.back(), tmp);
      if (hiding[i]) M::hp_axpy(item.rand, c, host_rand_poly<Fr>(rands, rand_stride, i));
      if (marlin && item.bound >= 0 && hiding[i]) M::hp_axpy(item.srand, c, host_rand_poly<Fr>(shifted_rands, rand_stride, i));
    }
    item.dev = lc_dev.back().p;
    lcs.push_back(std::move(item));
  }
  // one opening per point, the combinations queried there in label (= index) order
  for (size_t p = 0; p < n_points; p++) {
    std::vector<size_t> which;
    for (size_t q = 0; q < n_queries; q++)
      if (query_point[q] == p) {
        B2M_REQUIRE(query_lc[q] < n_lcs, B2M_ERR_INVALID_ARG, "query %zu names linear combination %zu of %zu", q, query_lc[q], n_lcs);
        which.push_back(query_lc[q]);
      }
    std::sort(which.begin(), which.end());
    which.erase(std::unique(which.begin(), which.end()), which.end());
    B2M_REQUIRE(!which.empty(), B2M_ERR_INVALID_ARG, "point %zu is not queried", p);
    std::vector<OpenItem<Fr>> items;
    for (size_t l : which) items.push_back(lcs[l]);
    Fr z;
    memcpy(z.l, points + 4 * p, sizeof(z.l));
    pc_open_point_dev<Fr, Fq>(srs, msm, pc, items, max_degree_bound, z, xi, out_w_xy + p * (2 * Fq::N / 2), out_has_random_v + p, out_random_v + 4 * p);
  }
}

}  // namespace b2m
