// Kernels and member definitions of Msm<Fr, Fq>; included only by the inst_msm_*.cu units.
#pragma once
#include "msm.cuh"
#include "devmem.cuh"
#include "scan.cuh"
#include "msm_affine.cuh"
#include "comm.cuh"

#include <algorithm>

namespace b2m {

template <class Fq>
__device__ __forceinline__ Affine<Fq> ld_affine(const Affine<Fq>* p) {
  Affine<Fq> r;
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint32_t* d = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
  for (int i = 0; i < 2 * Fq::N / 4; i++) {
    uint4 v = __ldg(q + i);
    d[4 * i] = v.x; d[4 * i + 1] = v.y; d[4 * i + 2] = v.z; d[4 * i + 3] = v.w;
  }
  return r;
}
// Out-of-line group operations for everything except the accumulate kernel: keeps the cold kernels
// small (and the build fast); the hot loop in msm_accumulate_kernel stays fully inlined.
template <class Fq> __device__ __noinline__ void g1_add(XYZZ<Fq>& a, const XYZZ<Fq>& b) { a.add(b); }
template <class Fq> __device__ __noinline__ void g1_add_mixed(XYZZ<Fq>& a, const Affine<Fq>& b) { a.add_mixed(b); }
template <class Fq> __device__ __noinline__ void g1_dbl(XYZZ<Fq>& a) { a = a.dbl(); }
template <class Fq> __device__ __noinline__ Fq fq_inverse(const Fq& a) { return a.inverse_fast(); }  // binary Euclid: ~1/5 of the Fermat ladder's latency
template <class Fq> __device__ __noinline__ Affine<Fq> g1_to_affine(const XYZZ<Fq>& p) {
  if (p.is_inf()) return Affine<Fq>::inf();
  Fq izzz = fq_inverse(p.ZZZ);
  Fq izz = (p.ZZ * izzz).sqr();
  return Affine<Fq>{p.X * izz, p.Y * izzz};
}
template <class Fq> __device__ __noinline__ XYZZ<Fq> g1_scalar_mul(const Affine<Fq>& p, const uint32_t* k, int nlimbs) {
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  bool started = false;
  for (int i = nlimbs - 1; i >= 0; i--) {
    for (int b = 31; b >= 0; b--) {
      if (started) g1_dbl(acc);
      if ((k[i] >> b) & 1u) {
        g1_add_mixed(acc, p);
        started = true;
      }
    }
  }
  return acc;
}

// ---- key-load time: window tables ---------------------------------------------------------
// tables[w * n + i] = 2^(c*w) * P_i  (affine).  One thread per power; window w from window w-1.
template <class Fq>
__global__ void msm_precompute_kernel(Affine<Fq>* tables, size_t n, int c, int W) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Affine<Fq> cur = ld_affine(tables + i);
  for (int w = 1; w < W; w++) {
    XYZZ<Fq> acc = XYZZ<Fq>::from_affine(cur);
    for (int k = 0; k < c; k++) g1_dbl(acc);
    cur = g1_to_affine(acc);
    st_words(tables + (size_t)w * n + i, cur);
  }
}

// Multi-GPU key load: keep the powers of this rank's residue class, tables[k] = all[k * world + rank].
template <class Fq>
__global__ void msm_take_residue_kernel(const Affine<Fq>* all, size_t n_loc, int rank, int world, Affine<Fq>* tables) {
  size_t k = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (k >= n_loc) return;
  st_words(tables + k, ld_affine(all + k * (size_t)world + rank));
}

// ---- 1. digits ----------------------------------------------------------------------------
// digits[w * nt + i] = (|d| - 1) | sign << 31, or MSM_NO_DIGIT for d == 0; hist[|d| - 1]++.
// Scalars come in two groups: i < n from `scalars` (the polynomial), the rest from `scalars2`
// (the few blinding coefficients that multiply the gamma powers), nt = n + n2.
template <class Fr>
__global__ void msm_digits_kernel(const Fr* scalars, size_t sstride, const Fr* scalars2, bool MONT, size_t n, size_t nt, int c, int W,
                                  uint32_t* digits, uint32_t* hist) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= nt) return;
  Fr s = i < n ? ld_fr(scalars + i * sstride) : ld_fr(scalars2 + (i - n));
  if (MONT) s = s.to_canonical();
  const uint32_t half = 1u << (c - 1);
  uint32_t carry = 0;
  for (int w = 0; w < W; w++) {
    int bit = w * c;
    int limb = bit >> 5, off = bit & 31;
    uint32_t raw = 0;
    if (limb < Fr::N) {
      raw = s.l[limb] >> off;
      if (off + c > 32 && limb + 1 < Fr::N) raw |= s.l[limb + 1] << (32 - off);
      raw &= (1u << c) - 1;
    }
    uint32_t v = raw + carry;
    uint32_t out;
    if (v > half) {
      uint32_t mag = (1u << c) - v;  // d = v - 2^c < 0
      carry = 1;
      out = (mag - 1) | 0x80000000u;
    } else {
      carry = 0;
      out = v ? (v - 1) : MSM_NO_DIGIT;
    }
    digits[(size_t)w * nt + i] = out;
    if (out != MSM_NO_DIGIT) atomicAdd(hist + (out & 0x7fffffffu), 1u);
  }
}

// ---- 2. exclusive scan of u32: scan.cuh -------------------------------------------------------

// ---- 3. scatter -------------------------------------------------------------------------------
// Counting sort by bucket: sorted[pos] = {(absolute table index) | sign << 31, bucket | window << 24}.
static __global__ void msm_scatter_kernel(const uint32_t* digits, size_t n, size_t nt, size_t base_off, size_t idx2, int W,
                                          uint32_t* cursor, uint2* sorted) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= nt) return;
  uint32_t abs_idx = (uint32_t)(i < n ? base_off + i : idx2 + (i - n));
  for (int w = 0; w < W; w++) {
    uint32_t d = digits[(size_t)w * nt + i];
    if (d == MSM_NO_DIGIT) continue;
    uint32_t bkt = d & 0x7fffffffu;
    uint32_t pos = atomicAdd(cursor + bkt, 1u);
    sorted[pos] = make_uint2(abs_idx | (d & 0x80000000u), bkt | ((uint32_t)w << MSM_BKT_BITS));  // one 8-byte scattered store
  }
}

// ---- 4. accumulate ----------------------------------------------------------------------------
// Balanced bucket accumulation: the references are sorted by bucket, and every thread owns the same
// number (MSM_Q) of consecutive references, so all lanes of a warp run the same number of XYZZ mixed
// additions whatever the bucket-size distribution.  A run of references that covers a whole bucket
// is stored straight into buckets[b]; the (at most two) runs per thread that cut a bucket are stored
// as partials and stitched together by msm_stitch_kernel.  The next point is prefetched while the
// current one is being added.
constexpr int MSM_Q = 64;      // nominal references per thread; the launch picks q near it so the grid is whole waves
constexpr int MSM_Q_MIN = 32;  // buffers are sized for at least this many references per thread
template <class Fq>
__global__ void __launch_bounds__(128)  // 178 registers, 2 CTAs/SM; forcing 3 CTAs/SM (168 regs + spills) measured 5 % slower
msm_accumulate_kernel(const Affine<Fq>* __restrict__ tables, size_t table_stride, const uint32_t* __restrict__ offsets,
                      const uint32_t* __restrict__ ends, const uint2* __restrict__ sorted, const uint32_t* __restrict__ total_refs_p,
                      const uint32_t q, XYZZ<Fq>* __restrict__ buckets, XYZZ<Fq>* __restrict__ part_pt,
                      uint32_t* __restrict__ part_bkt) {
  const uint32_t total = *total_refs_p;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t start64 = (uint64_t)t * q;
  // partial slots 2t (head) and 2t+1 (tail) default to "none"
  uint32_t head_b = MSM_NO_DIGIT, tail_b = MSM_NO_DIGIT;
  if (start64 < total) {
    const uint32_t start = (uint32_t)start64;
    const uint32_t end = (total - start > q) ? start + q : total;
    uint2 rb = __ldg(sorted + start);
    uint32_t ref = rb.x;
    uint32_t cur_b = rb.y & MSM_BKT_MASK;
    uint32_t seg_start = start;
    Affine<Fq> p = ld_affine(tables + (size_t)(rb.y >> MSM_BKT_BITS) * table_stride + (ref & 0x7fffffffu));
    XYZZ<Fq> acc = XYZZ<Fq>::inf();
    for (uint32_t e = start; e < end; e++) {
      Affine<Fq> cur = p;
      const bool neg = ref >> 31;
      uint32_t next_b = cur_b;
      if (e + 1 < end) {
        rb = __ldg(sorted + e + 1);
        ref = rb.x;
        next_b = rb.y & MSM_BKT_MASK;
        p = ld_affine(tables + (size_t)(rb.y >> MSM_BKT_BITS) * table_stride + (ref & 0x7fffffffu));
      }
      acc.add_mixed(cur, neg);
      if (e + 1 == end || next_b != cur_b) {
        // run [seg_start, e] of bucket cur_b ends here
        const bool whole = (seg_start == offsets[cur_b]) && (e + 1 == ends[cur_b]);
        if (whole) {
          st_words(buckets + cur_b, acc);
        } else if (seg_start == start && head_b == MSM_NO_DIGIT) {
          st_words(part_pt + 2 * (size_t)t, acc);
          head_b = cur_b;
        } else {
          st_words(part_pt + 2 * (size_t)t + 1, acc);
          tail_b = cur_b;
        }
        acc = XYZZ<Fq>::inf();
        seg_start = e + 1;
        cur_b = next_b;
      }
    }
  }
  part_bkt[2 * (size_t)t] = head_b;
  part_bkt[2 * (size_t)t + 1] = tail_b;
}
// ---- 4a. batched-affine levels (msm_affine.cuh) ------------------------------------------------------
// cnt[b] = ceil(points of bucket b / 2): sizes of the next level; cnt[B] = 0 so that its scan ends with the total.
static __global__ void msm_level_counts_kernel(const uint32_t* off_in, uint32_t B, uint32_t* cnt) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > B) return;
  cnt[b] = b < B ? (off_in[b + 1] - off_in[b] + 1u) / 2u : 0u;
}
template <class Fq, bool L0>
__global__ void __launch_bounds__(256) msm_affine_plan_kernel(const AffLevel<Fq> A) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < A.nthreads) aff_plan_thread<Fq, L0>(A, t);
}
template <class Fq, int MINB, bool PF>
__global__ void __launch_bounds__(128, MINB) msm_affine_level_kernel(const AffLevel<Fq> A, const Affine<Fq>* __restrict__ base) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < A.nthreads) aff_level_thread<Fq, PF>(A, base, t);
}

// software-pipelined variant (msm_affine.cuh aff_level_thread_sp): variants 8 (3 CTAs/SM), 9 (2), 10 (4)
template <class Fq, int MINB, int PHASE, bool PIPE = true>
__global__ void __launch_bounds__(128, MINB) msm_affine_level_sp_kernel(const AffLevel<Fq> A, const Affine<Fq>* __restrict__ base) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < A.nthreads) aff_level_thread_sp<Fq, PHASE, PIPE>(A, base, t);
}

// v[i] <- 1 / v[i] for all i < n (no zero among them): Montgomery's trick in two levels -- 4 values per thread, a prefix and a
// suffix product scan across the warp (shuffles), ONE inversion per warp (lane 31), back-substitution.  Used by the split level
// kernels to invert all chain products of a level together.
template <class Fq>
__device__ __forceinline__ Fq shfl_fq(const Fq& a, int src_lane) {
  Fq r;
#pragma unroll
  for (int i = 0; i < Fq::N; i++) r.l[i] = __shfl_sync(0xffffffffu, a.l[i], src_lane);
  return r;
}
template <class Fq>
__global__ void __launch_bounds__(128) fq_batch_inverse_kernel(Fq* v, size_t n) {
  constexpr int G = 4;
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const size_t i0 = t * G;
  Fq e[G], pre[G];
  Fq run = Fq::one();
#pragma unroll
  for (int k = 0; k < G; k++) {
    e[k] = i0 + k < n ? ld_words(v + i0 + k) : Fq::one();
    pre[k] = run;
    run = run * e[k];
  }
  // inclusive prefix / suffix products of `run` across the warp
  Fq pin = run, sin = run;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const Fq up = shfl_fq(pin, lane - d < 0 ? lane : lane - d);
    const Fq dn = shfl_fq(sin, lane + d > 31 ? lane : lane + d);
    if (lane >= d) pin = pin * up;
    if (lane + d <= 31) sin = sin * dn;
  }
  Fq tinv = Fq::one();
  if (lane == 31) tinv = fq_inverse(pin);  // 1 / (product of the warp's 128 values)
  tinv = shfl_fq(tinv, 31);
  Fq before = shfl_fq(pin, lane == 0 ? 0 : lane - 1), after = shfl_fq(sin, lane == 31 ? 31 : lane + 1);
  if (lane == 0) before = Fq::one();
  if (lane == 31) after = Fq::one();
  Fq inv_run = tinv * before * after;  // 1 / (this thread's 4 values)
#pragma unroll
  for (int k = G - 1; k >= 0; k--) {
    const Fq ek = inv_run * pre[k];
    inv_run = inv_run * e[k];
    if (i0 + k < n) st_words(v + i0 + k, ek);
  }
}

// Partials are ordered by bucket (they follow the sorted references).  The first partial of each bucket
// sums the ones that follow it and stores the bucket; a bucket cut into many partials (skewed scalar
// distributions, e.g. a polynomial whose coefficients are nearly all equal) is queued for
// msm_stitch_runs_kernel, which reduces it with a whole warp.
struct MsmLongRun {
  uint32_t first, last, bucket;  // partial slots [first, last]
  uint32_t dst;                  // MSM_NO_DIGIT: the run's sum is the bucket; else: chunk-partial slot it goes to
};
constexpr uint32_t MSM_RUN_CHUNK = 256;  // slots one warp folds; longer runs are cut into chunks + one second-stage entry
constexpr uint32_t MSM_RUN_SHORT = 12;   // runs of up to this many slots are folded by ONE thread each (many short runs: the
                                         // full top window of an XYZZ-only pass gives every one of its 2^14 buckets a 6-12 slot run)
template <class Fq>
__global__ void __launch_bounds__(128)
msm_stitch_kernel(const XYZZ<Fq>* part_pt, const uint32_t* part_bkt, size_t nthreads, const uint32_t q, const uint32_t* offsets,
                  const uint32_t* ends, XYZZ<Fq>* buckets, MsmLongRun* long_runs, MsmLongRun* final_runs, MsmLongRun* short_runs, uint32_t* n_long,
                  uint32_t long_cap, uint32_t chunk_cap) {
  // One thread per accumulate-thread u.  A run of partials starts either in u's tail slot (a bucket that
  // begins inside u's range and continues into u + 1) or in u's head slot when the bucket begins exactly at
  // u's first reference; u can hold only one of the two.  The common run is the pair (tail of u, head of
  // u + 1): every lane does exactly one addition.  Longer runs go to msm_stitch_runs_kernel.
  size_t u = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (u >= nthreads) return;
  uint32_t first = 2u * (uint32_t)u + 1u;
  uint32_t b = part_bkt[first];
  if (b == MSM_NO_DIGIT) {
    first = 2u * (uint32_t)u;
    b = part_bkt[first];
    if (b == MSM_NO_DIGIT || offsets[b] != (uint32_t)u * q) return;  // not a run start
  }
  const uint32_t t1 = (ends[b] - 1u) / q;  // thread holding the bucket's last reference
  const uint32_t last = 2u * t1;                          // its head slot closes the run
  if (t1 > (uint32_t)u + 1u) {
    // n_long[0]: queued (first-stage) entries, [1]: second-stage entries, [2]: chunk-partial slots handed out, [3]: short runs
    const uint32_t nslots = last - first + 1u;
    if (nslots <= MSM_RUN_SHORT) {
      const uint32_t slot = atomicAdd(n_long + 3, 1u);
      if (slot < long_cap) {
        short_runs[slot] = MsmLongRun{first, last, b, MSM_NO_DIGIT};
        return;
      }
    } else if (nslots <= MSM_RUN_CHUNK) {
      const uint32_t slot = atomicAdd(n_long, 1u);
      if (slot < long_cap) {
        long_runs[slot] = MsmLongRun{first, last, b, MSM_NO_DIGIT};
        return;
      }
    } else {
      const uint32_t nch = (nslots + MSM_RUN_CHUNK - 1u) / MSM_RUN_CHUNK;
      const uint32_t c0 = atomicAdd(n_long + 2, nch);
      const uint32_t base = atomicAdd(n_long, nch);
      if (c0 + nch <= chunk_cap && base + nch <= long_cap) {
        for (uint32_t k = 0; k < nch; k++) {
          const uint32_t f = first + k * MSM_RUN_CHUNK;
          const uint32_t l = (last - f >= MSM_RUN_CHUNK) ? f + MSM_RUN_CHUNK - 1u : last;
          long_runs[base + k] = MsmLongRun{f, l, b, c0 + k};
        }
        final_runs[atomicAdd(n_long + 1, 1u)] = MsmLongRun{c0, c0 + nch - 1u, b, MSM_NO_DIGIT};  // (at most chunk_cap entries)
        return;
      }
      for (uint32_t k = 0; k < nch && base + k < long_cap; k++) long_runs[base + k] = MsmLongRun{1u, 0u, b, MSM_NO_DIGIT};  // empty entries
    }
    XYZZ<Fq> acc = ld_words(part_pt + first);  // overflow of a queue: fold serially
    for (uint32_t k = first + 1; k <= last; k++)
      if (part_bkt[k] == b) g1_add(acc, ld_words(part_pt + k));
    st_words(buckets + b, acc);
    return;
  }
  XYZZ<Fq> acc = ld_words(part_pt + first);
  g1_add(acc, ld_words(part_pt + last));
  st_words(buckets + b, acc);
}
// Runs longer than a pair (heavy buckets: with a short top window -- e.g. 3 bits at c = 18, which is what an 8-GPU
// shard of a 2^20 key picks -- ALL references of that window land in eight buckets of n / 8 references, each cut into
// thousands of partials).  One WARP per queued entry: the lanes stride over the entry's slots, then a 5-step tree through
// shared memory; runs of more than MSM_RUN_CHUNK slots were queued as chunks whose sums a second launch (FINAL) adds up.
// (Round 1 folded runs of up to 256 slots serially in one thread -- 256 dependent XYZZ additions, ~2 ms of latency per
// MSM -- and longer ones in one block each: `msm_stitch` grew from 1.3 ms to 8-13 ms per proof on 4 and 8 GPUs.)
// short runs: one thread per run, all lanes busy
template <class Fq>
__global__ void __launch_bounds__(128)
msm_stitch_short_kernel(const XYZZ<Fq>* part_pt, const uint32_t* part_bkt, const MsmLongRun* runs, const uint32_t* n_runs, uint32_t cap,
                        XYZZ<Fq>* buckets) {
  uint32_t count = *n_runs;
  if (count > cap) count = cap;
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < count; r += gridDim.x * blockDim.x) {
    const MsmLongRun run = runs[r];
    XYZZ<Fq> acc = ld_words(part_pt + run.first);
    for (uint32_t k = run.first + 1; k <= run.last; k++)
      if (part_bkt[k] == run.bucket) g1_add(acc, ld_words(part_pt + k));
    st_words(buckets + run.bucket, acc);
  }
}
template <class Fq, bool FINAL>
__global__ void __launch_bounds__(128)
msm_stitch_runs_kernel(const XYZZ<Fq>* part_pt, const uint32_t* part_bkt, const MsmLongRun* runs, const uint32_t* n_runs, uint32_t cap,
                       XYZZ<Fq>* buckets, XYZZ<Fq>* chunk_pt) {
  __shared__ uint4 sm_raw[128 * sizeof(XYZZ<Fq>) / 16];
  XYZZ<Fq>* sm = reinterpret_cast<XYZZ<Fq>*>(sm_raw) + (threadIdx.x & ~31u);  // this warp's 32 slots
  const uint32_t lane = threadIdx.x & 31u;
  uint32_t count = *n_runs;
  if (count > cap) count = cap;
  const uint32_t warps = gridDim.x * (blockDim.x >> 5);
  for (uint32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < count; r += warps) {
    const MsmLongRun run = runs[r];
    if (run.first > run.last) continue;  // (placeholder left by an overflowing queue)
    XYZZ<Fq> acc = XYZZ<Fq>::inf();
    for (uint32_t k = run.first + lane; k <= run.last; k += 32) {
      if (FINAL) g1_add(acc, ld_words(chunk_pt + k));
      else if (part_bkt[k] == run.bucket) g1_add(acc, ld_words(part_pt + k));
    }
    sm[lane] = acc;
    __syncwarp();
    for (uint32_t s2 = 16; s2 >= 1; s2 >>= 1) {
      if (lane < s2) {
        XYZZ<Fq> t = sm[lane];
        g1_add(t, sm[lane + s2]);
        sm[lane] = t;
      }
      __syncwarp();
    }
    if (lane == 0) st_words(run.dst == MSM_NO_DIGIT ? buckets + run.bucket : chunk_pt + run.dst, sm[0]);
    __syncwarp();
  }
}

// ---- 5. reduce ----------------------------------------------------------------------------------
// sum_b (b + 1) B_b for a BATCH of bucket arrays at once (the MSMs of one commit round), built from
// log-depth trees so that the latency-bound tail is paid once per round, not once per MSM.
// View bucket index b = hi * L + lo  (R = B / L rows of L columns):
//     sum_b b B_b = L * sum_hi hi * Rsum[hi] + sum_lo lo * Csum[lo],
//     Rsum[hi] = sum_lo B[hi][lo]  (row tree),   Csum[lo] = sum_hi B[hi][lo]  (column tree),
// and each of the two short weighted sums is done by bit planes: sum_i i V_i = sum_k 2^k sum_{i: bit k} V_i.

// Both trees in two launches each, shaped for LATENCY as much as throughput (an XYZZ addition is ~9 us of dependent
// multiplications, and the reduction sits on the critical path of every round: the host needs the commitments to draw the next
// challenges).  Stage 1: one thread per (position, segment) adds K = 8 consecutive summands serially -- this is where the 2^19
// buckets are read, one pass per axis.  Stage 2: one WARP per position folds the remaining len / 8 partials (strided loads, then a
// 5-level tree through shared memory), rows and columns in the same launch.  Depth: 8 + <= 4 + 5 additions per tree (round 1's
// pairwise kernels: 10 launches per tree; a 3-stage serial variant: 36 additions deep).
//     stage 1: out[(g * ni + i) * nseg + s] = sum_{k < K} in[g * group_stride + (s * K + k) * stride_k + i * stride_i]
template <class Fq>
__global__ void __launch_bounds__(128) msm_segsum_kernel(const XYZZ<Fq>* __restrict__ in, XYZZ<Fq>* __restrict__ out, size_t groups, size_t nseg,
                                                         uint32_t K, size_t ni, size_t stride_k, size_t stride_i, size_t group_stride) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (t >= groups * nseg * ni) return;
  // thread order: position fastest for the column sums (stride_i == 1: coalesced), segment fastest for the row sums
  size_t i, sg, g;
  if (stride_i == 1) {
    i = t % ni;
    const size_t gs = t / ni;
    sg = gs % nseg;
    g = gs / nseg;
  } else {
    sg = t % nseg;
    const size_t gi = t / nseg;
    i = gi % ni;
    g = gi / ni;
  }
  const XYZZ<Fq>* p = in + g * group_stride + sg * K * stride_k + i * stride_i;
  XYZZ<Fq> acc = ld_words(p);
  for (uint32_t k = 1; k < K; k++) acc.add(ld_words(p + (size_t)k * stride_k));
  st_words(out + (g * ni + i) * nseg + sg, acc);
}
// stage 2: out[pos] = sum_{s < nseg} in[pos * nseg + s] for two arrays at once (row partials then column partials)
struct MsmFoldJob {
  const void* in;
  void* out;
  size_t positions, nseg;
};
template <class Fq>
__global__ void __launch_bounds__(128) msm_fold_kernel(MsmFoldJob a, MsmFoldJob b) {
  __shared__ uint4 sm_raw[128 * sizeof(XYZZ<Fq>) / 16];
  XYZZ<Fq>* sm = reinterpret_cast<XYZZ<Fq>*>(sm_raw) + (threadIdx.x & ~31u);
  const uint32_t lane = threadIdx.x & 31u;
  size_t w = blockIdx.x * (size_t)(blockDim.x >> 5) + (threadIdx.x >> 5);
  const MsmFoldJob* job = &a;
  if (w >= a.positions) {
    w -= a.positions;
    job = &b;
  }
  if (w >= job->positions) return;  // (whole warps leave together)
  const XYZZ<Fq>* in = reinterpret_cast<const XYZZ<Fq>*>(job->in) + w * job->nseg;
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  for (size_t k = lane; k < job->nseg; k += 32) g1_add(acc, ld_words(in + k));
  sm[lane] = acc;
  __syncwarp();
  for (uint32_t s2 = 16; s2 >= 1; s2 >>= 1) {
    if (lane < s2) {
      XYZZ<Fq> t = sm[lane];
      g1_add(t, sm[lane + s2]);
      sm[lane] = t;
    }
    __syncwarp();
  }
  if (lane == 0) st_words(reinterpret_cast<XYZZ<Fq>*>(job->out) + w, sm[0]);
}
// planes[j][p] for p in [0, nbits]: p < nbits -> sum of V[j][i] over i with bit p set; p == nbits -> sum of all.
// Row planes (blockIdx.x <= rbits) and column planes in one launch.
template <class Fq>
__global__ void __launch_bounds__(256) msm_bitplane_kernel(const XYZZ<Fq>* rsum, size_t R, int rbits, XYZZ<Fq>* rplanes, const XYZZ<Fq>* csum,
                                                           size_t L, int cbits, XYZZ<Fq>* cplanes) {
  __shared__ uint4 sm_raw[256 * sizeof(XYZZ<Fq>) / 16];
  XYZZ<Fq>* sm = reinterpret_cast<XYZZ<Fq>*>(sm_raw);
  const bool rows = (int)blockIdx.x <= rbits;
  const int p = rows ? blockIdx.x : blockIdx.x - (rbits + 1);
  const int nbits = rows ? rbits : cbits;
  const size_t len = rows ? R : L;
  const size_t j = blockIdx.y;
  const XYZZ<Fq>* vec = (rows ? rsum : csum) + j * len;
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  for (size_t i = threadIdx.x; i < len; i += 256)
    if (p == nbits || ((i >> p) & 1)) g1_add(acc, ld_words(vec + i));
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s >= 1; s >>= 1) {
    if ((int)threadIdx.x < s) {
      XYZZ<Fq> t = sm[threadIdx.x];
      g1_add(t, sm[threadIdx.x + s]);
      sm[threadIdx.x] = t;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) st_words((rows ? rplanes : cplanes) + j * (nbits + 1) + p, sm[0]);
}
struct MsmFinishJob {
  const void* extra;  // XYZZ[n_extra] further terms (hiding commitments, shifted parts)
  int n_extra;
  void* out_xyzz;     // XYZZ* or null
  void* out_affine;   // Affine* or null
};
struct MsmFinishJobs {
  MsmFinishJob j[MSM_MAX_BATCH];
};
// One block per job: warp 0 folds the row planes, warp 1 the column planes (Horner over the bits), then
// result = L * Wr + Wc + (sum of all buckets) + extras.  has_buckets = 0: only the extras (empty MSM).
template <class Fq>
__global__ void __launch_bounds__(64) msm_finish_kernel(const XYZZ<Fq>* rplanes, int rbits, const XYZZ<Fq>* cplanes, int cbits,
                                                        int has_buckets, MsmFinishJobs jobs) {
  __shared__ uint4 sm_raw[2 * sizeof(XYZZ<Fq>) / 16];
  XYZZ<Fq>* sm = reinterpret_cast<XYZZ<Fq>*>(sm_raw);
  const int j = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    XYZZ<Fq> acc = XYZZ<Fq>::inf();
    if (has_buckets) {
      const XYZZ<Fq>* pl = warp == 0 ? rplanes + (size_t)j * (rbits + 1) : cplanes + (size_t)j * (cbits + 1);
      int nb = warp == 0 ? rbits : cbits;
      for (int k = nb - 1; k >= 0; k--) {
        g1_dbl(acc);
        g1_add(acc, ld_words(pl + k));
      }
      if (warp == 0) {
        for (int k = 0; k < cbits; k++) g1_dbl(acc);   // * L
        g1_add(acc, ld_words(pl + rbits));               // + sum of all buckets (weights are b + 1)
      }
    }
    sm[warp] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    XYZZ<Fq> total = sm[0];
    g1_add(total, sm[1]);
    const XYZZ<Fq>* extra = reinterpret_cast<const XYZZ<Fq>*>(jobs.j[j].extra);
    for (int i = 0; i < jobs.j[j].n_extra; i++) g1_add(total, ld_words(extra + i));
    if (jobs.j[j].out_xyzz) st_words(reinterpret_cast<XYZZ<Fq>*>(jobs.j[j].out_xyzz), total);
    if (jobs.j[j].out_affine) st_words(reinterpret_cast<Affine<Fq>*>(jobs.j[j].out_affine), g1_to_affine(total));
  }
}

// Multi-GPU: out_j = sum_r partial[r][j] + extras (every rank computes the same sum in the same order).
template <class Fq>
__global__ void __launch_bounds__(32) msm_combine_kernel(const XYZZ<Fq>* all, int world, int nj, MsmFinishJobs jobs) {
  const int j = blockIdx.x;
  if (threadIdx.x != 0) return;
  XYZZ<Fq> total = XYZZ<Fq>::inf();
  for (int r = 0; r < world; r++) g1_add(total, ld_words(all + (size_t)r * nj + j));
  const XYZZ<Fq>* extra = reinterpret_cast<const XYZZ<Fq>*>(jobs.j[j].extra);
  for (int i = 0; i < jobs.j[j].n_extra; i++) g1_add(total, ld_words(extra + i));
  if (jobs.j[j].out_xyzz) st_words(reinterpret_cast<XYZZ<Fq>*>(jobs.j[j].out_xyzz), total);
  if (jobs.j[j].out_affine) st_words(reinterpret_cast<Affine<Fq>*>(jobs.j[j].out_affine), g1_to_affine(total));
}

// ---- fixed-base scalar multiplication (`KZG10::setup`: powers_of_g, powers_of_gamma_g) ---------------------------------
// [U ark-ec FixedBaseMSM::get_window_table / multi_scalar_mul]: one table of j * 2^(8 k) * g (32 windows x 255 multiples,
// 786 KB: L2-resident), then every scalar costs at most 32 mixed additions instead of a 255-step double-and-add; the results
// are normalised together (Montgomery's trick over FB_NORM points per thread: `ProjectiveCurve::batch_normalization`).
constexpr int FB_WIN = 8, FB_WINDOWS = 32, FB_NORM = 16;
template <class Fq>
__global__ void fixed_base_table_kernel(Affine<Fq> g, Affine<Fq>* table) {  // table[k * 256 + j] = j * 2^(8 k) * g  (j = 0: infinity)
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= FB_WINDOWS * 256) return;
  const int k = t >> 8, j = t & 255;
  uint32_t sc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  sc[k >> 2] = (uint32_t)j << (8 * (k & 3));
  st_words(table + t, j ? g1_to_affine(g1_scalar_mul<Fq>(g, sc, 8)) : Affine<Fq>::inf());
}
// out[i] = scalar_i * g with scalar_i = scalars[i] (canonical), or beta^(first + i) when scalars == nullptr
template <class Fr, class Fq>
__global__ void __launch_bounds__(128) fixed_base_mul_kernel(const Affine<Fq>* __restrict__ table, const Fr* scalars, Fr beta, size_t first, size_t n,
                                                             XYZZ<Fq>* out) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Fr k = scalars ? ld_fr(scalars + i) : beta.pow_u64(first + i).to_canonical();
  XYZZ<Fq> acc = XYZZ<Fq>::inf();
  for (int w = 0; w < FB_WINDOWS && w * FB_WIN < 32 * Fr::N; w++) {
    const uint32_t d = (k.l[w >> 2] >> (8 * (w & 3))) & 255u;
    if (d) g1_add_mixed(acc, ld_affine(table + w * 256 + d));
  }
  st_words(out + i, acc);
}
// pts[i] (XYZZ) -> affine: x = X / ZZ, y = Y / ZZZ with one inversion per FB_NORM points
template <class Fq>
__global__ void __launch_bounds__(128) batch_normalize_kernel(const XYZZ<Fq>* pts, size_t n, Affine<Fq>* out) {
  const size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t i0 = t * FB_NORM;
  if (i0 >= n) return;
  const int cnt = (int)(n - i0 < (size_t)FB_NORM ? n - i0 : FB_NORM);
  Fq pref[FB_NORM];
  Fq run = Fq::one();
  for (int k = 0; k < cnt; k++) {
    const Fq zzz = ld_words(&pts[i0 + k].ZZZ);
    pref[k] = run;
    if (!zzz.is_zero()) run = run * zzz;  // (infinity stays out of the product)
  }
  Fq inv = fq_inverse(run);
  for (int k = cnt - 1; k >= 0; k--) {
    const XYZZ<Fq> p = ld_words(pts + i0 + k);
    if (p.is_inf()) {
      st_words(out + i0 + k, Affine<Fq>::inf());
      continue;
    }
    const Fq izzz = inv * pref[k];
    inv = inv * p.ZZZ;
    const Fq izz = (p.ZZ * izzz).sqr();
    st_words(out + i0 + k, Affine<Fq>{p.X * izz, p.Y * izzz});
  }
}

// ---- ark-serialize uncompressed form of G1 points (SRS files) ----------------------------------------------------------------
template <class Fq>
__global__ void g1_canonical_kernel(const Affine<Fq>* in, size_t n, Affine<Fq>* out, bool to_bytes) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  Affine<Fq> p = ld_words(in + i);
  if (to_bytes) {
    const bool inf = p.is_inf();
    p.x = p.x.to_canonical();
    p.y = p.y.to_canonical();
    if (inf) p.y.l[Fq::N - 1] |= 1u << 30;  // SWFlags::Infinity: bit 6 of the last byte
  } else {
    const bool inf = (p.y.l[Fq::N - 1] >> 30) & 1u;
    p.y.l[Fq::N - 1] &= 0x3fffffffu;
    p.x = Fq::from_canonical(p.x);
    p.y = Fq::from_canonical(p.y);
    if (inf) p = Affine<Fq>::inf();
  }
  st_words(out + i, p);
}

// ---- host driver ------------------------------------------------------------------------------
template <class Fr, class Fq>
int Msm<Fr, Fq>::pick_window(size_t n) {
  // n = powers of this key resident on ONE GPU.  The bucket pass costs n * ceil(256 / c) additions per MSM, the reduction
  // ~0.8 ns per bucket plus a latency floor; measured (profiles/r02_scaling_notes.md, 2^20-constraint proofs and their per-rank
  // equivalents): c = 20 (13 windows, 2^19 buckets) wins from 2^21 powers per GPU on, c = 16 (16 windows, 2^15 buckets, a full
  // top window) below that -- 4 and 8 GPUs on a 2^22-power key, or a single GPU on a small one -- and c ~ log2(n) - 1 for tiny keys.
  int lg = 0;
  while (((size_t)1 << (lg + 1)) <= n) lg++;
  int c = lg >= 21 ? 20 : (lg >= 17 ? 16 : lg - 1);
  if (c < MSM_MIN_WINDOW) c = MSM_MIN_WINDOW;
  if (c > 20) c = 20;
  // The top window only holds what is left of the scalar: (BITS + 1) - (W - 1) c bits.  When that is a handful of bits
  // (c = 18: 4, c = 17: 1) EVERY scalar sends its top-window reference to one of a few buckets -- eight buckets of n / 8
  // references each at c = 18 -- which the balanced accumulation then cuts into thousands of partials.  Step to the
  // nearest width whose top window is reasonably full.
  auto top_bits = [](int w) {
    const int W = (Fr::Params::BITS + 1 + w - 1) / w;
    return Fr::Params::BITS + 1 - (W - 1) * w;
  };
  if (top_bits(c) < 6) {
    if (c + 1 <= 20 && top_bits(c + 1) >= 6) c = c + 1;
    else if (c - 1 >= MSM_MIN_WINDOW && top_bits(c - 1) >= 6) c = c - 1;
    else if (c - 2 >= MSM_MIN_WINDOW && top_bits(c - 2) >= 6) c = c - 2;
  }
  return c;
}

template <class Fr, class Fq>
Msm<Fr, Fq>::Msm(Ctx& cx, const Affine<Fq>* host_powers, size_t n, const Affine<Fq>* host_extra, size_t n_extra_bases, int window_bits)
    : ctx(&cx), n_extra(n_extra_bases), n_srs_global(n) {
  // Multi-GPU: GPU r keeps only the powers i = r (mod world) -- every contiguous slice of the key, whatever its
  // offset and length, then splits evenly over the GPUs, and table memory and build time drop by `world`.
  tab_world = cx.world > 1 ? cx.world : 1;
  tab_rank = cx.world > 1 ? cx.rank : 0;
  n_srs = n > (size_t)tab_rank ? (n - tab_rank + tab_world - 1) / tab_world : 0;
  stride = n_srs + n_extra;
  B2M_REQUIRE(n >= 1 && stride < ((size_t)1 << 31), B2M_ERR_INVALID_ARG, "SRS size %zu out of range", n);
  c = window_bits > 0 ? window_bits : pick_window(n / (size_t)tab_world);  // sharded MSMs see n / world pairs per rank
  B2M_REQUIRE(c >= MSM_MIN_WINDOW && c <= 24, B2M_ERR_INVALID_ARG, "window bits %d out of range [%d, 24]", c, MSM_MIN_WINDOW);
  W = (Fr::Params::BITS + 1 + c - 1) / c;
  B2M_REQUIRE(W <= 32, B2M_ERR_INVALID_ARG, "too many windows (%d)", W);
  tables = DBuf<Affine<Fq>>(cx, (size_t)W * stride);
  if (tab_world == 1) {
    tables.upload(host_powers, n);
  } else if (n_srs) {
    DBuf<Affine<Fq>> all(cx, n);
    all.upload(host_powers, n);
    msm_take_residue_kernel<Fq><<<div_up(n_srs, 256), 256, 0, cx.stream>>>(all.p, n_srs, tab_rank, tab_world, tables.p);
    B2M_CHECK_LAUNCH();
    cx.launches++;
  }
  if (n_extra) B2M_CUDA(cudaMemcpyAsync(tables.p + n_srs, host_extra, n_extra * sizeof(Affine<Fq>), cudaMemcpyHostToDevice, cx.stream));
  if (stride) {  // (a rank can own none of a tiny key's powers)
    msm_precompute_kernel<Fq><<<div_up(stride, 128), 128, 0, cx.stream>>>(tables.p, stride, c, W);
    B2M_CHECK_LAUNCH();
    cx.launches++;
  }
  cx.sync();
  B2M_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&acc_ctas_per_sm, msm_accumulate_kernel<Fq>, 128, 0));
  if (acc_ctas_per_sm < 1) acc_ctas_per_sm = 1;
  if (const char* e = getenv("B2M_MSM_AFFINE_LEVELS")) affine_levels = atoi(e);
  if (const char* e = getenv("B2M_MSM_AFFINE_T")) affine_T = affine_T_upper = atoi(e);
  if (const char* e = getenv("B2M_MSM_AFFINE_T_UPPER")) affine_T_upper = atoi(e);
  if (const char* e = getenv("B2M_MSM_AFFINE_CTAS")) affine_ctas = atoi(e);
  if (const char* e = getenv("B2M_MSM_AFFINE_CTAS_UPPER")) affine_ctas_upper = atoi(e);
  if (const char* e = getenv("B2M_MSM_AFFINE_MIN_REFS")) affine_min_refs = (size_t)atoll(e);
  if (const char* e = getenv("B2M_MSM_AFFINE_MAP")) affine_map = atoi(e);

  if (affine_levels < 0) affine_levels = 0;
  if (affine_levels > MSM_MAX_AFFINE_LEVELS) affine_levels = MSM_MAX_AFFINE_LEVELS;
  if (affine_T < 1) affine_T = 1;
  if (affine_T > 1024) affine_T = 1024;
  if (affine_T_upper < 1) affine_T_upper = 1;
  if (affine_T_upper > 1024) affine_T_upper = 1024;
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::run(const Fr* scalars, bool mont, size_t n, size_t base_off, const XYZZ<Fq>* extra, int n_extra,
                      XYZZ<Fq>* out_xyzz, Affine<Fq>* out_affine) {
  MsmJob<Fr, Fq> job{scalars, mont, n, base_off, nullptr, 0, 0, extra, n_extra, out_xyzz, out_affine};
  run_batch(&job, 1);
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::run_batch(const MsmJob<Fr, Fq>* jobs_in, int nj) {
  Ctx& cx = *ctx;
  B2M_REQUIRE(nj >= 1 && nj <= MSM_MAX_BATCH, B2M_ERR_INVALID_ARG, "MSM batch of %d jobs", nj);
  // Multi-GPU (comm.cuh): the prover runs replicated, so every rank holds the full scalar vectors, but only the
  // window tables of the powers i = rank (mod world).  Rank r takes the pairs of its residue class out of every
  // MSM (a strided read of the scalars, a contiguous run of table slots), reduces them to one XYZZ point, and
  // one all-gather of 192 B per MSM per rank exchanges the partial sums.
  MsmJob<Fr, Fq> local[MSM_MAX_BATCH];
  const bool sharded = cx.world > 1;
  B2M_REQUIRE((sharded ? cx.world : 1) == tab_world && (sharded ? cx.rank : 0) == tab_rank, B2M_ERR_INVALID_ARG,
              "this key's tables were built for rank %d of %d; create the SRS after b2m_ctx_attach_comm", tab_rank, tab_world);
  DBuf<XYZZ<Fq>> partial, gathered;
  if (sharded) {
    partial = DBuf<XYZZ<Fq>>(cx, nj);
    gathered = DBuf<XYZZ<Fq>>(cx, (size_t)nj * cx.world);
  }
  for (int j = 0; j < nj; j++) {
    local[j] = jobs_in[j];
    B2M_REQUIRE(jobs_in[j].base_off + jobs_in[j].n <= n_srs_global, B2M_ERR_DEGREE_TOO_LARGE,
                "MSM slice [%zu, %zu) exceeds the SRS (%zu powers)", jobs_in[j].base_off, jobs_in[j].base_off + jobs_in[j].n, n_srs_global);
    if (sharded) {
      // pairs i of the slice with base_off + i = rank (mod world): first one at i = skip, then every world-th
      const size_t G = (size_t)cx.world, off = jobs_in[j].base_off, n = jobs_in[j].n;
      const size_t skip = ((size_t)cx.rank + G - off % G) % G;
      const size_t cnt = n > skip ? (n - skip + G - 1) / G : 0;
      local[j].scalars = jobs_in[j].scalars + skip;
      local[j].scalar_stride = G;
      local[j].base_off = (off + skip) / G;  // table slot of power off + skip = slot * world + rank
      local[j].n = cnt;
      if (cx.rank != 0) { local[j].scalars2 = nullptr; local[j].n2 = 0; }  // the blinding terms go to rank 0
      local[j].extra = nullptr; local[j].n_extra = 0;
      local[j].out_xyzz = partial.p + j; local[j].out_affine = nullptr;
    }
  }
  const MsmJob<Fr, Fq>* jobs = local;
  size_t max_n = 0;
  for (int j = 0; j < nj; j++) {
    B2M_REQUIRE(jobs[j].n == 0 || jobs[j].base_off + jobs[j].n <= n_srs, B2M_ERR_DEGREE_TOO_LARGE, "MSM slot range [%zu, %zu) exceeds the tables (%zu)",
                jobs[j].base_off, jobs[j].base_off + jobs[j].n, n_srs);
    B2M_REQUIRE(jobs[j].n2 == 0 || jobs[j].extra_base + jobs[j].n2 <= n_extra, B2M_ERR_INVALID_ARG, "extra bases out of range");
    max_n = std::max(max_n, jobs[j].n + jobs[j].n2);
  }
  // 32-bit positions: the sorted references, their offsets and the per-thread ranges index W * n references
  B2M_REQUIRE((size_t)W * max_n < ((size_t)1 << 32), B2M_ERR_DEGREE_TOO_LARGE, "MSM of %zu pairs x %d windows exceeds 2^32 bucket references", max_n, W);
  MsmFinishJobs fj;
  for (int j = 0; j < nj; j++) fj.j[j] = MsmFinishJob{jobs[j].extra, jobs[j].n_extra, jobs[j].out_xyzz, jobs[j].out_affine};
  auto exchange = [&]() {  // multi-GPU: gather the per-rank partial sums and fold them (plus the extras) on every rank
    if (!sharded) return;
    size_t spx = cx.span_begin("msm_allgather", (double)nj);
    all_gather_bytes(cx, partial.p, gathered.p, (size_t)nj * sizeof(XYZZ<Fq>));
    MsmFinishJobs oj;
    for (int j = 0; j < nj; j++) oj.j[j] = MsmFinishJob{jobs_in[j].extra, jobs_in[j].n_extra, jobs_in[j].out_xyzz, jobs_in[j].out_affine};
    msm_combine_kernel<Fq><<<nj, 32, 0, cx.stream>>>(gathered.p, cx.world, nj, oj);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    cx.span_end(spx);
  };
  if (max_n == 0) {
    msm_finish_kernel<Fq><<<nj, 64, 0, cx.stream>>>(nullptr, 0, nullptr, 0, 0, fj);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    exchange();
    return;
  }
  const uint32_t B = 1u << (c - 1);
  const int cbits = (c - 1 + 1) / 2, rbits = (c - 1) - cbits;  // L = 2^cbits columns, R = 2^rbits rows
  const size_t L = (size_t)1 << cbits, R = (size_t)1 << rbits;
  DBuf<XYZZ<Fq>> buckets(cx, (size_t)nj * B);
  {
    // Software pipeline over the jobs on three streams.  The counting sorts (memory / atomic bound, ~40 registers per thread)
    // run ahead on the side stream.  The bucket passes (levels, accumulate, stitch: integer-ALU bound) alternate between two
    // lanes, cx.stream and cx.lane1, so that the stages of one pass that leave most SMs idle -- the batch inversions, the
    // short plan / count / scan launches, the stitch, the partial last wave of every kernel -- run under the other pass's
    // throughput kernels.  Jobs are issued largest first: the k-th issued job, order[k], sorts into slot k % slots and runs
    // its bucket pass on lane k % 2.  Every job writes its own bucket array, so neither order nor lane changes a result.
    // Sort slots: a slot is read by its job's bucket pass (level 0, or accumulate and stitch) until the pass ends (ev_acc).
    // With two passes in flight, three slots let the sort of job k + 2 run while k and k + 1 are still on the lanes; the
    // sort of k + 3 waits for the end of k.  Everything else a bucket pass writes exists once per lane (LaneScratch).
    const size_t max_refs = (size_t)W * max_n;
    const size_t max_threads = (max_refs + MSM_Q_MIN - 1) / MSM_Q_MIN + 256;  // launches round up to whole blocks
    const int slots = std::min(nj, 3), lanes = std::min(nj, 2);
    const cudaStream_t lane_stream[2] = {cx.stream, cx.lane1};
    int order[MSM_MAX_BATCH];
    for (int j = 0; j < nj; j++) order[j] = j;
    std::stable_sort(order, order + nj, [&](int a, int b) { return jobs[a].n + jobs[a].n2 > jobs[b].n + jobs[b].n2; });
    DBuf<uint32_t> digits[3], hist[3], offsets[3], cursor[3];
    DBuf<uint2> sorted[3];
    for (int s = 0; s < slots; s++) {
      digits[s] = DBuf<uint32_t>(cx, max_refs); hist[s] = DBuf<uint32_t>(cx, B + 1); offsets[s] = DBuf<uint32_t>(cx, B + 1);
      cursor[s] = DBuf<uint32_t>(cx, B); sorted[s] = DBuf<uint2>(cx, max_refs);
    }
    const uint32_t long_cap = 1u << 18;
    const uint32_t chunk_cap = (uint32_t)(4 * max_threads / MSM_RUN_CHUNK + 4);  // every chunk but a run's last covers MSM_RUN_CHUNK slots
    // batched-affine levels (msm_affine.cuh): level l has at most bound[l] points
    const int LV = max_refs >= affine_min_refs ? affine_levels : 0;  // (the largest job of the batch decides the buffers)
    // the level-0 plan packs (window * stride + index) | sign << 31 into 32 bits (msm_affine.cuh aff_plan_thread)
    B2M_REQUIRE(LV == 0 || (size_t)W * stride < ((size_t)1 << 31), B2M_ERR_DEGREE_TOO_LARGE,
                "window tables of %d x %zu entries exceed the 31-bit index of the batched-affine plan", W, stride);
    size_t bound[MSM_MAX_AFFINE_LEVELS + 1];
    bound[0] = max_refs;
    for (int l = 1; l <= LV; l++) bound[l] = (bound[l - 1] + B) / 2 + 1;
    const size_t T_max = (size_t)std::max(affine_T, affine_T_upper), T_min = (size_t)std::min(affine_T, affine_T_upper);
    const size_t slots_l0 = LV > 0 ? T_max * ((bound[1] + T_max - 1) / T_max + 128) : 0;  // >= T * nthreads at every level, for either mapping
    struct LaneScratch {
      DBuf<uint32_t> part_bkt, n_long;  // n_long: queued long-run entries, second-stage entries, chunk slots, short runs
      DBuf<MsmLongRun> long_runs, short_runs, final_runs;
      DBuf<XYZZ<Fq>> chunk_pt, part_pt;
      DBuf<Affine<Fq>> lvl_pts[2];
      DBuf<uint32_t> lvl_off[2], lvl_cnt;
      DBuf<uint2> lvl_refs;
      DBuf<uint4> lvl_meta;
      DBuf<Fq> lvl_pref, lvl_inv;
    } lane[2];
    for (int i = 0; i < lanes; i++) {
      LaneScratch& ls = lane[i];
      ls.part_bkt = DBuf<uint32_t>(cx, 2 * max_threads); ls.n_long = DBuf<uint32_t>(cx, 4);
      ls.long_runs = DBuf<MsmLongRun>(cx, long_cap); ls.short_runs = DBuf<MsmLongRun>(cx, long_cap);
      ls.final_runs = DBuf<MsmLongRun>(cx, chunk_cap);
      ls.chunk_pt = DBuf<XYZZ<Fq>>(cx, chunk_cap);
      ls.part_pt = DBuf<XYZZ<Fq>>(cx, 2 * max_threads);
      if (LV > 0) {
        ls.lvl_pts[0] = DBuf<Affine<Fq>>(cx, bound[1]);
        if (LV > 1) ls.lvl_pts[1] = DBuf<Affine<Fq>>(cx, bound[2]);
        ls.lvl_off[0] = DBuf<uint32_t>(cx, B + 1); ls.lvl_off[1] = DBuf<uint32_t>(cx, B + 1); ls.lvl_cnt = DBuf<uint32_t>(cx, B + 1);
        ls.lvl_refs = DBuf<uint2>(cx, bound[LV]);
        ls.lvl_meta = DBuf<uint4>(cx, slots_l0);
        ls.lvl_pref = DBuf<Fq>(cx, slots_l0);
        ls.lvl_inv = DBuf<Fq>(cx, slots_l0 / T_min + 256);
      }
    }
    buckets.zero();  // empty buckets are never written: all-zero XYZZ is the point at infinity
    // events are indexed by issue position k
    cudaEvent_t ev_ready, ev_join, ev_sorted[MSM_MAX_BATCH], ev_acc[MSM_MAX_BATCH];
    B2M_CUDA(cudaEventCreateWithFlags(&ev_ready, cudaEventDisableTiming));
    B2M_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
    for (int k = 0; k < nj; k++) {
      B2M_CUDA(cudaEventCreateWithFlags(&ev_sorted[k], cudaEventDisableTiming));
      B2M_CUDA(cudaEventCreateWithFlags(&ev_acc[k], cudaEventDisableTiming));
    }
    B2M_CUDA(cudaEventRecord(ev_ready, cx.stream));  // buffers exist (stream-ordered allocation) and inputs are final
    B2M_CUDA(cudaStreamWaitEvent(cx.side, ev_ready, 0));
    if (lanes > 1) B2M_CUDA(cudaStreamWaitEvent(cx.lane1, ev_ready, 0));
    for (int k = 0; k < nj; k++) {
      const int j = order[k];
      const size_t n = jobs[j].n, nt = jobs[j].n + jobs[j].n2;
      const int s = k % slots;
      LaneScratch& ls = lane[k % 2];
      StreamSwap on_lane(cx, lane_stream[k % 2]);  // this job's DBufs, scans and spans follow its lane
      if (nt == 0) {
        // no sort and no pass; ev_acc[k] still has to mean "slot s is free": the slot's last user may be on the other lane
        if (k >= slots) B2M_CUDA(cudaStreamWaitEvent(cx.stream, ev_acc[k - slots], 0));
        B2M_CUDA(cudaEventRecord(ev_acc[k], cx.stream));
        continue;
      }
      {
        StreamSwap on_side(cx, cx.side);
        if (k >= slots) B2M_CUDA(cudaStreamWaitEvent(cx.side, ev_acc[k - slots], 0));  // the slot's previous user is done
        hist[s].zero();
        size_t sp0 = cx.span_begin("msm_sort", (double)n);
        msm_digits_kernel<Fr><<<div_up(nt, 256), 256, 0, cx.stream>>>(jobs[j].scalars, jobs[j].scalar_stride, jobs[j].scalars2, jobs[j].mont, n, nt, c, W,
                                                                      digits[s].p, hist[s].p);
        B2M_CHECK_LAUNCH();
        exclusive_scan_u32(cx, hist[s].p, offsets[s].p, B + 1);  // hist[B] = 0: offsets[B] = number of references
        B2M_CUDA(cudaMemcpyAsync(cursor[s].p, offsets[s].p, B * sizeof(uint32_t), cudaMemcpyDeviceToDevice, cx.stream));
        msm_scatter_kernel<<<div_up(nt, 256), 256, 0, cx.stream>>>(digits[s].p, n, nt, jobs[j].base_off, n_srs + jobs[j].extra_base, W,
                                                                    cursor[s].p, sorted[s].p);
        B2M_CHECK_LAUNCH();
        cx.launches += 2;
        cx.span_end(sp0);
        B2M_CUDA(cudaEventRecord(ev_sorted[k], cx.side));
      }
      B2M_CUDA(cudaStreamWaitEvent(cx.stream, ev_sorted[k], 0));
      // source of the XYZZ bucket pass: the sorted references into the window tables, or -- after LV batched-affine
      // levels -- the last level's points with one reference each
      const Affine<Fq>* src_tables = tables.p;
      size_t src_stride = stride;
      const uint32_t* src_off = offsets[s].p;
      const uint2* src_sorted = sorted[s].p;
      size_t refs = (size_t)W * nt;  // upper bound on the reference count (zero digits are rare)
      if (LV > 0 && refs >= affine_min_refs) {
        size_t spl = cx.span_begin("msm_affine_levels", (double)n);
        bound[0] = refs;
        for (int l = 1; l <= LV; l++) bound[l] = (bound[l - 1] + B) / 2 + 1;
        const uint32_t* off_in = offsets[s].p;
        for (int l = 0; l < LV; l++) {
          uint32_t* off_out = ls.lvl_off[l & 1].p;
          msm_level_counts_kernel<<<div_up((size_t)B + 1, 256), 256, 0, cx.stream>>>(off_in, B, ls.lvl_cnt.p);
          B2M_CHECK_LAUNCH();
          cx.launches++;
          exclusive_scan_u32(cx, ls.lvl_cnt.p, off_out, (size_t)B + 1);
          const uint32_t lane_step = affine_map ? 32u : 1u;
          const size_t T_l = (size_t)(l == 0 ? affine_T : affine_T_upper);  // additions per thread (and per chain) at this level
          const uint32_t nthreads = (uint32_t)(lane_step * ((bound[l + 1] + (size_t)lane_step * T_l - 1) / ((size_t)lane_step * T_l)));
          AffLevel<Fq> A{tables.p, stride, sorted[s].p, l > 0 ? ls.lvl_pts[(l - 1) & 1].p : nullptr, off_in, off_out, B, ls.lvl_pts[l & 1].p,
                         l == LV - 1 ? ls.lvl_refs.p : nullptr, ls.lvl_pref.p, ls.lvl_meta.p, (uint32_t)T_l, nthreads, lane_step, ls.lvl_inv.p};
          if (l == 0)
            msm_affine_plan_kernel<Fq, true><<<div_up(nthreads, 256), 256, 0, cx.stream>>>(A);
          else
            msm_affine_plan_kernel<Fq, false><<<div_up(nthreads, 256), 256, 0, cx.stream>>>(A);
          const Affine<Fq>* base = l == 0 ? tables.p : ls.lvl_pts[(l - 1) & 1].p;
          const unsigned grid = div_up(nthreads, 128);
          // Kernel variant (B2M_MSM_AFFINE_CTAS / _UPPER; every variant gives the same bytes, profiles/r02_level_kernel_notes.md):
          //   4 (default), 5: fused kernel, loads at use, compiled for that many resident CTAs per SM; 3: operands prefetched (3 CTAs/SM)
          //   8, 9: fused, branch-free and software-pipelined addition pass (3 / 2 CTAs/SM)
          //   11-13: split -- denominator pass + inversion at 5 CTAs/SM, then the addition pass pipelined at 3 / 2 CTAs/SM or plain at 4
          //   21, 22: split with ONE batch inversion of all chain products of the level between the passes
          const int variant = l == 0 ? affine_ctas : affine_ctas_upper;
          static const char* const lvl_names[MSM_MAX_AFFINE_LEVELS] = {"msm_aff_level0", "msm_aff_level1", "msm_aff_level2", "msm_aff_level3",
                                                                       "msm_aff_level4", "msm_aff_level5"};
          const size_t spk = cx.span_begin(lvl_names[l], (double)n);
          switch (variant) {
            case 3: msm_affine_level_kernel<Fq, 3, true><<<grid, 128, 0, cx.stream>>>(A, base); break;
            case 5: msm_affine_level_kernel<Fq, 5, false><<<grid, 128, 0, cx.stream>>>(A, base); break;
            case 8: msm_affine_level_sp_kernel<Fq, 3, 0><<<grid, 128, 0, cx.stream>>>(A, base); break;
            case 9: msm_affine_level_sp_kernel<Fq, 2, 0><<<grid, 128, 0, cx.stream>>>(A, base); break;
            case 11: case 12: case 13:
              msm_affine_level_sp_kernel<Fq, 5, 1><<<grid, 128, 0, cx.stream>>>(A, base);
              if (variant == 11) msm_affine_level_sp_kernel<Fq, 3, 2><<<grid, 128, 0, cx.stream>>>(A, base);
              else if (variant == 12) msm_affine_level_sp_kernel<Fq, 2, 2><<<grid, 128, 0, cx.stream>>>(A, base);
              else msm_affine_level_sp_kernel<Fq, 4, 2, false><<<grid, 128, 0, cx.stream>>>(A, base);
              cx.launches++;
              break;
            // split with the level-wide batch inversion between the two passes (21: plain addition pass at 4 CTAs/SM, 22: pipelined at 3)
            case 21: case 22:
              msm_affine_level_sp_kernel<Fq, 6, 3><<<grid, 128, 0, cx.stream>>>(A, base);
              fq_batch_inverse_kernel<Fq><<<div_up(div_up(nthreads, 4), 128), 128, 0, cx.stream>>>(ls.lvl_inv.p, nthreads);
              if (variant == 21) msm_affine_level_sp_kernel<Fq, 4, 2, false><<<grid, 128, 0, cx.stream>>>(A, base);
              else msm_affine_level_sp_kernel<Fq, 3, 2><<<grid, 128, 0, cx.stream>>>(A, base);
              cx.launches += 2;
              break;
            default: msm_affine_level_kernel<Fq, 4, false><<<grid, 128, 0, cx.stream>>>(A, base); break;
          }
          cx.span_end(spk);
          B2M_CHECK_LAUNCH();
          cx.launches += 2;
          off_in = off_out;
        }
        cx.span_end(spl);
        src_tables = ls.lvl_pts[(LV - 1) & 1].p;
        src_stride = 0;
        src_off = off_in;
        src_sorted = ls.lvl_refs.p;
        refs = bound[LV];
      }
      const uint32_t* src_ends = src_off + 1;   // buckets are contiguous: bucket b ends where b + 1 starts
      const uint32_t* src_total = src_off + B;
      size_t sp = cx.span_begin("msm_accumulate_kernel", (double)n);
      // References per thread: near MSM_Q, chosen so that the grid is a whole number of waves of
      // (SMs x resident CTAs) -- every thread does the same work, so a partial last wave is pure loss.
      const size_t wave = (size_t)cx.sm_count * acc_ctas_per_sm * 128;
      size_t waves = (refs + wave * MSM_Q / 2) / (wave * MSM_Q);
      if (waves < 1) waves = 1;
      uint32_t q = (uint32_t)((refs + waves * wave - 1) / (waves * wave));
      if (q < (uint32_t)MSM_Q_MIN) q = MSM_Q_MIN;
      const size_t nthreads = (refs + q - 1) / q;
      msm_accumulate_kernel<Fq><<<div_up(nthreads, 128), 128, 0, cx.stream>>>(src_tables, src_stride, src_off, src_ends, src_sorted,
                                                                               src_total, q, buckets.p + (size_t)j * B, ls.part_pt.p,
                                                                               ls.part_bkt.p);
      B2M_CHECK_LAUNCH();
      cx.launches++;
      cx.span_end(sp);
      size_t sp1 = cx.span_begin("msm_stitch", (double)n);
      ls.n_long.zero();
      msm_stitch_kernel<Fq><<<div_up(nthreads, 128), 128, 0, cx.stream>>>(ls.part_pt.p, ls.part_bkt.p, nthreads, q, src_off, src_ends,
                                                                           buckets.p + (size_t)j * B, ls.long_runs.p, ls.final_runs.p, ls.short_runs.p, ls.n_long.p,
                                                                           long_cap, chunk_cap);
      msm_stitch_short_kernel<Fq><<<2 * cx.sm_count, 128, 0, cx.stream>>>(ls.part_pt.p, ls.part_bkt.p, ls.short_runs.p, ls.n_long.p + 3, long_cap,
                                                                          buckets.p + (size_t)j * B);
      msm_stitch_runs_kernel<Fq, false><<<4 * cx.sm_count, 128, 0, cx.stream>>>(ls.part_pt.p, ls.part_bkt.p, ls.long_runs.p, ls.n_long.p, long_cap,
                                                                                buckets.p + (size_t)j * B, ls.chunk_pt.p);
      msm_stitch_runs_kernel<Fq, true><<<cx.sm_count, 128, 0, cx.stream>>>(ls.part_pt.p, ls.part_bkt.p, ls.final_runs.p, ls.n_long.p + 1, chunk_cap,
                                                                           buckets.p + (size_t)j * B, ls.chunk_pt.p);
      B2M_CHECK_LAUNCH();
      cx.launches += 4;
      cx.span_end(sp1);
      B2M_CUDA(cudaEventRecord(ev_acc[k], cx.stream));
    }
    if (lanes > 1) {
      // Join lane 1 into cx.stream.  Every buffer of this block is freed at its closing brace below, on cx.stream (a DBuf is
      // freed on the stream that is current when it is destroyed), and lane 1's scratch, the sort slots and `buckets` are
      // read or written on lane 1: those frees, and the reduction after this block, are ordered behind lane 1's work only
      // through this wait.  No buffer that lane 1 uses may be destroyed before this point.  (The side stream needs no join
      // of its own: each of its sorts ends in an ev_sorted that a lane waits for.)
      B2M_CUDA(cudaEventRecord(ev_join, cx.lane1));
      B2M_CUDA(cudaStreamWaitEvent(cx.stream, ev_join, 0));
    }
    cudaEventDestroy(ev_ready);
    cudaEventDestroy(ev_join);
    for (int k = 0; k < nj; k++) {
      cudaEventDestroy(ev_sorted[k]);
      cudaEventDestroy(ev_acc[k]);
    }
  }
  double units = 0;
  for (int j = 0; j < nj; j++) units += (double)jobs[j].n;
  size_t sp2 = cx.span_begin("msm_reduce", units);
  DBuf<XYZZ<Fq>> rsum(cx, (size_t)nj * R), csum(cx, (size_t)nj * L);
  {
    // stage 1: K summands per thread (K = 8, or the whole axis when it is shorter); stage 2: one warp per position
    const uint32_t Kr = (uint32_t)std::min<size_t>(L, 8), Kc = (uint32_t)std::min<size_t>(R, 8);
    const size_t seg_r = L / Kr, seg_c = R / Kc;  // partials per row / per column
    DBuf<XYZZ<Fq>> part_r(cx, (size_t)nj * R * seg_r), part_c(cx, (size_t)nj * L * seg_c);
    msm_segsum_kernel<Fq><<<div_up((size_t)nj * R * seg_r, 128), 128, 0, cx.stream>>>(buckets.p, part_r.p, (size_t)nj, seg_r, Kr, R, 1, L, B);
    msm_segsum_kernel<Fq><<<div_up((size_t)nj * L * seg_c, 128), 128, 0, cx.stream>>>(buckets.p, part_c.p, (size_t)nj, seg_c, Kc, L, L, 1, B);
    const MsmFoldJob fr{part_r.p, rsum.p, (size_t)nj * R, seg_r}, fc{part_c.p, csum.p, (size_t)nj * L, seg_c};
    msm_fold_kernel<Fq><<<div_up(((size_t)nj * R + (size_t)nj * L) * 32, 128), 128, 0, cx.stream>>>(fr, fc);
    B2M_CHECK_LAUNCH();
    cx.launches += 3;
  }
  DBuf<XYZZ<Fq>> rplanes(cx, (size_t)nj * (rbits + 1)), cplanes(cx, (size_t)nj * (cbits + 1));
  msm_bitplane_kernel<Fq><<<dim3(rbits + 1 + cbits + 1, nj), 256, 0, cx.stream>>>(rsum.p, R, rbits, rplanes.p, csum.p, L, cbits, cplanes.p);
  B2M_CHECK_LAUNCH();
  cx.launches++;
  msm_finish_kernel<Fq><<<nj, 64, 0, cx.stream>>>(rplanes.p, rbits, cplanes.p, cbits, 1, fj);
  B2M_CHECK_LAUNCH();
  cx.launches++;
  cx.span_end(sp2);
  exchange();
  // the DBufs are stream-ordered: their frees are enqueued behind the kernels above
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::run_host(size_t base_off, const uint64_t* scalars, size_t n, uint64_t* out_xy, int* out_is_inf) {
  Ctx& cx = *ctx;
  DBuf<Fr> sc(cx, n ? n : 1);
  if (n) sc.upload(reinterpret_cast<const Fr*>(scalars), n);
  DBuf<Affine<Fq>> res(cx, 1);
  run(sc.p, false, n, base_off, nullptr, 0, nullptr, res.p);
  Affine<Fq> h;
  res.download(&h, 1);
  memcpy(out_xy, &h, sizeof(h));
  if (out_is_inf) *out_is_inf = h.is_inf() ? 1 : 0;
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::read_power(size_t i, uint64_t* out_xy) {
  B2M_REQUIRE(i < n_srs_global, B2M_ERR_INVALID_ARG, "power %zu of %zu", i, n_srs_global);
  B2M_REQUIRE(tab_world == 1, B2M_ERR_UNSUPPORTED, "read_power on a sharded key (the power lives on rank %zu)", i % (size_t)tab_world);
  Affine<Fq> h;
  B2M_CUDA(cudaMemcpyAsync(&h, tables.p + i, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
  ctx->sync();
  memcpy(out_xy, &h, sizeof(h));
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::fixed_base_host(Ctx& cx, const uint64_t* g_xy, const uint64_t* scalars, const uint64_t* beta, size_t first, size_t n, uint64_t* out) {
  Affine<Fq> g;
  memcpy(&g, g_xy, sizeof(g));
  Fr b = Fr::zero();
  if (beta) {
    memcpy(&b, beta, sizeof(b));
    b = Fr::from_canonical(b);
  }
  if (n == 0) return;
  DBuf<Affine<Fq>> table(cx, FB_WINDOWS * 256);
  fixed_base_table_kernel<Fq><<<div_up(FB_WINDOWS * 256, 64), 64, 0, cx.stream>>>(g, table.p);
  B2M_CHECK_LAUNCH();
  cx.launches++;
  // in slices, so that a 2^26-power key needs neither 13 GB of XYZZ scratch nor one giant staging copy
  const size_t slice = (size_t)1 << 22;
  DBuf<XYZZ<Fq>> acc(cx, std::min(n, slice));
  DBuf<Affine<Fq>> aff(cx, std::min(n, slice));
  DBuf<Fr> sc;
  if (scalars) sc = DBuf<Fr>(cx, std::min(n, slice));
  for (size_t at = 0; at < n; at += slice) {
    const size_t m = std::min(slice, n - at);
    if (scalars) sc.upload(reinterpret_cast<const Fr*>(scalars) + at, m);
    fixed_base_mul_kernel<Fr, Fq><<<div_up(m, 128), 128, 0, cx.stream>>>(table.p, scalars ? sc.p : nullptr, b, first + at, m, acc.p);
    batch_normalize_kernel<Fq><<<div_up(div_up(m, FB_NORM), 128), 128, 0, cx.stream>>>(acc.p, m, aff.p);
    B2M_CHECK_LAUNCH();
    cx.launches += 2;
    aff.download(reinterpret_cast<Affine<Fq>*>(out) + at, m);
  }
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::g1_to_bytes(Ctx& cx, const Affine<Fq>* dev_pts, const uint64_t* host_pts, size_t n, uint8_t* out) {
  const size_t slice = (size_t)1 << 22;
  DBuf<Affine<Fq>> in, conv(cx, std::min(n, slice) + 1);
  if (!dev_pts) in = DBuf<Affine<Fq>>(cx, std::min(n, slice) + 1);
  for (size_t at = 0; at < n; at += slice) {
    const size_t m = std::min(slice, n - at);
    const Affine<Fq>* src = dev_pts ? dev_pts + at : in.p;
    if (!dev_pts) in.upload(reinterpret_cast<const Affine<Fq>*>(host_pts) + at, m);
    g1_canonical_kernel<Fq><<<div_up(m, 256), 256, 0, cx.stream>>>(src, m, conv.p, true);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    conv.download(reinterpret_cast<Affine<Fq>*>(out) + at, m);
  }
}
template <class Fr, class Fq>
void Msm<Fr, Fq>::g1_from_bytes(Ctx& cx, const uint8_t* bytes, size_t n, uint64_t* out_xy) {
  const size_t slice = (size_t)1 << 22;
  DBuf<Affine<Fq>> in(cx, std::min(n, slice) + 1), conv(cx, std::min(n, slice) + 1);
  for (size_t at = 0; at < n; at += slice) {
    const size_t m = std::min(slice, n - at);
    in.upload(reinterpret_cast<const Affine<Fq>*>(bytes) + at, m);
    g1_canonical_kernel<Fq><<<div_up(m, 256), 256, 0, cx.stream>>>(in.p, m, conv.p, false);
    B2M_CHECK_LAUNCH();
    cx.launches++;
    conv.download(reinterpret_cast<Affine<Fq>*>(out_xy) + at, m);
  }
}

template <class Fr, class Fq>
void Msm<Fr, Fq>::g1_powers_host(Ctx& cx, const uint64_t* g_xy, const uint64_t* beta, size_t n, uint64_t* out) {
  fixed_base_host(cx, g_xy, nullptr, beta, 0, n, out);
}

}  // namespace b2m
