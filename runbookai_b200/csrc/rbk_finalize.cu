// rbk_finalize.cu — everything around the fused scan that makes the result EXACT:
//   prep_queries   : per query  bf16 copy for the scan, fp64 copy + exact ||q||^2 (the
//                    reference's `normA`, embedder.ts:175-180), error bound, start threshold
//   finalize       : K2 (select the k' best approximate candidates of a query across the
//                    per-CTA lists) + K4 (re-score them in fp64 in the reference's exact
//                    operation order, embedder.ts:173-183) + the final ordering of
//                    VectorStore.search (score desc, stable = slot asc; `>= minScore`;
//                    vector-store.ts:212,218,221) + the proof that no other row can belong
//                    to the answer
//   exact fallback : K0, exhaustive fp64 scan for the (rare) queries whose proof failed
//   merge_shards   : merge of per-GPU result lists after the all-gather (SURVEY.md §8e)
#include <cuda_bf16.h>
#include <limits.h>

#include "rbk_internal.h"
#include "rbk_ptx.cuh"

namespace rbk {

namespace {

constexpr uint32_t kFull = 0xFFFFFFFFu;

__device__ __forceinline__ double bf16_to_f64(uint32_t h) { return static_cast<double>(__uint_as_float(h << 16)); }

// dot(q, row) accumulated in index order, multiply then add, no FMA (embedder.ts:177-178).
__device__ __forceinline__ double exact_dot(const double* __restrict__ q, const uint16_t* __restrict__ row, int d) {
  double dot = 0.0;
  const uint4* p = reinterpret_cast<const uint4*>(row);
  int i = 0;
  for (; i + 8 <= d; i += 8) {
    const uint4 v = __ldg(p + (i >> 3));
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      dot = __dadd_rn(dot, __dmul_rn(__ldg(q + i + 2 * j), bf16_to_f64(w[j] & 0xFFFFu)));
      dot = __dadd_rn(dot, __dmul_rn(__ldg(q + i + 2 * j + 1), bf16_to_f64(w[j] >> 16)));
    }
  }
  for (; i < d; ++i) dot = __dadd_rn(dot, __dmul_rn(__ldg(q + i), bf16_to_f64(row[i])));
  return dot;
}
// same, f64 sidecar row
__device__ __forceinline__ double exact_dot_f64(const double* __restrict__ q, const double* __restrict__ row, int d) {
  double dot = 0.0;
  for (int i = 0; i < d; ++i) dot = __dadd_rn(dot, __dmul_rn(__ldg(q + i), __ldg(row + i)));
  return dot;
}
// embedder.ts:183  dotProduct / (Math.sqrt(normA) * Math.sqrt(normB))
__device__ __forceinline__ double exact_cosine(double dot, double na, double nb) {
  return __ddiv_rn(dot, __dmul_rn(__dsqrt_rn(na), __dsqrt_rn(nb)));
}

// --------------------------------------------------------------------------- prep
// kNorm2: also compute the reference's normA (one SEQUENTIAL fp64 chain over d elements, ~30 cycles each: 12 us
// at d = 768).  A search does not need it here: only the finalize kernel reads it, and computes it itself on an
// otherwise idle thread beside the candidates' dot chains - so the chain left the critical path of every search.
// The exact-scores path, which has no finalize, asks for it.
// scratch (nullable): the per-launch scan scratch of the FIRST sub-batch - hist [Bs][kHistBins] | maxbin [Bs] |
// gthr [Bs] | progress [n_progress] - zeroed here, one row per query block, instead of by a separate memset node.
template <typename SrcT, bool kNorm2>
__global__ void __launch_bounds__(128) prep_queries_kernel(const SrcT* __restrict__ src, int d, int dpad,
                                                           double min_score, double acc_eps,
                                                           const float* __restrict__ eps_c, QueryBuffers qb,
                                                           unsigned int* __restrict__ scratch, int Bs, int n_progress) {
  const int q = blockIdx.x;
  const int tid = threadIdx.x;
  if (scratch != nullptr && q < Bs) {
    uint4* row = reinterpret_cast<uint4*>(scratch + static_cast<size_t>(q) * kHistBins);
    for (int i = tid; i < kHistBins / 4; i += blockDim.x) row[i] = make_uint4(0u, 0u, 0u, 0u);
    unsigned int* tail = scratch + static_cast<size_t>(Bs) * kHistBins;
    if (tid == 0) {
      tail[q] = 0u;        // maxbin
      tail[Bs + q] = 0u;   // gthr
    }
    if (q == 0)
      for (int i = tid; i < n_progress; i += blockDim.x) tail[2 * Bs + i] = 0u;
  }
  const SrcT* s = src + static_cast<size_t>(q) * d;
  // The scan's copy is bf16(q * 2^e), e chosen so that the largest |element| lands in [1, 2) (DESIGN.md §6: every
  // tensor-core product and partial sum is then a normal fp32 number for rows inside the norm window, whatever the
  // query's own scale - cosine does not depend on it).  Scaling by 2^e is exact in fp64.  q_f64, normA and the
  // validity test stay on the unscaled query: they define the reference's result.
  __shared__ double red_m[4];
  double amax = 0.0;
  for (int i0 = tid; i0 < d; i0 += 8 * blockDim.x) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * blockDim.x;
      if (i < d) amax = fmax(amax, fabs(static_cast<double>(__ldg(s + i))));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) amax = fmax(amax, __shfl_xor_sync(kFull, amax, o));
  if ((tid & 31) == 0) red_m[tid >> 5] = amax;
  __syncthreads();
  amax = fmax(fmax(red_m[0], red_m[1]), fmax(red_m[2], red_m[3]));
  const int e = (amax > 0.0 && amax < INFINITY) ? -ilogb(amax) : 0;
  // ||bf16(qs)||^2, ||qs - bf16(qs)||^2, ||qs||^2 of the scaled copy qs (any order: bounds only); ||q||^2 unscaled
  double sb = 0.0, sd = 0.0, ss = 0.0, sq = 0.0;
  // 8 elements per thread and pass, ALL loads first: the stores below may alias the source as far as the compiler
  // knows, so a load -> store loop exposed one global round trip per element (the kernel took 7.8 us for this)
  for (int i0 = tid; i0 < dpad; i0 += 8 * blockDim.x) {
    double xs[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * blockDim.x;
      xs[u] = i < d ? static_cast<double>(__ldg(s + i)) : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int i = i0 + u * blockDim.x;
      if (i >= dpad) continue;
      uint16_t b = 0;
      if (i < d) {
        const double x = xs[u];
        qb.q_f64[static_cast<size_t>(q) * d + i] = x;
        const double xs2 = scalbn(x, e);
        const __nv_bfloat16 h = __float2bfloat16_rn(__double2float_rn(xs2));
        b = __bfloat16_as_ushort(h);
        const double xb = static_cast<double>(__bfloat162float(h));
        sb += xb * xb;
        sd += (xs2 - xb) * (xs2 - xb);
        ss += xs2 * xs2;
        sq += x * x;
      }
      qb.q_bf16[static_cast<size_t>(q) * dpad + i] = b;
    }
  }
  __shared__ double red_b[4], red_d[4], red_s[4];
  __shared__ double s_na;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sb += __shfl_xor_sync(kFull, sb, o);
    sd += __shfl_xor_sync(kFull, sd, o);
    ss += __shfl_xor_sync(kFull, ss, o);
  }
  if ((tid & 31) == 0) {
    red_b[tid >> 5] = sb;
    red_d[tid >> 5] = sd;
    red_s[tid >> 5] = ss;
  }
  // the reference's normA: index order, multiply then add.  The chain is sequential by contract, so its
  // operands are staged in smem first (a dependent global load per element cost ~23 ns each).
  __shared__ double s_x[512];
  double na = 0.0;
  if (kNorm2) {
    for (int c0 = 0; c0 < d; c0 += 512) {
      const int len = d - c0 < 512 ? d - c0 : 512;
      __syncthreads();
      for (int i = tid; i < len; i += blockDim.x) s_x[i] = static_cast<double>(s[c0 + i]);
      __syncthreads();
      if (tid == 0)
        for (int i = 0; i < len; ++i) na = __dadd_rn(na, __dmul_rn(s_x[i], s_x[i]));
    }
  } else {
    // any-order sum of squares of the f64 query (accumulated above): only its sign/finiteness and the ratio below
    // (bounds) are used
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(kFull, sq, o);
    __shared__ double red_q[4];
    if ((tid & 31) == 0) red_q[tid >> 5] = sq;
    __syncthreads();
    na = red_q[0] + red_q[1] + red_q[2] + red_q[3];
  }
  if (tid == 0) s_na = na;
  __syncthreads();
  if (tid == 0) {
    const double na = s_na;
    const double nb2 = red_b[0] + red_b[1] + red_b[2] + red_b[3];
    const double nd2 = red_d[0] + red_d[1] + red_d[2] + red_d[3];
    const double ns2 = red_s[0] + red_s[1] + red_s[2] + red_s[3];
    const bool ok = nb2 > 0.0 && nb2 < INFINITY && na > 0.0 && na < INFINITY;
    const double inv = ok ? 1.0 / sqrt(nb2) : 0.0;
    // angle(qs, bf16(qs)) <= asin(||qs - bf16(qs)|| / ||qs||); cosine is 1-Lipschitz in the angle
    double ang = 0.0;
    if (ok && nd2 > 0.0) {
      const double ratio = sqrt(nd2 / ns2) * (1.0 + 1e-9) * (1.0 + 1e-12 * d);   // any-order sums: widen
      ang = ratio < 1.0 ? asin(ratio) * (1.0 + 1e-9) : 3.2;
    }
    // + corpus-side term (rbk_ingest.cu): the quantisation angle of an f64 sidecar's rows, and 3.2 (no bound) once
    // a row's norm has left the scan's window; 0 for bf16-exact corpora inside the window
    const double eps = acc_eps + ang + (eps_c != nullptr ? static_cast<double>(*eps_c) * (1.0 + 1e-6) : 0.0);
    if (kNorm2) qb.q_norm2[q] = na;   // (else: written by the finalize kernel, bit-exact)
    qb.q_eps[q] = eps;
    const float invf = ok ? static_cast<float>(inv) : __uint_as_float(0x7FC00000u);
    qb.q_inv_norm[q] = invf;
    float thr;
    if (!ok) {
      thr = INFINITY;  // zero / non-finite query: cosine is NaN for every row (S3) -> nothing matches
    } else if (min_score == -INFINITY) {
      thr = -INFINITY;
    } else {
      // a row can only reach min_score if approx > min_score - eps; go to the raw domain
      // (divide by inv_norm_q) and step two ulps down so rounding never hides a row.
      const double raw = (min_score - eps) / static_cast<double>(invf);
      float t = static_cast<float>(raw);
      t = nextafterf(nextafterf(t, -INFINITY), -INFINITY);
      thr = t;
    }
    qb.thr_init[q] = thr;
  }
}

// --------------------------------------------------------------------------- finalize
constexpr int kFinThreads = 256;

constexpr int kQChunk = 512;    // query elements staged per re-rank chunk
// Candidate keys of one query are staged in dynamic smem (key_cap keys, chosen per launch: large for few
// queries, small for many so that 8 blocks fit an SM); a query with more keys streams them from L2.

// Visit every candidate key of one query: from the smem staging buffer when it holds them all,
// else straight from the per-unit lists (qb, r, qrow), r in [0, R), in L2.
template <typename F>
__device__ __forceinline__ void for_each_key(const unsigned long long* __restrict__ cand, const int* s_cnt,
                                             const unsigned long long* s_keys, int M, bool staged, int R, int qb,
                                             int qrow, int block_m, F&& f) {
  if (staged) {
    for (int i = threadIdx.x; i < M; i += kFinThreads) f(s_keys[i]);
    return;
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < R; r += kFinThreads / 32) {
    const unsigned long long* l =
        cand + (static_cast<size_t>(qb * R + r) * block_m + qrow) * static_cast<size_t>(kListCap);
    const int c = s_cnt[r];
    for (int i = lane; i < c; i += 32) f(__ldcg(l + i));
  }
}

__global__ void __launch_bounds__(kFinThreads) finalize_kernel(FinalizeParams p) {
  const int ql = blockIdx.x;  // query index inside this launch
  const int tid = threadIdx.x;
  const int qb = ql / p.block_m, qrow = ql % p.block_m;

  __shared__ int s_cnt[160];
  __shared__ int s_off[161];
  extern __shared__ __align__(16) unsigned long long s_keys[];   // p.key_cap keys; later the re-rank's row chunks
  __shared__ unsigned int s_hist[256];
  __shared__ unsigned long long s_sel[kMaxKPrime];
  __shared__ double s_score[kMaxKPrime];
  __shared__ int s_row[kMaxKPrime];
  __shared__ int s_valid[kMaxKPrime];
  __shared__ int s_total, s_nsel, s_nvalid, s_bin, s_want, s_done;
  __shared__ unsigned long long s_prefix, s_minkey;
  __shared__ double s_ekth;

  if (tid == 0) {
    s_total = 0;
    s_nsel = 0;
    s_nvalid = 0;
    s_ekth = 0.0;
    s_done = 0;
    s_minkey = ~0ull;
  }
  __syncthreads();
  int local = 0;
  for (int r = tid; r < p.R; r += kFinThreads) {
    const int c = p.cand_cnt[(qb * p.R + r) * p.block_m + qrow];
    s_cnt[r] = c;
    local += c;
  }
  if (local) atomicAdd(&s_total, local);
  __syncthreads();
  const int M = s_total;
  const int kprime = p.kprime;
  // Stage the query's keys in smem with every load in flight at once: flat key index ->
  // (list, offset) by binary search in the prefix sums.  (Walking the lists one after the
  // other costs one L2 round trip per list and pass: 60-125 us per block, measured.)
  const bool staged = M <= p.key_cap;
  if (staged) {
    if (tid < 32) {   // exclusive scan of up to 160 counts, 5 per lane
      int v[5], sum = 0;
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int r = tid * 5 + j;
        v[j] = r < p.R ? s_cnt[r] : 0;
        sum += v[j];
      }
      int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(kFull, incl, o);
        if (tid >= o) incl += t;
      }
      int run = incl - sum;
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        const int r = tid * 5 + j;
        if (r <= p.R) s_off[r] = run;
        run += v[j];
      }
    }
    __syncthreads();
    // four independent loads in flight per thread (a load -> store loop exposes one L2 round trip per key)
    for (int i0 = tid; i0 < M; i0 += 4 * kFinThreads) {
      unsigned long long kv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * kFinThreads;
        kv[u] = 0ull;
        if (i < M) {
          int lo = 0, hi = p.R - 1;   // last r with s_off[r] <= i
          while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (s_off[mid] <= i) lo = mid;
            else hi = mid - 1;
          }
          const unsigned long long* l =
              p.cand + (static_cast<size_t>(qb * p.R + lo) * p.block_m + qrow) * static_cast<size_t>(kListCap);
          kv[u] = __ldcg(l + (i - s_off[lo]));
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * kFinThreads;
        if (i < M) s_keys[i] = kv[u];
      }
    }
    __syncthreads();
  }

  // ---- K2: radix select of the k'-th largest 64-bit key (keys are unique) ----
  unsigned long long pivot = 0ull;
  if (M >= kprime) {
    if (tid == 0) {
      s_prefix = 0ull;
      s_want = kprime;
    }
    unsigned long long mask = 0ull;
    for (int pass = 7; pass >= 0; --pass) {
      const int shift = pass * 8;
      s_hist[tid] = 0u;
      __syncthreads();
      const unsigned long long prefix = s_prefix;
      for_each_key(p.cand, s_cnt, s_keys, M, staged, p.R, qb, qrow, p.block_m, [&](unsigned long long k) {
        if ((k & mask) == prefix) atomicAdd(&s_hist[static_cast<unsigned>(k >> shift) & 255u], 1u);
      });
      __syncthreads();
      if (tid < 32) {
        // lane L owns bins [255-8L-7, 255-8L]; scan from the top bin down
        const int top = 255 - 8 * tid;
        unsigned int mine = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) mine += s_hist[top - j];
        unsigned int incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned int v = __shfl_up_sync(kFull, incl, o);
          if (tid >= o) incl += v;
        }
        const unsigned int want = static_cast<unsigned int>(s_want);
        const bool crosses = (incl >= want) && (incl - mine < want);
        if (crosses) {
          unsigned int cum = incl - mine;
          int b = top;
          for (int j = 0; j < 8; ++j, --b) {
            const unsigned int h = s_hist[b];
            if (cum + h >= want) break;
            cum += h;
          }
          s_bin = b;
          s_want = static_cast<int>(want - cum);
          // every key left in this bin is wanted: the bin's lower edge is already a valid pivot
          s_done = (s_hist[b] == want - cum) ? 1 : 0;
        }
      }
      __syncthreads();
      if (tid == 0) s_prefix = prefix | (static_cast<unsigned long long>(s_bin) << shift);
      mask |= 0xFFull << shift;
      __syncthreads();
      if (s_done) break;   // uniform: read after the barrier
    }
    pivot = s_prefix;
  }
  for_each_key(p.cand, s_cnt, s_keys, M, staged, p.R, qb, qrow, p.block_m, [&](unsigned long long k) {
    if (k >= pivot) {
      const int pos = atomicAdd(&s_nsel, 1);
      if (pos < kMaxKPrime) s_sel[pos] = k;
      atomicMin(&s_minkey, k);   // the k'-th best key itself (the pivot may be only a bin edge after an early exit)
    }
  });
  __syncthreads();
  const int nsel = s_nsel < kMaxKPrime ? s_nsel : kMaxKPrime;
  // every row that is NOT a candidate has raw score <= tau_raw (or was cut by thr_init)
  const float tau_raw = M >= kprime ? key_score(s_minkey) : -INFINITY;

  // ---- K4: exact fp64 re-score of the candidates ----
  // The arithmetic is a sequential chain per candidate (parity contract), so global-load latency
  // must not sit inside it: all threads stage a K-chunk of every candidate row (and of the query)
  // into smem with the loads in flight together, then each candidate's thread walks its chunk.
  // The key staging buffer is dead by now (selection is in s_sel) and is reused for the rows.
  // Cycle stamps (a clock64 probe build, round 2; 625k-row shard, B=256, d=768, 32 candidates): this phase is
  // 26 k of the block's 44 k cycles = 34 cycles per element for conversion + DMUL + DADD in one warp.  Three
  // rearrangements of the same operations were measured and ALL lost: widening bf16 -> binary64 with integer
  // instructions instead of F2F (51 k cycles), forming the next group's 8 products ahead of the current group's
  // 8 dependent adds by hand (38 k), and letting all 256 threads form the products into shared memory so that the
  // chain thread only adds (65 k with 16-byte row loads, 110 k element-wise).  Whatever issues them, fp64-pipe
  // instructions cost this kernel 11-27 cycles each; the loop below issues the fewest.
  // The reference's normA (embedder.ts:179: index order, multiply then add) is one more sequential fp64 chain over
  // the query.  The last thread of the block - idle, at most kMaxKPrime threads carry candidates - walks it over the
  // same staged query chunks the candidates' dot chains read, so it costs the search nothing.
  __shared__ double s_na;
  double na_chain = 0.0;
  const double* qv = p.q.q_f64 + static_cast<size_t>(ql) * p.d;
  __shared__ double s_q[kQChunk];
  unsigned char* s_rows = reinterpret_cast<unsigned char*>(s_keys);
  int my_row = 0;
  double dot = 0.0;
  if (tid < nsel) my_row = static_cast<int>(key_row(s_sel[tid]));
  if (p.rows_f64 == nullptr) {
    int chunk = nsel > 0 ? ((p.key_cap * 8 / nsel - 16) / 2) & ~7 : kQChunk;
    chunk = chunk < kQChunk ? chunk : kQChunk;
    const int chunk16 = chunk >> 3;                                   // 16-byte units per row chunk
    const int row_stride = (chunk16 | 1) << 4;                        // odd number of 16-B units: conflict-free walks
    for (int c0 = 0; c0 < p.d; c0 += chunk) {
      const int len = p.d - c0 < chunk ? p.d - c0 : chunk;            // elements of this chunk
      const int len16 = (len + 7) >> 3;                               // rows are zero padded to dpad (multiple of 8)
      __syncthreads();                                                // previous chunk fully consumed
      for (int i0 = tid; i0 < nsel * len16; i0 += 4 * kFinThreads) {   // 4 row pieces in flight per thread
        uint4 pv[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int i = i0 + b * kFinThreads;
          pv[b] = make_uint4(0u, 0u, 0u, 0u);
          if (i < nsel * len16) {
            const int rr = i / len16, u = i - rr * len16;
            const int row = static_cast<int>(key_row(s_sel[rr]));
            pv[b] = __ldg(reinterpret_cast<const uint4*>(p.rows + static_cast<size_t>(row) * p.dpad + c0) + u);
          }
        }
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int i = i0 + b * kFinThreads;
          if (i < nsel * len16) {
            const int rr = i / len16, u = i - rr * len16;
            *reinterpret_cast<uint4*>(s_rows + rr * row_stride + u * 16) = pv[b];
          }
        }
      }
      for (int i = tid; i < len; i += kFinThreads) s_q[i] = __ldg(qv + c0 + i);
      __syncthreads();
      if (tid < nsel) {
        const unsigned char* mine = s_rows + tid * row_stride;
        int i = 0;
        for (; i + 8 <= len; i += 8) {
          const uint4 v = *reinterpret_cast<const uint4*>(mine + i * 2);
          const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            dot = __dadd_rn(dot, __dmul_rn(s_q[i + 2 * j], bf16_to_f64(w[j] & 0xFFFFu)));
            dot = __dadd_rn(dot, __dmul_rn(s_q[i + 2 * j + 1], bf16_to_f64(w[j] >> 16)));
          }
        }
        for (; i < len; ++i)
          dot = __dadd_rn(dot, __dmul_rn(s_q[i], bf16_to_f64(reinterpret_cast<const uint16_t*>(mine)[i])));
      }
      if (tid == kFinThreads - 1)
        for (int i = 0; i < len; ++i) na_chain = __dadd_rn(na_chain, __dmul_rn(s_q[i], s_q[i]));
    }
  } else {
    // exact source = the f64 sidecar: same staging, 8-byte elements (odd stride in doubles: conflict-free)
    double* s_rows64 = reinterpret_cast<double*>(s_keys);
    int chunk = nsel > 0 ? (p.key_cap / nsel - 1) : kQChunk;          // doubles per row chunk
    chunk = chunk < kQChunk ? chunk : kQChunk;
    const int row_stride = chunk | 1;
    for (int c0 = 0; c0 < p.d; c0 += chunk) {
      const int len = p.d - c0 < chunk ? p.d - c0 : chunk;
      __syncthreads();
      for (int i = tid; i < nsel * len; i += kFinThreads) {
        const int rr = i / len, u = i - rr * len;
        const int row = static_cast<int>(key_row(s_sel[rr]));
        s_rows64[rr * row_stride + u] = __ldg(p.rows_f64 + static_cast<size_t>(row) * p.d + c0 + u);
      }
      for (int i = tid; i < len; i += kFinThreads) s_q[i] = __ldg(qv + c0 + i);
      __syncthreads();
      if (tid < nsel) {
        const double* mine = s_rows64 + tid * row_stride;
        for (int i = 0; i < len; ++i) dot = __dadd_rn(dot, __dmul_rn(s_q[i], mine[i]));
      }
      if (tid == kFinThreads - 1)
        for (int i = 0; i < len; ++i) na_chain = __dadd_rn(na_chain, __dmul_rn(s_q[i], s_q[i]));
    }
  }
  if (tid == kFinThreads - 1) {
    s_na = na_chain;
    p.q.q_norm2[ql] = na_chain;   // kept for the exhaustive fallback of a flagged query
  }
  __syncthreads();
  const double na = s_na;
  if (tid < nsel) {
    const double sc = exact_cosine(dot, na, p.row_norm2[my_row]);
    s_score[tid] = sc;
    s_row[tid] = my_row;
    const int ok = sc >= p.min_score ? 1 : 0;  // vector-store.ts:212 (NaN fails; -inf = no threshold)
    s_valid[tid] = ok;
    if (ok) atomicAdd(&s_nvalid, 1);
  }
  __syncthreads();
  const int nvalid = s_nvalid;
  const int count = nvalid < p.k_fetch ? nvalid : p.k_fetch;
  // ---- final order: score desc, ties -> lower slot (stable sort over insertion order) ----
  if (tid < nsel && s_valid[tid]) {
    const double sc = s_score[tid];
    const int row = s_row[tid];
    int rank = 0;
    for (int j = 0; j < nsel; ++j) {
      if (!s_valid[j]) continue;
      const double sj = s_score[j];
      rank += (sj > sc || (sj == sc && s_row[j] < row)) ? 1 : 0;
    }
    if (rank < p.k_fetch) {
      p.out_slots[static_cast<size_t>(ql) * p.k_fetch + rank] = p.slot.global(row);
      p.out_scores[static_cast<size_t>(ql) * p.k_fetch + rank] = sc;
    }
    if (rank == p.k_fetch - 1) s_ekth = sc;
  }
  for (int i = count + tid; i < p.k_fetch; i += kFinThreads) {
    p.out_slots[static_cast<size_t>(ql) * p.k_fetch + i] = -1;
    p.out_scores[static_cast<size_t>(ql) * p.k_fetch + i] = __longlong_as_double(0x7FF8000000000000ll);
  }
  __syncthreads();
  if (tid == 0) {
    p.out_counts[ql] = count;
    // ---- proof of exactness (DESIGN.md §6) ----
    bool ok;
    if (!(p.q.q_eps[ql] < 2.0)) {
      // cosines lie in [-1, 1]: a bound this wide (a row outside the scan's norm window, DESIGN.md §6) says nothing
      // about the rows the scan dropped - NaN accumulators included - so nothing is proven
      ok = false;
    } else if (tau_raw == -INFINITY) {
      ok = true;  // nothing was ever dropped except by thr_init (provably below min_score)
    } else {
      const double bound = static_cast<double>(tau_raw) * static_cast<double>(p.q.q_inv_norm[ql]) + p.q.q_eps[ql];
      if (count == p.k_fetch) ok = s_ekth > bound;       // every outsider scores strictly below the k-th hit
      else ok = bound < p.min_score;                      // no outsider can pass the threshold
    }
    p.flags[ql] = ok ? 0 : 1;
  }
}

// --------------------------------------------------------------------------- exact fallback (K0)
constexpr int kExThreads = 256;
constexpr int kExBuf = 1024;

struct ExactTopK {
  double score[kExBuf];
  int row[kExBuf];
  int n;
  int have_thr;
  double thr_score;
  int thr_row;
};

__device__ __forceinline__ bool hit_before(double sa, int ra, double sb, int rb) {
  return sa > sb || (sa == sb && ra < rb);
}

// Block-wide: sort the buffer by (score desc, row asc), keep the best K.
__device__ void exact_compact(ExactTopK& t, int K) {
  const int tid = threadIdx.x;
  __syncthreads();
  const int n = t.n;
  for (int i = n + tid; i < kExBuf; i += kExThreads) {
    t.score[i] = -INFINITY;
    t.row[i] = INT_MAX;
  }
  __syncthreads();
  for (int k2 = 2; k2 <= kExBuf; k2 <<= 1) {
    for (int s = k2 >> 1; s > 0; s >>= 1) {
      for (int i = tid; i < kExBuf; i += kExThreads) {
        const int j = i ^ s;
        if (j > i) {
          const bool desc = (i & k2) == 0;
          const bool j_first = hit_before(t.score[j], t.row[j], t.score[i], t.row[i]);
          if (desc ? j_first : !j_first) {
            const double ts = t.score[i];
            t.score[i] = t.score[j];
            t.score[j] = ts;
            const int tr = t.row[i];
            t.row[i] = t.row[j];
            t.row[j] = tr;
          }
        }
      }
      __syncthreads();
    }
  }
  if (tid == 0) {
    const int keep = n < K ? n : K;
    t.n = keep;
    if (keep == K) {
      t.have_thr = 1;
      t.thr_score = t.score[K - 1];
      t.thr_row = t.row[K - 1];
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void exact_push(ExactTopK& t, double sc, int row) {
  if (t.have_thr && !hit_before(sc, row, t.thr_score, t.thr_row)) return;
  const int pos = atomicAdd(&t.n, 1);
  t.score[pos] = sc;
  t.row[pos] = row;
}

__global__ void __launch_bounds__(kExThreads) exact_scan_kernel(ExactParams p) {
  __shared__ ExactTopK t;
  const int tid = threadIdx.x;
  const int f = blockIdx.y;
  const int q = p.fail_list[f];
  if (tid == 0) {
    t.n = 0;
    t.have_thr = 0;
  }
  __syncthreads();
  const int64_t chunk = (p.n_rows + p.n_blocks - 1) / p.n_blocks;
  const int64_t r0 = blockIdx.x * chunk;
  const int64_t r1 = r0 + chunk < p.n_rows ? r0 + chunk : p.n_rows;
  const double* qv = p.q_f64 + static_cast<size_t>(q) * p.d;
  const double na = p.q_norm2[q];
  for (int64_t base = r0; base < r1; base += kExThreads) {
    if (t.n > kExBuf - kExThreads) exact_compact(t, p.k_fetch);  // uniform: t.n read after a barrier
    const int64_t row = base + tid;
    if (row < r1) {
      const bool dead = (p.dead_bits[row >> 5] >> (row & 31)) & 1u;
      if (!dead) {   // zero-norm rows give NaN and fail the compare below, like in the reference (S3)
        const double dot = p.rows_f64 != nullptr
                               ? exact_dot_f64(qv, p.rows_f64 + static_cast<size_t>(row) * p.d, p.d)
                               : exact_dot(qv, p.rows + static_cast<size_t>(row) * p.dpad, p.d);
        const double sc = exact_cosine(dot, na, p.row_norm2[row]);
        if (sc >= p.min_score) exact_push(t, sc, static_cast<int>(row));
      }
    }
    __syncthreads();
  }
  exact_compact(t, p.k_fetch);
  const size_t o = (static_cast<size_t>(f) * p.n_blocks + blockIdx.x) * p.k_fetch;
  for (int i = tid; i < t.n; i += kExThreads) {
    p.part_scores[o + i] = t.score[i];
    p.part_rows[o + i] = t.row[i];
  }
  if (tid == 0) p.part_cnt[f * p.n_blocks + blockIdx.x] = t.n;
}

__global__ void __launch_bounds__(kExThreads) exact_merge_kernel(ExactParams p) {
  __shared__ ExactTopK t;
  const int tid = threadIdx.x;
  const int f = blockIdx.x;
  const int q = p.fail_list[f];
  if (tid == 0) {
    t.n = 0;
    t.have_thr = 0;
  }
  __syncthreads();
  const int total = p.n_blocks * p.k_fetch;
  for (int base = 0; base < total; base += kExThreads) {
    if (t.n > kExBuf - kExThreads) exact_compact(t, p.k_fetch);
    const int i = base + tid;
    if (i < total) {
      const int b = i / p.k_fetch, e = i % p.k_fetch;
      if (e < p.part_cnt[f * p.n_blocks + b]) {
        const size_t o = (static_cast<size_t>(f) * p.n_blocks + b) * p.k_fetch + e;
        exact_push(t, p.part_scores[o], p.part_rows[o]);
      }
    }
    __syncthreads();
  }
  exact_compact(t, p.k_fetch);
  const int n = t.n;
  for (int i = tid; i < p.k_fetch; i += kExThreads) {
    const size_t o = static_cast<size_t>(q) * p.k_fetch + i;
    if (i < n) {
      p.out_slots[o] = p.slot.global(t.row[i]);
      p.out_scores[o] = t.score[i];
    } else {
      p.out_slots[o] = -1;
      p.out_scores[o] = __longlong_as_double(0x7FF8000000000000ll);
    }
  }
  if (tid == 0) p.out_counts[q] = n;
}

// --------------------------------------------------------------------------- all exact scores (large-k path)
// One thread per (row, query): the reference's fp64 cosine of EVERY row, NaN for tombstoned / zero rows.  Serves
// requests for more hits than the scan's candidate lists hold (k_fetch > RBK_MAX_K_FETCH): the host then applies
// `>= minScore`, the stable sort and the cut literally (vector-store.ts:212-221).  Rare and small (RunbookAI's
// corpora are 10^4-10^5 chunks when somebody asks for 1000 results), so simplicity wins over bandwidth here.
__global__ void __launch_bounds__(256) exact_scores_kernel(const uint16_t* __restrict__ rows,
                                                           const double* __restrict__ rows_f64,
                                                           const double* __restrict__ row_norm2,
                                                           const unsigned int* __restrict__ dead_bits, int64_t n_rows,
                                                           int d, int dpad, const double* __restrict__ q_f64,
                                                           const double* __restrict__ q_norm2,
                                                           double* __restrict__ out) {
  const int64_t row = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int q = blockIdx.y;
  if (row >= n_rows) return;
  double sc = __longlong_as_double(0x7FF8000000000000ll);
  if (!((dead_bits[row >> 5] >> (row & 31)) & 1u)) {
    const double* qv = q_f64 + static_cast<size_t>(q) * d;
    const double dot = rows_f64 != nullptr ? exact_dot_f64(qv, rows_f64 + static_cast<size_t>(row) * d, d)
                                           : exact_dot(qv, rows + static_cast<size_t>(row) * dpad, d);
    sc = exact_cosine(dot, q_norm2[q], row_norm2[row]);
  }
  out[static_cast<size_t>(q) * n_rows + row] = sc;
}

// --------------------------------------------------------------------------- shard merge
// Lists are sorted by (score desc, slot asc); slots are globally unique, so the rank of an
// entry in the merged order is its own index plus, for every other list, the number of
// entries of that list that come before it (binary search).
__global__ void __launch_bounds__(128) merge_shards_kernel(int G, int B, int k, const char* __restrict__ slots_base,
                                                           const char* __restrict__ scores_base,
                                                           const char* __restrict__ counts_base,
                                                           const char* __restrict__ flags_base, size_t slots_stride,
                                                           size_t scores_stride, size_t counts_stride,
                                                           size_t flags_stride, long long* out_slots,
                                                           double* out_scores, int* out_counts, int* out_flags) {
  // shard g's arrays start g * stride bytes after shard 0's (dense [G][...] arrays: stride = array size;
  // packed per-rank blocks, e.g. straight out of ONE all-gather: the same block stride for all three)
  auto slots_of = [&](int g) { return reinterpret_cast<const long long*>(slots_base + g * slots_stride); };
  auto scores_of = [&](int g) { return reinterpret_cast<const double*>(scores_base + g * scores_stride); };
  auto count_of = [&](int g, int b) { return reinterpret_cast<const int*>(counts_base + g * counts_stride)[b]; };
  const int b = blockIdx.x;
  int total = 0;
  for (int g = 0; g < G; ++g) total += count_of(g, b);
  const int n_out = total < k ? total : k;
  for (int i = threadIdx.x; i < G * k; i += blockDim.x) {
    const int g = i / k, e = i % k;
    if (e >= count_of(g, b)) continue;
    const size_t o = static_cast<size_t>(b) * k;
    const double sc = scores_of(g)[o + e];
    const long long sl = slots_of(g)[o + e];
    int rank = e;
    for (int g2 = 0; g2 < G; ++g2) {
      if (g2 == g) continue;
      const double* s2p = scores_of(g2) + o;
      const long long* l2p = slots_of(g2) + o;
      int lo = 0, hi = count_of(g2, b);
      while (lo < hi) {  // first index whose entry does NOT come before (sc, sl)
        const int mid = (lo + hi) >> 1;
        const double s2 = s2p[mid];
        const long long l2 = l2p[mid];
        if (s2 > sc || (s2 == sc && l2 < sl)) lo = mid + 1;
        else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) {
      out_slots[o + rank] = sl;
      out_scores[o + rank] = sc;
    }
  }
  for (int i = n_out + threadIdx.x; i < k; i += blockDim.x) {
    out_slots[static_cast<size_t>(b) * k + i] = -1;
    out_scores[static_cast<size_t>(b) * k + i] = __longlong_as_double(0x7FF8000000000000ll);
  }
  if (threadIdx.x == 0) {
    out_counts[b] = n_out;
    if (out_flags != nullptr) {
      // "not provably exact" travels with the lists: a query is dirty if any shard's proof failed.  out_flags[B]
      // counts dirty queries across calls (the caller zeroes it), so a pipelined caller can check once at the end.
      int dirty = 0;
      for (int g = 0; g < G; ++g) dirty |= reinterpret_cast<const int*>(flags_base + g * flags_stride)[b];
      out_flags[b] = dirty;
      if (dirty) atomicAdd(out_flags + B, 1);
    }
  }
}

}  // namespace

cudaError_t launch_prep_queries(const void* src, int src_type, int B, int d, int dpad, double min_score,
                                const float* eps_c, const QueryBuffers& qb, cudaStream_t stream, bool with_norm2,
                                unsigned int* scratch, int Bs, int n_progress) {
  if (B <= 0) return cudaSuccess;
  const double acc_eps = accumulation_eps(d);
  const double* sd = static_cast<const double*>(src);
  const float* sf = static_cast<const float*>(src);
  if (src_type == 0) {
    if (with_norm2)
      prep_queries_kernel<double, true><<<B, 128, 0, stream>>>(sd, d, dpad, min_score, acc_eps, eps_c, qb, scratch, Bs, n_progress);
    else
      prep_queries_kernel<double, false><<<B, 128, 0, stream>>>(sd, d, dpad, min_score, acc_eps, eps_c, qb, scratch, Bs, n_progress);
  } else {
    if (with_norm2)
      prep_queries_kernel<float, true><<<B, 128, 0, stream>>>(sf, d, dpad, min_score, acc_eps, eps_c, qb, scratch, Bs, n_progress);
    else
      prep_queries_kernel<float, false><<<B, 128, 0, stream>>>(sf, d, dpad, min_score, acc_eps, eps_c, qb, scratch, Bs, n_progress);
  }
  return cudaGetLastError();
}

cudaError_t launch_finalize(const FinalizeParams& p_in, cudaStream_t stream) {
  if (p_in.B <= 0) return cudaSuccess;
  FinalizeParams p = p_in;
  // >= 2048 keys (16 KB: room for 128 candidate rows x 56 elements per re-rank chunk)
  p.key_cap = p.B <= 160 ? 16384 : (p.B <= 320 ? 8192 : 2048);
  const size_t smem = static_cast<size_t>(p.key_cap) * 8;
  cudaError_t e = cudaFuncSetAttribute(finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16384 * 8);
  if (e != cudaSuccess) return e;
  finalize_kernel<<<p.B, kFinThreads, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_exact_fallback(const ExactParams& p, cudaStream_t stream) {
  if (p.n_fail <= 0) return cudaSuccess;
  dim3 grid(p.n_blocks, p.n_fail);
  exact_scan_kernel<<<grid, kExThreads, 0, stream>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  exact_merge_kernel<<<p.n_fail, kExThreads, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_exact_scores(const uint16_t* rows, const double* rows_f64, const double* row_norm2,
                                const unsigned int* dead_bits, int64_t n_rows, int d, int dpad, const double* q_f64,
                                const double* q_norm2, int B, double* out, cudaStream_t stream) {
  if (B <= 0 || n_rows <= 0) return cudaSuccess;
  dim3 grid(static_cast<unsigned>((n_rows + 255) / 256), static_cast<unsigned>(B));
  exact_scores_kernel<<<grid, 256, 0, stream>>>(rows, rows_f64, row_norm2, dead_bits, n_rows, d, dpad, q_f64, q_norm2,
                                                out);
  return cudaGetLastError();
}

cudaError_t launch_merge_shards(int G, int B, int k_fetch, const void* slots, const void* scores, const void* counts,
                                const void* flags, size_t slots_stride, size_t scores_stride, size_t counts_stride,
                                size_t flags_stride, long long* out_slots, double* out_scores, int* out_counts,
                                int* out_flags, cudaStream_t stream) {
  if (B <= 0) return cudaSuccess;
  merge_shards_kernel<<<B, 128, 0, stream>>>(G, B, k_fetch, static_cast<const char*>(slots),
                                             static_cast<const char*>(scores), static_cast<const char*>(counts),
                                             static_cast<const char*>(flags), slots_stride, scores_stride,
                                             counts_stride, flags_stride, out_slots, out_scores, out_counts,
                                             flags ? out_flags : nullptr);
  return cudaGetLastError();
}

}  // namespace rbk
