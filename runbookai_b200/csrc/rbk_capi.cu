// rbk_capi.cu — the C ABI of include/rbk_knn.h: index lifetime, mutation, batched search.
// Host-side orchestration only; the device work is in rbk_ingest.cu / rbk_scan.cu /
// rbk_finalize.cu.  No torch, no CPU compute path: every entry point that needs a GPU
// fails with RBK_ECUDA when there is none.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "rbk_index_impl.h"

using namespace rbk;

namespace rbk {
namespace impl {
thread_local std::string g_err_storage;
rbk_status fail(rbk_status st, const std::string& msg) {
  g_err_storage = msg;
  return st;
}
rbk_status cuda_fail(cudaError_t e, const char* what) {
  // a sticky error (trap in a kernel) poisons the context; report it verbatim
  return fail(e == cudaErrorMemoryAllocation ? RBK_ENOMEM : RBK_ECUDA,
              std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")");
}
const char* last_error() { return g_err_storage.c_str(); }
}  // namespace impl
}  // namespace rbk
using namespace rbk::impl;

namespace {


typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

// 2D bf16 row-major [rows][dpad] tensor, box = box_cols columns (one swizzle row: 64 -> 128 B, 32 -> 64 B)
// x box_rows.
rbk_status encode_rows_tmap(CUtensorMap* out, const void* base, int64_t rows, int dpad, int box_rows,
                            int box_cols = kBlockK) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return fail(RBK_ECUDA, "cuTensorMapEncodeTiled is not available from this driver");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(dpad), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(dpad) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE,
                  box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_64B
                                 : (box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE),
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[160];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed: CUresult %d (rows=%lld dpad=%d)", (int)r,
             (long long)rows, dpad);
    return fail(RBK_ECUDA, buf);
  }
  return RBK_OK;
}

int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

// Page-locked (or managed) host memory: cudaMemcpyAsync from it returns before the bytes have been read, unlike a copy
// from pageable memory, which the driver stages before returning.
bool host_source_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

cudaEvent_t get_event(rbk_index* ix, size_t i) {
  while (ix->ev.size() <= i) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    ix->ev.push_back(e);
  }
  return ix->ev[i];
}

// Fold finished (start, stop) pairs into the running totals.  wait = true: block on the pending ones.
void resolve_scan_events(rbk_index* ix, bool wait) {
  while (ix->tev_tail < ix->tev_head) {
    cudaEvent_t* pr = ix->tev[ix->tev_tail % rbk_index::kTimingRing];
    if (wait) cudaEventSynchronize(pr[1]);
    else if (cudaEventQuery(pr[1]) != cudaSuccess) { cudaGetLastError(); break; }
    float t = 0.f;
    if (cudaEventElapsedTime(&t, pr[0], pr[1]) == cudaSuccess) {
      ix->stats.scan_ms_total += t;
      ix->stats.scans_timed++;
      ix->stats.last_scan_ms = t;
    }
    ix->tev_tail++;
  }
}
// Next (start, stop) pair of the ring; created on first use.
cudaEvent_t* next_scan_events(rbk_index* ix) {
  if (ix->tev_head - ix->tev_tail >= rbk_index::kTimingRing) {   // ring full: the oldest finished long ago
    cudaEvent_t* old = ix->tev[ix->tev_tail % rbk_index::kTimingRing];
    cudaEventSynchronize(old[1]);
    resolve_scan_events(ix, false);
  }
  cudaEvent_t* pr = ix->tev[ix->tev_head % rbk_index::kTimingRing];
  if (!pr[0]) {
    cudaEventCreate(&pr[0]);
    cudaEventCreate(&pr[1]);
  }
  ix->tev_head++;
  return pr;
}

int64_t inv_norm_len(int64_t cap) { return round_up(cap, kBlockN) + kBlockN; }

rbk_status ensure_capacity(rbk_index* ix, int64_t need) {
  if (need <= ix->cap) return RBK_OK;
  if (need >= (1ll << 31) - 2 * kBlockN) return fail(RBK_EINVAL, "an index shard holds at most 2^31 rows");
  // whole 256-row tiles: the corpus tensor maps cover round_up(n_rows, 256) rows, so that no TMA box ever hangs over
  // the end of the tensor (the TMA unit zero-fills out-of-bounds rows one by one - see ensure_query_scratch)
  int64_t ncap = round_up(std::max<int64_t>(need, std::max<int64_t>(ix->cap * 2, 1024)), kBlockN);
  uint16_t* rows = nullptr;
  float* inv = nullptr;
  double* n2 = nullptr;
  unsigned int* dead = nullptr;
  double* r64 = nullptr;
  const size_t dead_words = static_cast<size_t>((ncap + 31) / 32);
  cudaError_t e;
  if (ix->keep_f64 &&
      (e = cudaMalloc(reinterpret_cast<void**>(&r64), static_cast<size_t>(ncap) * ix->dim * 8)) != cudaSuccess)
    return cuda_fail(e, "cudaMalloc(f64 sidecar)");
  if ((e = cudaMalloc(reinterpret_cast<void**>(&rows), static_cast<size_t>(ncap) * ix->dpad * 2)) != cudaSuccess ||
      (e = cudaMalloc(reinterpret_cast<void**>(&inv), static_cast<size_t>(inv_norm_len(ncap)) * 4)) != cudaSuccess ||
      (e = cudaMalloc(reinterpret_cast<void**>(&n2), static_cast<size_t>(ncap) * 8)) != cudaSuccess ||
      (e = cudaMalloc(reinterpret_cast<void**>(&dead), dead_words * 4)) != cudaSuccess) {
    cudaFree(rows);
    cudaFree(inv);
    cudaFree(n2);
    cudaFree(dead);
    cudaFree(r64);
    return cuda_fail(e, "cudaMalloc(index storage)");
  }
  cudaStream_t st = ix->stream;
  CK(cudaMemsetAsync(inv, 0xFF, static_cast<size_t>(inv_norm_len(ncap)) * 4, st));  // all-ones = NaN
  CK(cudaMemsetAsync(dead, 0, dead_words * 4, st));
  // rows not (yet) appended are read by the scan as part of the last tile (their 1/||c|| is NaN: they never match)
  CK(cudaMemsetAsync(rows + static_cast<size_t>(ix->n_rows) * ix->dpad, 0,
                     static_cast<size_t>(ncap - ix->n_rows) * ix->dpad * 2, st));
  if (ix->n_rows > 0) {
    CK(cudaMemcpyAsync(rows, ix->rows, static_cast<size_t>(ix->n_rows) * ix->dpad * 2, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(inv, ix->inv_norm, static_cast<size_t>(ix->n_rows) * 4, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(n2, ix->norm2, static_cast<size_t>(ix->n_rows) * 8, cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(dead, ix->dead_bits, static_cast<size_t>((ix->n_rows + 31) / 32) * 4,
                       cudaMemcpyDeviceToDevice, st));
    if (r64)
      CK(cudaMemcpyAsync(r64, ix->rows_f64, static_cast<size_t>(ix->n_rows) * ix->dim * 8, cudaMemcpyDeviceToDevice,
                         st));
  }
  CK(cudaStreamSynchronize(st));
  cudaFree(ix->rows);
  cudaFree(ix->inv_norm);
  cudaFree(ix->norm2);
  cudaFree(ix->dead_bits);
  cudaFree(ix->rows_f64);
  ix->rows_f64 = r64;
  ix->rows = rows;
  ix->inv_norm = inv;
  ix->norm2 = n2;
  ix->dead_bits = dead;
  ix->cap = ncap;
  return RBK_OK;
}

// src: host (is_device = false) or device rows of `elem` bytes (8 = f64, 4 = f32, 2 = bf16).
rbk_status append_rows(rbk_index* ix, const void* src, bool is_device, int elem, int64_t n, int64_t* first_out) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  if (n < 0 || (n > 0 && !src)) return fail(RBK_EINVAL, "bad rows argument");
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  if (first_out) *first_out = ix->n_rows;
  if (n == 0) return RBK_OK;
  rbk_status st = ensure_capacity(ix, ix->n_rows + n);
  if (st != RBK_OK) return st;
  const int src_type = elem == 8 ? 0 : (elem == 4 ? 1 : 2);
  uint16_t* dst0 = ix->rows + static_cast<size_t>(ix->n_rows) * ix->dpad;
  double* dst64 = ix->keep_f64 ? ix->rows_f64 + static_cast<size_t>(ix->n_rows) * ix->dim : nullptr;
  if (is_device) {
    if (elem == 2 && ix->dpad == ix->dim && !ix->keep_f64) {
      CK(cudaMemcpyAsync(dst0, src, static_cast<size_t>(n) * ix->dim * 2, cudaMemcpyDeviceToDevice, ix->stream));
    } else {
      CK(launch_convert_rows(src, src_type, n, ix->dim, ix->dpad, dst0, dst64, ix->stream));
      ix->stats.kernel_launches++;
    }
  } else {
    const size_t row_bytes = static_cast<size_t>(ix->dim) * elem;
    const int64_t chunk_rows = std::max<int64_t>(1, std::min<int64_t>(n, (64ll << 20) / static_cast<int64_t>(row_bytes)));
    CK(ix->stage.ensure(static_cast<size_t>(chunk_rows) * row_bytes));
    for (int64_t r0 = 0; r0 < n; r0 += chunk_rows) {
      const int64_t nr = std::min<int64_t>(chunk_rows, n - r0);
      const unsigned char* hp = static_cast<const unsigned char*>(src) + static_cast<size_t>(r0) * row_bytes;
      CK(cudaMemcpyAsync(ix->stage.p, hp, static_cast<size_t>(nr) * row_bytes, cudaMemcpyHostToDevice, ix->stream));
      CK(launch_convert_rows(ix->stage.p, src_type, nr, ix->dim, ix->dpad, dst0 + static_cast<size_t>(r0) * ix->dpad,
                             dst64 ? dst64 + static_cast<size_t>(r0) * ix->dim : nullptr, ix->stream));
      ix->stats.kernel_launches++;
      // the staging buffer is reused by the next chunk; pageable H2D copies are already
      // synchronous with respect to the host buffer, the kernel is ordered by the stream
    }
  }
  CK(launch_row_norms(ix->rows, ix->keep_f64 ? ix->rows_f64 : nullptr, ix->n_rows, n, ix->dim, ix->dpad, ix->inv_norm,
                      ix->norm2, ix->d_counter + 1, ix->stream));
  ix->stats.kernel_launches += ix->keep_f64 ? 2 : 1;
  // Host sources: pageable H2D copies have consumed the caller's buffer when cudaMemcpyAsync returns and everything
  // after is stream-ordered, so an append costs no host round trip.  Device sources are read by the copy/convert
  // kernel itself, and page-locked host sources by a copy that really is asynchronous: the caller may free or reuse
  // either as soon as we return, so wait for those.
  if (is_device || host_source_is_pinned(src)) CK(cudaStreamSynchronize(ix->stream));
  ix->n_rows += n;
  ix->n_live += n;
  return RBK_OK;
}

int pick_kprime(const rbk_index* ix, int k_fetch) {
  if (ix->kprime_override > 0) return ix->kprime_override;
  int kp = static_cast<int>(round_up(k_fetch + ix->margin, 16));
  return std::min(kp, kMaxKPrime);
}

rbk_status refresh_corpus_tmap(rbk_index* ix) {
  const int64_t map_rows = round_up(ix->n_rows, kBlockN);   // whole tiles (<= cap): no out-of-bounds box rows
  if (ix->tmap_c_base == ix->rows && ix->tmap_c_rows == map_rows) return RBK_OK;
  rbk_status st = encode_rows_tmap(&ix->tmap_c, ix->rows, map_rows, ix->dpad, kBlockN);
  if (st != RBK_OK) return st;
  st = encode_rows_tmap(&ix->tmap_c_half, ix->rows, map_rows, ix->dpad, kBlockN / 2);
  if (st != RBK_OK) return st;
  st = encode_rows_tmap(&ix->tmap_c_quarter, ix->rows, map_rows, ix->dpad, kBlockN / 4);
  if (st != RBK_OK) return st;
#ifdef RBK_EXPERIMENTAL
  st = encode_rows_tmap(&ix->tmap_c_half32, ix->rows, map_rows, ix->dpad, kBlockN / 2, 32);
  if (st != RBK_OK) return st;
  st = encode_rows_tmap(&ix->tmap_c_pf, ix->rows, map_rows, ix->dpad, kBlockN / 2, 256);
  if (st != RBK_OK) return st;
  st = encode_rows_tmap(&ix->tmap_c_r32, ix->rows, map_rows, ix->dpad, scan3_box_rows());
  if (st != RBK_OK) return st;
#endif
  ix->tmap_c_base = ix->rows;
  ix->tmap_c_rows = map_rows;
  return RBK_OK;
}

}  // namespace

// ---- shared with rbk_group.cu (declared in rbk_index_impl.h) ----
namespace rbk {
namespace impl {

rbk_status ensure_query_scratch(rbk_index* ix, int B, int elem) {
  CK(ix->q_raw.ensure(static_cast<size_t>(B) * ix->dim * elem));
  // rows padded to whole query blocks: the scan's TMA boxes are 128 query rows, and a box that hangs over the end of
  // the tensor is zero-FILLED by the TMA unit row by row - measured: a B = 1 scan over 1M rows took 0.295 ms against
  // 0.239 ms at B = 128 for the same bytes.  With the map covering whole blocks the pad rows are ordinary (zeroed
  // once here) memory; they only ever feed accumulator rows of queries that do not exist.
  {
    const size_t want = static_cast<size_t>(round_up(B, 2 * kBlockM)) * ix->dpad;
    if (want > ix->q_bf16.n) {
      CK(ix->q_bf16.ensure(want));
      CK(cudaMemsetAsync(ix->q_bf16.p, 0, ix->q_bf16.n * sizeof(uint16_t), ix->stream));
    }
  }
  CK(ix->q_f64.ensure(static_cast<size_t>(B) * ix->dim));
  CK(ix->q_norm2.ensure(B));
  CK(ix->q_eps.ensure(B));
  CK(ix->q_inv_norm.ensure(B));
  CK(ix->thr_init.ensure(B));
  CK(ix->flags.ensure(B));
  CK(ix->cand.ensure(static_cast<size_t>(ix->sm_count) * kBlockM * kListCap * kMaxHalves));
  CK(ix->cand_cnt.ensure(static_cast<size_t>(ix->sm_count) * kBlockM * kMaxHalves));
  // hist [kMaxSubBatch][kHistBins] | maxbin [kMaxSubBatch] | gthr [kMaxSubBatch] | progress [sm_count + 8]:
  // one buffer, one memset
  CK(ix->hist.ensure(static_cast<size_t>(kMaxSubBatch) * kHistBins + 2 * kMaxSubBatch + ix->sm_count + 8));
  return RBK_OK;
}

rbk_status check_search_args(rbk_index* ix, int B, bool have_q, int query_dim, int k_fetch, double min_score) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  if (B < 0 || (B > 0 && !have_q)) return fail(RBK_EINVAL, "bad queries argument");
  if (k_fetch < 1 || k_fetch > RBK_MAX_K_FETCH) return fail(RBK_EINVAL, "k_fetch must be in [1, 112]");
  if (query_dim != ix->dim) return fail(RBK_EDIM, "Vectors must have the same length");  // embedder.ts:170
  if (min_score != min_score) return fail(RBK_EINVAL, "min_score is NaN");
  return RBK_OK;
}

}  // namespace impl
}  // namespace rbk

namespace {

QueryBuffers query_buffers(rbk_index* ix, int q0) {
  QueryBuffers qb;
  qb.q_bf16 = ix->q_bf16.p + static_cast<size_t>(q0) * ix->dpad;
  qb.q_f64 = ix->q_f64.p + static_cast<size_t>(q0) * ix->dim;
  qb.q_norm2 = ix->q_norm2.p + q0;
  qb.q_inv_norm = ix->q_inv_norm.p + q0;
  qb.q_eps = ix->q_eps.p + q0;
  qb.thr_init = ix->thr_init.p + q0;
  return qb;
}

// Launch the scan (+ optionally finalize) for every sub-batch.  d_q: device queries.
rbk_status run_scan(rbk_index* ix, const void* d_q, int src_type, int B, int k_fetch, double min_score,
                    long long* d_slots, double* d_scores, int* d_counts, int* d_flags, float* dbg) {
  const int kprime = pick_kprime(ix, k_fetch);
  ix->stats.last_kprime = kprime;
  // (also zeroes the scan scratch of the first sub-batch; normA is left to the finalize kernel)
  const int Bs0 = std::min(kMaxSubBatch, B);
  CK(launch_prep_queries(d_q, src_type, B, ix->dim, ix->dpad, min_score, reinterpret_cast<const float*>(ix->d_counter + 1),
                         query_buffers(ix, 0), ix->stream, /*with_norm2=*/d_counts == nullptr, ix->hist.p, Bs0,
                         ix->sm_count + 8));
  ix->stats.kernel_launches++;
  if (ix->n_rows == 0) {
    // nothing to scan: finalize would read unwritten lists; emit empty results directly
    if (d_counts) {
      CK(cudaMemsetAsync(d_counts, 0, sizeof(int) * B, ix->stream));
      CK(cudaMemsetAsync(d_slots, 0xFF, sizeof(long long) * B * k_fetch, ix->stream));   // -1
      CK(cudaMemsetAsync(d_scores, 0xFF, sizeof(double) * B * k_fetch, ix->stream));     // NaN
      CK(cudaMemsetAsync(d_flags, 0, sizeof(int) * B, ix->stream));
    }
    return RBK_OK;
  }
  rbk_status st = refresh_corpus_tmap(ix);
  if (st != RBK_OK) return st;
  const int n_tiles = static_cast<int>((ix->n_rows + kBlockN - 1) / kBlockN);
  for (int q0 = 0; q0 < B; q0 += kMaxSubBatch) {
    const int Bs = std::min(kMaxSubBatch, B - q0);
    // more than one 128-query block: CTA pairs (256 queries per pair) halve the corpus bytes per query
    const bool pairs = Bs > kBlockM && !ix->force_1cta;
    const int block_m = pairs ? 2 * kBlockM : kBlockM;
    const int QB = (Bs + block_m - 1) / block_m;
    const int units = pairs ? ix->sm_count / 2 : ix->sm_count;
    int R = std::max(1, std::min(units / QB, n_tiles));
    // EXPERIMENTAL builds only (RBK_KNN_CLUSTER4=1): clusters of two pairs, one operand of every k-block multicast
    // (rbk_scan4.cu) - the kernel whose tensor pipe runs at 97 % - on every SM that can host a 4-CTA cluster (33
    // clusters = 132 of the 148 SMs of a B200), and CONCURRENTLY the pair kernel (rbk_scan2.cu) on the SMs that
    // cannot, over its own slice of the corpus.  Measured within 2 % of the pair kernel alone (power-bound), so the
    // default build launches the pair kernel on all SMs.  An even number of query blocks: the pairs of a cluster
    // take different blocks and share the corpus tile; odd: same block, alternate tiles, shared query slab.
#ifdef RBK_EXPERIMENTAL
    const bool aligned = pairs ? scan_smem_base_is_aligned() : false;
    const int max_cl = (pairs && ix->cluster4) ? scan4_max_clusters(aligned) : 0;
#else
    const int max_cl = 0;
#endif
    const bool use4 = max_cl > 0 && n_tiles >= 2;
    const bool share_c = use4 && (QB % 2) == 0;
    int RC = 0, R4 = 0, R2 = 0, T2 = 0;   // cluster ranges; list units per query block of each kernel; tiles of the tail
    if (use4) {
      const int n_cols = share_c ? QB / 2 : QB;
      RC = std::max(1, std::min(max_cl / n_cols, share_c ? n_tiles : n_tiles / 2));
      R4 = share_c ? RC : 2 * RC;
      // the tail: pairs on the SMs left over, if the scan is long enough to be worth a second launch
      const int spare_pairs = (ix->sm_count - 4 * RC * n_cols) / 2;
      R2 = ix->tail_pairs >= 0 ? std::min(ix->tail_pairs, spare_pairs / QB) : spare_pairs / QB;
      if (n_tiles < 16 * (R4 + R2)) R2 = 0;
      if (R2 > 0) {
        // a pair of the tail needs tail_rho x the time of a cluster pair per tile (no multicast: 82 % vs 97 % tensor
        // duty): tiles in proportion to capacity, so that both launches finish together
        const double cap4 = R4, cap2 = R2 / ix->tail_rho;
        T2 = static_cast<int>(n_tiles * cap2 / (cap4 + cap2) + 0.5);
        if (T2 < R2) R2 = T2 = 0;
      }
      R = R4 + R2;
    }
    CUtensorMap tmap_q, tmap_q64;
    const int q_rows = static_cast<int>(round_up(Bs, block_m));   // whole query blocks: no out-of-bounds box rows
    st = encode_rows_tmap(&tmap_q, ix->q_bf16.p + static_cast<size_t>(q0) * ix->dpad, q_rows, ix->dpad, kBlockM);
    if (st != RBK_OK) return st;
    if (use4) {   // (never in the default build)
      st = encode_rows_tmap(&tmap_q64, ix->q_bf16.p + static_cast<size_t>(q0) * ix->dpad, q_rows, ix->dpad, kBlockM / 2);
      if (st != RBK_OK) return st;
    }
    ScanParams sp;
    sp.inv_norm_c = ix->inv_norm;
    sp.thr_init = ix->thr_init.p + q0;
    sp.inv_norm_q = ix->q_inv_norm.p + q0;
    {
      // per-launch scratch, zeroed with one memset: hist rows of this sub-batch, then maxbin, gthr, progress
      unsigned int* base = ix->hist.p;
      sp.hist = base;
      sp.maxbin = reinterpret_cast<int*>(base + static_cast<size_t>(Bs) * kHistBins);
      sp.gthr = reinterpret_cast<unsigned int*>(sp.maxbin + Bs);
      sp.progress = sp.maxbin + 2 * Bs;
      if (q0 > 0)   // the first sub-batch's scratch was zeroed by the prep kernel
        CK(cudaMemsetAsync(base, 0,
                           sizeof(unsigned int) * (static_cast<size_t>(Bs) * kHistBins + 2 * Bs + ix->sm_count + 8),
                           ix->stream));
    }
    sp.cand = ix->cand.p;
    sp.cand_cnt = ix->cand_cnt.p;
    sp.dbg_scores = dbg ? dbg + static_cast<size_t>(q0) * ix->n_rows : nullptr;
    sp.n_rows = static_cast<int>(ix->n_rows);
    sp.B = Bs;
    sp.kprime = kprime;
    sp.num_kb = (ix->dpad + kBlockK - 1) / kBlockK;
    sp.dpad = ix->dpad;
    sp.QB = QB;
    sp.R = R;
    sp.RC = RC;
    sp.n_tiles = n_tiles;
    sp.tile_begin = 0;
    sp.tile_count = n_tiles - T2;
    sp.R_local = R;
    sp.unit_base = 0;
    sp.prog_base = 0;
    cudaEvent_t* tev = ix->capturing ? nullptr : next_scan_events(ix);
    if (tev) CK(cudaEventRecord(tev[0], ix->stream));
    sp.prefetch_tiles = ix->prefetch_tiles;
    sp.perf_probe = ix->perf_probe;
    sp.max_lead_tiles = ix->max_lead_tiles;
#ifdef RBK_EXPERIMENTAL
    const bool resident = pairs && !ix->force_streamed && scan2_resident_fits(ix->dpad);
    const bool ts = pairs && ix->use_ts && scan3_fits(ix->dpad);
#else
    const bool resident = false, ts = false;
#endif
    // lists per (unit, query): the default pair kernel splits every tile between two sets of epilogue warps
    // Eight epilogue warps (two lists per unit and query): measured in one box against four, +7-10 % at
    // B=256 up to 1M rows and +10-17 % at B=1024 up to 0.5M rows (where the filter is busy: thresholds still
    // rising, appends frequent), +-1 % on long scans (cfg3).  RBK_KNN_HALVES=1 forces the narrow epilogue.
    int halves = 1;
    if (pairs && !ts && ix->hybrid_res_kb < 0) {
      halves = ix->epi_halves > 0 ? std::min(ix->epi_halves, kMaxHalves) : kMaxHalves;
    }
    // Start-up seeds (rbk_epilogue.cuh): two per thread and tile when many units feed one query's histogram
    // (>= 4 k' seeds in total) - pair kernel only: measured in one box, B=256 scans 2 % (1M rows) to 9 % (65k
    // rows) faster than with two seeds per 32-column chunk, but the 1-CTA kernel at B=1 became bimodal (0.03 /
    // 0.07 ms at 65k rows): with one or two tiles per unit and only two seeds from each, a unit that reads the
    // histogram before ~k'/2 peers have seeded finds no threshold and floods its lists.
    sp.seed_tile = ix->seed_tile >= 0 ? ix->seed_tile : ((pairs && R * 2 * halves >= 4 * kprime) ? 1 : 0);
#ifdef RBK_EXPERIMENTAL
    if (use4) {
      if (R2 > 0) CK(cudaEventRecord(ix->ev_fork, ix->stream));   // scratch zeroed, queries prepared
      CK(launch_scan4(tmap_q, tmap_q64, ix->tmap_c_half, ix->tmap_c_quarter, sp, share_c, aligned, ix->stream,
                      &ix->stats.last_ring_stages));
      if (R2 > 0) {
        // launched SECOND, on its own stream: the cluster kernel's CTAs are placed first, the tail's pairs land on
        // the SMs no 4-CTA cluster fits on.  (Were they ever placed the other way round the result would still be
        // right - the kernels only exchange lower bounds - just slower.)
        ScanParams st2 = sp;
        st2.tile_begin = n_tiles - T2;
        st2.tile_count = T2;
        st2.R_local = R2;
        st2.unit_base = R4;
        st2.prog_base = RC * (share_c ? QB / 2 : QB);
        CK(cudaStreamWaitEvent(ix->side_stream, ix->ev_fork, 0));
        CK(launch_scan2(tmap_q, ix->tmap_c_half, ix->tmap_c_half, st2, false, halves, ix->side_stream, nullptr));
        CK(cudaEventRecord(ix->ev_join, ix->side_stream));
        CK(cudaStreamWaitEvent(ix->stream, ix->ev_join, 0));
        ix->stats.kernel_launches++;
      }
    } else if (pairs && !ts && ix->hybrid_res_kb >= 0)
      CK(launch_scan2h(tmap_q, ix->tmap_c_half, sp, ix->hybrid_res_kb, ix->hybrid_slots, ix->stream));
    else if (ts)
      CK(launch_scan3(ix->tmap_c_r32, sp, ix->q_bf16.p + static_cast<size_t>(q0) * ix->dpad, ix->stream));
    else if (pairs)
      CK(launch_scan2(tmap_q, (resident && scan2_resident_k() == 32) ? ix->tmap_c_half32 : ix->tmap_c_half,
                      ix->tmap_c_pf, sp, resident, halves, ix->stream, &ix->stats.last_ring_stages));
    else CK(launch_scan(tmap_q, ix->tmap_c, sp, ix->stream));
#else
    if (pairs)
      CK(launch_scan2(tmap_q, ix->tmap_c_half, ix->tmap_c_half, sp, false, halves, ix->stream,
                      &ix->stats.last_ring_stages));
    else CK(launch_scan(tmap_q, ix->tmap_c, sp, ix->stream));
#endif
    if (tev) CK(cudaEventRecord(tev[1], ix->stream));
    ix->stats.scan_launches++;
    ix->stats.kernel_launches++;
    if (d_counts) {
      FinalizeParams fp;
      fp.cand = ix->cand.p;
      fp.cand_cnt = ix->cand_cnt.p;
      fp.QB = QB;
      fp.R = R * halves;   // finalize sees every list as a unit of its own
      fp.kprime = kprime;
      fp.k_fetch = k_fetch;
      fp.B = Bs;
      fp.d = ix->dim;
      fp.dpad = ix->dpad;
      fp.q0 = q0;
      fp.block_m = block_m;
      fp.min_score = min_score;
      fp.rows = ix->rows;
      fp.rows_f64 = ix->rows_f64;
      fp.row_norm2 = ix->norm2;
      fp.n_rows = ix->n_rows;
      fp.slot = ix->slot;
      fp.q = query_buffers(ix, q0);
      fp.out_slots = d_slots + static_cast<size_t>(q0) * k_fetch;
      fp.out_scores = d_scores + static_cast<size_t>(q0) * k_fetch;
      fp.out_counts = d_counts + q0;
      fp.flags = d_flags + q0;
      CK(launch_finalize(fp, ix->stream));
      ix->stats.kernel_launches++;
    }
  }
  return RBK_OK;
}

rbk_status run_fallback(rbk_index* ix, const std::vector<int>& fails, int k_fetch, double min_score,
                        long long* d_slots, double* d_scores, int* d_counts) {
  const int nf = static_cast<int>(fails.size());
  const int nb = std::max(1, std::min<int>(ix->sm_count * 2, static_cast<int>((ix->n_rows + 255) / 256)));
  CK(ix->fail_list.ensure(nf));
  CK(ix->part_scores.ensure(static_cast<size_t>(nf) * nb * k_fetch));
  CK(ix->part_rows.ensure(static_cast<size_t>(nf) * nb * k_fetch));
  CK(ix->part_cnt.ensure(static_cast<size_t>(nf) * nb));
  CK(cudaMemcpyAsync(ix->fail_list.p, fails.data(), sizeof(int) * nf, cudaMemcpyHostToDevice, ix->stream));
  ExactParams ep;
  ep.fail_list = ix->fail_list.p;
  ep.n_fail = nf;
  ep.d = ix->dim;
  ep.dpad = ix->dpad;
  ep.k_fetch = k_fetch;
  ep.min_score = min_score;
  ep.rows = ix->rows;
  ep.rows_f64 = ix->rows_f64;
  ep.row_norm2 = ix->norm2;
  ep.dead_bits = ix->dead_bits;
  ep.n_rows = ix->n_rows;
  ep.slot = ix->slot;
  ep.q_f64 = ix->q_f64.p;
  ep.q_norm2 = ix->q_norm2.p;
  ep.part_scores = ix->part_scores.p;
  ep.part_rows = ix->part_rows.p;
  ep.part_cnt = ix->part_cnt.p;
  ep.n_blocks = nb;
  ep.out_slots = d_slots;
  ep.out_scores = d_scores;
  ep.out_counts = d_counts;
  CK(launch_exact_fallback(ep, ix->stream));
  // pageable source: the copy above has completed its host read before returning
  ix->stats.kernel_launches += 2;
  ix->stats.fallback_queries += nf;
  return RBK_OK;
}

}  // namespace

namespace rbk {
namespace impl {
// Enqueue-only search of device-resident queries (caller holds the lock).  No host synchronisation: the
// exactness flags land in d_flags and are the caller's to check (rbk_index_search_device_async, rbk_group.cu).
rbk_status enqueue_search(rbk_index* ix, const void* d_q, int src_type, int B, int k_fetch, double min_score,
                          long long* d_slots, double* d_scores, int* d_counts, int* d_flags) {
  ix->stats.searches++;
  ix->stats.queries += B;
  return run_scan(ix, d_q, src_type, B, k_fetch, min_score, d_slots, d_scores, d_counts, d_flags, nullptr);
}
}  // namespace impl
}  // namespace rbk

namespace {

void drop_graph(rbk_index* ix) {
  if (ix->graph_exec) cudaGraphExecDestroy(ix->graph_exec);
  ix->graph_exec = nullptr;
}

// Small-batch fast path of search_core (caller holds the lock; scratch, o_block and h_block are allocated): replay
// - or first capture - the graph of one whole search.  *done = true: results and flags are in h_block and every
// query is proven exact.  *done = false: something needs the general path (a query's proof failed), which the
// caller then runs from scratch.
rbk_status search_graph(rbk_index* ix, const void* q_host, int elem, int B, int k_fetch, double min_score,
                        size_t blk, size_t off_flags, bool* done) {
  *done = false;
  const size_t q_bytes = static_cast<size_t>(B) * ix->dim * elem;
  CK(ix->h_q.ensure(q_bytes));
  rbk_index::GraphKey key;
  memset(&key, 0, sizeof key);   // compared with memcmp: padding must be defined
  const void* ptrs[20] = {ix->rows, ix->inv_norm, ix->norm2, ix->rows_f64, ix->dead_bits, ix->d_counter, ix->q_raw.p,
                          ix->q_bf16.p, ix->q_f64.p, ix->q_norm2.p, ix->q_eps.p, ix->q_inv_norm.p, ix->thr_init.p,
                          ix->cand.p, ix->cand_cnt.p, ix->hist.p, ix->o_block.p, ix->h_block.p, ix->h_q.p, nullptr};
  memcpy(key.ptr, ptrs, sizeof ptrs);
  key.n_rows = ix->n_rows;
  key.min_score = min_score;
  key.B = B;
  key.k_fetch = k_fetch;
  key.elem = elem;
  key.margin = ix->margin;
  key.slot = ix->slot;
  key.stream = ix->stream;
  unsigned char* base = ix->o_block.p;
  const size_t nout = static_cast<size_t>(B) * k_fetch;
  if (!ix->graph_exec || memcmp(&key, &ix->graph_key, sizeof key) != 0) {
    drop_graph(ix);
    cudaGraph_t graph = nullptr;
    CK(cudaStreamBeginCapture(ix->stream, cudaStreamCaptureModeThreadLocal));
    ix->capturing = true;
    cudaError_t e = cudaMemcpyAsync(ix->q_raw.p, ix->h_q.p, q_bytes, cudaMemcpyHostToDevice, ix->stream);
    rbk_status st = RBK_OK;
    if (e == cudaSuccess)
      st = run_scan(ix, ix->q_raw.p, elem == 8 ? 0 : 1, B, k_fetch, min_score, reinterpret_cast<long long*>(base),
                    reinterpret_cast<double*>(base + nout * 8), reinterpret_cast<int*>(base + nout * 16),
                    reinterpret_cast<int*>(base + off_flags), nullptr);
    if (e == cudaSuccess && st == RBK_OK)
      e = cudaMemcpyAsync(ix->h_block.p, ix->o_block.p, blk, cudaMemcpyDeviceToHost, ix->stream);
    ix->capturing = false;
    const cudaError_t e2 = cudaStreamEndCapture(ix->stream, &graph);   // always leave capture mode
    if (st != RBK_OK) {
      if (graph) cudaGraphDestroy(graph);
      return st;
    }
    if (e != cudaSuccess || e2 != cudaSuccess || !graph) {
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      ix->use_graph = false;   // capture not possible here (e.g. the caller's stream is itself capturing): general
      return RBK_OK;           // path from now on, no retry per search
    }
    e = cudaGraphInstantiate(&ix->graph_exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) {
      ix->graph_exec = nullptr;
      cudaGetLastError();
      ix->use_graph = false;
      return RBK_OK;
    }
    memcpy(&ix->graph_key, &key, sizeof key);
  }
  memcpy(ix->h_q.p, q_host, q_bytes);
  CK(cudaEventRecord(get_event(ix, 0), ix->stream));
  CK(cudaGraphLaunch(ix->graph_exec, ix->stream));
  CK(cudaEventRecord(get_event(ix, 1), ix->stream));
  CK(cudaStreamSynchronize(ix->stream));   // the one host round trip
  ix->stats.searches++;
  ix->stats.queries += B;
  ix->stats.scan_launches++;
  ix->stats.kernel_launches += 3;           // prep, scan, finalize (inside the graph)
  ix->stats.graph_replays++;
  const int* h_flags = reinterpret_cast<const int*>(ix->h_block.p + off_flags);
  for (int b = 0; b < B; ++b)
    if (h_flags[b]) return RBK_OK;          // a proof failed: the general path re-answers the batch
  float total = 0.f;
  cudaEventElapsedTime(&total, get_event(ix, 0), get_event(ix, 1));
  ix->stats.last_total_ms = total;
  *done = true;
  return RBK_OK;
}

// Whole search, synchronous.  q_host/q_dev: exactly one is non-null.  Host outputs (h_*) may be null
// (device-output variant); device outputs may be null (host variant uses index scratch).
rbk_status search_core(rbk_index* ix, const void* q_host, const void* q_dev, int elem, int B, int query_dim,
                       int k_fetch, double min_score, long long* d_slots, double* d_scores, int* d_counts,
                       int64_t* h_slots, double* h_scores, int32_t* h_counts, float* ms_out) {
  rbk_status st = check_search_args(ix, B, q_host || q_dev, query_dim, k_fetch, min_score);
  if (st != RBK_OK) return st;
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  if (ms_out) *ms_out = 0.f;
  if (B == 0) {
    ix->stats.searches++;
    return RBK_OK;
  }
  st = ensure_query_scratch(ix, B, elem);
  if (st != RBK_OK) return st;
  const size_t nout = static_cast<size_t>(B) * k_fetch;
  // Host-output calls use ONE packed device block (slots | scores | counts | flags) mirrored by one pinned
  // host block, so results and exactness flags come back in a single D2H copy.
  const size_t off_scores = nout * 8, off_counts = nout * 16, off_flags = off_counts + static_cast<size_t>(B) * 4;
  const size_t blk = off_flags + static_cast<size_t>(B) * 4;
  const bool packed = d_slots == nullptr;
  int* d_flags = ix->flags.p;
  const int* h_flags = nullptr;
  if (packed) {
    CK(ix->o_block.ensure(blk));
    CK(ix->h_block.ensure(blk));
    unsigned char* base = ix->o_block.p;
    d_slots = reinterpret_cast<long long*>(base);
    d_scores = reinterpret_cast<double*>(base + off_scores);
    d_counts = reinterpret_cast<int*>(base + off_counts);
    d_flags = reinterpret_cast<int*>(base + off_flags);
    h_flags = reinterpret_cast<const int*>(ix->h_block.p + off_flags);
  } else {
    CK(ix->h_flags.ensure(B));
    h_flags = ix->h_flags.p;
  }
  if (packed && q_host && B <= kBlockM && ix->n_rows > 0 && ix->use_graph) {
    bool done = false;
    st = search_graph(ix, q_host, elem, B, k_fetch, min_score, blk, off_flags, &done);
    if (st != RBK_OK) return st;
    if (done) {
      if (ms_out) *ms_out = ix->stats.last_total_ms;
      memcpy(h_slots, ix->h_block.p, sizeof(int64_t) * nout);
      memcpy(h_scores, ix->h_block.p + off_scores, sizeof(double) * nout);
      memcpy(h_counts, ix->h_block.p + off_counts, sizeof(int32_t) * B);
      return RBK_OK;
    }
  }
  resolve_scan_events(ix, false);
  const double scan_ms0 = ix->stats.scan_ms_total;
  CK(cudaEventRecord(get_event(ix, 0), ix->stream));
  const void* d_q = q_dev;
  if (q_host) {
    CK(cudaMemcpyAsync(ix->q_raw.p, q_host, static_cast<size_t>(B) * ix->dim * elem, cudaMemcpyHostToDevice,
                       ix->stream));
    d_q = ix->q_raw.p;
  }
  const int src_type = elem == 8 ? 0 : 1;
  st = enqueue_search(ix, d_q, src_type, B, k_fetch, min_score, d_slots, d_scores, d_counts, d_flags);
  if (st != RBK_OK) return st;
  auto copy_back = [&]() -> cudaError_t {
    if (packed) return cudaMemcpyAsync(ix->h_block.p, ix->o_block.p, blk, cudaMemcpyDeviceToHost, ix->stream);
    return cudaMemcpyAsync(ix->h_flags.p, d_flags, sizeof(int) * B, cudaMemcpyDeviceToHost, ix->stream);
  };
  CK(copy_back());
  CK(cudaEventRecord(get_event(ix, 1), ix->stream));
  CK(cudaStreamSynchronize(ix->stream));   // the ONE host round trip of an exact batch
  std::vector<int> fails;
  for (int b = 0; b < B; ++b)
    if (h_flags[b]) fails.push_back(b);
  if (!fails.empty() && ix->retry_wide && ix->stats.last_kprime < kMaxKPrime) {
    // A proof fails when more rows tie with the k_fetch-th hit (within the scan's error bound) than the
    // candidate margin holds - duplicated chunks, typically.  Before paying an exhaustive fp64 pass per failing
    // query, scan the batch once more at scan speed with the widest margin (k' = 128): groups of up to ~100
    // near-ties then fit among the candidates and the proof goes through.  Results of the queries that had
    // already passed are recomputed to the same values (both passes are exact).
    ix->kprime_override = kMaxKPrime;
    st = run_scan(ix, d_q, src_type, B, k_fetch, min_score, d_slots, d_scores, d_counts, d_flags, nullptr);
    ix->kprime_override = 0;
    if (st != RBK_OK) return st;
    CK(copy_back());
    CK(cudaEventRecord(get_event(ix, 1), ix->stream));
    CK(cudaStreamSynchronize(ix->stream));
    ix->stats.retry_batches++;
    fails.clear();
    for (int b = 0; b < B; ++b)
      if (h_flags[b]) fails.push_back(b);
  }
  if (!fails.empty()) {
    st = run_fallback(ix, fails, k_fetch, min_score, d_slots, d_scores, d_counts);
    if (st != RBK_OK) return st;
    // the exhaustive answers are exact by construction: clear the flags the caller may forward
    CK(cudaMemsetAsync(d_flags, 0, sizeof(int) * B, ix->stream));
    if (packed) CK(copy_back());
    CK(cudaEventRecord(get_event(ix, 1), ix->stream));
    CK(cudaStreamSynchronize(ix->stream));
  }
  float total = 0.f;
  cudaEventElapsedTime(&total, get_event(ix, 0), get_event(ix, 1));
  resolve_scan_events(ix, true);   // the stream is idle: every pair is final
  ix->stats.last_total_ms = total;
  ix->stats.last_scan_ms = static_cast<float>(ix->stats.scan_ms_total - scan_ms0);
  if (ms_out) *ms_out = total;
  if (h_slots) {
    memcpy(h_slots, ix->h_block.p, sizeof(int64_t) * nout);
    memcpy(h_scores, ix->h_block.p + off_scores, sizeof(double) * nout);
    memcpy(h_counts, ix->h_block.p + off_counts, sizeof(int32_t) * B);
  }
  return RBK_OK;
}

}  // namespace

// =========================================================================== C ABI
extern "C" {

int rbk_abi_version(void) { return RBK_ABI_VERSION; }
const char* rbk_last_error(void) { return rbk::impl::last_error(); }

rbk_status rbk_index_create(int32_t dim, int32_t device, int64_t capacity_hint, rbk_index** out) {
  return rbk_index_create_ex(dim, device, capacity_hint, 0, out);
}

rbk_status rbk_index_create_ex(int32_t dim, int32_t device, int64_t capacity_hint, uint32_t flags, rbk_index** out) {
  if (!out) return fail(RBK_EINVAL, "out is null");
  if (flags & ~static_cast<uint32_t>(RBK_INDEX_KEEP_F64)) return fail(RBK_EINVAL, "unknown flag");
  *out = nullptr;
  if (dim < 1 || dim > (1 << 20)) return fail(RBK_EINVAL, "dim out of range");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(RBK_ECUDA, std::string("no CUDA device (this engine has no CPU path): ") +
                               (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
  if (device < 0 || device >= ndev) return fail(RBK_EINVAL, "device ordinal out of range");
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(RBK_ECUDA, std::string("this build targets sm_100a (Blackwell B200); device is ") + prop.name);
  DeviceGuard dg(device);
  rbk_index* ix = new (std::nothrow) rbk_index();
  if (!ix) return fail(RBK_ENOMEM, "out of host memory");
  ix->dim = dim;
  // row pitch = whole 64-element k-blocks (128 bytes): no TMA box hangs over the end of a row either
  ix->dpad = static_cast<int>(round_up(dim, kBlockK));
  ix->device = device;
  ix->keep_f64 = (flags & RBK_INDEX_KEEP_F64) != 0;
  ix->sm_count = prop.multiProcessorCount;
  memset(&ix->stats, 0, sizeof ix->stats);
  ix->stats.sm_count = ix->sm_count;
#ifdef RBK_EXPERIMENTAL   // A/B switches of development builds; the shipped library reads no environment
  if (const char* m = getenv("RBK_KNN_CLUSTER4")) ix->cluster4 = atoi(m);
  if (const char* m = getenv("RBK_KNN_GRAPH")) ix->use_graph = atoi(m) != 0;
  if (const char* m = getenv("RBK_KNN_TAIL_PAIRS")) ix->tail_pairs = atoi(m);
  if (const char* m = getenv("RBK_KNN_TAIL_RHO")) ix->tail_rho = std::max(0.5, std::min(3.0, atof(m)));
  if (const char* m = getenv("RBK_KNN_MARGIN")) ix->margin = std::max(0, std::min(96, atoi(m)));
  if (const char* m = getenv("RBK_KNN_FORCE_1CTA")) ix->force_1cta = atoi(m) != 0;
  if (const char* m = getenv("RBK_KNN_RESIDENT")) ix->force_streamed = atoi(m) == 0;
  if (const char* m = getenv("RBK_KNN_TS")) ix->use_ts = atoi(m) != 0;
  if (const char* m = getenv("RBK_KNN_MAX_LEAD")) ix->max_lead_tiles = std::max(1, atoi(m));
  if (const char* m = getenv("RBK_KNN_SEED_TILE")) ix->seed_tile = atoi(m);
  if (const char* m = getenv("RBK_KNN_RETRY_WIDE")) ix->retry_wide = atoi(m) != 0;
  if (const char* m = getenv("RBK_KNN_HALVES")) ix->epi_halves = std::max(0, atoi(m));
  if (const char* m = getenv("RBK_KNN_PERF_PROBE")) ix->perf_probe = atoi(m);   // breaks results; timing only
  if (const char* m = getenv("RBK_KNN_HYBRID_KB")) ix->hybrid_res_kb = atoi(m);
  if (const char* m = getenv("RBK_KNN_HYBRID_SLOTS")) ix->hybrid_slots = atoi(m);
  if (const char* m = getenv("RBK_KNN_PREFETCH_TILES")) ix->prefetch_tiles = std::max(0, std::min(64, atoi(m)));
#endif
  e = cudaStreamCreateWithFlags(&ix->own_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete ix;
    return cuda_fail(e, "cudaStreamCreate");
  }
  ix->stream = ix->own_stream;
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ix->side_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ix->ev_join, cudaEventDisableTiming);
  if (e != cudaSuccess) {
    rbk_index_destroy(ix);
    return cuda_fail(e, "cudaStreamCreate");
  }
  e = cudaMalloc(reinterpret_cast<void**>(&ix->d_counter), 2 * sizeof(int));
  if (e == cudaSuccess) e = cudaMemset(ix->d_counter, 0, 2 * sizeof(int));
  if (e != cudaSuccess) {
    rbk_index_destroy(ix);
    return cuda_fail(e, "cudaMalloc");
  }
  rbk_status st = ensure_capacity(ix, std::max<int64_t>(capacity_hint, 1024));
  if (st != RBK_OK) {
    rbk_index_destroy(ix);
    return st;
  }
  *out = ix;
  return RBK_OK;
}

void rbk_index_destroy(rbk_index* ix) {
  if (!ix) return;
  {
    DeviceGuard dg(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    cudaFree(ix->rows);
    cudaFree(ix->inv_norm);
    cudaFree(ix->norm2);
    cudaFree(ix->dead_bits);
    cudaFree(ix->rows_f64);
    cudaFree(ix->d_counter);
    ix->stage.release();
    ix->d_slots.release();
    ix->q_raw.release();
    ix->q_bf16.release();
    ix->q_f64.release();
    ix->q_norm2.release();
    ix->q_eps.release();
    ix->q_inv_norm.release();
    ix->thr_init.release();
    ix->cand.release();
    ix->cand_cnt.release();
    ix->hist.release();
    ix->maxbin.release();
    ix->progress.release();
    ix->flags.release();
    ix->fail_list.release();
    ix->o_counts.release();
    ix->part_rows.release();
    ix->part_cnt.release();
    ix->o_slots.release();
    ix->o_scores.release();
    ix->part_scores.release();
    ix->dbg.release();
    ix->o_block.release();
    ix->h_block.release();
    ix->h_flags.release();
    ix->h_counts.release();
    ix->h_slots.release();
    ix->h_scores.release();
    ix->h_f32.release();
    drop_graph(ix);
    ix->h_q.release();
    for (cudaEvent_t e : ix->ev) cudaEventDestroy(e);
    for (auto& pr : ix->tev)
      for (cudaEvent_t e : pr)
        if (e) cudaEventDestroy(e);
    if (ix->side_stream) {
      cudaStreamSynchronize(ix->side_stream);
      cudaStreamDestroy(ix->side_stream);
    }
    if (ix->ev_fork) cudaEventDestroy(ix->ev_fork);
    if (ix->ev_join) cudaEventDestroy(ix->ev_join);
    if (ix->own_stream) cudaStreamDestroy(ix->own_stream);
  }
  delete ix;
}

rbk_status rbk_index_set_stream(rbk_index* ix, void* cuda_stream) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  CK(cudaStreamSynchronize(ix->stream));
  ix->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ix->own_stream;
  return RBK_OK;
}

rbk_status rbk_index_set_slot_base(rbk_index* ix, int64_t slot_base) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  if (slot_base < 0) return fail(RBK_EINVAL, "slot_base must be >= 0");
  std::lock_guard<std::mutex> lk(ix->mu);
  ix->slot.base = slot_base;
  return RBK_OK;
}

rbk_status rbk_index_append_f64(rbk_index* ix, const double* rows, int64_t n, int64_t* first) {
  return append_rows(ix, rows, false, 8, n, first);
}
rbk_status rbk_index_append_f32(rbk_index* ix, const float* rows, int64_t n, int64_t* first) {
  return append_rows(ix, rows, false, 4, n, first);
}
rbk_status rbk_index_append_bf16(rbk_index* ix, const uint16_t* rows, int64_t n, int64_t* first) {
  return append_rows(ix, rows, false, 2, n, first);
}
rbk_status rbk_index_append_bf16_device(rbk_index* ix, const void* dev_rows, int64_t n, int64_t* first) {
  return append_rows(ix, dev_rows, true, 2, n, first);
}
rbk_status rbk_index_append_f64_device(rbk_index* ix, const void* dev_rows, int64_t n, int64_t* first) {
  return append_rows(ix, dev_rows, true, 8, n, first);
}

rbk_status rbk_index_overwrite_f64_batch(rbk_index* ix, const int64_t* slots, int64_t n, const double* rows) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  if (n < 0 || (n > 0 && (!slots || !rows))) return fail(RBK_EINVAL, "bad argument");
  if (n == 0) return RBK_OK;
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  for (int64_t i = 0; i < n; ++i)
    if (slots[i] < 0 || slots[i] >= ix->n_rows) return fail(RBK_EINVAL, "slot out of range");
  // The same slot twice in one batch is Map.set twice: the LAST value wins (and two thread blocks scattering into one
  // row would race).  Keep each slot's last occurrence; the common case (no repeats) copies nothing.
  std::vector<int64_t> u_slots;
  std::vector<double> u_rows;
  if (n > 1) {
    std::unordered_map<int64_t, int64_t> last;
    last.reserve(static_cast<size_t>(n) * 2);
    for (int64_t i = 0; i < n; ++i) last[slots[i]] = i;
    if (static_cast<int64_t>(last.size()) != n) {
      u_slots.reserve(last.size());
      u_rows.resize(last.size() * static_cast<size_t>(ix->dim));
      for (int64_t i = 0; i < n; ++i) {
        if (last[slots[i]] != i) continue;
        memcpy(u_rows.data() + u_slots.size() * static_cast<size_t>(ix->dim), rows + static_cast<size_t>(i) * ix->dim,
               static_cast<size_t>(ix->dim) * 8);
        u_slots.push_back(slots[i]);
      }
      slots = u_slots.data();
      rows = u_rows.data();
      n = static_cast<int64_t>(u_slots.size());
    }
  }
  // one H2D of the slots, one of the rows (chunked through the staging buffer), two kernels per chunk that scatter
  // into the named slots and skip tombstoned ones on the device, ONE host round trip for the whole batch
  const size_t row_bytes = static_cast<size_t>(ix->dim) * 8;
  const int64_t chunk_rows = std::max<int64_t>(1, std::min<int64_t>(n, (64ll << 20) / static_cast<int64_t>(row_bytes)));
  CK(ix->stage.ensure(static_cast<size_t>(chunk_rows) * row_bytes));
  CK(ix->d_slots.ensure(static_cast<size_t>(n)));
  CK(cudaMemcpyAsync(ix->d_slots.p, slots, sizeof(int64_t) * n, cudaMemcpyHostToDevice, ix->stream));
  CK(cudaMemsetAsync(ix->d_counter, 0, sizeof(int), ix->stream));
  for (int64_t r0 = 0; r0 < n; r0 += chunk_rows) {
    const int64_t nr = std::min<int64_t>(chunk_rows, n - r0);
    CK(cudaMemcpyAsync(ix->stage.p, reinterpret_cast<const unsigned char*>(rows) + static_cast<size_t>(r0) * row_bytes,
                       static_cast<size_t>(nr) * row_bytes, cudaMemcpyHostToDevice, ix->stream));
    CK(launch_convert_rows(ix->stage.p, 0, nr, ix->dim, ix->dpad, ix->rows, ix->keep_f64 ? ix->rows_f64 : nullptr,
                           ix->stream, ix->d_slots.p + r0, ix->dead_bits, ix->d_counter));
    CK(launch_row_norms(ix->rows, ix->keep_f64 ? ix->rows_f64 : nullptr, 0, nr, ix->dim, ix->dpad, ix->inv_norm,
                        ix->norm2, ix->d_counter + 1, ix->stream, ix->d_slots.p + r0, ix->dead_bits));
    ix->stats.kernel_launches += ix->keep_f64 ? 3 : 2;
  }
  int dead = 0;
  CK(cudaMemcpyAsync(&dead, ix->d_counter, sizeof(int), cudaMemcpyDeviceToHost, ix->stream));
  CK(cudaStreamSynchronize(ix->stream));
  if (dead > 0) {
    // a tombstoned slot stays dead: the host never overwrites a deleted id (S9b: a re-added id is appended)
    char buf[96];
    snprintf(buf, sizeof buf, "slot is tombstoned (%d of %lld rows skipped)", dead, static_cast<long long>(n));
    return fail(RBK_EINVAL, buf);
  }
  return RBK_OK;
}

rbk_status rbk_index_overwrite_f64(rbk_index* ix, int64_t slot, const double* row) {
  if (!row) return fail(RBK_EINVAL, "null argument");
  return rbk_index_overwrite_f64_batch(ix, &slot, 1, row);
}

rbk_status rbk_index_tombstone(rbk_index* ix, const int64_t* slots, int64_t n) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  if (n < 0 || (n > 0 && !slots)) return fail(RBK_EINVAL, "bad slots argument");
  if (n == 0) return RBK_OK;
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  for (int64_t i = 0; i < n; ++i)
    if (slots[i] < 0 || slots[i] >= ix->n_rows) return fail(RBK_EINVAL, "slot out of range");
  CK(ix->d_slots.ensure(static_cast<size_t>(n)));
  CK(cudaMemcpyAsync(ix->d_slots.p, slots, sizeof(int64_t) * n, cudaMemcpyHostToDevice, ix->stream));
  CK(cudaMemsetAsync(ix->d_counter, 0, sizeof(int), ix->stream));
  CK(launch_tombstone(ix->d_slots.p, n, ix->n_rows, ix->inv_norm, ix->dead_bits, ix->d_counter, ix->stream));
  ix->stats.kernel_launches++;
  int killed = 0;
  CK(cudaMemcpyAsync(&killed, ix->d_counter, sizeof(int), cudaMemcpyDeviceToHost, ix->stream));
  CK(cudaStreamSynchronize(ix->stream));
  ix->n_live -= killed;
  return RBK_OK;
}

rbk_status rbk_index_clear(rbk_index* ix) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  CK(cudaMemsetAsync(ix->inv_norm, 0xFF, static_cast<size_t>(inv_norm_len(ix->cap)) * 4, ix->stream));
  CK(cudaMemsetAsync(ix->dead_bits, 0, static_cast<size_t>((ix->cap + 31) / 32) * 4, ix->stream));
  CK(cudaMemsetAsync(ix->d_counter, 0, 2 * sizeof(int), ix->stream));   // also resets the corpus-side error bound
  CK(cudaStreamSynchronize(ix->stream));
  ix->n_rows = 0;
  ix->n_live = 0;
  return RBK_OK;
}

int64_t rbk_index_count(const rbk_index* ix) { return ix ? ix->n_live : 0; }
int64_t rbk_index_size(const rbk_index* ix) { return ix ? ix->n_rows : 0; }
int32_t rbk_index_dim(const rbk_index* ix) { return ix ? ix->dim : 0; }

rbk_status rbk_index_read_rows_bf16(rbk_index* ix, int64_t first, int64_t n, uint16_t* out) {
  if (!ix || (n > 0 && !out)) return fail(RBK_EINVAL, "null argument");
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  if (first < 0 || n < 0 || first + n > ix->n_rows) return fail(RBK_EINVAL, "row range out of bounds");
  if (n == 0) return RBK_OK;
  CK(cudaMemcpy2DAsync(out, static_cast<size_t>(ix->dim) * 2, ix->rows + static_cast<size_t>(first) * ix->dpad,
                       static_cast<size_t>(ix->dpad) * 2, static_cast<size_t>(ix->dim) * 2, static_cast<size_t>(n),
                       cudaMemcpyDeviceToHost, ix->stream));
  CK(cudaStreamSynchronize(ix->stream));
  return RBK_OK;
}

rbk_status rbk_index_search_f64(rbk_index* ix, const double* queries, int32_t B, int32_t query_dim, int32_t k_fetch,
                                double min_score, int64_t* out_slots, double* out_scores, int32_t* out_counts,
                                float* kernel_ms_out) {
  if (B > 0 && (!out_slots || !out_scores || !out_counts)) return fail(RBK_EINVAL, "null output");
  return search_core(ix, queries, nullptr, 8, B, query_dim, k_fetch, min_score, nullptr, nullptr, nullptr, out_slots,
                     out_scores, out_counts, kernel_ms_out);
}
rbk_status rbk_index_search_f32(rbk_index* ix, const float* queries, int32_t B, int32_t query_dim, int32_t k_fetch,
                                double min_score, int64_t* out_slots, double* out_scores, int32_t* out_counts,
                                float* kernel_ms_out) {
  if (B > 0 && (!out_slots || !out_scores || !out_counts)) return fail(RBK_EINVAL, "null output");
  return search_core(ix, queries, nullptr, 4, B, query_dim, k_fetch, min_score, nullptr, nullptr, nullptr, out_slots,
                     out_scores, out_counts, kernel_ms_out);
}
rbk_status rbk_index_search_device(rbk_index* ix, const void* dev_queries_f32, int32_t B, int32_t k_fetch,
                                   double min_score, void* dev_out_slots, void* dev_out_scores,
                                   void* dev_out_counts) {
  if (B > 0 && (!dev_queries_f32 || !dev_out_slots || !dev_out_scores || !dev_out_counts))
    return fail(RBK_EINVAL, "null device pointer");
  return search_core(ix, nullptr, dev_queries_f32, 4, B, ix ? ix->dim : 0, k_fetch, min_score,
                     static_cast<long long*>(dev_out_slots), static_cast<double*>(dev_out_scores),
                     static_cast<int*>(dev_out_counts), nullptr, nullptr, nullptr, nullptr);
}

rbk_status rbk_index_exact_scores_f64(rbk_index* ix, const double* queries, int32_t B, int32_t query_dim,
                                      double* out_scores) {
  if (!ix) return fail(RBK_EINVAL, "null index");
  if (B < 0 || (B > 0 && (!queries || !out_scores))) return fail(RBK_EINVAL, "bad argument");
  if (query_dim != ix->dim) return fail(RBK_EDIM, "Vectors must have the same length");  // embedder.ts:170
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  if (B == 0 || ix->n_rows == 0) return RBK_OK;
  rbk_status st = ensure_query_scratch(ix, B, 8);
  if (st != RBK_OK) return st;
  const size_t n = static_cast<size_t>(B) * ix->n_rows;
  CK(ix->o_scores.ensure(n));
  CK(cudaMemcpyAsync(ix->q_raw.p, queries, static_cast<size_t>(B) * ix->dim * 8, cudaMemcpyHostToDevice, ix->stream));
  // the prep kernel gives the f64 copy and the reference's normA; its scan-side outputs are unused here
  CK(launch_prep_queries(ix->q_raw.p, 0, B, ix->dim, ix->dpad, -INFINITY, nullptr, query_buffers(ix, 0), ix->stream,
                         /*with_norm2=*/true, nullptr, 0, 0));
  CK(launch_exact_scores(ix->rows, ix->rows_f64, ix->norm2, ix->dead_bits, ix->n_rows, ix->dim, ix->dpad, ix->q_f64.p,
                         ix->q_norm2.p, B, ix->o_scores.p, ix->stream));
  ix->stats.kernel_launches += 2;
  CK(cudaMemcpyAsync(out_scores, ix->o_scores.p, n * 8, cudaMemcpyDeviceToHost, ix->stream));
  CK(cudaStreamSynchronize(ix->stream));
  return RBK_OK;
}

rbk_status rbk_index_search_device_async(rbk_index* ix, const void* dev_queries_f32, int32_t B, int32_t k_fetch,
                                         double min_score, void* dev_out_slots, void* dev_out_scores,
                                         void* dev_out_counts, void* dev_out_flags) {
  if (B > 0 && (!dev_queries_f32 || !dev_out_slots || !dev_out_scores || !dev_out_counts || !dev_out_flags))
    return fail(RBK_EINVAL, "null device pointer");
  rbk_status st = check_search_args(ix, B, true, ix ? ix->dim : 0, k_fetch, min_score);
  if (st != RBK_OK) return st;
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  if (B == 0) return RBK_OK;
  st = ensure_query_scratch(ix, B, 4);
  if (st != RBK_OK) return st;
  return enqueue_search(ix, dev_queries_f32, 1, B, k_fetch, min_score, static_cast<long long*>(dev_out_slots),
                        static_cast<double*>(dev_out_scores), static_cast<int*>(dev_out_counts),
                        static_cast<int*>(dev_out_flags));
}

rbk_status rbk_merge_topk_device(int32_t device, void* cuda_stream, int32_t G, int32_t B, int32_t k_fetch,
                                 const void* dev_slots, const void* dev_scores, const void* dev_counts,
                                 void* dev_out_slots, void* dev_out_scores, void* dev_out_counts) {
  if (G < 1 || B < 0 || k_fetch < 1) return fail(RBK_EINVAL, "bad merge shape");
  if (B == 0) return RBK_OK;
  if (!dev_slots || !dev_scores || !dev_counts || !dev_out_slots || !dev_out_scores || !dev_out_counts)
    return fail(RBK_EINVAL, "null device pointer");
  DeviceGuard dg(device);
  const size_t nk = static_cast<size_t>(B) * k_fetch;
  CK(launch_merge_shards(G, B, k_fetch, dev_slots, dev_scores, dev_counts, nullptr, nk * 8, nk * 8,
                         static_cast<size_t>(B) * 4, 0, static_cast<long long*>(dev_out_slots),
                         static_cast<double*>(dev_out_scores), static_cast<int*>(dev_out_counts), nullptr,
                         static_cast<cudaStream_t>(cuda_stream)));
  return RBK_OK;
}

int64_t rbk_packed_block_bytes(int32_t B, int32_t k_fetch) {
  const int64_t nk = static_cast<int64_t>(B) * k_fetch;
  return nk * 16 + 2 * (((static_cast<int64_t>(B) * 4 + 15) / 16) * 16);   // slots | scores | counts | flags
}
int64_t rbk_packed_flags_offset(int32_t B, int32_t k_fetch) {
  const int64_t nk = static_cast<int64_t>(B) * k_fetch;
  return nk * 16 + ((static_cast<int64_t>(B) * 4 + 15) / 16) * 16;
}

rbk_status rbk_merge_topk_packed_device(int32_t device, void* cuda_stream, int32_t G, int32_t B, int32_t k_fetch,
                                        const void* dev_blocks, void* dev_out_slots, void* dev_out_scores,
                                        void* dev_out_counts, void* dev_out_flags) {
  if (G < 1 || B < 0 || k_fetch < 1) return fail(RBK_EINVAL, "bad merge shape");
  if (B == 0) return RBK_OK;
  if (!dev_blocks || !dev_out_slots || !dev_out_scores || !dev_out_counts)
    return fail(RBK_EINVAL, "null device pointer");
  DeviceGuard dg(device);
  const size_t nk = static_cast<size_t>(B) * k_fetch;
  const size_t stride = static_cast<size_t>(rbk_packed_block_bytes(B, k_fetch));
  const char* base = static_cast<const char*>(dev_blocks);
  CK(launch_merge_shards(G, B, k_fetch, base, base + nk * 8, base + nk * 16,
                         dev_out_flags ? base + rbk_packed_flags_offset(B, k_fetch) : nullptr, stride, stride, stride,
                         stride, static_cast<long long*>(dev_out_slots), static_cast<double*>(dev_out_scores),
                         static_cast<int*>(dev_out_counts), static_cast<int*>(dev_out_flags),
                         static_cast<cudaStream_t>(cuda_stream)));
  return RBK_OK;
}

rbk_status rbk_index_stats(rbk_index* ix, rbk_stats* out) {
  if (!ix || !out) return fail(RBK_EINVAL, "null argument");
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  resolve_scan_events(ix, false);   // fold in every scan that has finished; never blocks
  *out = ix->stats;
  return RBK_OK;
}

rbk_status rbk_index_debug_scores_f32(rbk_index* ix, const float* queries, int32_t B, float* out_scores) {
  if (!ix || !queries || !out_scores || B < 1) return fail(RBK_EINVAL, "bad argument");
  std::lock_guard<std::mutex> lk(ix->mu);
  DeviceGuard dg(ix->device);
  if (ix->n_rows == 0) return RBK_OK;
  rbk_status st = ensure_query_scratch(ix, B, 4);
  if (st != RBK_OK) return st;
  const size_t n = static_cast<size_t>(B) * ix->n_rows;
  CK(ix->dbg.ensure(n));
  CK(cudaMemsetAsync(ix->dbg.p, 0xFF, n * 4, ix->stream));
  CK(cudaMemcpyAsync(ix->q_raw.p, queries, static_cast<size_t>(B) * ix->dim * 4, cudaMemcpyHostToDevice, ix->stream));
  st = run_scan(ix, ix->q_raw.p, 1, B, 16, -INFINITY, nullptr, nullptr, nullptr, nullptr, ix->dbg.p);
  if (st != RBK_OK) return st;
  std::vector<float> invq(B);
  CK(cudaMemcpyAsync(out_scores, ix->dbg.p, n * 4, cudaMemcpyDeviceToHost, ix->stream));
  CK(cudaMemcpyAsync(invq.data(), ix->q_inv_norm.p, sizeof(float) * B, cudaMemcpyDeviceToHost, ix->stream));
  CK(cudaStreamSynchronize(ix->stream));
  for (int b = 0; b < B; ++b)
    for (int64_t r = 0; r < ix->n_rows; ++r) out_scores[static_cast<size_t>(b) * ix->n_rows + r] *= invq[b];
  return RBK_OK;
}

}  // extern "C"
