// rbk_internal.h — declarations shared by the kernels and the C-ABI translation unit.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace rbk {

// ---- tiling of the fused scan (rbk_scan.cu) ----
constexpr int kBlockM = 128;      // queries per CTA (UMMA M, TMEM lanes)
constexpr int kBlockN = 256;      // corpus rows per tile (UMMA N, TMEM columns)
constexpr int kBlockK = 64;       // bf16 elements per pipeline stage (one 128-byte swizzle row)
constexpr int kStages = 4;        // smem ring depth
constexpr int kListCap = 256;     // entries per (CTA, query) candidate list
constexpr int kMaxKPrime = 128;   // candidates kept per query (k_fetch + margin)
constexpr int kScanThreads = 192; // warp0 TMA, warp1 MMA/TMEM, warps2-5 epilogue
// the CTA-pair kernel (rbk_scan2.cu) can run 8 epilogue warps: two column halves per tile, two lists per (unit, query)
constexpr int kMaxHalves = 2;
constexpr int kMaxSubBatch = 1024;  // queries per scan launch (8 query blocks)
constexpr int kMaxLeadTiles = 4;    // lockstep: max tiles a CTA may lead the slowest peer of its range (A/B on cfg3
                                    // under the power cap: 8 -> 74.2 k, 4 -> 76.4 k, 2 -> 77.4 k q/s; short kernels: 8 best by 2 %)
constexpr int kHistBins = 1024;     // per-query score histogram, cosine in [-1,1] -> bin width 1/512

// The default build ships ONE scan path per batch size (scan_kernel for B <= 128, the streamed CTA-pair kernel
// above).  -DRBK_EXPERIMENTAL additionally compiles the measured-and-rejected variants of DESIGN.md §7 (query-
// resident / hybrid / TMEM-query pair kernels, the timing probes) and the environment switches that select them.
#ifdef RBK_EXPERIMENTAL
constexpr bool kExperimental = true;
#else
constexpr bool kExperimental = false;
#endif

struct ScanParams {
  const float* inv_norm_c;  // [rows padded to kBlockN], NaN = dead / out of range
  const float* thr_init;    // [B] initial threshold, raw domain (acc * inv_norm_c); -inf = none
  const float* inv_norm_q;  // [B] 1/||bf16(q)||
  unsigned int* hist;       // [B][kHistBins] scores of all appended rows (zeroed per launch)
  int* maxbin;              // [B] highest occupied histogram bin (zeroed per launch)
  unsigned int* gthr;       // [B] best published threshold per query, f32_ordered (0 = none; zeroed per launch)
  int* progress;            // [R][QB] tiles issued by each CTA's producer (zeroed per launch)
  unsigned long long* cand; // [QB][R][kBlockM][kListCap] packed keys
  int* cand_cnt;            // [QB][R][kBlockM]
  float* dbg_scores;        // nullable: [B][n_rows] raw-domain scores (validation aid)
  int n_rows;
  int B;        // queries in this launch
  int kprime;
  int num_kb;   // k-blocks per tile = ceil(dpad / kBlockK)
  int dpad;     // padded row length (elements)
  int prefetch_tiles;  // query-resident pair kernel: L2 prefetch distance in tiles (0 = off)
  int max_lead_tiles;  // lockstep: tiles a producer may lead the slowest peer of its range
  int seed_tile;       // start-up seeding: 1 = count each thread's two best rows of its first tile, 0 = two per chunk
  int perf_probe;      // 0 = normal.  TIMING EXPERIMENTS ONLY (results are wrong): 1 = epilogue drains TMEM but does not filter
  int QB;       // query blocks
  int R;        // list units per query block (CTAs / CTA pairs that scan different tiles for the same queries)
  int RC;       // cluster kernel: corpus ranges = clusters per column (R = RC when the pairs of a cluster share the
                // corpus tile, 2 * RC when they share the query slab and alternate tiles)
  int n_tiles;  // ceil(n_rows / kBlockN)
  // A scan may be split over two concurrent launches (the cluster kernel on the SMs that can host 4-CTA clusters, the
  // pair kernel on the rest): each launch covers tiles [tile_begin, tile_begin + tile_count) with R_local ranges,
  // its units are numbered unit_base.. inside the query block's R lists, its pacing slots start at prog_base.
  int tile_begin, tile_count;
  int R_local;   // corpus ranges of THIS launch (1-CTA / pair kernels; the cluster kernel uses RC)
  int unit_base;
  int prog_base;
};

cudaError_t launch_scan(const CUtensorMap& tmap_q, const CUtensorMap& tmap_c, const ScanParams& p,
                        cudaStream_t stream);
size_t scan_smem_bytes();
// CTA-pair variants (B > 128): QB counts 256-query blocks, R pairs per block.  tmap_c has 128-row boxes:
// 64 columns / SWIZZLE_128B for the streamed kernel, 32 columns / SWIZZLE_64B for the query-resident one.
// tmap_pf: un-swizzled 128-row x 256-col boxes, used only for L2 prefetch.
cudaError_t launch_scan2(const CUtensorMap& tmap_q, const CUtensorMap& tmap_c, const CUtensorMap& tmap_pf,
                         const ScanParams& p, bool resident, int halves, cudaStream_t stream,
                         int* ring_stages_out = nullptr);
// Cluster-of-two-pairs kernel with one operand multicast (rbk_scan4.cu).  tmap_q128 / tmap_c128: 128-row boxes,
// tmap_q64 / tmap_c64: 64-row boxes (the multicast halves), all 64 columns / SWIZZLE_128B.
cudaError_t launch_scan4(const CUtensorMap& tmap_q128, const CUtensorMap& tmap_q64, const CUtensorMap& tmap_c128,
                         const CUtensorMap& tmap_c64, const ScanParams& p, bool share_c, bool smem_aligned,
                         cudaStream_t stream, int* ring_stages_out = nullptr);
int scan4_max_clusters(bool smem_aligned);   // resident 4-CTA clusters of that kernel on the current device
bool scan_smem_base_is_aligned();            // is the dynamic smem window 1024-byte aligned (7-stage ring possible)?
// CTA-pair kernel with the query operand in TMEM (rbk_scan3.cu): dpad <= 768.  tmap_c: 32-row x 64-col boxes.
cudaError_t launch_scan3(const CUtensorMap& tmap_c, const ScanParams& p, const uint16_t* q_bf16, cudaStream_t stream);
bool scan3_fits(int dpad);
int scan3_box_rows();   // corpus rows per CTA per TMA box of the TMEM-query kernel
bool scan2_resident_fits(int dpad);
// Hybrid pair kernel: res_kb resident query panels, the rest + the corpus through n_slots 16-KB ring slots.
cudaError_t launch_scan2h(const CUtensorMap& tmap_q, const CUtensorMap& tmap_c_half, const ScanParams& p, int res_kb,
                          int n_slots, cudaStream_t stream);
int scan2_resident_k();   // corpus columns per stage of the resident kernel (64 or 32)

// ---- ingest (rbk_ingest.cu) ----
// src element type: 0 = f64, 1 = f32, 2 = bf16 bits.  src is device memory, row pitch = d.
// dst_f64 (nullable): exact-source sidecar rows, pitch d.
// slot_map (nullable, bulk overwrite): dst_rows / dst_f64 are the index's row 0 and source row r lands in row
// slot_map[r]; rows whose slot is tombstoned (dead_bits) are skipped and counted in *n_dead.
cudaError_t launch_convert_rows(const void* src, int src_type, int64_t n_rows, int d, int dpad,
                                uint16_t* dst_rows, double* dst_f64, cudaStream_t stream,
                                const int64_t* slot_map = nullptr, const unsigned int* dead_bits = nullptr,
                                int* n_dead = nullptr);
// Norms of rows [first_row, first_row + n_items) of the index (or, with slot_map, of rows slot_map[i]; tombstoned
// ones skipped).  All array arguments are the index's BASE pointers.  rows_f64_base (nullable): when given,
// norm2 comes from it and the bf16-vs-f64 angle bound is max-ed into *eps_c_max (float bits in an int).  Any index:
// a row whose norm is outside the scan's window (DESIGN.md §6) max-es 3.2 into *eps_c_max.
cudaError_t launch_row_norms(const uint16_t* rows_base, const double* rows_f64_base, int64_t first_row,
                             int64_t n_items, int d, int dpad, float* inv_norm_base, double* norm2_base,
                             int* eps_c_max, cudaStream_t stream, const int64_t* slot_map = nullptr,
                             const unsigned int* dead_bits = nullptr);
cudaError_t launch_tombstone(const int64_t* dev_slots, int64_t n, int64_t n_rows, float* inv_norm,
                             unsigned int* dead_bits, int* n_killed, cudaStream_t stream);

// ---- query preparation + finalize + exhaustive fallback + shard merge (rbk_finalize.cu) ----
struct QueryBuffers {
  uint16_t* q_bf16;    // [B][dpad]
  double* q_f64;       // [B][d]
  double* q_norm2;     // [B] exact sequential sum of squares of the f64 query (reference's normA)
  float* q_inv_norm;   // [B] 1/||bf16(q * 2^e)||, e per query (approximate-score scaling of the scan's copy)
  double* q_eps;       // [B] bound on |approx - exact| cosine for this query
  float* thr_init;     // [B]
};
// src_type: 0 = f64, 1 = f32 (device pointers, row pitch d)
// eps_c (nullable): device float, corpus-side term of the error bound (rbk_ingest.cu: the quantisation angle of f64
// sidecar rows; 3.2 once a row's norm has left the scan's window).
// with_norm2: also run the sequential normA chain (only the exact-scores path, which has no finalize kernel; a
// search leaves it to finalize).  scratch (nullable): hist | maxbin | gthr | progress of the first sub-batch (Bs
// queries, n_progress pacing slots), zeroed by the kernel.
cudaError_t launch_prep_queries(const void* src, int src_type, int B, int d, int dpad, double min_score,
                                const float* eps_c, const QueryBuffers& qb, cudaStream_t stream, bool with_norm2,
                                unsigned int* scratch, int Bs, int n_progress);

// local row -> global slot.  Contiguous shards: slot_base + row.  A group that deals rows out block-cyclically over
// G devices (rbk_group.cu): device g's local row r is global slot ((r / block) * G + g) * block + r % block - still
// monotonic in r, so per-shard lists stay sorted by global slot among equal scores.
struct SlotLayout {
  int64_t base = 0;
  int32_t block = 0, G = 1, g = 0;   // block == 0: contiguous
  __host__ __device__ int64_t global(int64_t row) const {
    if (block == 0) return base + row;
    return ((row / block) * G + g) * block + row % block;
  }
};

struct FinalizeParams {
  const unsigned long long* cand;
  const int* cand_cnt;
  int QB, R, kprime, k_fetch, B, d, dpad;
  int block_m;  // queries per list block: 128 (1-CTA scan) or 256 (CTA-pair scan)
  int key_cap;  // keys staged in smem per query (set by launch_finalize)
  int q0;  // global index of the first query of this launch (sub-batch offset)
  double min_score;
  const uint16_t* rows;
  const double* rows_f64;   // nullable: exact-source sidecar (pitch d); the re-rank reads it instead of `rows`
  const double* row_norm2;
  int64_t n_rows;
  SlotLayout slot;
  QueryBuffers q;  // pointers already offset to the sub-batch
  long long* out_slots;   // [B][k_fetch]
  double* out_scores;     // [B][k_fetch]
  int* out_counts;        // [B]
  int* flags;             // [B] 1 = not provably exact -> exhaustive fallback
};
cudaError_t launch_finalize(const FinalizeParams& p, cudaStream_t stream);

struct ExactParams {
  const int* fail_list;  // [n_fail] query indices
  int n_fail;
  int d, dpad, k_fetch;
  double min_score;
  const uint16_t* rows;
  const double* rows_f64;   // nullable: exact-source sidecar
  const double* row_norm2;
  const unsigned int* dead_bits;  // tombstones
  int64_t n_rows;
  SlotLayout slot;
  const double* q_f64;
  const double* q_norm2;
  double* part_scores;   // [n_fail][n_blocks][k_fetch]
  int* part_rows;        // [n_fail][n_blocks][k_fetch]
  int* part_cnt;         // [n_fail][n_blocks]
  int n_blocks;
  long long* out_slots;
  double* out_scores;
  int* out_counts;
};
cudaError_t launch_exact_fallback(const ExactParams& p, cudaStream_t stream);

// Exact fp64 cosine of every row for B prepared queries: out [B][n_rows], NaN = tombstoned / zero row.
cudaError_t launch_exact_scores(const uint16_t* rows, const double* rows_f64, const double* row_norm2,
                                const unsigned int* dead_bits, int64_t n_rows, int d, int dpad, const double* q_f64,
                                const double* q_norm2, int B, double* out, cudaStream_t stream);

// slots/scores/counts/flags point at shard 0's arrays; shard g's arrays start g * <stride> bytes later.
// flags (nullable): per-shard exactness flags i32[B]; out_flags: i32[B+1] ([b] = OR over shards, [B] += dirty queries).
cudaError_t launch_merge_shards(int G, int B, int k_fetch, const void* slots, const void* scores, const void* counts,
                                const void* flags, size_t slots_stride, size_t scores_stride, size_t counts_stride,
                                size_t flags_stride, long long* out_slots, double* out_scores, int* out_counts,
                                int* out_flags, cudaStream_t stream);

// Bound on the fp32 tensor-core accumulation + scaling error of an approximate cosine.
inline double accumulation_eps(int d) { return (double)(d + 8) * (1.0 / 4194304.0); }  // (d+8) * 2^-22

}  // namespace rbk
