// rbk_ingest.cu — K3: corpus ingest.  Replaces VectorStore.loadEmbeddings /
// bufferToFloatArray (reference src/knowledge/store/vector-store.ts:56-88): rows arrive as
// little-endian float64 (the SQLite BLOB layout), float32 or bf16 and are stored as bf16
// rows of pitch dpad (= dim rounded up to 8 elements, zero padded) plus, per row,
//   inv_norm (fp32)  1/||row||           for the approximate scan (NaN = never matches)
//   norm2    (fp64)  sum of squares accumulated in index order, multiply-then-add — the
//                    reference's `normB` (embedder.ts:175-181) bit for bit, reused by the
//                    exact re-rank so it is not recomputed per query.
// Both kernels are HBM-bound streams: 16-byte vector loads/stores, no reuse.
#include <cuda_bf16.h>

#include "rbk_internal.h"

namespace rbk {

namespace {

__device__ __forceinline__ uint16_t f64_to_bf16_bits(double x) {
  // f64 -> f32 (RNE) -> bf16 (RNE); documented in DESIGN.md §3.
  return __bfloat16_as_ushort(__float2bfloat16_rn(__double2float_rn(x)));
}
__device__ __forceinline__ uint16_t f32_to_bf16_bits(float x) {
  return __bfloat16_as_ushort(__float2bfloat16_rn(x));
}

// One thread produces 8 consecutive output elements (one 16-byte store).
template <typename SrcT>
__global__ void __launch_bounds__(256) convert_rows_kernel(const SrcT* __restrict__ src, int64_t n_rows, int d,
                                                           int dpad, uint16_t* __restrict__ dst,
                                                           double* __restrict__ dst_f64, bool aligned,
                                                           const int64_t* __restrict__ slot_map,
                                                           const unsigned int* __restrict__ dead_bits,
                                                           int* __restrict__ n_dead) {
  // slot_map == nullptr: source row r -> destination row r of dst (an append).  slot_map != nullptr (bulk
  // overwrite): dst/dst_f64 are the index's row 0 and source row r goes to row slot_map[r]; tombstoned slots are
  // skipped and counted (once per row) in *n_dead.
  const int groups = dpad >> 3;
  const int64_t total = n_rows * groups;
  for (int64_t g = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; g < total;
       g += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t srow = g / groups;
    const int c0 = static_cast<int>(g - srow * groups) << 3;
    const SrcT* s = src + srow * d + c0;
    int64_t row = srow;
    if (slot_map != nullptr) {
      row = slot_map[srow];
      if ((dead_bits[row >> 5] >> (row & 31)) & 1u) {
        if (c0 == 0) atomicAdd(n_dead, 1);
        continue;
      }
    }
    uint16_t o[8];
    if (c0 >= d) {
      // pad columns (the row pitch is a whole number of 64-element k-blocks): zeros, and nothing to read
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = 0;
    } else if (aligned) {
      if constexpr (sizeof(SrcT) == 8) {
        const double2* s2 = reinterpret_cast<const double2*>(s);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double2 v = __ldg(s2 + j);
          o[2 * j] = f64_to_bf16_bits(v.x);
          o[2 * j + 1] = f64_to_bf16_bits(v.y);
        }
      } else if constexpr (sizeof(SrcT) == 4) {
        const float4* s4 = reinterpret_cast<const float4*>(s);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const float4 v = __ldg(s4 + j);
          o[4 * j] = f32_to_bf16_bits(v.x);
          o[4 * j + 1] = f32_to_bf16_bits(v.y);
          o[4 * j + 2] = f32_to_bf16_bits(v.z);
          o[4 * j + 3] = f32_to_bf16_bits(v.w);
        }
      } else {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(s));
        *reinterpret_cast<uint4*>(o) = v;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        uint16_t b = 0;
        if (c0 + j < d) {
          if constexpr (sizeof(SrcT) == 8) b = f64_to_bf16_bits(static_cast<double>(s[j]));
          else if constexpr (sizeof(SrcT) == 4) b = f32_to_bf16_bits(static_cast<float>(s[j]));
          else b = static_cast<uint16_t>(s[j]);
        }
        o[j] = b;
      }
    }
    if (dst_f64 != nullptr) {   // exact-source sidecar: the original values, widened to f64 (pitch d)
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (c0 + j < d) {
          double x;
          if constexpr (sizeof(SrcT) == 8) x = static_cast<double>(s[j]);
          else if constexpr (sizeof(SrcT) == 4) x = static_cast<double>(static_cast<float>(s[j]));
          else x = static_cast<double>(__uint_as_float(static_cast<uint32_t>(s[j]) << 16));
          dst_f64[row * d + c0 + j] = x;
        }
      }
    }
    uint4 out;
    out.x = o[0] | (static_cast<uint32_t>(o[1]) << 16);
    out.y = o[2] | (static_cast<uint32_t>(o[3]) << 16);
    out.z = o[4] | (static_cast<uint32_t>(o[5]) << 16);
    out.w = o[6] | (static_cast<uint32_t>(o[7]) << 16);
    *reinterpret_cast<uint4*>(dst + row * dpad + c0) = out;
  }
}

__device__ __forceinline__ double bf16_bits_to_f64(uint32_t h) {
  return static_cast<double>(__uint_as_float(h << 16));
}

// ---- K3b: per-row norms.  The accumulation ORDER is part of the parity contract (norm2 must be the reference's
// normB, embedder.ts:180: index order, multiply then add), so each row is one sequential fp64 chain owned by one
// thread - but the chain must not wait on memory, and the loads must be coalesced.  A block of kNormRows threads
// (= rows) therefore stages a K-chunk of all its rows in shared memory with 16-byte loads in which consecutive
// lanes read consecutive 16-byte pieces of the SAME row (full 128-byte lines, every byte of the chunk requested
// exactly once, many loads in flight per thread), and only then does every thread walk its own row's chunk out
// of shared memory (row pitch = an odd number of 16-byte units: conflict-free).  Several blocks per SM overlap
// one block's staging with the others' arithmetic.  (Round 1 had one thread read its row straight from global
// memory: adjacent threads 2*dpad bytes apart, one dependent 16-byte load per 8 elements of the chain.)
// slot_map == nullptr: item i is row first_row + i.  slot_map != nullptr (bulk overwrite): item i is row
// slot_map[i]; items whose slot is tombstoned are skipped.
constexpr int kNormRows = 128;          // rows (= threads) per block
constexpr int kNormChunk = 128;         // bf16 elements per staged chunk (256 B per row)
constexpr int kNormPitch16 = kNormChunk / 8 + 1;   // 17 x 16 B per row in smem: odd -> conflict-free walks
constexpr double kNormLo = 0x1p-60, kNormHi = 0x1p100;   // the scan's row-norm window

__global__ void __launch_bounds__(kNormRows) row_norms_kernel(const uint16_t* __restrict__ rows_base,
                                                              const double* __restrict__ rows_f64_base,
                                                              const int64_t* __restrict__ slot_map,
                                                              const unsigned int* __restrict__ dead_bits,
                                                              int64_t first_row, int64_t n_items, int d, int dpad,
                                                              float* __restrict__ inv_norm_base,
                                                              double* __restrict__ norm2_base,
                                                              int* __restrict__ eps_c_max) {
  __shared__ uint4 s_chunk[kNormRows * kNormPitch16];
  __shared__ long long s_row[kNormRows];
  const int tid = threadIdx.x;
  const int64_t item0 = static_cast<int64_t>(blockIdx.x) * kNormRows;
  {
    const int64_t item = item0 + tid;
    long long row = -1;
    if (item < n_items) {
      row = slot_map ? slot_map[item] : first_row + item;
      if (slot_map && ((dead_bits[row >> 5] >> (row & 31)) & 1u)) row = -1;   // tombstoned slots stay dead
    }
    s_row[tid] = row;
  }
  __syncthreads();
  const long long my_row = s_row[tid];
  double acc = 0.0;
  const int n16 = dpad >> 3;                         // 16-byte pieces per row
  constexpr int kPieces = kNormChunk / 8;            // 16-byte pieces per row and chunk; = pieces per thread and chunk
  // piece index i of a chunk -> (row i / len16, unit i % len16): consecutive lanes = consecutive units of a row;
  // all of a thread's 16 loads are in flight before the first is stored.  (Tried and measured on B200, 4M x 768:
  // keeping the NEXT chunk's pieces in registers while this one is walked - no change, the kernel is not waiting on
  // memory; forming x*x with one fp32 multiply and widening it to binary64 with integer shifts instead of two F2F
  // conversions and a DMUL - 50 % SLOWER, the per-element range check costs more issue slots than the fp64 pipe
  // saves.  The sequential fp64 chain per row, which the parity contract imposes, is what bounds this kernel.)
  uint4 v[kPieces];
  auto load_chunk = [&](int c0) {
    const int len16 = n16 - c0 < kPieces ? n16 - c0 : kPieces;
#pragma unroll
    for (int u = 0; u < kPieces; ++u) {
      const int i = tid + u * kNormRows;
      v[u] = make_uint4(0u, 0u, 0u, 0u);
      if (i < kNormRows * len16) {
        const int rr = i / len16, un = i - rr * len16;
        const long long row = s_row[rr];
        if (row >= 0) v[u] = __ldg(reinterpret_cast<const uint4*>(rows_base + row * dpad) + c0 + un);
      }
    }
  };
  for (int c0 = 0; c0 < n16; c0 += kPieces) {
    const int len16 = n16 - c0 < kPieces ? n16 - c0 : kPieces;
    load_chunk(c0);
#pragma unroll
    for (int u = 0; u < kPieces; ++u) {
      const int i = tid + u * kNormRows;
      if (i < kNormRows * len16) {
        const int rr = i / len16, un = i - rr * len16;
        s_chunk[rr * kNormPitch16 + un] = v[u];
      }
    }
    __syncthreads();
    if (my_row >= 0) {
      const uint4* mine = s_chunk + tid * kNormPitch16;
      for (int g = 0; g < len16; ++g) {   // pad columns are zero: adding 0*0 is exact
        const uint4 w4 = mine[g];
        const uint32_t w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double lo = bf16_bits_to_f64(w[j] & 0xFFFFu);
          const double hi = bf16_bits_to_f64(w[j] >> 16);
          acc = __dadd_rn(acc, __dmul_rn(lo, lo));
          acc = __dadd_rn(acc, __dmul_rn(hi, hi));
        }
      }
    }
    __syncthreads();
  }
  if (my_row < 0) return;
  const bool ok = acc > 0.0 && acc < INFINITY;
  inv_norm_base[my_row] = ok ? static_cast<float>(1.0 / sqrt(acc)) : __uint_as_float(0x7FC00000u);
  if (rows_f64_base == nullptr) norm2_base[my_row] = acc;
  // The scan's error bound holds for ||row|| in [kNormLo, kNormHi] (DESIGN.md §6): outside it the fp32 accumulator
  // may overflow or lose products to underflow.  Such a row voids the bound for the whole index (3.2 > any cosine
  // distance), so every proof fails and the exhaustive fp64 kernel answers.
  if (ok && !(acc >= kNormLo * kNormLo && acc <= kNormHi * kNormHi)) atomicMax(eps_c_max, __float_as_int(3.2f));
}

// Exact-source sidecar indexes (RBK_INDEX_KEEP_F64): norm2 comes from the f64 row (the reference's normB for
// the values it really stores), again as one sequential chain per row fed from shared memory, and the angle
// between the f64 row and its bf16 rounding - an upper bound on how far the scan's approximate cosine of this
// row can be from its true cosine, on top of the other error terms - is folded into *eps_c_max.
constexpr int kNorm64Chunk = 32;        // doubles per staged chunk (256 B per row)
constexpr int kNorm64Pitch = kNorm64Chunk + 1;

__global__ void __launch_bounds__(kNormRows) row_norms_f64_kernel(const uint16_t* __restrict__ rows_base,
                                                                  const double* __restrict__ rows_f64_base,
                                                                  const int64_t* __restrict__ slot_map,
                                                                  const unsigned int* __restrict__ dead_bits,
                                                                  int64_t first_row, int64_t n_items, int d, int dpad,
                                                                  double* __restrict__ norm2_base,
                                                                  int* __restrict__ eps_c_max) {
  __shared__ double s_x[kNormRows * kNorm64Pitch];
  __shared__ uint16_t s_b[kNormRows * (kNorm64Chunk + 2)];
  __shared__ long long s_row[kNormRows];
  const int tid = threadIdx.x;
  const int64_t item0 = static_cast<int64_t>(blockIdx.x) * kNormRows;
  {
    const int64_t item = item0 + tid;
    long long row = -1;
    if (item < n_items) {
      row = slot_map ? slot_map[item] : first_row + item;
      if (slot_map && ((dead_bits[row >> 5] >> (row & 31)) & 1u)) row = -1;
    }
    s_row[tid] = row;
  }
  __syncthreads();
  const long long my_row = s_row[tid];
  double n2 = 0.0, diff2 = 0.0;
  for (int c0 = 0; c0 < d; c0 += kNorm64Chunk) {
    const int len = d - c0 < kNorm64Chunk ? d - c0 : kNorm64Chunk;
    for (int i = tid; i < kNormRows * len; i += kNormRows) {   // consecutive lanes = consecutive elements of a row
      const int rr = i / len, e = i - rr * len;
      const long long row = s_row[rr];
      double x = 0.0;
      uint16_t bq = 0;
      if (row >= 0) {
        x = __ldg(rows_f64_base + row * d + c0 + e);
        bq = __ldg(rows_base + row * dpad + c0 + e);
      }
      s_x[rr * kNorm64Pitch + e] = x;
      s_b[rr * (kNorm64Chunk + 2) + e] = bq;
    }
    __syncthreads();
    if (my_row >= 0) {
      const double* mine = s_x + tid * kNorm64Pitch;
      const uint16_t* mb = s_b + tid * (kNorm64Chunk + 2);
      for (int i = 0; i < len; ++i) {
        const double v = mine[i];
        n2 = __dadd_rn(n2, __dmul_rn(v, v));   // the reference's normB for the f64 row
        const double e = v - bf16_bits_to_f64(mb[i]);
        diff2 += e * e;
      }
    }
    __syncthreads();
  }
  if (my_row < 0) return;
  norm2_base[my_row] = n2;
  float eps = 0.f;
  if (diff2 > 0.0) {
    const double ratio = (n2 > 0.0 && n2 < INFINITY) ? sqrt(diff2 / n2) * (1.0 + 1e-9) : 2.0;
    eps = static_cast<float>((ratio < 1.0 ? asin(ratio) : 3.2) * (1.0 + 1e-6));
    eps = nextafterf(eps, INFINITY);
  }
  if (eps > 0.f) atomicMax(eps_c_max, __float_as_int(eps));   // non-negative floats order like ints
}

__global__ void tombstone_kernel(const int64_t* __restrict__ slots, int64_t n, int64_t n_rows,
                                 float* __restrict__ inv_norm, unsigned int* __restrict__ dead_bits,
                                 int* __restrict__ n_killed) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const int64_t s = slots[i];
  if (s < 0 || s >= n_rows) return;
  const unsigned int bit = 1u << (s & 31);
  const unsigned int old = atomicOr(dead_bits + (s >> 5), bit);
  if (!(old & bit)) {
    inv_norm[s] = __uint_as_float(0x7FC00000u);
    atomicAdd(n_killed, 1);
  }
}

int grid_for(int64_t items, int threads, int max_blocks) {
  int64_t b = (items + threads - 1) / threads;
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return static_cast<int>(b);
}

}  // namespace

cudaError_t launch_convert_rows(const void* src, int src_type, int64_t n_rows, int d, int dpad, uint16_t* dst_rows,
                                double* dst_f64, cudaStream_t stream, const int64_t* slot_map,
                                const unsigned int* dead_bits, int* n_dead) {
  if (n_rows <= 0) return cudaSuccess;
  const int64_t total = n_rows * (dpad >> 3);
  const int grid = grid_for(total, 256, 148 * 16);
  // vector loads need d % 8 == 0 (every 8-group starts 16-byte aligned) and an aligned base
  const bool aligned = (d & 7) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
  if (src_type == 0)
    convert_rows_kernel<double><<<grid, 256, 0, stream>>>(static_cast<const double*>(src), n_rows, d, dpad, dst_rows,
                                                          dst_f64, aligned, slot_map, dead_bits, n_dead);
  else if (src_type == 1)
    convert_rows_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(src), n_rows, d, dpad, dst_rows,
                                                         dst_f64, aligned, slot_map, dead_bits, n_dead);
  else
    convert_rows_kernel<uint16_t><<<grid, 256, 0, stream>>>(static_cast<const uint16_t*>(src), n_rows, d, dpad,
                                                            dst_rows, dst_f64, aligned, slot_map, dead_bits, n_dead);
  return cudaGetLastError();
}

cudaError_t launch_row_norms(const uint16_t* rows_base, const double* rows_f64_base, int64_t first_row, int64_t n_items,
                             int d, int dpad, float* inv_norm_base, double* norm2_base, int* eps_c_max,
                             cudaStream_t stream, const int64_t* slot_map, const unsigned int* dead_bits) {
  if (n_items <= 0) return cudaSuccess;
  const unsigned blocks = static_cast<unsigned>((n_items + kNormRows - 1) / kNormRows);
  row_norms_kernel<<<blocks, kNormRows, 0, stream>>>(rows_base, rows_f64_base, slot_map, dead_bits, first_row, n_items,
                                                     d, dpad, inv_norm_base, norm2_base, eps_c_max);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || rows_f64_base == nullptr) return e;
  row_norms_f64_kernel<<<blocks, kNormRows, 0, stream>>>(rows_base, rows_f64_base, slot_map, dead_bits, first_row,
                                                         n_items, d, dpad, norm2_base, eps_c_max);
  return cudaGetLastError();
}

cudaError_t launch_tombstone(const int64_t* dev_slots, int64_t n, int64_t n_rows, float* inv_norm,
                             unsigned int* dead_bits, int* n_killed, cudaStream_t stream) {
  if (n <= 0) return cudaSuccess;
  tombstone_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(dev_slots, n, n_rows, inv_norm,
                                                                              dead_bits, n_killed);
  return cudaGetLastError();
}

}  // namespace rbk
