// Epilogues over the count matrix that every reference notebook runs on the host right after
// sampling (SURVEY.md 8f rows 3 and 4): library-size normalisation and log transform
// (compare_axolotl.ipynb cell 14: `(X.T / scalings).T`, minimal_example.ipynb cell 6:
// `np.log(X + 1)`) and compaction of the (N, G) matrix into CSR for the on-disk formats
// single-cell tools read (tree_utils.py:59-173 writes dense text only).
//
// Both are pure streaming passes (HBM-bound): one 128-bit load per gene quad, rows walked by
// warps so that every warp touches 512 contiguous bytes.
#include <algorithm>
#include "pst_common.cuh"

namespace pst {
namespace {

// ---------------------------------------------------------------------------------------------
// out[i][g] = f(X[i][g], scaling[i]);  mode 0: X/s   1: log(X/s + 1)   2: log(X + 1)
// ---------------------------------------------------------------------------------------------
// grid.x walks the gene quads of a row, grid.y strides over rows: no 64-bit division per item
template <int MODE, bool VEC>
__global__ void __launch_bounds__(256)
transform_kernel(const int32_t *__restrict__ X, int64_t n, int64_t G, int64_t ldx,
                 const float *__restrict__ scaling, float *__restrict__ out, int64_t ldo) {
  const int64_t Q = (G + 3) / 4;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g0 = q * 4;
    for (int64_t row = blockIdx.y; row < n; row += gridDim.y) {
      // one correctly rounded reciprocal per item, then multiplies: within 1.5 ulp of x / s
      const float inv = (MODE == PST_TRANSFORM_LOG1P) ? 1.0f : 1.0f / __ldg(scaling + row);
      const int32_t *src = X + row * ldx + g0;
      float *dst = out + row * ldo + g0;
      if (VEC) {
        const int4 v = __ldcs(reinterpret_cast<const int4 *>(src));
        float4 o = make_float4((float)v.x * inv, (float)v.y * inv, (float)v.z * inv, (float)v.w * inv);
        if (MODE != PST_TRANSFORM_NORMALIZE)
          o = make_float4(log1pf(o.x), log1pf(o.y), log1pf(o.z), log1pf(o.w));
        __stcs(reinterpret_cast<float4 *>(dst), o);
      } else {
        for (int j = 0; j < 4 && g0 + j < G; ++j) {
          const float o = (float)src[j] * inv;
          dst[j] = (MODE != PST_TRANSFORM_NORMALIZE) ? log1pf(o) : o;
        }
      }
    }
  }
}

// one gene quad of row `src` (zeros past G)
template <bool VEC>
__device__ __forceinline__ int4 load_quad(const int32_t *__restrict__ src, int64_t q, int64_t Q, int64_t G) {
  int4 v = make_int4(0, 0, 0, 0);
  if (q < Q) {
    if (VEC) {
      v = __ldcs(reinterpret_cast<const int4 *>(src + q * 4));
    } else {
      const int64_t g = q * 4;
      v.x = src[g];
      if (g + 1 < G) v.y = src[g + 1];
      if (g + 2 < G) v.z = src[g + 2];
      if (g + 3 < G) v.w = src[g + 3];
    }
  }
  return v;
}

// ---------------------------------------------------------------------------------------------
// CSR fill: one warp per row, 128 genes per step; a lane owns a gene quad, so column order inside
// the row is preserved by an exclusive warp prefix of the lanes' nonzero counts.
// Nonzero number p of the matrix (indptr[0] <= p < indptr[n]) goes to indices/data[p - base]: a
// chunk of rows fills its own window of the streams.  IDX / VAL are the stored widths; SAT: values
// are stored as min(v, 65535) and every v >= 65535 is also listed exactly as (p, v) in the overflow
// list (slot from atomicAdd(ovf_count), written when below ovf_cap).
// ---------------------------------------------------------------------------------------------
constexpr int32_t kCsrSat = 65535;

template <typename IDX, typename VAL, bool SAT, bool VEC>
__global__ void __launch_bounds__(256)
csr_fill_kernel(const int32_t *__restrict__ X, int64_t n, int64_t G, int64_t ldx,
                const int64_t *__restrict__ indptr, int64_t base, IDX *__restrict__ indices,
                VAL *__restrict__ data, int64_t *__restrict__ ovf_pos, int32_t *__restrict__ ovf_value,
                int64_t ovf_cap, unsigned long long *__restrict__ ovf_count, uint32_t *__restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t Q = (G + 3) / 4;
  for (int64_t row = warp0; row < n; row += n_warps) {
    int64_t pos = indptr[row];
    const int64_t end = indptr[row + 1];
    const int32_t *src = X + row * ldx;
#pragma unroll 4
    for (int64_t q0 = 0; q0 < Q; q0 += 32) {
      const int64_t q = q0 + lane;
      const int4 v = load_quad<VEC>(src, q, Q, G);
      // exclusive prefix of the lanes' nonzero counts (0..4) from three ballots of the count's bits
      const int c = (v.x != 0) + (v.y != 0) + (v.z != 0) + (v.w != 0);
      const unsigned b0 = __ballot_sync(0xffffffffu, c & 1), b1 = __ballot_sync(0xffffffffu, c & 2),
                     b2 = __ballot_sync(0xffffffffu, c & 4);
      const int excl = __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt);
      const int total = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
      int64_t w = pos + excl;
      if (pos + total <= end) {                   // indptr is consistent with the matrix
        const int32_t g = (int32_t)(q * 4);
        const int32_t vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (vv[j] != 0) {
            indices[w - base] = (IDX)(g + j);
            if (SAT && vv[j] >= kCsrSat) {        // rare: one atomic per listed count
              const unsigned long long slot = atomicAdd(ovf_count, 1ull);
              if ((int64_t)slot < ovf_cap) { ovf_pos[slot] = w; ovf_value[slot] = vv[j]; }
              data[w - base] = (VAL)kCsrSat;
            } else {
              data[w - base] = (VAL)vv[j];
            }
            ++w;
          }
        }
      }
      pos += total;
    }
    if (lane == 0 && pos != end) atomicOr(flags, (uint32_t)PST_FLAG_ROW);   // indptr does not match X
  }
}

// ---------------------------------------------------------------------------------------------
// Row sizes of the CSR form: row_nnz[i] = nonzeros of row i; *sat_count += elements >= 65535.  One
// warp per row, four 128-bit streaming loads in flight per lane; a lane keeps its own counts and the
// warp sums them once per row (one REDUX instead of ballots per step: only the total is needed here),
// the saturated elements once per warp with a single atomic.
// ---------------------------------------------------------------------------------------------
template <bool VEC>
__global__ void __launch_bounds__(256)
csr_row_count_kernel(const int32_t *__restrict__ X, int64_t n, int64_t G, int64_t ldx,
                     int32_t *__restrict__ row_nnz, unsigned long long *__restrict__ sat_count) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t Q = (G + 3) / 4;
  unsigned sat = 0;
  for (int64_t row = warp0; row < n; row += n_warps) {
    const int32_t *src = X + row * ldx;
    unsigned c = 0;
    for (int64_t q0 = 0; q0 < Q; q0 += 128) {
      int4 v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = load_quad<VEC>(src, q0 + 32 * j + lane, Q, G);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        c += (v[j].x != 0) + (v[j].y != 0) + (v[j].z != 0) + (v[j].w != 0);
        sat += (v[j].x >= kCsrSat) + (v[j].y >= kCsrSat) + (v[j].z >= kCsrSat) + (v[j].w >= kCsrSat);
      }
    }
    c = __reduce_add_sync(0xffffffffu, c);
    if (lane == 0) row_nnz[row] = (int32_t)c;
  }
  sat = __reduce_add_sync(0xffffffffu, sat);
  if (lane == 0 && sat != 0 && sat_count != nullptr) atomicAdd(sat_count, (unsigned long long)sat);
}

// ---------------------------------------------------------------------------------------------
// indptr[0] = 0, indptr[i + 1] = row_nnz[0] + ... + row_nnz[i]: one CTA walks the rows in tiles of
// 1024 x 8; each thread sums its 8 rows, the block scans the thread sums (warp shuffles + one word per
// warp in shared memory) and carries the tile total into the next tile.  n is one shard's cells (a
// few million at most: a few hundred microseconds), so no grid-wide scan is needed.
// ---------------------------------------------------------------------------------------------
constexpr int kScanThreads = 1024, kScanItems = 8;

__global__ void __launch_bounds__(kScanThreads)
csr_row_offsets_kernel(const int32_t *__restrict__ row_nnz, int64_t n, int64_t *__restrict__ indptr) {
  __shared__ long long warp_sum[kScanThreads / 32];
  __shared__ long long carry_s;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  long long carry = 0;
  if (t == 0) indptr[0] = 0;
  for (int64_t tile = 0; tile < n; tile += (int64_t)kScanThreads * kScanItems) {
    const int64_t i0 = tile + (int64_t)t * kScanItems;
    int32_t v[kScanItems];
    long long s = 0;
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) {
      v[j] = (i0 + j < n) ? row_nnz[i0 + j] : 0;
      s += v[j];
    }
    long long incl = s;                                         // inclusive scan of the thread sums
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const long long o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) warp_sum[wid] = incl;
    __syncthreads();
    if (wid == 0) {
      long long ws = warp_sum[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const long long o = __shfl_up_sync(0xffffffffu, ws, d);
        if (lane >= d) ws += o;
      }
      warp_sum[lane] = ws;                                      // inclusive over warps
      if (lane == 31) carry_s = carry + ws;
    }
    __syncthreads();
    long long run = carry + (wid ? warp_sum[wid - 1] : 0) + incl - s;
#pragma unroll
    for (int j = 0; j < kScanItems; ++j) {
      run += v[j];
      if (i0 + j < n) indptr[i0 + j + 1] = run;
    }
    carry = carry_s;
    __syncthreads();                                            // warp_sum / carry_s are rewritten next tile
  }
}

// ---------------------------------------------------------------------------------------------
// narrow transfer formats: out = min(X, SAT) as uint8 (SAT = 255) or uint16 (SAT = 65535); every
// element that reads SAT also has an entry (flat index, exact value) in the overflow list, so the
// int32 matrix can be rebuilt exactly
// ---------------------------------------------------------------------------------------------
template <typename OUT, bool VEC>
__global__ void __launch_bounds__(256)
narrow_kernel(const int32_t *__restrict__ X, int64_t n, int64_t G, int64_t ldx, OUT *__restrict__ out, int64_t ldo,
              int64_t row0, int64_t *__restrict__ ovf_index, int32_t *__restrict__ ovf_value, int64_t ovf_cap,
              unsigned long long *__restrict__ ovf_count) {
  constexpr int SAT = (sizeof(OUT) == 1) ? 255 : 65535;
  const int64_t Q = (G + 3) / 4;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < Q; q += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g0 = q * 4;
    for (int64_t row = blockIdx.y; row < n; row += gridDim.y) {
      const int32_t *src = X + row * ldx + g0;
      OUT *dst = out + row * ldo + g0;
      int v[4] = {0, 0, 0, 0};
      if (VEC) {
        const int4 w = __ldcs(reinterpret_cast<const int4 *>(src));
        v[0] = w.x; v[1] = w.y; v[2] = w.z; v[3] = w.w;
      } else {
        for (int j = 0; j < 4 && g0 + j < G; ++j) v[j] = src[j];
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (v[j] >= SAT && g0 + j < G) {                              // rare: one atomic per listed count
          const unsigned long long slot = atomicAdd(ovf_count, 1ull);
          if ((int64_t)slot < ovf_cap) { ovf_index[slot] = (row0 + row) * G + g0 + j; ovf_value[slot] = v[j]; }
          v[j] = SAT;
        }
      }
      if (VEC) {
        if (sizeof(OUT) == 1) {
          __stcs(reinterpret_cast<unsigned *>(dst),
                 (unsigned)v[0] | ((unsigned)v[1] << 8) | ((unsigned)v[2] << 16) | ((unsigned)v[3] << 24));
        } else {
          __stcs(reinterpret_cast<uint2 *>(dst), make_uint2((unsigned)v[0] | ((unsigned)v[1] << 16),
                                                            (unsigned)v[2] | ((unsigned)v[3] << 16)));
        }
      } else {
        for (int j = 0; j < 4 && g0 + j < G; ++j) dst[j] = (OUT)v[j];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// The indptr member of a streamed CSR file: out[i] = *running + indptr[i + 1] (i < n) in the index dtype,
// then *running += indptr[n].  indptr is a chunk's local row pointer (indptr[0] = 0), so the chunks'
// outputs concatenate, after the file's leading 0, to the whole matrix's row pointer.  One CTA: the
// running total is read before and written after every thread's stores.
// ---------------------------------------------------------------------------------------------
template <typename OUT>
__global__ void __launch_bounds__(1024)
csr_indptr_kernel(const int64_t *__restrict__ indptr, int64_t n, int64_t *__restrict__ running, OUT *__restrict__ out) {
  const int64_t base = *running;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) out[i] = (OUT)(base + indptr[i + 1]);
  __syncthreads();
  if (threadIdx.x == 0) *running = base + indptr[n];
}

// ---------------------------------------------------------------------------------------------
// Text of a chunk of rows, one formatter per on-disk text format (the Text policies below).  Row i of the
// chunk is cell number Text::cell(first, i) of the file.  Text::row_bytes gives each row's text length,
// pst_csr_row_offsets scans them into the chunk's text pointer and text_format_kernel writes the text.  Both
// walk a row with one warp, a lane owning a gene quad, like the CSR kernels above.
// ---------------------------------------------------------------------------------------------
constexpr int kTextWarps = 4;                          // warps per block of text_format_kernel

__device__ __forceinline__ int dec_digits32(uint32_t v) {
  return 1 + (v >= 10u) + (v >= 100u) + (v >= 1000u) + (v >= 10000u) + (v >= 100000u) + (v >= 1000000u) +
         (v >= 10000000u) + (v >= 100000000u) + (v >= 1000000000u);
}

__device__ __forceinline__ int dec_digits64(uint64_t v) {     // once per row
  int d = 1;
  for (; v >= 10u; v /= 10u) ++d;
  return d;
}

// the d decimal digits of v at p, two at a time from the table "00" ... "99"
template <typename U>
__device__ __forceinline__ void put_dec(char *p, U v, int d, const char *__restrict__ pairs) {
  char *e = p + d;
  while (v >= 100u) {
    const U q = v / 100u;
    const unsigned r = (unsigned)(v - q * 100u);
    e -= 2;
    e[0] = pairs[2 * r];
    e[1] = pairs[2 * r + 1];
    v = q;
  }
  if (v >= 10u) {
    e[-2] = pairs[2 * (unsigned)v];
    e[-1] = pairs[2 * (unsigned)v + 1];
  } else {
    e[-1] = (char)('0' + (unsigned)v);
  }
}

// Matrix Market text (the 10x `matrix.mtx.gz`, genes x cells): cell first + i + 1, and each nonzero
// X[i][g] = v is the line "<g+1> <cell> <v>\n", genes ascending; a row without nonzeros has no text.  The
// cell field is put once per row into the warp's `field` and copied into each line.
struct MtxText {
  static constexpr int kGene = 42;                     // longest line: 10 + 19 + 10 digits, 3 separators
  static constexpr int kLabel = 0;                     // staging bytes of a row before its first gene
  __device__ static uint64_t cell(int64_t first, int64_t row) { return (uint64_t)(first + row + 1); }
  // the text of gene g1 - 1 (in: g1 <= G) with value v, cell field of cl digits
  __device__ static int gene(int32_t v, uint32_t g1, bool, int cl) {
    return v != 0 ? dec_digits32(g1) + cl + dec_digits32((uint32_t)v) + 3 : 0;
  }
  __device__ static int other(int) { return 0; }       // bytes of a row outside its genes' text
  __device__ static int label(char *, char *field, uint64_t cell, int cl, const char *pairs) {
    put_dec(field, cell, cl, pairs);
    return 0;
  }
  __device__ static void put(char *p, int32_t v, uint32_t g1, int cl, const char *field, const char *pairs) {
    const int dg = dec_digits32(g1);
    put_dec(p, g1, dg, pairs);
    p[dg] = ' ';
    p += dg + 1;
    for (int c = 0; c < cl; ++c) p[c] = field[c];
    p[cl] = ' ';
    p += cl + 1;
    const int dv = dec_digits32((uint32_t)v);
    put_dec(p, (uint32_t)v, dv, pairs);
    p[dv] = '\n';
  }
  __device__ static int end(char *) { return 0; }
};

// Dense tab-separated text (the reference's `_simulation.txt`, tree_utils.save_matrices): the row of cell
// first + i is "cell_<first+i>", then "\t<v>" for every gene including zeros, then "\n".
struct TsvText {
  static constexpr int kGene = 11;                     // a tab and up to 10 digits
  static constexpr int kLabel = 5 + 20;                // "cell_" and up to 20 digits
  __device__ static uint64_t cell(int64_t first, int64_t row) { return (uint64_t)(first + row); }
  __device__ static int gene(int32_t v, uint32_t, bool in, int) { return in ? 1 + dec_digits32((uint32_t)v) : 0; }
  __device__ static int other(int cl) { return 5 + cl + 1; }
  __device__ static int label(char *s, char *, uint64_t cell, int cl, const char *pairs) {
    s[0] = 'c'; s[1] = 'e'; s[2] = 'l'; s[3] = 'l'; s[4] = '_';
    put_dec(s + 5, cell, cl, pairs);
    return 5 + cl;
  }
  __device__ static void put(char *p, int32_t v, uint32_t, int, const char *, const char *pairs) {
    p[0] = '\t';
    put_dec(p + 1, (uint32_t)v, dec_digits32((uint32_t)v), pairs);
  }
  __device__ static int end(char *s) { *s = '\n'; return 1; }
};

// the staging of each warp: a partial 16-byte piece carried over, a row's label and the text of 128 genes
template <class Text>
__host__ __device__ constexpr int text_stage() { return (16 + Text::kLabel + 128 * Text::kGene + 15) / 16 * 16; }

// row_bytes[i] = Text::other(digits(cell)) + sum over the row's genes of Text::gene: csr_row_count_kernel's walk
// (four 128-bit streaming loads in flight per lane, one REDUX per row)
template <class Text, bool VEC>
__global__ void __launch_bounds__(256)
text_row_bytes_kernel(const int32_t *__restrict__ X, int64_t n, int64_t G, int64_t ldx, int64_t first,
                      int32_t *__restrict__ row_bytes) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t Q = (G + 3) / 4;
  for (int64_t row = warp0; row < n; row += n_warps) {
    const int32_t *src = X + row * ldx;
    const int cl = dec_digits64(Text::cell(first, row));
    unsigned b = 0;
    for (int64_t q0 = 0; q0 < Q; q0 += 128) {
      int4 v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = load_quad<VEC>(src, q0 + 32 * j + lane, Q, G);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t g0 = (q0 + 32 * j + lane) * 4;
        const int32_t vv[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) b += (unsigned)Text::gene(vv[k], (uint32_t)g0 + k + 1u, g0 + k < G, cl);
      }
    }
    b = __reduce_add_sync(0xffffffffu, b);
    if (lane == 0) row_bytes[row] = (int32_t)(b + (unsigned)Text::other(cl));
  }
}

// The text of row i at out + text_ptr[i].  Lane 0 puts the row's label into the warp's shared staging; then per
// tile of 128 genes a lane writes its genes' text into the staging at a warp-exclusive scan of their lengths,
// and the warp stores the staging's whole 16-byte pieces with 128-bit stores (512 contiguous bytes per
// instruction) and carries the last partial piece to the next tile.  A row's first and last pieces are shared
// with its neighbours' text: their bytes are stored one by one, only the row's own.  Writes nothing when
// text_ptr[n] > cap.
template <class Text, bool VEC>
__global__ void __launch_bounds__(kTextWarps * 32, 8)   // 8 blocks per SM: at most 64 registers, no spill
text_format_kernel(const int32_t *__restrict__ X, int64_t n, int64_t G, int64_t ldx, int64_t first,
                   const int64_t *__restrict__ text_ptr, int64_t cap, char *__restrict__ out) {
  __shared__ char pairs[200];
  __shared__ __align__(16) char stage[kTextWarps][text_stage<Text>()];
  __shared__ char cell_field[kTextWarps][20];
  if (text_ptr[n] > cap) return;                               // the same for every thread of the grid
  for (int t = threadIdx.x; t < 100; t += blockDim.x) {
    pairs[2 * t] = (char)('0' + t / 10);
    pairs[2 * t + 1] = (char)('0' + t % 10);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  char *s = stage[wid];
  char *cf = cell_field[wid];
  const int64_t Q = (G + 3) / 4;
  for (int64_t row = (int64_t)blockIdx.x * kTextWarps + wid; row < n; row += (int64_t)gridDim.x * kTextWarps) {
    const int64_t pos = text_ptr[row];
    if (pos == text_ptr[row + 1]) continue;                    // no text
    const uint64_t cell = Text::cell(first, row);
    const int cl = dec_digits64(cell);
    int64_t base = pos & ~(int64_t)15;                         // staging byte 0 belongs at out + base
    int head = (int)(pos & 15);                                // bytes before it that are not this row's
    int fill = head + (lane == 0 ? Text::label(s + head, cf, cell, cl, pairs) : 0);   // once per row
    fill = __shfl_sync(0xffffffffu, fill, 0);
    __syncwarp();
    const int32_t *src = X + row * ldx;
    for (int64_t q0 = 0; q0 < Q; q0 += 32) {
      const int64_t q = q0 + lane;
      const int4 v = load_quad<VEC>(src, q, Q, G);
      const int32_t vv[4] = {v.x, v.y, v.z, v.w};
      const uint32_t g = (uint32_t)(q * 4) + 1u;
      int len[4], tot = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        len[k] = Text::gene(vv[k], g + k, q * 4 + k < G, cl);
        tot += len[k];
      }
      int incl = tot;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += o;
      }
      const int T = __shfl_sync(0xffffffffu, incl, 31);
      if (T == 0) continue;
      int at = fill + incl - tot;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (len[k] != 0) {
          Text::put(s + at, vv[k], g + k, cl, cf, pairs);
          at += len[k];
        }
      }
      __syncwarp();
      const int have = fill + T, whole = have >> 4;
      for (int p = (head ? 1 : 0) + lane; p < whole; p += 32)
        __stcs(reinterpret_cast<int4 *>(out + base) + p, reinterpret_cast<const int4 *>(s)[p]);
      if (head && whole) {
        if (lane >= head && lane < 16) out[base + lane] = s[lane];
        head = 0;
      }
      const int rem = have - 16 * whole;
      const char carried = lane < rem ? s[16 * whole + lane] : 0;
      __syncwarp();
      if (lane < rem) s[lane] = carried;
      __syncwarp();
      base += 16 * whole;
      fill = rem;
    }
    if (lane == 0) fill += Text::end(s + fill);
    fill = __shfl_sync(0xffffffffu, fill, 0);
    __syncwarp();
    for (int p = lane; p < fill; p += 32)                      // the row's last piece (and, for a short row
      if (p >= head) out[base + p] = s[p];                     // that never filled one, its first)
    __syncwarp();                                              // the staging is rewritten by the next row
  }
}

// Pure-store kernel: the write-only HBM ceiling the count write is measured against (SURVEY.md 8d).  Same
// shape of traffic as the sampler's output: 128-bit stores, 512 contiguous bytes per warp instruction.
__global__ void __launch_bounds__(256) store_fill_kernel(int4 *__restrict__ out, int64_t n16, int32_t value) {
  const int4 v = make_int4(value, value, value, value);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) out[i] = v;
}

inline unsigned stream_grid(int64_t threads) {
  return (unsigned)std::max<int64_t>(1, std::min<int64_t>((threads + 255) / 256, (int64_t)num_sm() * 16));
}

// pst_mtx_row_bytes / pst_tsv_row_bytes: one warp per row
template <class Text>
void launch_text_row_bytes(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t first, int32_t *row_bytes,
                           void *stream) {
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && ((uintptr_t)X % 16 == 0);
  const unsigned grid = stream_grid(n * 32);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec) text_row_bytes_kernel<Text, true><<<grid, 256, 0, st>>>(X, n, G, ldx, first, row_bytes);
  else text_row_bytes_kernel<Text, false><<<grid, 256, 0, st>>>(X, n, G, ldx, first, row_bytes);
}

// pst_mtx_format / pst_tsv_format: kTextWarps rows per block
template <class Text>
void launch_text_format(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t first, const int64_t *text_ptr,
                        int64_t cap, char *out, void *stream) {
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && ((uintptr_t)X % 16 == 0);
  const unsigned grid = (unsigned)std::max<int64_t>(
      1, std::min<int64_t>((n + kTextWarps - 1) / kTextWarps, (int64_t)num_sm() * 16));
  cudaStream_t st = (cudaStream_t)stream;
  if (vec) text_format_kernel<Text, true><<<grid, kTextWarps * 32, 0, st>>>(X, n, G, ldx, first, text_ptr, cap, out);
  else text_format_kernel<Text, false><<<grid, kTextWarps * 32, 0, st>>>(X, n, G, ldx, first, text_ptr, cap, out);
}

constexpr int64_t kMtxMaxG = ((int64_t)1 << 31) / MtxText::kGene;       // a row's text fits int32
constexpr int64_t kTsvMaxG = (INT32_MAX - 32) / TsvText::kGene;          // G * 11 + 32 fits int32

}  // namespace
}  // namespace pst

using namespace pst;

extern "C" int pst_transform_counts(const int32_t *X, int64_t n, int64_t G, int64_t ldx, const float *scaling,
                                    int32_t mode, float *out, int64_t ldo, void *stream) {
  const char *fn = "pst_transform_counts";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && ldo >= G, fn, "need n, G >= 0, ldx >= G and ldo >= G");
  PST_REQUIRE(mode == PST_TRANSFORM_NORMALIZE || mode == PST_TRANSFORM_NORMALIZE_LOG1P ||
              mode == PST_TRANSFORM_LOG1P, fn, "unknown mode");
  if (n == 0 || G == 0) return 0;
  PST_REQUIRE(X && out, fn, "null pointer");
  PST_REQUIRE(scaling || mode == PST_TRANSFORM_LOG1P, fn, "scaling is required for the normalising modes");
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && ((uintptr_t)X % 16 == 0) &&
                   ((uintptr_t)out % 16 == 0);
  const int64_t qblocks = std::min<int64_t>((((G + 3) / 4) + 255) / 256, 64);
  const int64_t yblocks = std::max<int64_t>(1, std::min<int64_t>(n, ((int64_t)num_sm() * 16 + qblocks - 1) / qblocks));
  const dim3 grid((unsigned)qblocks, (unsigned)yblocks);
  cudaStream_t st = (cudaStream_t)stream;
#define PST_LAUNCH_TRANSFORM(M)                                                                  \
  do {                                                                                           \
    if (vec) transform_kernel<M, true><<<grid, 256, 0, st>>>(X, n, G, ldx, scaling, out, ldo);   \
    else transform_kernel<M, false><<<grid, 256, 0, st>>>(X, n, G, ldx, scaling, out, ldo);      \
  } while (0)
  if (mode == PST_TRANSFORM_NORMALIZE) PST_LAUNCH_TRANSFORM(PST_TRANSFORM_NORMALIZE);
  else if (mode == PST_TRANSFORM_NORMALIZE_LOG1P) PST_LAUNCH_TRANSFORM(PST_TRANSFORM_NORMALIZE_LOG1P);
  else PST_LAUNCH_TRANSFORM(PST_TRANSFORM_LOG1P);
#undef PST_LAUNCH_TRANSFORM
  return check_launch(fn);
}

extern "C" int pst_store_fill(int32_t *out, int64_t n, int32_t value, void *stream) {
  const char *fn = "pst_store_fill";
  PST_REQUIRE(n >= 0 && n % 4 == 0, fn, "n must be a non-negative multiple of 4");
  if (n == 0) return 0;
  PST_REQUIRE(out && (uintptr_t)out % 16 == 0, fn, "out must be a 16-byte aligned device pointer");
  store_fill_kernel<<<(unsigned)((int64_t)num_sm() * 8), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<int4 *>(out), n / 4, value);
  return check_launch(fn);
}

extern "C" int pst_csr_fill(const int32_t *X, int64_t n, int64_t G, int64_t ldx, const int64_t *indptr,
                            int32_t *indices, int32_t *data, uint32_t *flags, void *stream) {
  const char *fn = "pst_csr_fill";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G, fn, "need n, G >= 0 and ldx >= G");
  PST_REQUIRE(G < ((int64_t)1 << 31), fn, "column index does not fit int32");
  if (n == 0 || G == 0) return 0;
  PST_REQUIRE(X && indptr && indices && data && flags, fn, "null pointer");
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && ((uintptr_t)X % 16 == 0);
  const unsigned grid = stream_grid(n * 32);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec) csr_fill_kernel<int32_t, int32_t, false, true><<<grid, 256, 0, st>>>(
      X, n, G, ldx, indptr, 0, indices, data, nullptr, nullptr, 0, nullptr, flags);
  else csr_fill_kernel<int32_t, int32_t, false, false><<<grid, 256, 0, st>>>(
      X, n, G, ldx, indptr, 0, indices, data, nullptr, nullptr, 0, nullptr, flags);
  return check_launch(fn);
}

extern "C" int pst_csr_row_counts(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int32_t *row_nnz,
                                  uint64_t *sat_count, void *stream) {
  const char *fn = "pst_csr_row_counts";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G, fn, "need n, G >= 0 and ldx >= G");
  PST_REQUIRE(G < ((int64_t)1 << 31), fn, "a row's count does not fit int32");
  if (n == 0) return 0;
  PST_REQUIRE(X && row_nnz, fn, "null pointer");
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && ((uintptr_t)X % 16 == 0);
  const unsigned grid = stream_grid(n * 32);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long *sat = (unsigned long long *)sat_count;
  if (vec) csr_row_count_kernel<true><<<grid, 256, 0, st>>>(X, n, G, ldx, row_nnz, sat);
  else csr_row_count_kernel<false><<<grid, 256, 0, st>>>(X, n, G, ldx, row_nnz, sat);
  return check_launch(fn);
}

extern "C" int pst_csr_row_offsets(const int32_t *row_nnz, int64_t n, int64_t *indptr, void *stream) {
  const char *fn = "pst_csr_row_offsets";
  PST_REQUIRE(n >= 0, fn, "need n >= 0");
  PST_REQUIRE(indptr && (n == 0 || row_nnz), fn, "null pointer");
  csr_row_offsets_kernel<<<1, kScanThreads, 0, (cudaStream_t)stream>>>(row_nnz, n, indptr);
  return check_launch(fn);
}

extern "C" int pst_csr_pack(const int32_t *X, int64_t n, int64_t G, int64_t ldx, const int64_t *indptr,
                            int64_t base, void *indices, int32_t index_bits, void *data, int32_t data_bits,
                            int64_t *ovf_pos, int32_t *ovf_value, int64_t ovf_cap, uint64_t *ovf_count,
                            uint32_t *flags, void *stream) {
  const char *fn = "pst_csr_pack";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && base >= 0 && ovf_cap >= 0, fn,
              "need n, G, base, ovf_cap >= 0 and ldx >= G");
  PST_REQUIRE(index_bits == 16 || index_bits == 32 || index_bits == 64, fn, "index_bits must be 16, 32 or 64");
  PST_REQUIRE(data_bits == 16 || data_bits == 32 || data_bits == 64, fn, "data_bits must be 16, 32 or 64");
  PST_REQUIRE((index_bits < 64 && data_bits < 64) || (index_bits >= 32 && data_bits >= 32), fn,
              "64-bit widths go with 32- or 64-bit widths");
  PST_REQUIRE(index_bits != 16 || G <= 65536, fn, "16-bit column indices need G <= 65536");
  PST_REQUIRE(G < ((int64_t)1 << 31), fn, "column index does not fit int32");
  if (n == 0 || G == 0) return 0;
  PST_REQUIRE(X && indptr && indices && data && flags, fn, "null pointer");
  PST_REQUIRE(data_bits != 16 || (ovf_count && (ovf_cap == 0 || (ovf_pos && ovf_value))), fn,
              "16-bit values need the overflow list");
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && ((uintptr_t)X % 16 == 0);
  const unsigned grid = stream_grid(n * 32);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long *cnt = (unsigned long long *)ovf_count;
#define PST_LAUNCH_PACK(I, V, S)                                                                             \
  do {                                                                                                       \
    if (vec) csr_fill_kernel<I, V, S, true><<<grid, 256, 0, st>>>(X, n, G, ldx, indptr, base, (I *)indices,  \
                                                                  (V *)data, ovf_pos, ovf_value, ovf_cap,    \
                                                                  cnt, flags);                               \
    else csr_fill_kernel<I, V, S, false><<<grid, 256, 0, st>>>(X, n, G, ldx, indptr, base, (I *)indices,     \
                                                               (V *)data, ovf_pos, ovf_value, ovf_cap, cnt,  \
                                                               flags);                                       \
  } while (0)
  if (index_bits == 16 && data_bits == 16) PST_LAUNCH_PACK(uint16_t, uint16_t, true);
  else if (index_bits == 32 && data_bits == 16) PST_LAUNCH_PACK(int32_t, uint16_t, true);
  else if (index_bits == 16) PST_LAUNCH_PACK(uint16_t, int32_t, false);
  else if (index_bits == 32 && data_bits == 32) PST_LAUNCH_PACK(int32_t, int32_t, false);
  else if (index_bits == 32) PST_LAUNCH_PACK(int32_t, int64_t, false);
  else if (data_bits == 32) PST_LAUNCH_PACK(int64_t, int32_t, false);
  else PST_LAUNCH_PACK(int64_t, int64_t, false);
#undef PST_LAUNCH_PACK
  return check_launch(fn);
}

extern "C" int pst_narrow_counts(const int32_t *X, int64_t n, int64_t G, int64_t ldx, void *out, int64_t ldo,
                                 int32_t out_bits, int64_t row0, int64_t *ovf_index, int32_t *ovf_value,
                                 int64_t ovf_cap, uint64_t *ovf_count, void *stream) {
  const char *fn = "pst_narrow_counts";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && ldo >= G && row0 >= 0 && ovf_cap >= 0, fn,
              "need n, G, row0, ovf_cap >= 0, ldx >= G and ldo >= G");
  PST_REQUIRE(out_bits == 8 || out_bits == 16, fn, "out_bits must be 8 or 16");
  if (n == 0 || G == 0) return 0;
  PST_REQUIRE(X && out && ovf_count && (ovf_cap == 0 || (ovf_index && ovf_value)), fn, "null pointer");
  const int64_t obytes = out_bits / 8;
  const bool vec = (G % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && ((uintptr_t)X % 16 == 0) &&
                   ((uintptr_t)out % (4 * obytes) == 0);
  const int64_t qblocks = std::min<int64_t>((((G + 3) / 4) + 255) / 256, 64);
  const int64_t yblocks = std::max<int64_t>(1, std::min<int64_t>(n, ((int64_t)num_sm() * 16 + qblocks - 1) / qblocks));
  const dim3 grid((unsigned)qblocks, (unsigned)yblocks);
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long *cnt = (unsigned long long *)ovf_count;
#define PST_LAUNCH_NARROW(T, V) \
  narrow_kernel<T, V><<<grid, 256, 0, st>>>(X, n, G, ldx, (T *)out, ldo, row0, ovf_index, ovf_value, ovf_cap, cnt)
  if (out_bits == 8) { if (vec) PST_LAUNCH_NARROW(uint8_t, true); else PST_LAUNCH_NARROW(uint8_t, false); }
  else { if (vec) PST_LAUNCH_NARROW(uint16_t, true); else PST_LAUNCH_NARROW(uint16_t, false); }
#undef PST_LAUNCH_NARROW
  return check_launch(fn);
}

extern "C" int pst_csr_indptr_bytes(const int64_t *indptr, int64_t n, int64_t *running, void *out, int32_t out_bits,
                                    void *stream) {
  const char *fn = "pst_csr_indptr_bytes";
  PST_REQUIRE(n >= 0, fn, "need n >= 0");
  PST_REQUIRE(out_bits == 32 || out_bits == 64, fn, "out_bits must be 32 or 64");
  PST_REQUIRE(indptr && running && (n == 0 || out), fn, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (out_bits == 32) csr_indptr_kernel<int32_t><<<1, 1024, 0, st>>>(indptr, n, running, (int32_t *)out);
  else csr_indptr_kernel<int64_t><<<1, 1024, 0, st>>>(indptr, n, running, (int64_t *)out);
  return check_launch(fn);
}

extern "C" int pst_mtx_row_bytes(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t col0, int32_t *row_bytes,
                                 void *stream) {
  const char *fn = "pst_mtx_row_bytes";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && col0 >= 0, fn, "need n, G, col0 >= 0 and ldx >= G");
  PST_REQUIRE(G <= kMtxMaxG, fn, "a row's text does not fit int32");
  PST_REQUIRE(col0 <= INT64_MAX - n, fn, "cell numbers do not fit int64");
  if (n == 0) return 0;
  PST_REQUIRE(row_bytes && (G == 0 || X), fn, "null pointer");
  launch_text_row_bytes<MtxText>(X, n, G, ldx, col0, row_bytes, stream);
  return check_launch(fn);
}

extern "C" int pst_mtx_format(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t col0,
                              const int64_t *text_ptr, int64_t cap, char *out, void *stream) {
  const char *fn = "pst_mtx_format";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && col0 >= 0 && cap >= 0, fn, "need n, G, col0, cap >= 0 and ldx >= G");
  PST_REQUIRE(G <= kMtxMaxG, fn, "a row's text does not fit int32");
  PST_REQUIRE(col0 <= INT64_MAX - n, fn, "cell numbers do not fit int64");
  if (n == 0 || G == 0) return 0;
  PST_REQUIRE(X && text_ptr && out, fn, "null pointer");
  PST_REQUIRE((uintptr_t)out % 16 == 0, fn, "out must be 16-byte aligned");
  launch_text_format<MtxText>(X, n, G, ldx, col0, text_ptr, cap, out, stream);
  return check_launch(fn);
}

extern "C" int pst_tsv_row_bytes(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t row0, int32_t *row_bytes,
                                 void *stream) {
  const char *fn = "pst_tsv_row_bytes";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && row0 >= 0, fn, "need n, G, row0 >= 0 and ldx >= G");
  PST_REQUIRE(G <= kTsvMaxG, fn, "a row's text does not fit int32");
  PST_REQUIRE(row0 <= INT64_MAX - n, fn, "cell numbers do not fit int64");
  if (n == 0) return 0;
  PST_REQUIRE(row_bytes && (G == 0 || X), fn, "null pointer");
  launch_text_row_bytes<TsvText>(X, n, G, ldx, row0, row_bytes, stream);
  return check_launch(fn);
}

extern "C" int pst_tsv_format(const int32_t *X, int64_t n, int64_t G, int64_t ldx, int64_t row0,
                              const int64_t *text_ptr, int64_t cap, char *out, void *stream) {
  const char *fn = "pst_tsv_format";
  PST_REQUIRE(n >= 0 && G >= 0 && ldx >= G && row0 >= 0 && cap >= 0, fn, "need n, G, row0, cap >= 0 and ldx >= G");
  PST_REQUIRE(G <= kTsvMaxG, fn, "a row's text does not fit int32");
  PST_REQUIRE(row0 <= INT64_MAX - n, fn, "cell numbers do not fit int64");
  if (n == 0) return 0;
  PST_REQUIRE(text_ptr && out && (G == 0 || X), fn, "null pointer");
  PST_REQUIRE((uintptr_t)out % 16 == 0, fn, "out must be 16-byte aligned");
  launch_text_format<TsvText>(X, n, G, ldx, row0, text_ptr, cap, out, stream);
  return check_launch(fn);
}
