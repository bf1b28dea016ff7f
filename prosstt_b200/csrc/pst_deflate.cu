// Raw DEFLATE (RFC 1951) on the device for the compressed CSR file (`out="csr", path=..., compress=True`):
// the CSR streams of one chunk are compressed where they are made, so only compressed bytes cross PCIe
// and reach the disk.
//
// Huffman-only: the input is cut into blocks of B <= 32 KiB bytes; each becomes one dynamic-Huffman
// block over the literals 0..255 and end-of-block (no length / distance symbols: no match search), ended
// by an empty stored block (zlib's Z_SYNC_FLUSH marker), so every block ends on a byte boundary and any
// grouping of blocks concatenates into a valid stream.  A block whose Huffman form would not be smaller
// is one stored block instead, which bounds the output at input + 5 bytes per block.
//
// One CTA per block: the block is staged in shared memory, counted (per-warp histograms with
// warp-aggregated increments: zero bytes make one bin very hot), one thread builds the length-limited
// code and the block header, and the CTA writes the bit stream at the offsets of an exclusive scan of the
// code lengths.  Then the blocks' sizes are scanned and the blocks compacted into one output.  The
// CRC-32 of the input is built from per-thread CRCs moved to their place by the GF(2) shift
// x^(8 * bytes following them) mod P and XOR-ed together: the same word whatever the launch order.
//
// Segments (pst_deflate_segments, the zlib chunks of a Zarr store): the same blocks, and per segment of
// seg_blocks blocks its compressed offset (from the scan of the block sizes) and the Adler-32 of its input.
// The block kernel then sums its staged block instead of taking its CRC (ADLER), and a small kernel combines
// the blocks' sums of each segment as zlib's adler32_combine does.
#include <algorithm>
#include "pst_common.cuh"

namespace pst {
namespace {

constexpr int kDefThreads = 256;         // one thread per byte value in the histogram and the rank sort
constexpr int kMaxBlock = 32768;          // largest block: its stored form must stay below 65 535 bytes
constexpr int kStoredOverhead = 5;        // stored block header: 1 byte of BFINAL/BTYPE + padding, LEN, NLEN
constexpr int64_t kSlotPad = 16;          // per-block slot in the workspace: B + 16 bytes
constexpr int64_t kSumsAt = 8;            // a block's output is at most B + 5 bytes: its Adler sums at B + 8
constexpr uint32_t kCrcPoly = 0xEDB88320u;
constexpr uint32_t kAdlerMod = 65521;

// ---------------------------------------------------------------------------------------------
// CRC-32 (zlib's): table-driven per byte; multmodp / x2nmodp are zlib's GF(2) product and x^(2^k) powers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t multmodp(uint32_t a, uint32_t b) {
  uint32_t p = 0;
#pragma unroll 1
  for (uint32_t m = 1u << 31; m != 0; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1) ? (b >> 1) ^ kCrcPoly : b >> 1;
  }
  return p;
}

// crc moved past `bytes` zero bytes: crc32(A || B) = crc_shift(crc32(A), |B|) ^ crc32(B)
__device__ __forceinline__ uint32_t crc_shift(uint32_t crc, int64_t bytes, const uint32_t *x2n) {
  if (bytes == 0 || crc == 0) return crc;
  uint32_t p = 1u << 31;                  // x^0
  int k = 3;                              // 2^3 bits per byte
  for (uint64_t n = (uint64_t)bytes; n; n >>= 1, ++k)
    if (n & 1) p = multmodp(x2n[k & 31], p);
  return multmodp(p, crc);
}

// the byte table and x^(2^k) mod P in shared memory (one entry per thread; the 32 powers by thread 0)
__device__ void crc_tables(uint32_t *table, uint32_t *x2n) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    uint32_t c = (uint32_t)i;
    for (int j = 0; j < 8; ++j) c = (c & 1) ? (c >> 1) ^ kCrcPoly : c >> 1;
    table[i] = c;
  }
  if (threadIdx.x == 0) {
    uint32_t p = 1u << 30;                // x^1
    x2n[0] = p;
    for (int k = 1; k < 32; ++k) x2n[k] = p = multmodp(p, p);
  }
}

// ---------------------------------------------------------------------------------------------
// the staged block: byte i at word i/4 + i/128 (one pad word every 32), so that thread t reading its own
// contiguous segment of 128 bytes word by word hits bank (t + j) % 32
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int padded_word(int w) { return w + (w >> 5); }
__device__ __forceinline__ uint32_t staged_word(const uint32_t *s, int w) { return s[padded_word(w)]; }

// copy in[0, len) into the staged layout; bytes past len within the last word read 0
__device__ void stage_block(const uint8_t *__restrict__ in, int len, uint32_t *s) {
  const int words = (len + 3) >> 2;
  if (((uintptr_t)in & 15) == 0) {
    const int quads = len >> 4;
    for (int q = threadIdx.x; q < quads; q += blockDim.x) {
      const uint4 v = __ldcs(reinterpret_cast<const uint4 *>(in) + q);
      const int w = q * 4;                // four words of one 32-word group
      s[padded_word(w)] = v.x; s[padded_word(w + 1)] = v.y; s[padded_word(w + 2)] = v.z; s[padded_word(w + 3)] = v.w;
    }
    for (int w = quads * 4 + threadIdx.x; w < words; w += blockDim.x) {
      uint32_t v = 0;
      for (int j = 0; j < 4 && 4 * w + j < len; ++j) v |= (uint32_t)in[4 * w + j] << (8 * j);
      s[padded_word(w)] = v;
    }
  } else {
    for (int w = threadIdx.x; w < words; w += blockDim.x) {
      uint32_t v = 0;
      for (int j = 0; j < 4 && 4 * w + j < len; ++j) v |= (uint32_t)in[4 * w + j] << (8 * j);
      s[padded_word(w)] = v;
    }
  }
}

// thread t's segment [lo, hi) of a block of len bytes (seg bytes per thread, a multiple of 4)
__device__ __forceinline__ void segment(int len, int seg, int &lo, int &hi) {
  lo = min(len, (int)threadIdx.x * seg);
  hi = min(len, lo + seg);
}

// CRC-32 of the staged block (len bytes), valid in thread 0; `red` holds one word per warp
__device__ uint32_t block_crc(const uint32_t *s, int len, int seg, const uint32_t *table, const uint32_t *x2n,
                              uint32_t *red) {
  int lo, hi;
  segment(len, seg, lo, hi);
  uint32_t c = 0xFFFFFFFFu;
  for (int i = lo; i < hi; i += 4) {
    const uint32_t w = staged_word(s, i >> 2);
    const int k = min(4, hi - i);
    for (int j = 0; j < k; ++j) c = table[(c ^ (w >> (8 * j))) & 0xFF] ^ (c >> 8);
  }
  c = (hi > lo) ? crc_shift(c ^ 0xFFFFFFFFu, len - hi, x2n) : 0u;
  for (int d = 16; d; d >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, d);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
  __syncthreads();
  uint32_t all = 0;
  if (threadIdx.x == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) all ^= red[w];
  __syncthreads();
  return all;
}

// Adler-32 sums of the staged block (len bytes), valid in thread 0: x = sum b_i and y = sum (len - i) b_i, both
// mod 65521, so that adler32 = (1 + x) | ((len + y) << 16).  A thread's segment sums stay below 2^22 (at most 128
// bytes); each is moved to the block's end and reduced before the warps add them up.  `red` holds two words per warp.
__device__ uint2 block_adler(const uint32_t *s, int len, int seg, uint32_t *red) {
  int lo, hi;
  segment(len, seg, lo, hi);
  uint32_t x = 0, y = 0;                                           // y = sum (hi - i) b_i over the segment
  for (int i = lo; i < hi; i += 4) {
    const uint32_t w = staged_word(s, i >> 2);
    const int k = min(4, hi - i);
    for (int j = 0; j < k; ++j) { x += (w >> (8 * j)) & 0xFF; y += x; }
  }
  y = (uint32_t)(((uint64_t)y + (uint64_t)(len - hi) * x) % kAdlerMod);
  x %= kAdlerMod;
  for (int d = 16; d; d >>= 1) {
    x += __shfl_xor_sync(0xffffffffu, x, d);
    y += __shfl_xor_sync(0xffffffffu, y, d);
  }
  if ((threadIdx.x & 31) == 0) { red[2 * (threadIdx.x >> 5)] = x; red[2 * (threadIdx.x >> 5) + 1] = y; }
  __syncthreads();
  uint2 all = make_uint2(0, 0);
  if (threadIdx.x == 0) {
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { all.x += red[2 * w]; all.y += red[2 * w + 1]; }
    all.x %= kAdlerMod;
    all.y %= kAdlerMod;
  }
  __syncthreads();
  return all;
}

// ---------------------------------------------------------------------------------------------
// length-limited Huffman code (one thread).  key[0..n) holds the symbols' frequencies sorted ascending
// (ties by symbol), sym[] the symbols.  Moffat-Katajainen in place gives optimal lengths, the lengths
// over max_len are folded back by the Kraft-sum repair of miniz (tdefl_huffman_enforce_max_code_size),
// and the lengths go to the symbols from the most frequent down.  Deterministic.
// ---------------------------------------------------------------------------------------------
__device__ void huffman_lengths(uint32_t *key, const uint16_t *sym, int n, int max_len, uint8_t *len_out,
                                int *count /* 33 entries */) {
  if (n == 0) return;
  if (n == 1) { len_out[sym[0]] = 1; return; }
  key[0] += key[1];
  int root = 0, leaf = 2;
  for (int next = 1; next < n - 1; ++next) {
    if (leaf >= n || key[root] < key[leaf]) { key[next] = key[root]; key[root++] = next; }
    else key[next] = key[leaf++];
    if (leaf >= n || (root < next && key[root] < key[leaf])) { key[next] += key[root]; key[root++] = next; }
    else key[next] += key[leaf++];
  }
  key[n - 2] = 0;
  for (int next = n - 3; next >= 0; --next) key[next] = key[key[next]] + 1;
  int avbl = 1, used = 0, dpth = 0;
  root = n - 2;
  int next = n - 1;
  while (avbl > 0) {
    while (root >= 0 && (int)key[root] == dpth) { ++used; --root; }
    while (avbl > used) { key[next--] = dpth; --avbl; }
    avbl = 2 * used; ++dpth; used = 0;
  }
  for (int i = 0; i <= 32; ++i) count[i] = 0;
  for (int i = 0; i < n; ++i) count[min((int)key[i], 32)]++;
  for (int i = max_len + 1; i <= 32; ++i) { count[max_len] += count[i]; count[i] = 0; }
  uint32_t total = 0;
  for (int i = max_len; i > 0; --i) total += (uint32_t)count[i] << (max_len - i);
  while (total != (1u << max_len)) {
    count[max_len]--;
    for (int i = max_len - 1; i > 0; --i)
      if (count[i]) { count[i]--; count[i + 1] += 2; break; }
    total--;
  }
  for (int l = 1, j = n; l <= max_len; ++l)
    for (int c = count[l]; c > 0; --c) len_out[sym[--j]] = (uint8_t)l;
}

// canonical codes (RFC 1951 3.2.2), bit-reversed for the LSB-first stream
__device__ void canonical_codes(const uint8_t *len, int n, uint16_t *code, int *count /* 16 */, int *next /* 16 */) {
  for (int l = 0; l < 16; ++l) count[l] = 0;
  for (int s = 0; s < n; ++s) count[len[s]]++;
  count[0] = 0;
  int c = 0;
  for (int l = 1; l < 16; ++l) { c = (c + count[l - 1]) << 1; next[l] = c; }
  for (int s = 0; s < n; ++s) {
    const int l = len[s];
    if (l == 0) { code[s] = 0; continue; }
    code[s] = (uint16_t)(__brev((uint32_t)next[l]++) >> (32 - l));
  }
}

// bit writer of one thread into zeroed shared words (the header)
struct BitWriter {
  uint32_t *buf;
  int64_t pos;
  __device__ void put(uint32_t v, int n) {
    if (n == 0) return;
    const int64_t w = pos >> 5;
    const int o = (int)(pos & 31);
    buf[w] |= v << o;
    if (o + n > 32) buf[w + 1] |= v >> (32 - o);
    pos += n;
  }
};

__constant__ uint8_t kClOrder[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

// symbol s of freq[0..n) placed at its rank among the used symbols by (frequency, symbol): key / sym are
// the sorted input of huffman_lengths.  One thread per symbol.
__device__ void rank_place(const uint32_t *freq, int n, int s, uint32_t *key, uint16_t *sym) {
  const uint32_t f = freq[s];
  if (!f) return;
  int rank = 0;
  for (int u = 0; u < n; ++u) {
    const uint32_t g = freq[u];
    rank += (g != 0) && (g < f || (g == f && u < s));
  }
  key[rank] = f;
  sym[rank] = (uint16_t)s;
}

// the code lengths lens[0..n) run-length coded (RFC 1951 3.2.7) as (symbol, extra bits value) byte pairs
// into packed, each symbol counted in cl_freq[19]; returns the bytes written (one thread)
__device__ int rle_lengths(const uint8_t *lens, int n, uint8_t *packed, uint32_t *cl_freq) {
  for (int i = 0; i < 19; ++i) cl_freq[i] = 0;
  int np = 0, prev = 0xFF, rle_z = 0, rle_rep = 0;
  auto flush_rep = [&]() {
    if (rle_rep) {
      if (rle_rep < 3) {
        cl_freq[prev] += rle_rep;
        while (rle_rep--) { packed[np++] = (uint8_t)prev; packed[np++] = 0; }
      } else {
        cl_freq[16]++; packed[np++] = 16; packed[np++] = (uint8_t)(rle_rep - 3);
      }
      rle_rep = 0;
    }
  };
  auto flush_z = [&]() {
    if (rle_z) {
      if (rle_z < 3) {
        cl_freq[0] += rle_z;
        while (rle_z--) { packed[np++] = 0; packed[np++] = 0; }
      } else if (rle_z <= 10) {
        cl_freq[17]++; packed[np++] = 17; packed[np++] = (uint8_t)(rle_z - 3);
      } else {
        cl_freq[18]++; packed[np++] = 18; packed[np++] = (uint8_t)(rle_z - 11);
      }
      rle_z = 0;
    }
  };
  for (int i = 0; i < n; ++i) {
    const int l = lens[i];
    if (l == 0) {
      flush_rep();
      if (++rle_z == 138) flush_z();
    } else {
      flush_z();
      if (l != prev) { flush_rep(); cl_freq[l]++; packed[np++] = (uint8_t)l; packed[np++] = 0; }
      else if (++rle_rep == 6) flush_rep();
    }
    prev = l;
  }
  if (rle_rep) flush_rep(); else flush_z();
  return np;
}

// the code-length code of a block header (19 symbols, at most 7 bits) from rle_lengths' output
struct ClCode {
  uint8_t len[19];
  uint16_t code[19];
  uint32_t freq[19], key[19];
  uint16_t sym[19];
  int hclen;
};

// builds c from c.freq (one thread); returns the header's bits from HCLEN on: HCLEN, the code-length code
// lengths and the packed lengths with their extra bits
__device__ long long cl_build(ClCode &c, const uint8_t *packed, int np, int *count, int *next) {
  int cn = 0;
  for (int s = 0; s < 19; ++s) {
    c.len[s] = 0;
    if (!c.freq[s]) continue;
    int j = cn++;                                                  // insertion by (frequency, symbol)
    while (j > 0 && c.key[j - 1] > c.freq[s]) { c.key[j] = c.key[j - 1]; c.sym[j] = c.sym[j - 1]; --j; }
    c.key[j] = c.freq[s]; c.sym[j] = (uint16_t)s;
  }
  huffman_lengths(c.key, c.sym, cn, 7, c.len, count);
  canonical_codes(c.len, 19, c.code, count, next);
  c.hclen = 19;
  while (c.hclen > 4 && c.len[kClOrder[c.hclen - 1]] == 0) --c.hclen;
  long long bits = 4 + 3 * c.hclen;
  for (int i = 0; i < np; i += 2) {
    const int s = packed[i];
    bits += c.len[s] + (s == 16 ? 2 : s == 17 ? 3 : s == 18 ? 7 : 0);
  }
  return bits;
}

// HCLEN, the code-length code lengths and the packed code lengths
__device__ void cl_put(BitWriter &bw, const ClCode &c, const uint8_t *packed, int np) {
  bw.put(c.hclen - 4, 4);
  for (int i = 0; i < c.hclen; ++i) bw.put(c.len[kClOrder[i]], 3);
  for (int i = 0; i < np; i += 2) {
    const int s = packed[i];
    bw.put(c.code[s], c.len[s]);
    if (s >= 16) bw.put(packed[i + 1], s == 16 ? 2 : s == 17 ? 3 : 7);
  }
}

struct HuffShared {
  uint32_t hist[kDefThreads / 32][257];   // per-warp byte counts; bin 256 takes the bytes past the end
  uint32_t freq[257];
  uint32_t key[257];
  uint16_t sym[257];
  uint8_t len[258];                       // 257 literal/length lengths + the one distance code
  uint16_t code[257];
  uint8_t packed[2 * 258];                // run-length coded lengths: symbol, then its extra bits value
  ClCode cl;
  uint32_t crc_table[256];
  uint32_t x2n[32];
  int count[33], next[16];
  uint32_t red[2 * (kDefThreads / 32)];
  long long scan[kDefThreads / 32];
  int header_bits, stored;
  long long total_bits;
};

// ---------------------------------------------------------------------------------------------
// one CTA per block b: block bytes in[b*B, min((b+1)*B, n)), written to slot b of the workspace
// (B + 16 bytes), its size to sizes[b]; its CRC, shifted past the rest of the input, XOR-ed into *crc, or with
// ADLER its Adler sums (block_adler) at byte B + 8 of the slot
// ---------------------------------------------------------------------------------------------
template <bool ADLER>
__global__ void __launch_bounds__(kDefThreads)
deflate_block_kernel(const uint8_t *__restrict__ in, const int64_t *__restrict__ count, int64_t scale,
                     int64_t max_bytes, int block, uint8_t *__restrict__ slots, int32_t *__restrict__ sizes,
                     uint32_t *__restrict__ crc_out) {
  extern __shared__ __align__(16) uint32_t dyn[];
  __shared__ HuffShared sh;
  const int64_t n = count ? min(max_bytes, count[0] * scale) : max_bytes;
  const int64_t start = (int64_t)blockIdx.x * block;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (start >= n) {
    if (tid == 0) sizes[blockIdx.x] = 0;
    return;
  }
  const int len = (int)(n - start < block ? n - start : (int64_t)block);
  const int seg = block / kDefThreads;
  uint32_t *staged = dyn;                                          // padded_word(block / 4) words
  uint32_t *bits = dyn + padded_word(block / 4) + 4;               // block / 4 + 8 words
  const int bit_words = block / 4 + 8;
  stage_block(in + start, len, staged);
  for (int i = tid; i < bit_words; i += blockDim.x) bits[i] = 0;
  for (int i = tid; i < (kDefThreads / 32) * 257; i += blockDim.x) (&sh.hist[0][0])[i] = 0;
  if (!ADLER) crc_tables(sh.crc_table, sh.x2n);
  __syncthreads();

  // ---- histogram: word w of the block per thread and round, its four bytes aggregated over the warp
  const int words = (len + 3) >> 2;
  for (int r = 0; r < (words + kDefThreads - 1) / kDefThreads; ++r) {
    const int w = r * kDefThreads + tid;
    const uint32_t v = w < words ? staged_word(staged, w) : 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int b = (4 * w + j < len) ? (int)((v >> (8 * j)) & 0xFF) : 256;
      const unsigned peers = __match_any_sync(0xffffffffu, b);
      if (lane == __ffs(peers) - 1) sh.hist[wid][b] += __popc(peers);   // one leader per value and warp
      __syncwarp();
    }
  }
  uint32_t crc = 0;
  uint2 sums = make_uint2(0, 0);
  if (ADLER) sums = block_adler(staged, len, seg, sh.red);                           // synchronises
  else crc = block_crc(staged, len, seg, sh.crc_table, sh.x2n, sh.red);              // synchronises
  for (int s = tid; s < 257; s += blockDim.x) {
    uint32_t f = (s == 256) ? 1u : 0u;                             // end-of-block
    if (s < 256)
      for (int w = 0; w < kDefThreads / 32; ++w) f += sh.hist[w][s];
    sh.freq[s] = f;
    sh.len[s] = 0;
  }
  __syncthreads();
  // ---- sort the used symbols by (frequency, symbol): each finds its rank
  for (int s = tid; s < 257; s += blockDim.x) rank_place(sh.freq, 257, s, sh.key, sh.sym);
  const int used = __syncthreads_count(sh.freq[tid] != 0) + 1;    // + end-of-block (kDefThreads == 256)
  if (tid == 0) {
    // ---- literal/length code, its lengths run-length coded with the one distance code (length 1)
    huffman_lengths(sh.key, sh.sym, used, 15, sh.len, sh.count);
    sh.len[257] = 1;
    canonical_codes(sh.len, 257, sh.code, sh.count, sh.next);
    const int np = rle_lengths(sh.len, 258, sh.packed, sh.cl.freq);
    const long long hbits = 3 + 5 + 5 + cl_build(sh.cl, sh.packed, np, sh.count, sh.next);
    long long body = sh.len[256];
    for (int s = 0; s < 256; ++s) body += (long long)sh.freq[s] * sh.len[s];
    sh.header_bits = (int)hbits;
    sh.total_bits = hbits + body;
    // dynamic block + the empty stored block (3 bits, padding, 00 00 FF FF) against one stored block
    sh.stored = ((hbits + body + 3 + 7) / 8 + 4 >= (long long)len + kStoredOverhead);
    if (!sh.stored) {
      BitWriter bw{bits, 0};
      bw.put(0, 1);                                                // BFINAL = 0
      bw.put(2, 2);                                                // BTYPE = 10: dynamic Huffman
      bw.put(0, 5);                                                // HLIT = 257 - 257
      bw.put(0, 5);                                                // HDIST = 1 - 1
      cl_put(bw, sh.cl, sh.packed, np);
    }
  }
  __syncthreads();
  uint8_t *slot = slots + (int64_t)blockIdx.x * (block + kSlotPad);
  if (sh.stored) {
    if (tid == 0) {
      slot[0] = 0;                                                 // BFINAL = 0, BTYPE = 00, padding
      slot[1] = (uint8_t)(len & 0xFF); slot[2] = (uint8_t)(len >> 8);
      slot[3] = (uint8_t)(~len & 0xFF); slot[4] = (uint8_t)((~len >> 8) & 0xFF);
      sizes[blockIdx.x] = len + kStoredOverhead;
    }
    for (int i = tid; i < len; i += blockDim.x)
      slot[kStoredOverhead + i] = (uint8_t)(staged_word(staged, i >> 2) >> (8 * (i & 3)));
  } else {
    // ---- the literals: each thread's segment at the exclusive scan of the code lengths
    int lo, hi;
    segment(len, seg, lo, hi);
    long long mine = 0;
    for (int i = lo; i < hi; i += 4) {
      const uint32_t w = staged_word(staged, i >> 2);
      const int k = min(4, hi - i);
      for (int j = 0; j < k; ++j) mine += sh.len[(w >> (8 * j)) & 0xFF];
    }
    long long incl = mine;
    for (int d = 1; d < 32; d <<= 1) {
      const long long o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) sh.scan[wid] = incl;
    __syncthreads();
    long long off = sh.header_bits + incl - mine;
    for (int w = 0; w < wid; ++w) off += sh.scan[w];
    {
      uint64_t acc = 0;
      int nb = (int)(off & 31);
      int64_t wi = off >> 5;
      bool first = true;                                           // shared with the previous writer
      for (int i = lo; i < hi; i += 4) {
        const uint32_t w = staged_word(staged, i >> 2);
        const int k = min(4, hi - i);
        for (int j = 0; j < k; ++j) {
          const int b = (w >> (8 * j)) & 0xFF;
          acc |= (uint64_t)sh.code[b] << nb;
          nb += sh.len[b];
          if (nb >= 32) {
            if (first) atomicOr(&bits[wi], (uint32_t)acc); else bits[wi] = (uint32_t)acc;
            first = false;
            ++wi; acc >>= 32; nb -= 32;
          }
        }
      }
      if (nb > 0) atomicOr(&bits[wi], (uint32_t)acc);              // shared with the next writer
    }
    __syncthreads();
    if (tid == 0) {
      const long long end = sh.total_bits - sh.len[256];
      BitWriter bw{bits, end};
      bw.put(sh.code[256], sh.len[256]);                           // end-of-block
      bw.put(0, 3);                                                // empty stored block, then byte-align
      const int64_t at = (bw.pos + 7) >> 3;
      uint8_t *bb = reinterpret_cast<uint8_t *>(bits);
      bb[at] = 0; bb[at + 1] = 0; bb[at + 2] = 0xFF; bb[at + 3] = 0xFF;
      sizes[blockIdx.x] = (int32_t)(at + 4);
    }
    __syncthreads();
    const int nbytes = sizes[blockIdx.x];
    for (int w = tid; w < (nbytes + 3) / 4; w += blockDim.x) reinterpret_cast<uint32_t *>(slot)[w] = bits[w];
  }
  if (tid == 0) {
    if (ADLER) *reinterpret_cast<uint2 *>(slot + block + kSumsAt) = sums;
    else atomicXor(crc_out, crc_shift(crc, n - start - len, sh.x2n));
  }
}

// ---------------------------------------------------------------------------------------------
// LZ77 + Huffman (pst_deflate_lz_blocks): the same block framing, with length / distance codes.  The
// window is the block itself, so every block still decodes on its own.
//
// One CTA of kLzThreads per block; every step is a function of the block's bytes alone:
//  1. prev[p]: the nearest earlier position whose 3 bytes hash alike (zlib's hash chain).  Warp w walks
//     its region of the block 32 positions at a time with its own table of last positions: lanes that
//     hash alike find each other by __match_any_sync, the highest of them updates the table.  A position
//     first in its region with its hash then takes the table entry of the nearest earlier region.
//  2. Every position's longest match (the nearest on ties) over at most kMaxChain chain candidates.
//  3. Each segment of kLzSeg bytes is parsed greedily by one thread, matches cut at the segment's end,
//     into uint16 tokens in the block's token slot (global workspace); the symbols are counted.
//  4. Literal/length and distance codes (15-bit limited), the header, then each segment's tokens at the
//     exclusive scan of their bit lengths, as in deflate_block_kernel.
// ---------------------------------------------------------------------------------------------
constexpr int kLzThreads = 512;
constexpr int kLzWarps = kLzThreads / 32;
constexpr int kHashBits = 11;              // one table of 2^11 uint16 positions per warp: 64 KiB in all
constexpr int kLzSeg = 512;               // bytes parsed by one thread (a match is at most this long)
constexpr int kMaxChain = 8;              // chain candidates tried per position
constexpr int kNiceMatch = 64;            // a match this long ends the chain walk
constexpr int kMinMatch = 3, kMaxMatch = 258;
constexpr int kLitSyms = 286, kDistSyms = 30;
constexpr uint16_t kNone = 0xFFFF;

// the 4 bytes at byte i of the staged block (bytes past the block's end are not meaningful)
__device__ __forceinline__ uint32_t bytes4(const uint32_t *s, int i) {
  const int w = i >> 2;
  return __funnelshift_r(staged_word(s, w), staged_word(s, w + 1), 8 * (i & 3));
}

__device__ __forceinline__ int byte_at(const uint32_t *s, int i) { return (staged_word(s, i >> 2) >> (8 * (i & 3))) & 0xFF; }

__device__ __forceinline__ uint32_t hash3(const uint32_t *s, int i) {
  return ((bytes4(s, i) & 0xFFFFFFu) * 0x9E3779B1u) >> (32 - kHashBits);
}

// length of the common prefix of the bytes at p and q < p, at most maxl
__device__ __forceinline__ int match_len(const uint32_t *s, int p, int q, int maxl) {
  for (int l = 0; l < maxl; l += 4) {
    const uint32_t x = bytes4(s, p + l) ^ bytes4(s, q + l);
    if (x) return min(maxl, l + ((__ffs(x) - 1) >> 3));
  }
  return maxl;
}

// length symbol (257..285) of a match of l bytes, with its extra bits
__device__ __forceinline__ int len_sym(int l, int &ebits, int &evalue) {
  const int x = l - kMinMatch;
  if (x < 8 || x == 255) { ebits = evalue = 0; return x == 255 ? 285 : 257 + x; }
  const int nb = 31 - __clz(x);
  ebits = nb - 2; evalue = x & ((1 << ebits) - 1);
  return 257 + 4 * (nb - 1) + ((x >> ebits) & 3);
}

// distance symbol (0..29) of distance d, with its extra bits
__device__ __forceinline__ int dist_sym(int d, int &ebits, int &evalue) {
  const int x = d - 1;
  if (x < 4) { ebits = evalue = 0; return x; }
  const int nb = 31 - __clz(x);
  ebits = nb - 1; evalue = x & ((1 << ebits) - 1);
  return 2 * nb + ((x >> ebits) & 1);
}

__device__ __forceinline__ int len_extra(int s) { return (s >= 265 && s < 285) ? (s - 261) >> 2 : 0; }
__device__ __forceinline__ int dist_extra(int s) { return s >= 4 ? (s >> 1) - 1 : 0; }

struct LzShared {
  uint32_t freq[kLitSyms + kDistSyms];    // literal/length counts, then distance counts
  uint32_t key[kLitSyms], dkey[kDistSyms];
  uint16_t sym[kLitSyms], dsym[kDistSyms];
  uint8_t len[kLitSyms + kDistSyms];      // code lengths, distances from kLitSyms
  uint16_t code[kLitSyms + kDistSyms];
  uint8_t lens[kLitSyms + kDistSyms];     // the HLIT + HDIST lengths the header codes
  uint8_t packed[2 * (kLitSyms + kDistSyms)];
  ClCode cl;
  uint32_t crc_table[256];
  uint32_t x2n[32];
  int count[33], next[16];
  uint32_t red[2 * kLzWarps];
  long long scan[kLzWarps];
  int ntok[kMaxBlock / kLzSeg];           // tokens of each segment
  int header_bits, stored;
  long long total_bits;
};

// scratch region of the dynamic shared memory: the hash tables, then the match distances, then the bit stream
inline size_t lz_scratch_bytes(int32_t block) {
  return std::max<size_t>((size_t)kLzWarps << kHashBits, (size_t)block) * 2;
}

// one CTA per block b, as deflate_block_kernel; tokens: the block's slot of `block` uint16 entries
template <bool ADLER>
__global__ void __launch_bounds__(kLzThreads)
deflate_lz_block_kernel(const uint8_t *__restrict__ in, const int64_t *__restrict__ count, int64_t scale,
                        int64_t max_bytes, int block, uint8_t *__restrict__ slots, int32_t *__restrict__ sizes,
                        uint32_t *__restrict__ crc_out, uint16_t *__restrict__ tokens) {
  extern __shared__ __align__(16) uint32_t dyn[];
  __shared__ LzShared sh;
  const int64_t n = count ? min(max_bytes, count[0] * scale) : max_bytes;
  const int64_t start = (int64_t)blockIdx.x * block;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (start >= n) {
    if (tid == 0) sizes[blockIdx.x] = 0;
    return;
  }
  const int len = (int)(n - start < block ? n - start : (int64_t)block);
  uint32_t *staged = dyn;                                          // padded_word(block / 4) + 4 words
  uint16_t *prev = reinterpret_cast<uint16_t *>(dyn + padded_word(block / 4) + 4);   // block entries
  uint16_t *scratch = prev + block;                                // lz_scratch_bytes(block)
  stage_block(in + start, len, staged);
  if (tid == 0) staged[padded_word((len + 3) >> 2)] = 0;           // the word past the block's last one
  for (int i = tid; i < (kLzWarps << kHashBits); i += blockDim.x) scratch[i] = kNone;
  for (int s = tid; s < kLitSyms + kDistSyms; s += blockDim.x) { sh.freq[s] = (s == 256); sh.len[s] = 0; }
  if (!ADLER) crc_tables(sh.crc_table, sh.x2n);
  __syncthreads();

  // ---- 1. hash chains: warp w over its region, then the first positions of each region
  const int region = ((len + kLzWarps - 1) / kLzWarps + 31) & ~31;
  {
    uint16_t *tab = scratch + (wid << kHashBits);
    const int rhi = min(len, (wid + 1) * region);
    for (int base = wid * region; base < rhi; base += 32) {
      const int p = base + lane;
      const bool ok = p + kMinMatch <= len;
      const uint32_t h = ok ? hash3(staged, p) : (1u << kHashBits) + lane;
      const unsigned peers = __match_any_sync(0xffffffffu, h);
      uint16_t cand = kNone;
      if (ok) {
        const unsigned lower = peers & ((1u << lane) - 1);
        cand = lower ? (uint16_t)(base + 31 - __clz(lower)) : tab[h];
      }
      __syncwarp();
      if (ok && (peers >> lane) == 1u) tab[h] = (uint16_t)p;      // the last position of the step
      __syncwarp();
      if (p < rhi) prev[p] = cand;
    }
  }
  __syncthreads();
  for (int p = tid; p + kMinMatch <= len; p += blockDim.x) {
    if (prev[p] != kNone) continue;
    const uint32_t h = hash3(staged, p);
    for (int v = p / region - 1; v >= 0; --v) {
      const uint16_t c = scratch[(v << kHashBits) + h];
      if (c != kNone) { prev[p] = c; break; }
    }
  }
  __syncthreads();

  // ---- 2. longest match at every position: its distance, 0 for none (the tables are dead)
  uint16_t *mdist = scratch;
  for (int p = tid; p < len; p += blockDim.x) {
    const int maxl = min(kMaxMatch, len - p);
    int best = kMinMatch - 1, bestd = 0, cand = prev[p];
    for (int k = 0; k < kMaxChain && cand != kNone; ++k) {
      const int l = match_len(staged, p, cand, maxl);
      if (l > best) {
        best = l; bestd = p - cand;
        if (l >= kNiceMatch || l == maxl) break;
      }
      cand = prev[cand];
    }
    mdist[p] = (uint16_t)bestd;
  }
  __syncthreads();

  // ---- 3. greedy parse per segment: a literal is one token (the byte), a match two (256 + l - 3, d - 1)
  const int nseg = (len + kLzSeg - 1) / kLzSeg;
  uint16_t *tok = tokens + (int64_t)blockIdx.x * block;
  if (tid < nseg) {
    const int lo = tid * kLzSeg, hi = min(len, lo + kLzSeg);
    int o = lo, eb, ev;
    for (int p = lo; p < hi;) {
      const int d = mdist[p];
      const int l = d ? match_len(staged, p, p - d, min(kMaxMatch, hi - p)) : 0;
      if (l >= kMinMatch) {
        tok[o++] = (uint16_t)(256 + l - kMinMatch);
        tok[o++] = (uint16_t)(d - 1);
        atomicAdd(&sh.freq[len_sym(l, eb, ev)], 1u);
        atomicAdd(&sh.freq[kLitSyms + dist_sym(d, eb, ev)], 1u);
        p += l;
      } else {
        const int b = byte_at(staged, p);
        tok[o++] = (uint16_t)b;
        atomicAdd(&sh.freq[b], 1u);
        ++p;
      }
    }
    sh.ntok[tid] = o - lo;
  }
  __syncthreads();

  // ---- 4. the two codes and the header (the match distances are dead: the scratch holds the bit stream)
  uint32_t *bits = reinterpret_cast<uint32_t *>(scratch);
  const int bit_words = block / 4 + 8;
  for (int i = tid; i < bit_words; i += blockDim.x) bits[i] = 0;
  if (tid < kLitSyms) rank_place(sh.freq, kLitSyms, tid, sh.key, sh.sym);
  else if (tid >= 320 && tid < 320 + kDistSyms)                    // a warp of its own
    rank_place(sh.freq + kLitSyms, kDistSyms, tid - 320, sh.dkey, sh.dsym);
  __syncthreads();
  if (tid == 0) {
    int nl = 0, nd = 0;
    for (int s = 0; s < kLitSyms; ++s) nl += sh.freq[s] != 0;
    for (int s = 0; s < kDistSyms; ++s) nd += sh.freq[kLitSyms + s] != 0;
    huffman_lengths(sh.key, sh.sym, nl, 15, sh.len, sh.count);
    if (nd) huffman_lengths(sh.dkey, sh.dsym, nd, 15, sh.len + kLitSyms, sh.count);
    else sh.len[kLitSyms] = 1;                                     // no match: one unused distance code
    canonical_codes(sh.len, kLitSyms, sh.code, sh.count, sh.next);
    canonical_codes(sh.len + kLitSyms, kDistSyms, sh.code + kLitSyms, sh.count, sh.next);
    int hlit = kLitSyms, hdist = kDistSyms;
    while (hlit > 257 && sh.len[hlit - 1] == 0) --hlit;
    while (hdist > 1 && sh.len[kLitSyms + hdist - 1] == 0) --hdist;
    for (int i = 0; i < hlit; ++i) sh.lens[i] = sh.len[i];
    for (int i = 0; i < hdist; ++i) sh.lens[hlit + i] = sh.len[kLitSyms + i];
    const int np = rle_lengths(sh.lens, hlit + hdist, sh.packed, sh.cl.freq);
    const long long hbits = 3 + 5 + 5 + cl_build(sh.cl, sh.packed, np, sh.count, sh.next);
    long long body = 0;
    for (int s = 0; s < kLitSyms; ++s) body += (long long)sh.freq[s] * (sh.len[s] + len_extra(s));
    for (int s = 0; s < kDistSyms; ++s)
      body += (long long)sh.freq[kLitSyms + s] * (sh.len[kLitSyms + s] + dist_extra(s));
    sh.header_bits = (int)hbits;
    sh.total_bits = hbits + body;
    sh.stored = ((hbits + body + 3 + 7) / 8 + 4 >= (long long)len + kStoredOverhead);
    if (!sh.stored) {
      BitWriter bw{bits, 0};
      bw.put(0, 1);                                                // BFINAL = 0
      bw.put(2, 2);                                                // BTYPE = 10: dynamic Huffman
      bw.put(hlit - 257, 5);
      bw.put(hdist - 1, 5);
      cl_put(bw, sh.cl, sh.packed, np);
    }
  }
  __syncthreads();
  uint8_t *slot = slots + (int64_t)blockIdx.x * (block + kSlotPad);
  if (sh.stored) {
    if (tid == 0) {
      slot[0] = 0;
      slot[1] = (uint8_t)(len & 0xFF); slot[2] = (uint8_t)(len >> 8);
      slot[3] = (uint8_t)(~len & 0xFF); slot[4] = (uint8_t)((~len >> 8) & 0xFF);
      sizes[blockIdx.x] = len + kStoredOverhead;
    }
    for (int i = tid; i < len; i += blockDim.x) slot[kStoredOverhead + i] = (uint8_t)byte_at(staged, i);
  } else {
    // ---- each segment's tokens at the exclusive scan of their bit lengths
    const int t0 = tid * kLzSeg, t1 = tid < nseg ? t0 + sh.ntok[tid] : t0;
    long long mine = 0;
    int eb, ev;
    for (int i = t0; i < t1;) {
      const int x = tok[i++];
      if (x < 256) { mine += sh.len[x]; continue; }
      const int ls = len_sym(x - 256 + kMinMatch, eb, ev);
      mine += sh.len[ls] + eb;
      const int ds = dist_sym(tok[i++] + 1, eb, ev);
      mine += sh.len[kLitSyms + ds] + eb;
    }
    long long incl = mine;
    for (int d = 1; d < 32; d <<= 1) {
      const long long o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) sh.scan[wid] = incl;
    __syncthreads();
    long long off = sh.header_bits + incl - mine;
    for (int w = 0; w < wid; ++w) off += sh.scan[w];
    if (t1 > t0) {
      uint64_t acc = 0;
      int nb = (int)(off & 31);
      int64_t wi = off >> 5;
      bool first = true;                                           // shared with the previous writer
      auto put = [&](uint32_t v, int k) {
        acc |= (uint64_t)v << nb;
        nb += k;
        if (nb >= 32) {
          if (first) atomicOr(&bits[wi], (uint32_t)acc); else bits[wi] = (uint32_t)acc;
          first = false;
          ++wi; acc >>= 32; nb -= 32;
        }
      };
      for (int i = t0; i < t1;) {
        const int x = tok[i++];
        if (x < 256) { put(sh.code[x], sh.len[x]); continue; }
        const int ls = len_sym(x - 256 + kMinMatch, eb, ev);
        put(sh.code[ls], sh.len[ls]);
        put(ev, eb);
        const int ds = dist_sym(tok[i++] + 1, eb, ev);
        put(sh.code[kLitSyms + ds], sh.len[kLitSyms + ds]);
        put(ev, eb);
      }
      if (nb > 0) atomicOr(&bits[wi], (uint32_t)acc);              // shared with the next writer
    }
    __syncthreads();
    if (tid == 0) {
      BitWriter bw{bits, sh.total_bits - sh.len[256]};
      bw.put(sh.code[256], sh.len[256]);                           // end-of-block
      bw.put(0, 3);                                                // empty stored block, then byte-align
      const int64_t at = (bw.pos + 7) >> 3;
      uint8_t *bb = reinterpret_cast<uint8_t *>(bits);
      bb[at] = 0; bb[at + 1] = 0; bb[at + 2] = 0xFF; bb[at + 3] = 0xFF;
      sizes[blockIdx.x] = (int32_t)(at + 4);
    }
    __syncthreads();
    const int nbytes = sizes[blockIdx.x];
    for (int w = tid; w < (nbytes + 3) / 4; w += blockDim.x) reinterpret_cast<uint32_t *>(slot)[w] = bits[w];
  }
  const int seg = ((block / kLzThreads) + 3) & ~3;
  if (ADLER) {
    const uint2 sums = block_adler(staged, len, seg, sh.red);
    if (tid == 0) *reinterpret_cast<uint2 *>(slot + block + kSumsAt) = sums;
  } else {
    const uint32_t crc = block_crc(staged, len, seg, sh.crc_table, sh.x2n, sh.red);
    if (tid == 0) atomicXor(crc_out, crc_shift(crc, n - start - len, sh.x2n));
  }
}

// CRC-32 only: one CTA per block, as in deflate_block_kernel
__global__ void __launch_bounds__(kDefThreads)
crc_block_kernel(const uint8_t *__restrict__ in, int64_t n, int block, uint32_t *__restrict__ crc_out) {
  extern __shared__ __align__(16) uint32_t dyn[];
  __shared__ uint32_t table[256], x2n[32], red[kDefThreads / 32];
  const int64_t start = (int64_t)blockIdx.x * block;
  const int len = (int)(n - start < block ? n - start : (int64_t)block);
  stage_block(in + start, len, dyn);
  crc_tables(table, x2n);
  __syncthreads();
  const uint32_t crc = block_crc(dyn, len, block / kDefThreads, table, x2n, red);
  if (threadIdx.x == 0) atomicXor(crc_out, crc_shift(crc, n - start - len, x2n));
}

// block b's bytes from its slot to out + offsets[b]; CTA 0 also stores the total
__global__ void __launch_bounds__(kDefThreads)
deflate_compact_kernel(const uint8_t *__restrict__ slots, const int32_t *__restrict__ sizes,
                       const int64_t *__restrict__ offsets, int64_t nblocks, int block, uint8_t *__restrict__ out,
                       int64_t *__restrict__ out_bytes) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *out_bytes = offsets[nblocks];
  for (int64_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
    const int size = sizes[b];
    const uint8_t *src = slots + b * (block + kSlotPad);
    uint8_t *dst = out + offsets[b];
    for (int i = threadIdx.x; i < size; i += blockDim.x) dst[i] = src[i];
  }
}

// segment s = blocks [s*seg_blocks, (s+1)*seg_blocks): seg_offsets[s] = offsets of its first block (the total for
// s = nseg), seg_adler[s] = Adler-32 of its input, its blocks' sums combined as zlib's adler32_combine: for A || B,
// x = x_A + x_B and y = y_A + |B| x_A + y_B.  Blocks past the input length n are empty.
__global__ void __launch_bounds__(kDefThreads)
adler_segments_kernel(const uint8_t *__restrict__ slots, const int64_t *__restrict__ offsets,
                      const int64_t *__restrict__ count, int64_t scale, int64_t max_bytes, int block, int64_t nb,
                      int64_t seg_blocks, int64_t nseg, int64_t *__restrict__ seg_offsets,
                      uint32_t *__restrict__ seg_adler) {
  const int64_t n = count ? min(max_bytes, count[0] * scale) : max_bytes;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s <= nseg; s += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b0 = min(s * seg_blocks, nb);
    seg_offsets[s] = offsets[b0];
    if (s == nseg) continue;
    uint64_t x = 0, y = 0, total = 0;
    for (int64_t b = b0; b < min(nb, b0 + seg_blocks) && b * block < n; ++b) {
      const int64_t len = min((int64_t)block, n - b * block);
      const uint2 sums = *reinterpret_cast<const uint2 *>(slots + b * (block + kSlotPad) + block + kSumsAt);
      y = (y + (uint64_t)len * x + sums.y) % kAdlerMod;
      x = (x + sums.x) % kAdlerMod;
      total += (uint64_t)len;
    }
    seg_adler[s] = (uint32_t)((1 + x) % kAdlerMod) | ((uint32_t)((total + y) % kAdlerMod) << 16);
  }
}

inline int64_t n_blocks(int64_t n, int32_t block) { return (n + block - 1) / block; }
inline int64_t align16(int64_t v) { return (v + 15) / 16 * 16; }
inline size_t staged_bytes(int32_t block) { return (size_t)(block / 4 + block / 128 + 4) * 4; }

}  // namespace
}  // namespace pst

using namespace pst;

extern "C" int64_t pst_deflate_bound(int64_t n, int32_t block) {
  if (n < 0 || block <= 0) return -1;
  return n + kStoredOverhead * n_blocks(n, block);
}

extern "C" int64_t pst_deflate_workspace_bytes(int64_t n, int32_t block) {
  if (n < 0 || block <= 0) return -1;
  const int64_t nb = n_blocks(n, block);
  return align16(4 * nb) + align16(8 * (nb + 1)) + nb * (block + kSlotPad);
}

extern "C" int64_t pst_deflate_lz_workspace_bytes(int64_t n, int32_t block) {
  if (n < 0 || block <= 0) return -1;
  return pst_deflate_workspace_bytes(n, block) + n_blocks(n, block) * 2 * block;
}

// the dynamic shared memory limit of one kernel, raised once per device and thread
template <bool LZ, bool ADLER, typename K>
static void allow_smem(K kernel, size_t bytes) {
  static thread_local int configured_dev = -1;
  int dev = 0;
  cudaGetDevice(&dev);
  if (configured_dev != dev) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    configured_dev = dev;
  }
}

// pst_deflate_blocks (lz false) and pst_deflate_lz_blocks (lz true): the block kernel, the scan of the
// block sizes and the compaction; the LZ workspace has the token slots after the output slots.  With seg_offsets
// (pst_deflate_segments, pst_deflate_lz_segments) the block kernel takes Adler sums instead of the CRC, and
// adler_segments_kernel writes the segments' offsets and Adler-32s after the scan.
static int deflate_launch(const char *fn, bool lz, const void *in, const int64_t *count, int64_t scale,
                          int64_t max_bytes, int32_t block, void *out, int64_t *out_bytes, uint32_t *crc, void *work,
                          int64_t work_bytes, void *stream, int64_t seg_blocks = 0, int64_t *seg_offsets = nullptr,
                          uint32_t *seg_adler = nullptr) {
  const bool adler = seg_offsets != nullptr;
  PST_REQUIRE(max_bytes >= 0 && scale >= 0, fn, "need max_bytes, scale >= 0");
  PST_REQUIRE(block >= 1024 && block <= kMaxBlock && block % 1024 == 0, fn,
              "block must be a multiple of 1024 between 1024 and 32768");
  PST_REQUIRE(out_bytes && (adler ? seg_adler != nullptr : crc != nullptr), fn, "null pointer");
  PST_REQUIRE(!adler || seg_blocks >= 1, fn, "need seg_blocks >= 1");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t nb = n_blocks(max_bytes, block);
  if (!adler && cudaMemsetAsync(crc, 0, sizeof(uint32_t), st) != cudaSuccess) return check_launch(fn);
  if (nb == 0) {
    if (cudaMemsetAsync(out_bytes, 0, sizeof(int64_t), st) != cudaSuccess) return check_launch(fn);
    if (adler && cudaMemsetAsync(seg_offsets, 0, sizeof(int64_t), st) != cudaSuccess) return check_launch(fn);
    return 0;
  }
  PST_REQUIRE(in && out && work, fn, "null pointer");
  if (lz)
    PST_REQUIRE(work_bytes >= pst_deflate_lz_workspace_bytes(max_bytes, block), fn,
                "workspace smaller than pst_deflate_lz_workspace_bytes");
  else
    PST_REQUIRE(work_bytes >= pst_deflate_workspace_bytes(max_bytes, block), fn,
                "workspace smaller than pst_deflate_workspace_bytes");
  PST_REQUIRE(nb < (1ll << 31), fn, "too many blocks");
  int32_t *sizes = reinterpret_cast<int32_t *>(work);
  int64_t *offsets = reinterpret_cast<int64_t *>(static_cast<uint8_t *>(work) + align16(4 * nb));
  uint8_t *slots = static_cast<uint8_t *>(work) + align16(4 * nb) + align16(8 * (nb + 1));
  const uint8_t *src = static_cast<const uint8_t *>(in);
  if (lz) {
    const size_t most = staged_bytes(kMaxBlock) + 2 * kMaxBlock + lz_scratch_bytes(kMaxBlock);
    uint16_t *tokens = reinterpret_cast<uint16_t *>(slots + nb * (block + kSlotPad));
    const size_t smem = staged_bytes(block) + 2 * (size_t)block + lz_scratch_bytes(block);
    if (adler) {
      allow_smem<true, true>(deflate_lz_block_kernel<true>, most);
      deflate_lz_block_kernel<true><<<(unsigned)nb, kLzThreads, smem, st>>>(src, count, scale, max_bytes, block, slots,
                                                                            sizes, nullptr, tokens);
    } else {
      allow_smem<true, false>(deflate_lz_block_kernel<false>, most);
      deflate_lz_block_kernel<false><<<(unsigned)nb, kLzThreads, smem, st>>>(src, count, scale, max_bytes, block, slots,
                                                                             sizes, crc, tokens);
    }
  } else {
    const size_t most = staged_bytes(kMaxBlock) + (kMaxBlock / 4 + 8) * 4;
    const size_t smem = staged_bytes(block) + (size_t)(block / 4 + 8) * 4;
    if (adler) {
      allow_smem<false, true>(deflate_block_kernel<true>, most);
      deflate_block_kernel<true><<<(unsigned)nb, kDefThreads, smem, st>>>(src, count, scale, max_bytes, block, slots,
                                                                          sizes, nullptr);
    } else {
      allow_smem<false, false>(deflate_block_kernel<false>, most);
      deflate_block_kernel<false><<<(unsigned)nb, kDefThreads, smem, st>>>(src, count, scale, max_bytes, block, slots,
                                                                           sizes, crc);
    }
  }
  int rc = check_launch(fn);
  if (rc) return rc;
  rc = pst_csr_row_offsets(sizes, nb, offsets, stream);            // exclusive scan of the sizes
  if (rc) return rc;
  const unsigned grid = (unsigned)std::min<int64_t>(nb, (int64_t)num_sm() * 8);
  deflate_compact_kernel<<<grid, kDefThreads, 0, st>>>(slots, sizes, offsets, nb, block,
                                                       static_cast<uint8_t *>(out), out_bytes);
  if (adler) {
    const int64_t nseg = (nb + seg_blocks - 1) / seg_blocks;
    const unsigned sgrid = (unsigned)std::min<int64_t>((nseg + kDefThreads) / kDefThreads, (int64_t)num_sm() * 8);
    adler_segments_kernel<<<sgrid, kDefThreads, 0, st>>>(slots, offsets, count, scale, max_bytes, block, nb, seg_blocks,
                                                         nseg, seg_offsets, seg_adler);
  }
  return check_launch(fn);
}

extern "C" int pst_deflate_blocks(const void *in, const int64_t *count, int64_t scale, int64_t max_bytes,
                                  int32_t block, void *out, int64_t *out_bytes, uint32_t *crc, void *work,
                                  int64_t work_bytes, void *stream) {
  return deflate_launch("pst_deflate_blocks", false, in, count, scale, max_bytes, block, out, out_bytes, crc, work,
                        work_bytes, stream);
}

extern "C" int pst_deflate_lz_blocks(const void *in, const int64_t *count, int64_t scale, int64_t max_bytes,
                                     int32_t block, void *out, int64_t *out_bytes, uint32_t *crc, void *work,
                                     int64_t work_bytes, void *stream) {
  return deflate_launch("pst_deflate_lz_blocks", true, in, count, scale, max_bytes, block, out, out_bytes, crc,
                        work, work_bytes, stream);
}

extern "C" int pst_deflate_segments(const void *in, const int64_t *count, int64_t scale, int64_t max_bytes,
                                    int32_t block, int64_t seg_blocks, void *out, int64_t *out_bytes,
                                    int64_t *seg_offsets, uint32_t *seg_adler, void *work, int64_t work_bytes,
                                    void *stream) {
  const char *fn = "pst_deflate_segments";
  PST_REQUIRE(seg_offsets, fn, "null pointer");
  return deflate_launch(fn, false, in, count, scale, max_bytes, block, out, out_bytes, nullptr, work, work_bytes,
                        stream, seg_blocks, seg_offsets, seg_adler);
}

extern "C" int pst_deflate_lz_segments(const void *in, const int64_t *count, int64_t scale, int64_t max_bytes,
                                       int32_t block, int64_t seg_blocks, void *out, int64_t *out_bytes,
                                       int64_t *seg_offsets, uint32_t *seg_adler, void *work, int64_t work_bytes,
                                       void *stream) {
  const char *fn = "pst_deflate_lz_segments";
  PST_REQUIRE(seg_offsets, fn, "null pointer");
  return deflate_launch(fn, true, in, count, scale, max_bytes, block, out, out_bytes, nullptr, work, work_bytes,
                        stream, seg_blocks, seg_offsets, seg_adler);
}

extern "C" int pst_crc32(const void *in, int64_t n, uint32_t *crc, void *stream) {
  const char *fn = "pst_crc32";
  PST_REQUIRE(n >= 0, fn, "need n >= 0");
  PST_REQUIRE(crc && (n == 0 || in), fn, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if (cudaMemsetAsync(crc, 0, sizeof(uint32_t), st) != cudaSuccess) return check_launch(fn);
  if (n == 0) return 0;
  const int block = kMaxBlock;
  crc_block_kernel<<<(unsigned)n_blocks(n, block), kDefThreads, staged_bytes(block), st>>>(
      static_cast<const uint8_t *>(in), n, block, crc);
  return check_launch(fn);
}
