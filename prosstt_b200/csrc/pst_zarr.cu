// The fixed chunk grid of a Zarr array (out="zarr") cut across the engine's cell chunks on the device.
//
// An array of the store is written in chunks of C elements, but an engine chunk delivers any number of new values
// (its nonzeros, or its cells' row ends).  Each array keeps a carry: the tail of the values so far that does not
// fill a Zarr chunk yet, fewer than C elements.  pst_zarr_cut writes `carry || new values` into a segment buffer,
// whose whole chunks are what the engine chunk delivers, and records where the new carry lies in it.  The carry's
// place and length live in device memory, so the cut of chunk i needs no host read of chunk i - 1.
#include <algorithm>
#include "pst_common.cuh"

namespace pst {
namespace {

// seg = prev[prev_state[0] ..][: prev_state[1]] || src[: n_src], zero-padded to whole chunks when `final`; all
// lengths in 4-byte words.  Thread 0 writes the new state {offset, length} of the carry and the whole chunks.
__global__ void __launch_bounds__(256)
zarr_cut_kernel(const uint32_t *__restrict__ prev, const int64_t *__restrict__ prev_state,
                const uint32_t *__restrict__ src, const int64_t *__restrict__ count, int64_t scale, int64_t max_src,
                int64_t chunk_bytes, int final, uint32_t *__restrict__ seg, int64_t *__restrict__ state,
                int64_t *__restrict__ nchunks) {
  const int64_t carry_at = prev_state[0] >> 2, carry = prev_state[1] >> 2;
  const int64_t n_src = (count ? min(max_src, count[0] * scale) : max_src) >> 2;
  const int64_t total = carry + n_src, chunk = chunk_bytes >> 2;
  const int64_t whole = final ? (total + chunk - 1) / chunk : total / chunk;
  const int64_t end = final ? whole * chunk : total;
  for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < end; w += (int64_t)gridDim.x * blockDim.x)
    seg[w] = w < carry ? prev[carry_at + w] : w < total ? __ldcs(src + (w - carry)) : 0u;
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    state[0] = whole * chunk_bytes;
    state[1] = (end - whole * chunk) * 4;
    *nchunks = whole;
  }
}

}  // namespace
}  // namespace pst

using namespace pst;

extern "C" int64_t pst_zarr_seg_bytes(int64_t max_src, int64_t chunk_bytes) {
  if (max_src < 0 || chunk_bytes <= 0) return -1;
  return (max_src / chunk_bytes + 2) * chunk_bytes;
}

extern "C" int pst_zarr_cut(const void *prev, const int64_t *prev_state, const void *src, const int64_t *count,
                            int64_t scale, int64_t max_src, int64_t chunk_bytes, int32_t final, void *seg,
                            int64_t seg_bytes, int64_t *state, int64_t *nchunks, void *stream) {
  const char *fn = "pst_zarr_cut";
  PST_REQUIRE(max_src >= 0 && scale >= 0 && chunk_bytes > 0, fn, "need max_src, scale >= 0 and chunk_bytes > 0");
  PST_REQUIRE(max_src % 4 == 0 && scale % 4 == 0 && chunk_bytes % 4 == 0, fn,
              "max_src, scale and chunk_bytes must be multiples of 4");
  PST_REQUIRE(seg_bytes >= pst_zarr_seg_bytes(max_src, chunk_bytes), fn, "seg smaller than pst_zarr_seg_bytes");
  PST_REQUIRE(prev && prev_state && seg && state && nchunks && (max_src == 0 || src), fn, "null pointer");
  PST_REQUIRE(prev != seg && prev_state != state, fn, "prev and seg must be distinct buffers");
  PST_REQUIRE(((uintptr_t)prev | (uintptr_t)src | (uintptr_t)seg) % 4 == 0, fn, "buffers must be 4-byte aligned");
  const int64_t words = (max_src + 2 * chunk_bytes) / 4;
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((words + 255) / 256, (int64_t)num_sm() * 8));
  zarr_cut_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      static_cast<const uint32_t *>(prev), prev_state, static_cast<const uint32_t *>(src), count, scale, max_src,
      chunk_bytes, final ? 1 : 0, static_cast<uint32_t *>(seg), state, nchunks);
  return check_launch(fn);
}
