// Streamed exact temporal median: a clip added chunk by chunk, in any chunking and any order, gives the bytes of
// vu_temporal_median_u8 on the whole clip (np.median(stack, 0).astype(uint8)).
//
// State: one histogram of 256 16-bit counters per byte of the frame (512 B per element, independent of the clip
// length), laid out in tiles of MA_TILE = 128 elements.  A tile is 64 KB: [256 bins][64 words], each 32-bit word two
// counters.  Element e of a tile sits in column ((e >> 1) & 1) * 32 + (e >> 2), field e & 1: lane l of a warp, which
// loads bytes 4l..4l+3 of a frame, owns columns l and 32 + l, so the 32 lanes of a warp always update 32 different banks
// (and never the same word), whatever bins they hit.  A field never carries into its neighbour because the caller keeps
// the total at most 65535 frames.
//
// Add: one CTA per tile.  It reads the tile's histograms into shared memory (zeroes them when n_before == 0), counts
// the k frames - warp w takes frames w, w + 8, ..., a lane 4 elements per frame, MA_U frames in flight - with shared
// atomics, and writes the tile back.  Traffic: k * m bytes of frames plus 1024 * m bytes of state.
// Finish: one thread per column reads its 256 words once and returns the order statistics (n - 1) / 2 and n / 2 of
// both elements; even n gives (lo + hi) >> 1.
#include "vu_common.cuh"

namespace vu {
namespace {

constexpr int MA_TILE = 128;                   // elements per tile
constexpr int MA_COLS = MA_TILE / 2;           // words per bin row
constexpr int MA_WORDS = 256 * MA_COLS;        // words per tile (64 KB)
constexpr int MA_THREADS = 256;
constexpr int MA_WARPS = MA_THREADS / 32;
constexpr int MA_U = 8;                        // frames per lane in flight
constexpr int MA_V = MA_WORDS / 4 / MA_THREADS;   // 16-byte state vectors per thread

__global__ void __launch_bounds__(MA_THREADS, 3) median_accum_add_kernel(uint4* __restrict__ state, const uint8_t* __restrict__ frames, int k,
                                                                         long long m, int read_state, int aligned) {
  extern __shared__ __align__(16) unsigned hist[];   // [256][MA_COLS]
  uint4* sh = reinterpret_cast<uint4*>(hist);
  uint4* st = state + (long long)blockIdx.x * (MA_WORDS / 4);
  if (read_state) {
#pragma unroll 2
    for (int h = 0; h < MA_V; h += MA_V / 2) {
      uint4 v[MA_V / 2];
#pragma unroll
      for (int i = 0; i < MA_V / 2; ++i) v[i] = ldg_stream16(st + (h + i) * MA_THREADS + threadIdx.x);
#pragma unroll
      for (int i = 0; i < MA_V / 2; ++i) sh[(h + i) * MA_THREADS + threadIdx.x] = v[i];
    }
  } else {
#pragma unroll
    for (int i = 0; i < MA_V; ++i) sh[i * MA_THREADS + threadIdx.x] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long e0 = (long long)blockIdx.x * MA_TILE + 4 * lane;   // the lane's first element
  unsigned* col = hist + lane;
  if (aligned && (long long)(blockIdx.x + 1) * MA_TILE <= m) {
    // whole tile of 4-byte aligned frame rows: one coalesced 128-byte line per warp and frame
    const uint8_t* p = frames + e0;
    for (int f = warp; f < k; f += MA_U * MA_WARPS) {
      unsigned w[MA_U];
#pragma unroll
      for (int u = 0; u < MA_U; ++u) {
        const int ff = f + u * MA_WARPS;
        w[u] = ff < k ? __ldg(reinterpret_cast<const unsigned*>(p + (long long)ff * m)) : 0u;
      }
#pragma unroll
      for (int u = 0; u < MA_U; ++u) {
        if (f + u * MA_WARPS < k) {
#pragma unroll
          for (int q = 0; q < 4; ++q) atomicAdd(col + ((w[u] >> (8 * q)) & 255u) * MA_COLS + (q >> 1) * 32, 1u << (16 * (q & 1)));
        }
      }
    }
  } else {
    // the last, partial tile, or frames that are not 4-byte aligned: byte loads, elements past m are not counted
    for (int f = warp; f < k; f += MA_WARPS) {
      const uint8_t* p = frames + (long long)f * m + e0;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (e0 + q < m) atomicAdd(col + (unsigned)__ldg(p + q) * MA_COLS + (q >> 1) * 32, 1u << (16 * (q & 1)));
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < MA_V; ++i) st[i * MA_THREADS + threadIdx.x] = sh[i * MA_THREADS + threadIdx.x];
}

__global__ void __launch_bounds__(MA_COLS) median_accum_finish_kernel(const unsigned* __restrict__ state, long long m, int n,
                                                                      uint8_t* __restrict__ out) {
  const int c = threadIdx.x;
  const unsigned* col = state + (long long)blockIdx.x * MA_WORDS + c;
  const unsigned klo = (unsigned)(n - 1) >> 1, khi = (unsigned)n >> 1;   // 0-based ranks of the two middle values
  // value of order statistic r = number of bins whose running count is still <= r
  unsigned c0 = 0, c1 = 0, lo0 = 0, hi0 = 0, lo1 = 0, hi1 = 0;
#pragma unroll 16
  for (int b = 0; b < 256; ++b) {
    const unsigned w = __ldg(col + b * MA_COLS);
    c0 += w & 0xFFFFu;
    c1 += w >> 16;
    lo0 += c0 <= klo;
    hi0 += c0 <= khi;
    lo1 += c1 <= klo;
    hi1 += c1 <= khi;
  }
  const long long e = (long long)blockIdx.x * MA_TILE + 4 * (c & 31) + 2 * (c >> 5);
  if (e < m) out[e] = (uint8_t)((lo0 + hi0) >> 1);
  if (e + 1 < m) out[e + 1] = (uint8_t)((lo1 + hi1) >> 1);
}

int64_t ma_tiles(int64_t m) { return (m + MA_TILE - 1) / MA_TILE; }

}  // namespace
}  // namespace vu

using namespace vu;

extern "C" size_t vu_median_accum_bytes(int64_t m) { return m > 0 ? (size_t)ma_tiles(m) * MA_WORDS * 4 : 0; }

extern "C" int vu_median_accum_reset(void* state, int64_t m, vu_stream_t stream) {
  VU_REQUIRE(state && m >= 0);
  if (m == 0) return VU_OK;
  return record_cuda(cudaMemsetAsync(state, 0, vu_median_accum_bytes(m), S(stream)));
}

extern "C" int vu_median_accum_add_u8(void* state, int64_t m, const uint8_t* frames, int k, int n_before, vu_stream_t stream) {
  VU_REQUIRE(state && frames && m >= 0 && k >= 1 && n_before >= 0 && (int64_t)n_before + k <= 65535);
  VU_REQUIRE((reinterpret_cast<uintptr_t>(state) & 15) == 0);
  if (m == 0) return VU_OK;
  const int64_t tiles = ma_tiles(m);
  if (tiles > 0x7fffffff) return VU_ERR_UNSUPPORTED;
  // the shared-memory limit is a per-device attribute: set it once on every device that runs the add
  int dev = 0;
  int e = record_cuda(cudaGetDevice(&dev));
  if (e) return e;
  static uint64_t configured = 0;   // bit d: device d done (devices >= 64 set it on every call)
  if (dev >= 64 || !((configured >> dev) & 1u)) {
    e = record_cuda(cudaFuncSetAttribute(median_accum_add_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MA_WORDS * 4));
    if (e) return e;
    if (dev < 64) configured |= 1ull << dev;
  }
  // n_before == 0 skips reading the state - except in an add captured into a CUDA graph, whose replays must accumulate
  // whatever n_before was at capture
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  e = record_cuda(cudaStreamIsCapturing(S(stream), &cap));
  if (e) return e;
  const int read_state = n_before > 0 || cap != cudaStreamCaptureStatusNone;
  const int aligned = (reinterpret_cast<uintptr_t>(frames) % 4 == 0) && (m % 4 == 0);
  median_accum_add_kernel<<<(unsigned)tiles, MA_THREADS, MA_WORDS * 4, S(stream)>>>(static_cast<uint4*>(state), frames, k, m, read_state,
                                                                                   aligned);
  VU_RETURN_LAUNCH();
}

extern "C" int vu_median_accum_finish_u8(const void* state, int64_t m, int n, uint8_t* out, vu_stream_t stream) {
  VU_REQUIRE(state && out && m >= 0 && n >= 1 && n <= 65535);
  if (m == 0) return VU_OK;
  const int64_t tiles = ma_tiles(m);
  if (tiles > 0x7fffffff) return VU_ERR_UNSUPPORTED;
  median_accum_finish_kernel<<<(unsigned)tiles, MA_COLS, 0, S(stream)>>>(static_cast<const unsigned*>(state), m, n, out);
  VU_RETURN_LAUNCH();
}
