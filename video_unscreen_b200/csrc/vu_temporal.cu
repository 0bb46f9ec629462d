// Temporal background estimators (SURVEY.md section 8 rows a22, a23).
//
// vu_temporal_median_u8: exact per-element median over n frames.
//
// n <= 608: register-resident bit-wise binary search on the median value.  A
// warp owns a 64-byte (SPLIT=2) or 32-byte (SPLIT=4) segment of every frame;
// each lane loads its 4 bytes of up to 152 frames straight into registers (one
// coalesced LDG.32 per frame, all of them in flight at once), transposes 4x4
// byte blocks with PRMT so that a register holds 4 frames of ONE element, and
// then minimises the convex S(m) = sum_f |x_f - m| with a Fibonacci search: S
// costs one VABSDIFF4-with-accumulate per 4 frames per probe, 12 probes find
// the minimiser among 0..255 (see sad_search).  Frames are split over half /
// quarter warps and the partial sums meet in a shuffle.  Unused slots are
// padded with 0 on one side and 255 on the other, which keeps the middle order
// statistics where they are.  That is the direct kernel; on 16-byte aligned
// clips the TMA tile kernels run the same search on tiles staged in shared
// memory and read them byte-transposed with ldmatrix, so their registers hold
// 4 frames of one element without PRMT (vu_median_sad.cuh).
//
// n > 608: streaming 256-bin histograms in shared memory.  One warp owns a segment of
// 32*PX consecutive bytes of every frame; lane l owns PX of them and a private
// column of 256 packed counters laid out so that its bank is always `lane`
// (bin stride = WARPS*128 bytes): every increment is a conflict-free shared
// atomic, whatever the pixel values are.  Warps never synchronise with each
// other, so one warp's histogram scan overlaps the other warps' streaming.
// Two 16-bit counters per word (PX = 2, 64-byte segments), n <= 65535.
// The median is read back with a two-level scan (16 coarse groups, then 16
// bins); even n returns (lo + hi) >> 1 like np.median(...).astype(uint8).
//
// vu_masked_temporal_mean: tools/unscreen/bg_offline.py:106-125 as integer
// sums and counts per pixel, one float64 divide at the end.  The
// vu_masked_mean_accum_* calls keep those sums and counts in a state across
// chunks of the clip (the fused-dilation kernel, templated on ACCUM) and share
// the closed form of the end (mean_always / mean_byte).
#include <cstdlib>

#include "vu_common.cuh"
#include "vu_median_sad.cuh"

namespace vu {
namespace {

constexpr int WARPS = 7;
constexpr int MTHREADS = WARPS * 32;
constexpr int BIN_STRIDE = WARPS * 128;  // bytes between bins
constexpr int HIST_BYTES = 256 * BIN_STRIDE;

struct PolU16x2 {
  static constexpr int PX = 2;
  __device__ static __forceinline__ void add(unsigned char* base, unsigned w) {
#pragma unroll
    for (int j = 0; j < 2; ++j) atomicAdd(reinterpret_cast<unsigned*>(base + ((w >> (8 * j)) & 0xFFu) * BIN_STRIDE), 1u << (16 * j));
  }
  __device__ static __forceinline__ void unpack(unsigned w, unsigned* c) { c[0] = w & 0xFFFFu; c[1] = w >> 16; }
};

template <int PX>
__device__ __forceinline__ unsigned load_px(const uint8_t* p) {
  if (PX == 4) return __ldg(reinterpret_cast<const unsigned*>(p));
  return __ldg(reinterpret_cast<const unsigned short*>(p));
}

template <class P, int U>
__global__ void __launch_bounds__(MTHREADS, 1) median_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ out, int n, long long m,
                                                             int nseg, const uint8_t* __restrict__ flags) {
  extern __shared__ __align__(128) unsigned char smem[];
  constexpr int PX = P::PX;
  constexpr int SEG = 32 * PX;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned char* base = smem + warp * 128 + lane * 4;
  const unsigned klo = (unsigned)(n - 1) >> 1, khi = (unsigned)n >> 1;
  const int nb = n / U;
  // fix-up mode (flags != nullptr): only the segments the refine pass could not decide.  A warp scans 32 flags per
  // load and walks the set bits; without flags every segment of the warp's stride is processed.
  const int wid = blockIdx.x * WARPS + warp, nw = gridDim.x * WARPS;
  const int iters = flags ? (nseg + 32 * nw - 1) / (32 * nw) * 32 : (nseg + nw - 1) / nw;
  unsigned pending = 0;
  for (int it = 0; it < iters; ++it) {
    int seg;
    if (flags) {
      if ((it & 31) == 0) {
        const int s = ((it >> 5) * nw + wid) * 32 + lane;
        pending = __ballot_sync(0xffffffffu, s < nseg && flags[s] != 0);
      }
      if (pending == 0) { it |= 31; continue; }
      const int b = __ffs(pending) - 1;
      pending &= pending - 1;
      seg = ((it >> 5) * nw + wid) * 32 + b;
    } else {
      seg = it * nw + wid;
      if (seg >= nseg) break;
    }
#pragma unroll 8
    for (int b = 0; b < 256; ++b) *reinterpret_cast<unsigned*>(base + b * BIN_STRIDE) = 0u;
    __syncwarp();
    {
      const uint8_t* p = frames + (long long)seg * SEG + lane * PX;
      unsigned ra[U], rb[U];
      auto load = [&](unsigned(&r)[U]) {
#pragma unroll
        for (int u = 0; u < U; ++u) { r[u] = load_px<PX>(p); p += m; }
      };
      auto proc = [&](unsigned(&r)[U]) {
#pragma unroll
        for (int u = 0; u < U; ++u) P::add(base, r[u]);
      };
      if (nb > 0) load(ra);
      for (int i = 0; i < nb; i += 2) {
        if (i + 1 < nb) load(rb);
        proc(ra);
        if (i + 1 < nb) {
          if (i + 2 < nb) load(ra);
          proc(rb);
        }
      }
      for (int f = nb * U; f < n; ++f) { P::add(base, load_px<PX>(p)); p += m; }
    }
    __syncwarp();
    // two-level scan
    unsigned cum[PX], gsel[PX][2], before[PX][2];
#pragma unroll
    for (int j = 0; j < PX; ++j) { cum[j] = 0; gsel[j][0] = gsel[j][1] = 0; before[j][0] = before[j][1] = 0; }
#pragma unroll 1
    for (int g = 0; g < 16; ++g) {
      unsigned c[PX];
#pragma unroll
      for (int j = 0; j < PX; ++j) c[j] = 0;
#pragma unroll
      for (int b = 0; b < 16; ++b) {
        unsigned t[PX];
        P::unpack(*reinterpret_cast<unsigned*>(base + (g * 16 + b) * BIN_STRIDE), t);
#pragma unroll
        for (int j = 0; j < PX; ++j) c[j] += t[j];
      }
#pragma unroll
      for (int j = 0; j < PX; ++j) {
        const unsigned nc = cum[j] + c[j];
        if (nc <= klo) { gsel[j][0] = g + 1; before[j][0] = nc; }
        if (nc <= khi) { gsel[j][1] = g + 1; before[j][1] = nc; }
        cum[j] = nc;
      }
    }
    unsigned res = 0;
#pragma unroll
    for (int j = 0; j < PX; ++j) {
      unsigned med[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const unsigned k = q ? khi : klo;
        if (q == 1 && khi == klo) { med[1] = med[0]; continue; }
        const unsigned g = min(gsel[j][q], 15u);
        unsigned v = g * 16, c2 = before[j][q];
#pragma unroll 4
        for (int b = 0; b < 16; ++b) {
          unsigned t[PX];
          P::unpack(*reinterpret_cast<unsigned*>(base + (g * 16 + b) * BIN_STRIDE), t);
          c2 += t[j];
          if (c2 <= k) v = g * 16 + b + 1;
        }
        med[q] = min(v, 255u);
      }
      res |= ((med[0] + med[1]) >> 1) << (8 * j);
    }
    uint8_t* dst = out + (long long)seg * SEG;
    if (PX == 4) reinterpret_cast<unsigned*>(dst)[lane] = res;
    else reinterpret_cast<unsigned short*>(dst)[lane] = (unsigned short)res;
    __syncwarp();
  }
}

// ---- register-resident SAD search: vu_median_sad.cuh ------------------------
template <int SPLIT, int G, int GFULL, int SS, int CTAS>
int launch_median_sad(const uint8_t* frames, int n, int64_t m, int64_t nseg, uint8_t* out, vu_stream_t stream) {
  msad::median_sad_kernel<SPLIT, G, GFULL, SS, CTAS><<<(unsigned)((nseg + 3) / 4), 128, 0, S(stream)>>>(frames, out, n, m, (int)nseg, 0u);
  note_launch();
  return record_cuda(cudaGetLastError());
}

// TMA tile kernels: the clip as a 3-D tensor [n][m / 128][32] of 32-bit words, boxes of {TILE bytes, BOX_ROWS frames}
// with the 128-byte swizzle (the layout is described in vu_median_sad.cuh).  Tiles only cover whole 128-byte units.
using tma::encode_tiled_fn;
using tma::EncodeTiledFn;

// Does the whole tiles (TMA_WARPS segments of 16C bytes each) of the first nseg segments and sets *done to the number
// of segments they cover; the rest is the caller's.  pitch = bytes between consecutive frames of the (possibly
// subsampled) clip.  TRACE kernels record their timeline into `trace` (see vu_median_sad.cuh).
template <int C, int G, int SS, int TMA_WARPS, int TMA_CTAS, int PIPES = 1, bool TRACE = false>
int launch_median_sad_tma(const uint8_t* frames, int n, int64_t m, int64_t nseg, uint8_t* out, vu_stream_t stream, int64_t* done, int64_t pitch = 0,
                          unsigned long long* trace = nullptr) {
  using T = msad::TmaTile<C, G, TMA_WARPS>;
  const int64_t ntiles = nseg / TMA_WARPS;
  *done = 0;
  if (ntiles == 0) return VU_OK;
  if (pitch == 0) pitch = m;
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return VU_ERR_UNSUPPORTED;
  CUtensorMap tmap;
  const cuuint64_t dims[3] = {32, (cuuint64_t)(m / 128), (cuuint64_t)n};
  const cuuint64_t strides[2] = {128, (cuuint64_t)pitch};
  const cuuint32_t box[3] = {32, (cuuint32_t)T::COLS, (cuuint32_t)T::BOX_ROWS};
  const cuuint32_t estr[3] = {1, 1, 1};
  if (enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(frames), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return VU_ERR_UNSUPPORTED;
  auto kernel = msad::median_sad_tma_kernel<C, G, SS, TMA_WARPS, TMA_CTAS, PIPES, TRACE>;
  constexpr int smem = T::smem(PIPES);
  static bool configured = false;
  if (!configured) {
    int e = record_cuda(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (e) return e;
    configured = true;
  }
  const int64_t cap = (int64_t)device_sms() * TMA_CTAS, need = (ntiles + PIPES - 1) / PIPES;
  const int grid = (int)(need < cap ? need : cap);
  kernel<<<grid, PIPES * TMA_WARPS * 32, smem, S(stream)>>>(tmap, out, n, (int)ntiles, trace);
  note_launch();
  const int e = record_cuda(cudaGetLastError());
  if (e == VU_OK) *done = ntiles * TMA_WARPS;
  return e;
}

// elements that do not fill a whole segment (and unaligned inputs): one CTA
// per element, 256-bin shared histogram
__global__ void __launch_bounds__(256) median_tail_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ out, int n, long long m,
                                                          long long first) {
  __shared__ unsigned hist[256];
  const long long e = first + blockIdx.x;
  hist[threadIdx.x] = 0;
  __syncthreads();
  for (int f = threadIdx.x; f < n; f += 256) atomicAdd(&hist[__ldg(frames + (long long)f * m + e)], 1u);
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned klo = (unsigned)(n - 1) >> 1, khi = (unsigned)n >> 1;
    unsigned cum = 0, lo = 255, hi = 255;
    bool flo = false, fhi = false;
    for (int b = 0; b < 256; ++b) {
      cum += hist[b];
      if (!flo && cum > klo) { lo = b; flo = true; }
      if (!fhi && cum > khi) { hi = b; fhi = true; }
    }
    out[e] = (uint8_t)((lo + hi) >> 1);
  }
}

// ---- masked temporal mean -------------------------------------------------
// bg_offline.py:121-125 for one pixel, shared by the resident kernels and the accumulator's finish:
// mask_always = cnt <= min_count; bg = trunc(clip(sum / max(cnt, 1), 0, 255)), one float64 divide rounded once; 0
// where always masked
__device__ __forceinline__ bool mean_always(unsigned cnt, int min_count) { return cnt <= (unsigned)min_count; }
__device__ __forceinline__ unsigned mean_byte(unsigned sum, unsigned cnt, bool always) {
  const double q = fmin(fmax(__ddiv_rn((double)sum, (double)(cnt ? cnt : 1u)), 0.0), 255.0);
  return always ? 0u : (unsigned)(int)q;
}

constexpr int TT = 256;
__global__ void __launch_bounds__(TT) masked_mean_kernel(const uint8_t* __restrict__ frames, const uint8_t* __restrict__ masks, int n,
                                                         int64_t ngroups, int64_t npix, int min_count, uint8_t* __restrict__ bg_out,
                                                         uint8_t* __restrict__ always_out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
    unsigned sum[12], cnt[4];
#pragma unroll
    for (int i = 0; i < 12; ++i) sum[i] = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) cnt[i] = 0;
    const unsigned* f4 = reinterpret_cast<const unsigned*>(frames) + 3 * g;
    const unsigned* m4 = reinterpret_cast<const unsigned*>(masks) + g;
    const int64_t fstride = npix * 3 / 4, mstride = npix / 4;
#pragma unroll 4
    for (int f = 0; f < n; ++f) {
      int c[12];
      unpack12(__ldg(f4), __ldg(f4 + 1), __ldg(f4 + 2), c);
      const unsigned mw = __ldg(m4);
      f4 += fstride;
      m4 += mstride;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const unsigned mv = (mw >> (8 * i)) & 255u;
        const unsigned keep = 1u - mv / 255u;  // frame * (1 - mask // 255)
        sum[3 * i] += c[3 * i] * keep;
        sum[3 * i + 1] += c[3 * i + 1] * keep;
        sum[3 * i + 2] += c[3 * i + 2] * keep;
        cnt[i] += mv < 250u;               // count += (mask < 250)
      }
    }
    int o[12];
    unsigned aw = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool always = mean_always(cnt[i], min_count);
#pragma unroll
      for (int k = 0; k < 3; ++k) o[3 * i + k] = (int)mean_byte(sum[3 * i + k], cnt[i], always);
      aw |= (always ? 255u : 0u) << (8 * i);
    }
    unsigned w0, w1, w2;
    pack12(o, w0, w1, w2);
    unsigned* d4 = reinterpret_cast<unsigned*>(bg_out) + 3 * g;
    d4[0] = w0; d4[1] = w1; d4[2] = w2;
    reinterpret_cast<unsigned*>(always_out)[g] = aw;
  }
}

// The same at 16 pixels per thread: 4 x 128-bit loads per frame and thread (npix % 16 == 0, 16-byte aligned).  One
// 4-byte load per operand keeps too few bytes in flight for HBM; the sums stay in 64 registers.
__global__ void __launch_bounds__(TT) masked_mean16_kernel(const uint4* __restrict__ frames, const uint4* __restrict__ masks, int n, int64_t ngroups,
                                                           int min_count, uint4* __restrict__ bg_out, uint4* __restrict__ always_out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ngroups; g += stride) {
    unsigned sum[48], cnt[16];
#pragma unroll
    for (int i = 0; i < 48; ++i) sum[i] = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) cnt[i] = 0;
    const uint4* f16 = frames + 3 * g;
    const uint4* m16 = masks + g;
#pragma unroll 2
    for (int f = 0; f < n; ++f) {
      uint4 fv[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) fv[k] = ldg_stream16(f16 + k);
      const uint4 mv4 = ldg_stream16(m16);
      f16 += 3 * ngroups;
      m16 += ngroups;
      const unsigned* fw = reinterpret_cast<const unsigned*>(fv);
      const unsigned mw[4] = {mv4.x, mv4.y, mv4.z, mv4.w};
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const unsigned mv = (mw[i >> 2] >> (8 * (i & 3))) & 255u;
        const unsigned keep = mv == 255u ? 0u : 1u;   // frame * (1 - mask // 255)
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int b = 3 * i + k;
          sum[b] = __dp4a(fw[b >> 2], keep << (8 * (b & 3)), sum[b]);   // byte * keep + sum: one IDP.4A on the FMA pipe
        }
        cnt[i] += mv < 250u;                          // count += (mask < 250)
      }
    }
    unsigned ow[12], aw[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < 12; ++k) ow[k] = 0u;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const bool always = mean_always(cnt[i], min_count);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const int b = 3 * i + k;
        ow[b >> 2] |= mean_byte(sum[b], cnt[i], always) << (8 * (b & 3));
      }
      aw[i >> 2] |= (always ? 255u : 0u) << (8 * (i & 3));
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) bg_out[3 * g + k] = make_uint4(ow[4 * k], ow[4 * k + 1], ow[4 * k + 2], ow[4 * k + 3]);
    always_out[g] = make_uint4(aw[0], aw[1], aw[2], aw[3]);
  }
}

// The masked mean with the masks' dilate_mask(mask, 3, 2) (bg_offline.py:116) fused in.  The mean only asks two yes/no
// questions of a dilated mask value d: d == 255 (the frame is dropped) and d < 250 (the pixel counts).  A grey-scale
// dilation commutes with thresholds - max(taps) >= T  <=>  any tap >= T - so instead of dilating bytes the kernel
// thresholds the raw mask to two bit planes (m == 255, m >= 250) and dilates THOSE, 32 pixels per instruction: two
// passes of the 3x3 cross in shared memory, taps outside the image contributing nothing (SURVEY.md A.1).  The dilated
// masks never exist.  A CTA owns a tile of 128 x 16 pixels and walks through the frames; a thread owns 8 pixels of the
// tile and (200 of the 256 threads) one 16-pixel chunk of the staged mask (tile + halo).  The mask chunk of frame f + 1
// is requested as soon as that of frame f is thresholded, the frame pixels of f + 1 as soon as those of f are
// accumulated: both have the other half of an iteration to arrive.
constexpr int MD_TW = 128, MD_TH = 16, MD_HX = 16, MD_HY = 2;
constexpr int MD_ROWS = MD_TH + 2 * MD_HY;              // 20 staged rows
constexpr int MD_CHUNKS = (MD_TW + 2 * MD_HX) / 16;     // 10 staged 16-pixel chunks per row
constexpr int MD_WORDS = MD_CHUNKS / 2;                 // 5 words of 32 pixels
constexpr int MD_PITCH = MD_WORDS + 1;
static_assert(MD_ROWS * MD_CHUNKS <= 256, "one staged chunk per thread");

// bit 7 of every byte of t -> a nibble
__device__ __forceinline__ unsigned md_nibble(unsigned t) { return ((((t >> 7) & 0x01010101u) * 0x01020408u) >> 24) & 15u; }

constexpr int MD_FPI = 6;   // frames per iteration (and per pair of barriers)

// ACCUM: the sums and counts of these n frames are added to the accumulator state ({sum B, sum G, sum R, count} per
// pixel) instead of being turned into the background
template <bool ACCUM>
__global__ void __launch_bounds__(256, 2) masked_mean_dilate_kernel(const uint8_t* __restrict__ frames, const uint8_t* __restrict__ masks, int n, int h,
                                                                  int w, int min_count, uint8_t* __restrict__ bg_out,
                                                                  uint8_t* __restrict__ always_out, uint4* __restrict__ state) {
  // [stage: thresholded / dilated][frame of the iteration][plane][row][word]; plane 0: m == 255, plane 1: m >= 250
  __shared__ unsigned bits[2][MD_FPI][2][MD_ROWS][MD_PITCH];
  const int t = threadIdx.x;
  const int x0 = blockIdx.x * MD_TW, y0 = blockIdx.y * MD_TH;
  const int64_t npix = (int64_t)h * w;
  // own pixels: 8 of them
  const int ty = t >> 4, cx = t & 15;
  const int oy = y0 + ty, ox = x0 + 8 * cx;
  const bool own = oy < h && ox < w;
  // staged chunk
  const bool sval = t < MD_ROWS * MD_CHUNKS;
  const int sr = t / MD_CHUNKS, sc = t % MD_CHUNKS;
  const int gy = y0 - MD_HY + sr, gx = x0 - MD_HX + 16 * sc;
  const bool sin = sval && gy >= 0 && gy < h && gx >= 0 && gx < w;
  const uint8_t* mp = masks + (int64_t)gy * w + gx;
  const uint8_t* fp = frames + ((int64_t)oy * w + ox) * 3;
  unsigned sum[24], cnt[8];
#pragma unroll
  for (int i = 0; i < 24; ++i) sum[i] = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) cnt[i] = 0;
  uint4 cm[MD_FPI];
  uint2 cf[MD_FPI][3];
#pragma unroll
  for (int u = 0; u < MD_FPI; ++u)
#pragma unroll
    for (int k = 0; k < 3; ++k) cf[u][k] = make_uint2(0u, 0u);   // padding frames are added and taken back out: any value, but a defined one
  // a frame past the end of the clip behaves like a mask of 255 everywhere: dropped and not counted; chunks outside
  // the image are 0 everywhere: they add nothing to a dilation
  auto fetch_masks = [&](int f0) {
#pragma unroll
    for (int u = 0; u < MD_FPI; ++u) {
      if (f0 + u >= n) cm[u] = make_uint4(~0u, ~0u, ~0u, ~0u);
      else if (sin) cm[u] = ldg_stream16(mp + (int64_t)(f0 + u) * npix);
      else cm[u] = make_uint4(0u, 0u, 0u, 0u);
    }
  };
  auto fetch_frames = [&](int f0) {
#pragma unroll
    for (int u = 0; u < MD_FPI; ++u)
      if (own && f0 + u < n) {
#pragma unroll
        for (int k = 0; k < 3; ++k) cf[u][k] = __ldg(reinterpret_cast<const uint2*>(fp + (int64_t)(f0 + u) * npix * 3) + k);
      }
  };
  fetch_masks(0);
  fetch_frames(0);
  for (int f0 = 0; f0 < n; f0 += MD_FPI) {
    // threshold the staged chunks to the two planes, 16 bits each
    if (sval) {
#pragma unroll
      for (int u = 0; u < MD_FPI; ++u) {
        unsigned a = 0, b = 0;
        const unsigned ws[4] = {cm[u].x, cm[u].y, cm[u].z, cm[u].w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const unsigned x = ws[q], lo7 = x & 0x7F7F7F7Fu;
          a |= md_nibble((lo7 + 0x01010101u) & x) << (4 * q);     // byte == 255: bit 7 set and the low 7 bits carry
          b |= md_nibble((lo7 + 0x06060606u) & x) << (4 * q);     // byte >= 250
        }
        reinterpret_cast<unsigned short*>(bits[0][u][0][sr])[sc] = (unsigned short)a;
        reinterpret_cast<unsigned short*>(bits[0][u][1][sr])[sc] = (unsigned short)b;
      }
    }
    if (f0 + MD_FPI < n) fetch_masks(f0 + MD_FPI);
    __syncthreads();
    // two passes of the 3x3 cross at once: the radius-2 diamond, 13 taps (equal to the two passes also at the image
    // border: between two pixels of a rectangle at L1 distance 2 there is always an intermediate pixel inside it);
    // only the tile's own rows are needed
    for (int it = t; it < MD_FPI * 2 * MD_TH * MD_WORDS; it += 256) {
      const int dsel = it / (MD_TH * MD_WORDS), di = it % (MD_TH * MD_WORDS);
      const int dr = MD_HY + di / MD_WORDS, dj = di % MD_WORDS;
      const unsigned(*src)[MD_PITCH] = bits[0][dsel >> 1][dsel & 1];
      auto word = [&](int r, int j) -> unsigned { return (unsigned)j < (unsigned)MD_WORDS ? src[r][j] : 0u; };
      unsigned acc = word(dr - 2, dj) | word(dr + 2, dj);
#pragma unroll
      for (int d = -1; d <= 1; ++d) {
        const unsigned c = word(dr + d, dj), p = word(dr + d, dj - 1), q = word(dr + d, dj + 1);
        acc |= c | __funnelshift_l(p, c, 1) | __funnelshift_r(c, q, 1);
        if (d == 0) acc |= __funnelshift_l(p, c, 2) | __funnelshift_r(c, q, 2);
      }
      bits[1][dsel >> 1][dsel & 1][dr][dj] = acc;
    }
    __syncthreads();
    if (own) {
#pragma unroll
      for (int u = 0; u < MD_FPI; ++u) {
        const unsigned a = reinterpret_cast<const unsigned char*>(bits[1][u][0][ty + MD_HY])[cx + 2];
        const unsigned b = reinterpret_cast<const unsigned char*>(bits[1][u][1][ty + MD_HY])[cx + 2];
        const unsigned* fw = reinterpret_cast<const unsigned*>(cf[u]);
        // every byte is summed and every pixel counted (one IDP.4A with a constant selector each: FMA pipe, nothing on
        // the ALU pipe) ...
#pragma unroll
        for (int bi = 0; bi < 24; ++bi) sum[bi] = __dp4a(fw[bi >> 2], 1u << (8 * (bi & 3)), sum[bi]);
        // ... and the masked pixels - few - are taken back out: frame * (1 - dilated // 255), count += (dilated < 250)
        if (a | b) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if ((a >> i) & 1u) {
#pragma unroll
              for (int k = 0; k < 3; ++k) {
                const int bi = 3 * i + k;
                sum[bi] -= (fw[bi >> 2] >> (8 * (bi & 3))) & 255u;
              }
            }
            cnt[i] += (b >> i) & 1u;                               // here: the frames that do NOT count
          }
        }
      }
    }
    if (f0 + MD_FPI < n) fetch_frames(f0 + MD_FPI);
  }
  if (!own) return;
  const unsigned walked = (unsigned)((n + MD_FPI - 1) / MD_FPI * MD_FPI);   // frames of the walk, the padding ones included (never counted)
  if (ACCUM) {
    uint4* sp = state + (int64_t)oy * w + ox;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint4 s = sp[i];
      s.x += sum[3 * i];
      s.y += sum[3 * i + 1];
      s.z += sum[3 * i + 2];
      s.w += walked - cnt[i];
      sp[i] = s;
    }
    return;
  }
  unsigned ow[6], aw[2] = {0u, 0u};
#pragma unroll
  for (int k = 0; k < 6; ++k) ow[k] = 0u;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const unsigned c = walked - cnt[i];
    const bool always = mean_always(c, min_count);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int b = 3 * i + k;
      ow[b >> 2] |= mean_byte(sum[b], c, always) << (8 * (b & 3));
    }
    aw[i >> 2] |= (always ? 255u : 0u) << (8 * (i & 3));
  }
  uint2* bo = reinterpret_cast<uint2*>(bg_out + ((int64_t)oy * w + ox) * 3);
#pragma unroll
  for (int k = 0; k < 3; ++k) bo[k] = make_uint2(ow[2 * k], ow[2 * k + 1]);
  *reinterpret_cast<uint2*>(always_out + (int64_t)oy * w + ox) = make_uint2(aw[0], aw[1]);
}

// ---- masked-mean accumulator: state = {sum B, sum G, sum R, count} per pixel (uint32 each) ----
// k frames with ALREADY DILATED masks, any npix and alignment: one pixel per thread, byte loads
__global__ void __launch_bounds__(TT) masked_mean_accum_add_kernel(uint4* __restrict__ state, const uint8_t* __restrict__ frames,
                                                                   const uint8_t* __restrict__ masks, int k, int64_t npix) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += stride) {
    uint4 s = state[p];
    const uint8_t* f = frames + 3 * p;
    const uint8_t* mk = masks + p;
#pragma unroll 4
    for (int i = 0; i < k; ++i) {
      const unsigned mv = __ldg(mk + (int64_t)i * npix);
      const uint8_t* fp = f + (int64_t)i * 3 * npix;
      const unsigned keep = mv == 255u ? 0u : 1u;   // frame * (1 - mask // 255)
      s.x += __ldg(fp) * keep;
      s.y += __ldg(fp + 1) * keep;
      s.z += __ldg(fp + 2) * keep;
      s.w += mv < 250u;                             // count += (mask < 250)
    }
    state[p] = s;
  }
}

__global__ void __launch_bounds__(TT) masked_mean_accum_finish_kernel(const uint4* __restrict__ state, int64_t npix, int min_count,
                                                                      uint8_t* __restrict__ bg_out, uint8_t* __restrict__ always_out) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += stride) {
    const uint4 s = state[p];
    const bool always = mean_always(s.w, min_count);
    bg_out[3 * p] = (uint8_t)mean_byte(s.x, s.w, always);
    bg_out[3 * p + 1] = (uint8_t)mean_byte(s.y, s.w, always);
    bg_out[3 * p + 2] = (uint8_t)mean_byte(s.z, s.w, always);
    always_out[p] = always ? 255 : 0;
  }
}

template <class P, int U>
int launch_median(const uint8_t* frames, int n, int64_t m, int64_t nseg, uint8_t* out, vu_stream_t stream, const uint8_t* flags = nullptr) {
  static bool configured = false;
  if (!configured) {
    int e = record_cuda(cudaFuncSetAttribute(median_kernel<P, U>, cudaFuncAttributeMaxDynamicSharedMemorySize, HIST_BYTES));
    if (e) return e;
    configured = true;
  }
  int grid = device_sms();
  const int64_t need = (nseg + WARPS - 1) / WARPS;
  if (need < grid) grid = (int)need;
  median_kernel<P, U><<<grid, MTHREADS, HIST_BYTES, S(stream)>>>(frames, out, n, m, (int)nseg, flags);
  note_launch();
  return record_cuda(cudaGetLastError());
}

// n > 608 with a workspace: subsample estimate (tile kernel) + streaming refine + histogram fix-up of the undecided
// segments.  flags = one byte per 64-byte segment.  Returns VU_ERR_UNSUPPORTED when the TMA path is not available.
int launch_median_two_pass(const uint8_t* frames, int n, int64_t m, int64_t nseg, uint8_t* out, uint8_t* flags, vu_stream_t stream) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return VU_ERR_UNSUPPORTED;
  const int64_t ntiles = nseg / msad::RF_WARPS;
  if (ntiles == 0 || ntiles > 0x7fffffff) return VU_ERR_UNSUPPORTED;
  const int step = (n + 303) / 304;              // every step-th frame: at most 304 of them
  const int nsub = (n + step - 1) / step;
  const int64_t nsub_seg = ntiles * msad::RF_WARPS;   // the segments pass 2 refines: whole tiles of the subsample pass too
  int64_t done;                                       // = nsub_seg
  int e;
  if (nsub <= 152) e = launch_median_sad_tma<4, 19, 6, 4, 1, 4>(frames, nsub, m, nsub_seg, out, stream, &done, (int64_t)step * m);
  else if (nsub <= 232) e = launch_median_sad_tma<4, 29, 12, 4, 1, 3>(frames, nsub, m, nsub_seg, out, stream, &done, (int64_t)step * m);
  else e = launch_median_sad_tma<4, 38, 19, 4, 1, 2>(frames, nsub, m, nsub_seg, out, stream, &done, (int64_t)step * m);
  if (e) return e;
  CUtensorMap tmap;
  const cuuint64_t dims[2] = {(cuuint64_t)(m / 4), (cuuint64_t)n};
  const cuuint64_t strides[1] = {(cuuint64_t)m};
  const cuuint32_t box[2] = {(cuuint32_t)(msad::RF_TILE / 4), (cuuint32_t)msad::RF_ROWS};
  const cuuint32_t estr[2] = {1, 1};
  if (enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<uint8_t*>(frames), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
          CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return VU_ERR_UNSUPPORTED;
  static bool configured = false;
  if (!configured) {
    e = record_cuda(cudaFuncSetAttribute(msad::median_refine_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, msad::RF_SMEM));
    if (e) return e;
    configured = true;
  }
  const int nchunks = (n + msad::RF_ROWS - 1) / msad::RF_ROWS;
  const int grid = (int)(ntiles < device_sms() ? ntiles : device_sms());
  msad::median_refine_kernel<<<grid, msad::RF_WARPS * 32, msad::RF_SMEM, S(stream)>>>(tmap, out, flags, n, (int)ntiles, nchunks);
  note_launch();
  e = record_cuda(cudaGetLastError());
  if (e) return e;
  // segments that do not fill a tile are flagged wholesale; the histogram kernel then redoes every flagged segment
  if (done < nseg) {
    e = record_cuda(cudaMemsetAsync(flags + done, 1, (size_t)(nseg - done), S(stream)));
    if (e) return e;
  }
  return launch_median<PolU16x2, 32>(frames, n, m, nseg, out, stream, flags);
}

}  // namespace
}  // namespace vu

using namespace vu;

// VU_MEDIAN_DIRECT=1 keeps the TMA tile kernels out (tests run the direct kernels on aligned clips this way)
static const bool g_median_direct = [] {
  const char* e = getenv("VU_MEDIAN_DIRECT");
  return e && atoi(e) != 0;
}();

extern "C" size_t vu_temporal_median_workspace_bytes(int n, int64_t m) { return (n > 608 && m > 0) ? (size_t)(m / 64 + 64) : 0; }

extern "C" int vu_temporal_median_u8(const uint8_t* frames, int n, int64_t m, uint8_t* out, vu_stream_t stream) {
  return vu_temporal_median_u8_ws(frames, n, m, out, nullptr, 0, stream);
}

extern "C" int vu_temporal_median_u8_ws(const uint8_t* frames, int n, int64_t m, uint8_t* out, void* workspace, size_t workspace_bytes,
                                        vu_stream_t stream) {
  VU_REQUIRE(frames && out && m >= 0);
  if (n < 1 || n > 65535) return VU_ERR_UNSUPPORTED;
  if (m == 0) return VU_OK;
  // path: 0 = SAD search, half-warp split (n <= 304); 1 = SAD search, quarter-warp split (n <= 608);
  //       2 = shared-memory histograms with 16-bit counters.  The SAD kernels keep the frame stride in 32 bits.
  const bool fits32 = m < (1ll << 30);
  const int path = (n <= 304 && fits32) ? 0 : ((n <= 608 && fits32) ? 1 : 2);
  const int seg = path == 0 ? 64 : (path == 1 ? 32 : 64);
  const int align = path == 2 ? 2 : 4;
  // vector paths need element-aligned frame rows
  const bool ok = (reinterpret_cast<uintptr_t>(frames) % align == 0) && (reinterpret_cast<uintptr_t>(out) % align == 0) && (m % align == 0);
  int64_t nseg = ok ? m / seg : 0;
  if (nseg > 0x7fffffff) return VU_ERR_UNSUPPORTED;
  int64_t tiled = 0;   // bytes of every frame done by the tile kernels (frames / out are advanced past them)
  if (nseg > 0) {
    int e;
    // <SPLIT, G, GFULL, SS, CTAs/SM>: G = register groups of 4 frames per lane, the smallest variant that holds
    // ceil(n / SPLIT) frames; GFULL = groups whose first three rows are real frames over the whole n-range of the
    // variant; SS = stride of the four sample groups of the estimate (all real frames over the n-range)
    // 16-byte aligned frame rows: persistent TMA tile kernels (a pipeline of warps owns 256 adjacent bytes of every
    // frame, the next tile is fetched while the current one is searched); segments that do not fill a tile go to the
    // direct kernels below.
    // <C, G, SS, warps per pipeline (= segments per tile), CTAs per SM, pipelines per CTA>: C column blocks of 16 bytes
    // per warp (= seg / 16),
    // 4G words per lane; SS = stride of the stage-A sample words, which hold frames below 8P(3SS/2 + 1) (P = 4/C):
    // all real frames over the n-range of the variant
    const bool al16 = (reinterpret_cast<uintptr_t>(frames) % 16 == 0) && (m % 16 == 0);
    if (al16 && path != 2 && n > 80 && !g_median_direct) {
      int64_t done = 0;
      if (n <= 152) e = launch_median_sad_tma<4, 19, 6, 4, 1, 4>(frames, n, m, nseg, out, stream, &done);
      else if (n <= 232) e = launch_median_sad_tma<4, 29, 12, 4, 1, 3>(frames, n, m, nseg, out, stream, &done);
      else if (n <= 304) e = launch_median_sad_tma<4, 38, 19, 4, 1, 2>(frames, n, m, nseg, out, stream, &done);
      else if (n <= 464) e = launch_median_sad_tma<2, 29, 12, 8, 1>(frames, n, m, nseg, out, stream, &done);
      else e = launch_median_sad_tma<2, 38, 19, 8, 1>(frames, n, m, nseg, out, stream, &done);
      if (e == VU_OK) {
        frames += done * seg;
        out += done * seg;
        nseg -= done;
        tiled = done * seg;
      } else if (e != VU_ERR_UNSUPPORTED) {   // no tensor-map encoder in this driver: the direct kernels do everything
        return e;
      }
    }
    if (nseg == 0) {
      e = VU_OK;
    } else if (path == 0) {
      if (n <= 80) e = launch_median_sad<2, 10, 0, 0, 4>(frames, n, m, nseg, out, stream);
      else if (n <= 152) e = launch_median_sad<2, 19, 11, 2, 4>(frames, n, m, nseg, out, stream);
      else if (n <= 232) e = launch_median_sad<2, 29, 20, 5, 2>(frames, n, m, nseg, out, stream);
      else e = launch_median_sad<2, 38, 30, 8, 2>(frames, n, m, nseg, out, stream);
    } else if (path == 1) {
      e = n <= 464 ? launch_median_sad<4, 29, 20, 5, 2>(frames, n, m, nseg, out, stream) : launch_median_sad<4, 38, 30, 8, 2>(frames, n, m, nseg, out, stream);
    } else {
      // with a workspace, 16-byte aligned frame rows and a frame size the 32-bit tensor map can describe:
      // estimate + streaming refine + histogram fix-up; otherwise histograms for everything
      e = VU_ERR_UNSUPPORTED;
      if (workspace && workspace_bytes >= vu_temporal_median_workspace_bytes(n, m) && al16 && m < (1ll << 32) && !g_median_direct)
        e = launch_median_two_pass(frames, n, m, nseg, out, static_cast<uint8_t*>(workspace), stream);
      if (e == VU_ERR_UNSUPPORTED) e = launch_median<PolU16x2, 32>(frames, n, m, nseg, out, stream);
    }
    if (e) return e;
  }
  const int64_t first = nseg * seg;   // relative to the advanced pointers
  const int64_t rem = m - tiled;      // m stays the frame stride
  if (first < rem) {
    if (rem - first > 0x7fffffff) return VU_ERR_UNSUPPORTED;
    median_tail_kernel<<<(unsigned)(rem - first), 256, 0, S(stream)>>>(frames, out, n, m, first);
    note_launch();
    return record_cuda(cudaGetLastError());
  }
  return VU_OK;
}

extern "C" int vu_masked_temporal_mean_dilate32(const uint8_t* frames, const uint8_t* masks, int n, int h, int w, int min_count, uint8_t* bg_out,
                                                uint8_t* mask_always_out, vu_stream_t stream) {
  VU_REQUIRE(frames && masks && bg_out && mask_always_out && n >= 1 && h > 0 && w > 0);
  if (n > 16000000) return VU_ERR_UNSUPPORTED;  // 32-bit sums: 255 * n must fit
  const void* ptrs[] = {frames, masks, bg_out, mask_always_out};
  for (const void* p : ptrs)
    if (reinterpret_cast<uintptr_t>(p) & 15) return VU_ERR_UNSUPPORTED;
  if (w % 16 != 0 || (h + MD_TH - 1) / MD_TH > 65535) return VU_ERR_UNSUPPORTED;
  dim3 grid((w + MD_TW - 1) / MD_TW, (h + MD_TH - 1) / MD_TH);
  masked_mean_dilate_kernel<false><<<grid, 256, 0, S(stream)>>>(frames, masks, n, h, w, min_count, bg_out, mask_always_out, nullptr);
  VU_RETURN_LAUNCH();
}

// 32-bit sums: 255 * (frames added) must fit, the caller keeps the total at most 16,000,000 frames
extern "C" size_t vu_masked_mean_accum_bytes(int h, int w) { return (h > 0 && w > 0) ? (size_t)h * (size_t)w * 16 : 0; }

extern "C" int vu_masked_mean_accum_reset(void* state, int h, int w, vu_stream_t stream) {
  VU_REQUIRE(state && h > 0 && w > 0);
  return record_cuda(cudaMemsetAsync(state, 0, vu_masked_mean_accum_bytes(h, w), S(stream)));
}

extern "C" int vu_masked_mean_accum_add_dilate32(void* state, const uint8_t* frames, const uint8_t* masks, int k, int h, int w, vu_stream_t stream) {
  VU_REQUIRE(state && frames && masks && k >= 1 && h > 0 && w > 0);
  VU_REQUIRE((reinterpret_cast<uintptr_t>(state) & 15) == 0);
  if (k > 16000000) return VU_ERR_UNSUPPORTED;
  if (((reinterpret_cast<uintptr_t>(frames) | reinterpret_cast<uintptr_t>(masks)) & 15) != 0) return VU_ERR_UNSUPPORTED;
  if (w % 16 != 0 || (h + MD_TH - 1) / MD_TH > 65535) return VU_ERR_UNSUPPORTED;
  dim3 grid((w + MD_TW - 1) / MD_TW, (h + MD_TH - 1) / MD_TH);
  masked_mean_dilate_kernel<true><<<grid, 256, 0, S(stream)>>>(frames, masks, k, h, w, 0, nullptr, nullptr, static_cast<uint4*>(state));
  VU_RETURN_LAUNCH();
}

extern "C" int vu_masked_mean_accum_add(void* state, const uint8_t* frames, const uint8_t* masks_dilated, int k, int64_t npix, vu_stream_t stream) {
  VU_REQUIRE(state && frames && masks_dilated && k >= 1 && npix > 0);
  VU_REQUIRE((reinterpret_cast<uintptr_t>(state) & 15) == 0);
  if (k > 16000000) return VU_ERR_UNSUPPORTED;
  masked_mean_accum_add_kernel<<<grid_for(npix, TT, 8), TT, 0, S(stream)>>>(static_cast<uint4*>(state), frames, masks_dilated, k, npix);
  VU_RETURN_LAUNCH();
}

extern "C" int vu_masked_mean_accum_finish(const void* state, int64_t npix, int min_count, uint8_t* bg_out, uint8_t* mask_always_out,
                                           vu_stream_t stream) {
  VU_REQUIRE(state && bg_out && mask_always_out && npix > 0);
  VU_REQUIRE((reinterpret_cast<uintptr_t>(state) & 15) == 0);
  masked_mean_accum_finish_kernel<<<grid_for(npix, TT, 8), TT, 0, S(stream)>>>(static_cast<const uint4*>(state), npix, min_count, bg_out,
                                                                               mask_always_out);
  VU_RETURN_LAUNCH();
}

extern "C" int vu_masked_temporal_mean(const uint8_t* frames, const uint8_t* masks, int n, int64_t npix, int min_count, uint8_t* bg_out,
                                       uint8_t* mask_always_out, vu_stream_t stream) {
  VU_REQUIRE(frames && masks && bg_out && mask_always_out && n >= 1 && npix >= 0);
  if (n > 16000000) return VU_ERR_UNSUPPORTED;  // 32-bit sums: 255 * n must fit
  if (npix % 4 != 0) return VU_ERR_UNSUPPORTED;
  const void* ptrs[] = {frames, masks, bg_out, mask_always_out};
  for (const void* p : ptrs)
    if (reinterpret_cast<uintptr_t>(p) & 3) return VU_ERR_UNSUPPORTED;
  if (npix == 0) return VU_OK;
  const void* wide_ptrs[] = {frames, masks, bg_out, mask_always_out};
  bool wide = npix % 16 == 0;
  for (const void* p : wide_ptrs) wide = wide && (reinterpret_cast<uintptr_t>(p) & 15) == 0;
  if (wide)
    masked_mean16_kernel<<<grid_for(npix / 16, TT, 4), TT, 0, S(stream)>>>(reinterpret_cast<const uint4*>(frames), reinterpret_cast<const uint4*>(masks), n,
                                                                           npix / 16, min_count, reinterpret_cast<uint4*>(bg_out),
                                                                           reinterpret_cast<uint4*>(mask_always_out));
  else
    masked_mean_kernel<<<grid_for(npix / 4, TT, 8), TT, 0, S(stream)>>>(frames, masks, n, npix / 4, npix, min_count, bg_out, mask_always_out);
  VU_RETURN_LAUNCH();
}
