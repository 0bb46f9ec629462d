// Exact temporal median of up to 608 uint8 frames, data resident in registers
// (SURVEY.md section 8 row a23; new specification, no reference code).
//
// The median of x_1..x_n minimises the convex S(m) = sum_f |x_f - m|.
// VABSDIFF4 with accumulate evaluates S for 4 frames of one element per
// instruction, which makes "one probe of S" cost n/4 ALU-pipe instructions per
// element, and the ALU pipe (64 lanes/clk/SM) is what bounds this kernel.  The
// design goal is therefore the smallest number of probes:
//
//   stage A  the lower median of 16 frames spread over the whole clip is the
//            estimate (bisection on the slope of S, 8 steps x 8 instructions;
//            every frame-part does it for its share of the lane's elements);
//   stage B  Fibonacci search of the 20 values around the estimate on ALL
//            frames: 6 probes.  The bracket ends keep their S values, so the
//            search ends knowing S at both neighbours of the minimiser: a
//            strict minimum IS the median (odd n) / both middle order
//            statistics (even n), with no further probe;
//   even n   a neighbour with the same S belongs to the plateau [x_lo, x_hi]
//            of minimisers: its end is walked one probe at a time (one probe
//            for the usual plateau of two adjacent values), binary search for
//            long plateaus;
//   fallback if the minimiser of any element of the warp sits on the edge of
//            its window (estimate off by more than 8), the whole warp repeats
//            stage B over 0..255 (12 probes).  Always exact; only the speed
//            depends on the data.
//
// Layout of the direct kernel (the TMA tile kernel below has its own, and the
// search is written for both).  A warp owns SEG = 128/SPLIT consecutive bytes of every frame.  The
// frames are dealt to SPLIT lane groups ("parts"): part p holds frames
// f = SPLIT*i + p.  Lane l of a part holds its 4 bytes of all those frames: one
// coalesced LDG.32 per frame, every load of the warp in flight at once.  Slot
// (g, r) of a lane (register 4g+r) holds frame index i = r*Q + g with
// Q = ceil(ceil(n/SPLIT)/4), so that after the 4x4 byte transposes register
// 4g+j holds four frames of element j a quarter of the clip apart, and any few
// groups form a sample spread over the whole clip.  Unused slots are padded
// with 0 in one half of the parts and 255 in the other, which leaves the middle
// order statistics where they are; when the two pad counts differ by one (odd
// n) the surplus pad is taken out of S arithmetically (S += delta * m).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>
#include "vu_tma.cuh"

namespace vu {
namespace msad {

__device__ __forceinline__ unsigned sad_acc(unsigned a, unsigned b, unsigned c) {
  unsigned d;
  asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// 4x4 byte transposes: d[4g+j] <- byte j of the four registers of group g
// (tried: the same transposition with IDP.4A one-hot byte extraction + IMAD shifts to get it off the ALU pipe:
// 28 instead of 8 instructions per group, and the kernel got slower with every group moved over)
template <int G>
__device__ __forceinline__ void transpose_groups(unsigned (&d)[4 * G]) {
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const unsigned a = d[4 * g], b = d[4 * g + 1], c = d[4 * g + 2], e = d[4 * g + 3];
    const unsigned ab_lo = __byte_perm(a, b, 0x5140), ab_hi = __byte_perm(a, b, 0x7362);
    const unsigned ce_lo = __byte_perm(c, e, 0x5140), ce_hi = __byte_perm(c, e, 0x7362);
    d[4 * g] = __byte_perm(ab_lo, ce_lo, 0x5410);
    d[4 * g + 1] = __byte_perm(ab_lo, ce_lo, 0x7632);
    d[4 * g + 2] = __byte_perm(ab_hi, ce_hi, 0x5410);
    d[4 * g + 3] = __byte_perm(ab_hi, ce_hi, 0x7632);
  }
}

// ld.global.nc.u32 of [base + g * stride]: the 64-bit address is formed by ONE IMAD.WIDE.U32 with g as an immediate
// (FMA pipe), which keeps the address arithmetic of the ~150 loads per lane off the ALU pipe that bounds the search
template <int GI>
__device__ __forceinline__ unsigned ldg_strided(const uint8_t* base, unsigned stride) {
  unsigned long long addr;
  unsigned v;
  asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(addr) : "r"(stride), "n"(GI), "l"(base));
  asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(addr));
  return v;
}

template <int I, int N, class F>
__device__ __forceinline__ void static_for(F&& f) {
  if constexpr (I < N) {
    f(std::integral_constant<int, I>{});
    static_for<I + 1, N>(f);
  }
}

constexpr unsigned BIG = 0x7fffffffu;
constexpr unsigned FULL = 0xffffffffu;

// The search below is written for any register layout of this form: a lane holds E elements, register d[E*k + j]
// holds 4 frames of element j (k = 0..K-1), and the frames of one element are spread over the lanes that differ
// only in the lane bits XMASK (a contiguous run of bits, or 0 when one lane holds all frames of its elements).
__host__ __device__ constexpr int lowest_bit(unsigned x) { return x & 1u ? 0 : 1 + lowest_bit(x >> 1); }
template <unsigned XMASK>
__host__ __device__ constexpr int parts_of() { return XMASK ? (int)(XMASK >> lowest_bit(XMASK)) + 1 : 1; }   // lanes that share an element

// S(m[j]) over all frames of the warp's segment for the E elements of the lane.
// RANGE: probes outside 0..255 are allowed and evaluate to BIG.
template <int E, unsigned XMASK, int K, bool RANGE>
__device__ __forceinline__ void eval_s(const unsigned (&d)[E * K], const int (&m)[E], int delta, unsigned (&S)[E]) {
  constexpr int NA = E < 4 ? 4 / E : 1;   // accumulators per element: at least 4 independent VABSDIFF4 chains per lane
  static_assert(K % NA == 0, "words per element must split evenly over the accumulators");
  unsigned q[E], s[E][NA];
#pragma unroll
  for (int j = 0; j < E; ++j) {
    q[j] = (unsigned)(RANGE ? min(max(m[j], 0), 255) : m[j]) * 0x01010101u;
#pragma unroll
    for (int a = 0; a < NA; ++a) s[j][a] = 0;
  }
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int j = 0; j < E; ++j) s[j][k % NA] = sad_acc(d[E * k + j], q[j], s[j][k % NA]);
  }
#pragma unroll
  for (int j = 0; j < E; ++j) {
    unsigned t = s[j][0];
#pragma unroll
    for (int a = 1; a < NA; ++a) t += s[j][a];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
      if (XMASK & o) t += __shfl_xor_sync(FULL, t, o);
    t += (unsigned)(delta * m[j]);
    S[j] = (RANGE && (m[j] < 0 || m[j] > 255)) ? BIG : t;
  }
}

// Fibonacci search of the interior points a+1 .. a+F(K0)-1 of the bracket
// (a, a+F(K0)).  On return r is the minimiser among them, smin = S(r), and
// sl / sr are S(r-1) / S(r+1), or BIG where that neighbour is the bracket's
// original end (never evaluated).  2 + (K0 - 4) evaluations of S.
template <int E, unsigned XMASK, int K, bool RANGE>
__device__ __forceinline__ void fib_search(const unsigned (&d)[E * K], int delta, int k0, int fa, int fb, int fc, int (&a)[E], int (&r)[E],
                                           unsigned (&smin)[E], unsigned (&sl)[E], unsigned (&sr)[E]) {
  unsigned S1[E], S2[E];
  {
    int i1[E], i2[E];
#pragma unroll
    for (int j = 0; j < E; ++j) {
      i1[j] = a[j] + fb;
      i2[j] = a[j] + fa;
      sl[j] = sr[j] = BIG;
    }
    eval_s<E, XMASK, K, RANGE>(d, i1, delta, S1);
    eval_s<E, XMASK, K, RANGE>(d, i2, delta, S2);
  }
#pragma unroll 1
  for (int k = k0; k >= 5; --k) {
    int nidx[E];
    bool left[E];
#pragma unroll
    for (int j = 0; j < E; ++j) {
      left[j] = S1[j] <= S2[j];
      if (left[j]) {
        sr[j] = S2[j];
        S2[j] = S1[j];
        nidx[j] = a[j] + fc;
      } else {
        sl[j] = S1[j];
        a[j] += fb;
        S1[j] = S2[j];
        nidx[j] = a[j] + fb;
      }
    }
    unsigned Sn[E];
    eval_s<E, XMASK, K, RANGE>(d, nidx, delta, Sn);
#pragma unroll
    for (int j = 0; j < E; ++j) {
      if (left[j]) S1[j] = Sn[j];
      else S2[j] = Sn[j];
    }
    const int t = fb - fc;
    fa = fb;
    fb = fc;
    fc = t;
  }
  // k == 4: bracket (a, a+3), S1 = S(a+1), S2 = S(a+2)
#pragma unroll
  for (int j = 0; j < E; ++j) {
    if (S1[j] <= S2[j]) {
      r[j] = a[j] + 1;
      smin[j] = S1[j];
      sr[j] = S2[j];
    } else {
      r[j] = a[j] + 2;
      smin[j] = S2[j];
      sl[j] = S1[j];
    }
  }
}

template <int E>
__device__ __forceinline__ bool open_any(const int (&L)[E], const int (&R)[E]) {
  bool o = false;
#pragma unroll
  for (int j = 0; j < E; ++j) o |= L[j] < R[j];
  return o;
}

// SS = stride of the 4 sample words of stage A (0: no stage A, straight to the full search).
// Returns the median of element j in byte j.
template <int E, unsigned XMASK, int K, int SS>
__device__ __forceinline__ unsigned sad_median(const unsigned (&d)[E * K], int n, int delta) {
  int a[E], r[E];
  unsigned smin[E], sl[E], sr[E];
  bool full = (SS == 0);
  if (SS > 0) {
    // ---- stage A: every part (one of the lanes that share an element) estimates E/PARTS of the lane's elements as
    // the lower median of 16 of ITS frames (bisection on the slope of S), then the parts swap their estimates ----
    constexpr int PARTS = parts_of<XMASK>();
    constexpr int PSHIFT = XMASK ? lowest_bit(XMASK) : 0;
    constexpr int EPP = E / PARTS;   // elements per part
    const int lane = threadIdx.x & 31;
    const int part = (lane & XMASK) >> PSHIFT;
    unsigned smp[EPP][4];
#pragma unroll
    for (int e = 0; e < EPP; ++e)
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        unsigned v = d[E * (t * SS) + e];
#pragma unroll
        for (int p = 1; p < PARTS; ++p) v = (part == p) ? d[E * (t * SS) + p * EPP + e] : v;
        smp[e][t] = v;
      }
    int est[EPP];
#pragma unroll
    for (int e = 0; e < EPP; ++e) est[e] = 0;
#pragma unroll 1
    for (int bit = 128; bit > 0; bit >>= 1) {
#pragma unroll
      for (int e = 0; e < EPP; ++e) {
        const unsigned q1 = (unsigned)(est[e] | bit) * 0x01010101u, q0 = q1 - 0x01010101u;
        unsigned s0 = 0, s1 = 0;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          s0 = sad_acc(smp[e][t], q0, s0);
          s1 = sad_acc(smp[e][t], q1, s1);
        }
        if (s1 < s0) est[e] |= bit;
      }
    }
#pragma unroll
    for (int j = 0; j < E; ++j) {
      const int c = PARTS == 1 ? est[j] : __shfl_sync(FULL, est[j % EPP], (lane & ~XMASK) | ((j / EPP) << PSHIFT));
      a[j] = min(max(c - 10, -1), 235);   // interior a+1 .. a+20 within 0..255
    }
    // ---- stage B: the 20 values around the estimate ----
    fib_search<E, XMASK, K, false>(d, delta, 8, 13, 8, 5, a, r, smin, sl, sr);
    bool fail = false;
#pragma unroll
    for (int j = 0; j < E; ++j) fail |= (sl[j] == BIG && r[j] > 0) || (sr[j] == BIG && r[j] < 255);
    full = __any_sync(FULL, fail);
  }
  if (full) {
#pragma unroll
    for (int j = 0; j < E; ++j) a[j] = -1;
    fib_search<E, XMASK, K, true>(d, delta, 14, 233, 144, 89, a, r, smin, sl, sr);   // interior -1+1 .. 375: covers 0..255
  }
  int lo[E], hi[E];
#pragma unroll
  for (int j = 0; j < E; ++j) lo[j] = hi[j] = r[j];
  if (!(n & 1)) {
    // even n: minimisers form the plateau [x_lo, x_hi]
    bool openL[E], openR[E];
    bool any = false;
#pragma unroll
    for (int j = 0; j < E; ++j) {
      openL[j] = openR[j] = false;
      if (sl[j] == smin[j]) { lo[j] = r[j] - 1; openL[j] = lo[j] > 0; }
      if (sr[j] == smin[j]) { hi[j] = r[j] + 1; openR[j] = hi[j] < 255; }
      any |= openL[j] | openR[j];
    }
    // walk the open ends, one probe per lane and round
#pragma unroll 1
    for (int it = 0; it < 4 && __any_sync(FULL, any); ++it) {
      int idx[E];
      unsigned S[E];
#pragma unroll
      for (int j = 0; j < E; ++j) idx[j] = openL[j] ? lo[j] - 1 : (openR[j] ? hi[j] + 1 : r[j]);
      eval_s<E, XMASK, K, false>(d, idx, delta, S);
      any = false;
#pragma unroll
      for (int j = 0; j < E; ++j) {
        if (openL[j]) {
          if (S[j] == smin[j]) { --lo[j]; openL[j] = lo[j] > 0; }
          else openL[j] = false;
        } else if (openR[j]) {
          if (S[j] == smin[j]) { ++hi[j]; openR[j] = hi[j] < 255; }
          else openR[j] = false;
        }
        any |= openL[j] | openR[j];
      }
    }
    // long plateaus (e.g. two-valued data): binary search for the ends (S == smin is monotone on either side)
    if (__any_sync(FULL, any)) {
      int L[E], R[E];
#pragma unroll
      for (int j = 0; j < E; ++j) { R[j] = lo[j]; L[j] = openL[j] ? 0 : lo[j]; }
      while (__any_sync(FULL, open_any(L, R))) {
        int idx[E];
        unsigned S[E];
#pragma unroll
        for (int j = 0; j < E; ++j) idx[j] = (L[j] + R[j]) >> 1;
        eval_s<E, XMASK, K, false>(d, idx, delta, S);
#pragma unroll
        for (int j = 0; j < E; ++j)
          if (L[j] < R[j]) {
            const int mid = (L[j] + R[j]) >> 1;
            if (S[j] == smin[j]) R[j] = mid;
            else L[j] = mid + 1;
          }
      }
#pragma unroll
      for (int j = 0; j < E; ++j) { lo[j] = R[j]; L[j] = hi[j]; R[j] = openR[j] ? 255 : hi[j]; }
      while (__any_sync(FULL, open_any(L, R))) {
        int idx[E];
        unsigned S[E];
#pragma unroll
        for (int j = 0; j < E; ++j) idx[j] = (L[j] + R[j] + 1) >> 1;
        eval_s<E, XMASK, K, false>(d, idx, delta, S);
#pragma unroll
        for (int j = 0; j < E; ++j)
          if (L[j] < R[j]) {
            const int mid = (L[j] + R[j] + 1) >> 1;
            if (S[j] == smin[j]) L[j] = mid;
            else R[j] = mid - 1;
          }
      }
#pragma unroll
      for (int j = 0; j < E; ++j) hi[j] = L[j];
    }
  }
  unsigned res = 0;
#pragma unroll
  for (int j = 0; j < E; ++j) res |= (unsigned)((lo[j] + hi[j]) >> 1) << (8 * j);
  return res;
}

// pads: 0 in parts {0} (SPLIT 2) / {0,3} (SPLIT 4), 255 in the others: the two pad counts differ by at most one
template <int SPLIT>
__device__ __forceinline__ bool pad_high(int part) { return SPLIT == 2 ? part == 1 : (part == 1 || part == 2); }

// GFULL: groups whose rows 0..2 hold real frames for every n the variant is dispatched for (no bounds test on those loads).
// SPLIT * m must fit 32 bits.
template <int SPLIT, int G, int GFULL, int SS, int CTAS>
__global__ void __launch_bounds__(128, CTAS) median_sad_kernel(const uint8_t* __restrict__ frames, uint8_t* __restrict__ out, int n, long long m,
                                                               int nseg, unsigned zero) {
  constexpr int LPS = 32 / SPLIT;  // lanes per frame-part
  constexpr int SEG = LPS * 4;     // bytes of a frame one warp owns
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int part = lane / LPS, li = lane % LPS;
  const int seg = blockIdx.x * 4 + warp;
  if (seg >= nseg) return;
  const int cnt0 = (n + SPLIT - 1) / SPLIT;          // frames of part 0 (the largest part)
  const int cnt = (n - part + SPLIT - 1) / SPLIT;    // frames of this part
  const int Q = (cnt0 + 3) >> 2;
  const unsigned pad = pad_high<SPLIT>(part) ? 0xFFFFFFFFu : 0u;
  // surplus of 255-pads over 0-pads (-1, 0 or +1), taken out of S arithmetically
  int n0 = 0, n255 = 0;
#pragma unroll
  for (int p = 0; p < SPLIT; ++p) {
    const int c = 4 * G - (n - p + SPLIT - 1) / SPLIT;
    if (pad_high<SPLIT>(p)) n255 += c;
    else n0 += c;
  }
  const int delta = n255 - n0;
  // frame i of this part starts (SPLIT*i + part) * m bytes into the clip; slot (g, r) holds i = r*Q + g
  // (`zero` is 0: it gives every row its own copy of the stride, or the compiler shares g * stride between the
  // rows and goes back to 64-bit adds on the ALU pipe)
  unsigned gstride[4];
  const uint8_t* rowbase[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    rowbase[r] = frames + (long long)seg * SEG + li * 4 + ((long long)SPLIT * (r * Q) + part) * m;
    gstride[r] = (unsigned)(SPLIT * m) + (unsigned)r * zero;
  }
  unsigned d[4 * G];
  static_for<0, G>([&](auto gi) {
    constexpr int g = decltype(gi)::value;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const bool ok = (r < 3 && g < GFULL) ? true : (g < Q && r * Q + g < cnt);
      d[4 * g + r] = pad;
      if (ok) d[4 * g + r] = ldg_strided<g>(rowbase[r], gstride[r]);
    }
  });
  transpose_groups<G>(d);
  const unsigned res = sad_median<4, 32u - LPS, G, SS>(d, n, delta);
  if (part == 0) reinterpret_cast<unsigned*>(out + (long long)seg * SEG)[li] = res;
}


// ---- persistent tile kernel: TMA fetches the next tile while the current one is searched ---------------------------
//
// Measured on the B200 (tools/ldgsts_ubench.cu, fetch only): "one row per frame" streams at 2.8 TB/s when a warp
// fetches 64-byte rows on its own, at 5.9 TB/s with 128-byte rows and at 7.2 TB/s with 512-byte rows: requests must
// cover whole 128-byte lines, and the direct kernel above (64 bytes per frame and warp) cannot get there.  Here a CTA
// of WARPS warps owns tiles of WARPS adjacent segments of 16*C bytes (8 warps, C = 4: 512 bytes of every frame).  The
// clip is described to the TMA unit as a 3-D tensor [n frames][m/128 chunks][128 bytes], and boxes of {TILE bytes x
// BOX_ROWS frames} (cp.async.bulk.tensor.3d with the 128-byte swizzle, one elected thread, completion counted in bytes
// on an mbarrier) bring the tile into shared memory as rows of TILE bytes.  The swizzle works on 128-byte units: unit
// R = f*COLS + col (frame f, 128-byte column col) keeps its 16-byte chunk c at chunk c ^ (R & 7).  (With one box per
// 128-byte column the rows fetched were only 128 bytes long, and the fetch capped the kernel at ~4.5 TB/s.)  Frames past the end of the clip are zero-filled by the
// unit: pads are all 0 here and leave S through delta = -(number of pads).  The warps are only loosely coupled: a
// warp waits for the tile on the mbarrier, moves its segment to registers, bumps a counter and goes searching; the
// warp that bumps it last knows the buffer is free and launches the fetch of the next tile, which then lands while
// everybody searches.
//
// Layout.  ldmatrix.m16n16.trans.b8 reads a 16 x 16 byte block (16 row addresses, 16 bytes each) and hands lane l
// two words: rows 4*(l&3) .. +3 of block columns l>>2 and (l>>2)+8, i.e. "4 rows of one column" - four frames of one
// element when the rows are frames - with no byte transposes on the ALU pipe.  The rows of one block need not be
// adjacent: rows 4q .. 4q+3 (the ones lane quad member q receives) are 4 frames of the warp's 16-byte column block
// q % C.  So a lane holds E = 2 elements (columns i and i+8 of column block q % C, i = l>>2), and the frames of an
// element are dealt to the P = 4/C quad members q, q+C, ..: with C = 4 one lane holds every frame of its two elements
// and S needs no shuffle; with C = 2 two lanes hold half the frames each (shfl_xor 2).  Word k = 2j+M (matrix M of the
// j-th ldmatrix.x2) of quad member q holds frames 8Pj + 8(q/C) + 4((M^q)&1) + 0..3.  Banks: the swizzle of a row
// depends on f*COLS + col.  With COLS = 2 (C = 2) the 4 frames of a row group get 4 distinct swizzles and one 8-row
// phase of ldmatrix reads 8 distinct bank groups; with COLS = 4 (C = 4) only the frame's parity reaches the swizzle
// and a phase reads each bank group twice - as many wavefronts as the LDS.32 of the previous layout, and the rows of
// the tile stay 512 bytes long for the fetch.  The lane's row address only moves by a constant 8P*TILE bytes from one
// ldmatrix to the next (immediate offsets, no address arithmetic).  Stage A's sample words
// t*SS (t = 0..3) are four runs of 4 consecutive frames a quarter of the clip apart.
using tma::mbar_expect_tx;
using tma::mbar_init;
using tma::mbar_wait;
__device__ __forceinline__ void tma_load_2d(unsigned dst, const void* tmap, int c0, int c1, unsigned mbar) { tma::load_2d(dst, tmap, c0, c1, mbar); }

__device__ __forceinline__ void ldsm_x2_trans(unsigned addr, unsigned& r0, unsigned& r1, unsigned& r2, unsigned& r3) {
  asm volatile("ldmatrix.sync.aligned.m16n16.x2.trans.shared.b8 {%0, %1, %2, %3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr) : "memory");
}

// shape of the tile: shared by the kernel and the tensor map of its launcher
template <int C, int G, int WARPS>
struct TmaTile {
  static_assert(C == 2 || C == 4, "a warp owns 2 or 4 column blocks of 16 bytes");
  static constexpr int P = 4 / C;                 // lanes that share an element
  static constexpr int SEG = 16 * C;              // bytes of a frame one warp owns
  static constexpr int TILE = WARPS * SEG;        // bytes of a frame one CTA owns
  static constexpr int COLS = TILE / 128;         // 128-byte columns
  static constexpr int ROWS = 8 * P * G;          // frames in the buffer: G ldmatrix.x2 of 8P frames each
  static constexpr int row_boxes(int b) { return (ROWS % b == 0 && (ROWS / b) % 8 == 0 && ROWS / b <= 256) ? b : row_boxes(b + 1); }
  static constexpr int BOX_ROWS = ROWS / row_boxes(1);   // <= 256 rows, a multiple of 8: every box starts on 1024 bytes
  static constexpr int BYTES = ROWS * TILE;
  static constexpr int SMEM = BYTES + 1024 + 16;  // + alignment of the buffer to 1024 bytes (the swizzle's period) + mbarrier, counter
  static_assert(TILE % 128 == 0, "whole 128-byte columns");
};

// <C, G, SS, WARPS, CTAS>: C column blocks of 16 bytes per warp, 4G words per lane (2G per element), SS = stride of
// the stage-A sample words (all real frames for every n the variant is dispatched for).
template <int C, int G, int SS, int WARPS, int CTAS>
__global__ void __launch_bounds__(WARPS * 32, CTAS) median_sad_tma_kernel(const __grid_constant__ CUtensorMap tmap, uint8_t* __restrict__ out, int n,
                                                                          int ntiles) {
  extern __shared__ __align__(1024) uint8_t smem_tma[];
  using T = TmaTile<C, G, WARPS>;
  constexpr unsigned XMASK = 3u & ~(unsigned)(C - 1);   // lane bits of the quad members that share an element
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int delta = -(T::ROWS - n);
  const unsigned sraw = (unsigned)__cvta_generic_to_shared(smem_tma);
  const unsigned sdata = (sraw + 1023u) & ~1023u;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(smem_tma + (sdata - sraw) + T::BYTES);
  unsigned* count_p = reinterpret_cast<unsigned*>(mbar_p + 1);
  const unsigned mbar = (unsigned)__cvta_generic_to_shared(mbar_p);
  auto fetch = [&](int tile) {   // one thread
    mbar_expect_tx(mbar, T::BYTES);
#pragma unroll
    for (int r = 0; r < T::ROWS; r += T::BOX_ROWS) tma::load_3d(sdata + r * T::TILE, &tmap, 0, tile * T::COLS, r, mbar);
  };
  if (threadIdx.x == 0) {
    mbar_init(mbar, 1);
    *count_p = 0;
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  int tile = blockIdx.x;
  if (threadIdx.x == 0 && tile < ntiles) fetch(tile);
  // the row this lane addresses: row rho of matrix M, which lands in quad member qq = rho >> 2 as frame
  // 8Pj + f0 of column block qq % C
  unsigned laddr;
  {
    const int rho = lane & 15, M = lane >> 4, qq = rho >> 2;
    const int f0 = 8 * (qq / C) + 4 * ((M ^ qq) & 1) + (rho & 3);
    const int byte = warp * T::SEG + 16 * (qq % C);   // of the tile
    const int unit = f0 * T::COLS + (byte >> 7);
    laddr = sdata + unit * 128 + ((((byte >> 4) & 7) ^ (unit & 7)) << 4);
  }
  // the two elements of this lane: bytes q%C*16 + (l>>2) + {0, 8} of the warp's segment; quad members q < C write them
  const int q = lane & 3;
  const int ebyte = warp * T::SEG + 16 * (q % C) + (lane >> 2);
  unsigned parity = 0;
  for (; tile < ntiles; tile += gridDim.x) {
    mbar_wait(mbar, parity);
    parity ^= 1;
    unsigned d[4 * G];
#pragma unroll
    for (int j = 0; j < G; ++j) ldsm_x2_trans(laddr + j * (8 * T::P * T::TILE), d[4 * j], d[4 * j + 1], d[4 * j + 2], d[4 * j + 3]);
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      const unsigned old = atomicAdd(count_p, 1u);
      if (old % WARPS == WARPS - 1 && tile + (int)gridDim.x < ntiles) {
        __threadfence_block();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        fetch(tile + gridDim.x);
      }
    }
    const unsigned res = sad_median<2, XMASK, 2 * G, SS>(d, n, delta);
    if (q < C) {
      uint8_t* o = out + (long long)tile * T::TILE + ebyte;
      o[0] = (uint8_t)res;
      o[8] = (uint8_t)(res >> 8);
    }
  }
}

// ---- n > 608: estimate on a subsample, then ONE streaming pass that proves it ---------------------------------------
//
// More frames than the registers of a warp can hold.  Pass 1 is the tile kernel above on every s-th frame (a tensor
// map with row pitch s*m: at most 304 frames), which leaves the subsample's median in `out`.  Pass 2 (this kernel)
// streams ALL frames once, TMA chunk by chunk through a ring of shared-memory stages, and accumulates S(m) at the
// eight values m = e-4 .. e+3 around the estimate e of every element: 8 VABSDIFF4 + 2 PRMT per input word, just
// under what the ALU pipe can do at the HBM rate.  The minimiser of a convex function that is strictly inside the
// probed range is the global one, so a strict interior minimum is the median (odd n), and a plateau that ends
// inside the range gives both middle order statistics (even n).  Elements whose minimum touches the edge of the
// range are not decided here: the segment is flagged and the histogram kernel redoes the flagged segments.
// Frames are dealt to the two half-warps alternately; rows past the end of the clip are zero-filled by the TMA and
// leave S arithmetically (S -= pads * m).
constexpr int RF_WARPS = 8, RF_ROWS = 64, RF_STAGES = 4, RF_PROBES = 8;
constexpr int RF_TILE = RF_WARPS * 64;
constexpr int RF_STAGE_BYTES = RF_ROWS * RF_TILE;
constexpr int RF_SMEM = RF_STAGES * RF_STAGE_BYTES + RF_STAGES * 16;

__global__ void __launch_bounds__(RF_WARPS * 32, 1) median_refine_kernel(const __grid_constant__ CUtensorMap tmap, uint8_t* __restrict__ out,
                                                                         uint8_t* __restrict__ flags, int n, int ntiles, int nchunks) {
  extern __shared__ __align__(128) uint8_t smem_rf[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int part = lane >> 4, li = lane & 15;
  uint64_t* mbar_p = reinterpret_cast<uint64_t*>(smem_rf + RF_STAGES * RF_STAGE_BYTES);
  unsigned* count_p = reinterpret_cast<unsigned*>(mbar_p + RF_STAGES);
  const unsigned mbar0 = (unsigned)__cvta_generic_to_shared(mbar_p);
  const unsigned sdata = (unsigned)__cvta_generic_to_shared(smem_rf);
  const int my_tiles = blockIdx.x < ntiles ? (ntiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int J = my_tiles * nchunks;   // chunks this CTA streams, in order
  auto issue = [&](int j) {           // one thread
    const int tile = blockIdx.x + (j / nchunks) * gridDim.x, chunk = j % nchunks, st = j % RF_STAGES;
    mbar_expect_tx(mbar0 + 8 * st, RF_STAGE_BYTES);
    tma_load_2d(sdata + st * RF_STAGE_BYTES, &tmap, tile * (RF_TILE / 4), chunk * RF_ROWS, mbar0 + 8 * st);
  };
  if (threadIdx.x == 0) {
    for (int st = 0; st < RF_STAGES; ++st) {
      mbar_init(mbar0 + 8 * st, 1);
      count_p[st] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0)
    for (int j = 0; j < RF_STAGES && j < J; ++j) issue(j);
  const int delta = -(nchunks * RF_ROWS - n);   // zero rows past the clip
  unsigned acc[RF_PROBES][4], q[RF_PROBES][4];
  int a0[4];
  const uint8_t* lane_row = smem_rf + part * RF_TILE + warp * 64 + li * 4;   // rows 2i + part of a stage
  for (int j = 0; j < J; ++j) {
    const int tile = blockIdx.x + (j / nchunks) * gridDim.x, chunk = j % nchunks, st = j % RF_STAGES;
    const int64_t seg = (int64_t)tile * RF_WARPS + warp;
    if (chunk == 0) {
      const unsigned e = *reinterpret_cast<const unsigned*>(out + seg * 64 + li * 4);   // pass 1's estimates
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        a0[k] = min(max((int)((e >> (8 * k)) & 255u) - 4, 0), 256 - RF_PROBES);
#pragma unroll
        for (int p = 0; p < RF_PROBES; ++p) {
          q[p][k] = (unsigned)(a0[k] + p) * 0x01010101u;
          acc[p][k] = 0u;
        }
      }
    }
    mbar_wait(mbar0 + 8 * st, (unsigned)((j / RF_STAGES) & 1));
    const uint8_t* base = lane_row + st * RF_STAGE_BYTES;
#pragma unroll
    for (int h = 0; h < 2; ++h) {   // 2 x 16 rows of this part: 16 words, 4 groups
      unsigned d[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) d[i] = *reinterpret_cast<const unsigned*>(base + (2 * (16 * h + i)) * RF_TILE);
      transpose_groups<4>(d);
#pragma unroll
      for (int g = 0; g < 4; ++g)
#pragma unroll
        for (int p = 0; p < RF_PROBES; ++p)
#pragma unroll
          for (int k = 0; k < 4; ++k) acc[p][k] = sad_acc(d[4 * g + k], q[p][k], acc[p][k]);
    }
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      const unsigned old = atomicAdd(count_p + st, 1u);
      if (old % RF_WARPS == RF_WARPS - 1 && j + RF_STAGES < J) {
        __threadfence_block();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        issue(j + RF_STAGES);
      }
    }
    if (chunk == nchunks - 1) {
      unsigned res = 0;
      bool bad = false;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        unsigned S[RF_PROBES];
        unsigned smin = 0xFFFFFFFFu;
#pragma unroll
        for (int p = 0; p < RF_PROBES; ++p) {
          S[p] = acc[p][k] + __shfl_xor_sync(FULL, acc[p][k], 16) + (unsigned)(delta * (a0[k] + p));
          smin = min(smin, S[p]);
        }
        int lo = -1, hi = -1;   // first / last probe at the minimum
#pragma unroll
        for (int p = 0; p < RF_PROBES; ++p)
          if (S[p] == smin) {
            if (lo < 0) lo = p;
            hi = p;
          }
        // decided only if the minimum does not touch the edge of the probed range (or the edge of the byte range)
        bad |= (lo == 0 && a0[k] > 0) || (hi == RF_PROBES - 1 && a0[k] + RF_PROBES - 1 < 255);
        res |= (unsigned)((2 * a0[k] + lo + hi) >> 1) << (8 * k);
      }
      const bool any_bad = __any_sync(FULL, bad);
      if (part == 0) *reinterpret_cast<unsigned*>(out + seg * 64 + li * 4) = res;
      if (lane == 0) flags[seg] = any_bad ? 1 : 0;
    }
  }
}

}  // namespace msad
}  // namespace vu
