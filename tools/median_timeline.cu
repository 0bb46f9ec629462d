// Tile-kernel variants of the temporal median for tools/median_timeline.py: every <C, G, SS, WARPS, CTAS> variant the
// dispatch of vu_temporal_median_u8 has used or may use for n <= 608, each plain and with the TRACE timeline, launched
// through the library's own launcher (this file includes vu_temporal.cu; link it with vu_api.cu).
#include "../video_unscreen_b200/csrc/vu_temporal.cu"

namespace {
using Launch = int (*)(const uint8_t*, int, int64_t, int64_t, uint8_t*, vu_stream_t, int64_t*, int64_t, unsigned long long*);

struct Variant {
  const char* name;
  int max_n;   // frames the variant holds: 8P * G (P = 4 / C)
  int seg;     // bytes of a segment: 16C
  Launch plain, traced;
};

#define VARIANTP(C, G, SS, W, K, P) \
  { #C "," #G "," #SS "," #W "," #K "," #P, 8 * (4 / C) * G, 16 * C, vu::launch_median_sad_tma<C, G, SS, W, K, P, false>, \
    vu::launch_median_sad_tma<C, G, SS, W, K, P, true> }
#define VARIANT(C, G, SS, W, K) VARIANTP(C, G, SS, W, K, 1)

const Variant kVariants[] = {
    VARIANT(4, 38, 19, 8, 1), VARIANT(4, 38, 19, 4, 2), VARIANTP(4, 38, 19, 4, 1, 2), VARIANT(2, 19, 9, 8, 2),   // n <= 304
    VARIANT(4, 29, 12, 8, 1), VARIANT(4, 29, 12, 4, 2), VARIANT(4, 29, 12, 4, 3), VARIANTP(4, 29, 12, 4, 1, 3),  // n <= 232
    VARIANT(4, 19, 6, 8, 2),  VARIANT(4, 19, 6, 4, 2),  VARIANT(4, 19, 6, 4, 3),  VARIANT(4, 19, 6, 4, 4),
    VARIANTP(4, 19, 6, 4, 1, 4),                                                                                 // n <= 152
    VARIANT(2, 38, 19, 8, 1),                                                      // n <= 608
};
constexpr int kCount = sizeof(kVariants) / sizeof(kVariants[0]);
}  // namespace

extern "C" int mt_count() { return kCount; }
extern "C" const char* mt_name(int v) { return v >= 0 && v < kCount ? kVariants[v].name : nullptr; }
extern "C" int mt_max_n(int v) { return kVariants[v].max_n; }
extern "C" int mt_seg(int v) { return kVariants[v].seg; }

// One launch of variant v over the whole tiles of the clip (segments of mt_seg(v) bytes); *done = segments covered.
// trace != 0: the TRACE kernel, which needs msad::TRACE_WORDS words per warp and tile (see vu_median_sad.cuh).
extern "C" int mt_run(int v, const uint8_t* frames, int n, long long m, uint8_t* out, unsigned long long* trace, long long* done, void* stream) {
  if (v < 0 || v >= kCount || n > kVariants[v].max_n) return VU_ERR_INVALID_ARG;
  const Variant& k = kVariants[v];
  int64_t d = 0;
  const int e = (trace ? k.traced : k.plain)(frames, n, m, m / k.seg, out, reinterpret_cast<vu_stream_t>(stream), &d, 0, trace);
  *done = d;
  return e;
}
