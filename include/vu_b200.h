/*
 * vu_b200.h -- C ABI of the B200-native video_unscreen hot path.
 *
 * The reference (AnyiRao/video_unscreen) has no FFI: its boundary for this
 * path is Python-import level (SURVEY.md section 8b).  Every entry point below
 * names the reference function or inline lines it replaces; the Python package
 * `video_unscreen_b200.unscreen` binds them with ctypes and mirrors the
 * reference's signatures (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - every image pointer is a DEVICE pointer to dense, C-contiguous uint8:
 *     frames [n][h][w][3] in BGR order, masks [n][h][w]; no pitches.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *     Calls only enqueue work; nothing here synchronises or allocates.
 *   - workspaces are caller-provided; sizes come from the *_workspace_bytes
 *     twins.  Workspace pointers must be 256-byte aligned.
 *   - return value: VU_OK (0) or a negative vu_status.  No exceptions, no
 *     CPU fallback: if the device code cannot run, the call fails.
 */
#ifndef VU_B200_H
#define VU_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VU_ABI_VERSION 1

typedef void* vu_stream_t;

enum vu_status {
  VU_OK = 0,
  VU_ERR_INVALID_ARG = -1,
  VU_ERR_UNSUPPORTED = -2,
  VU_ERR_WORKSPACE = -3,
  VU_ERR_CUDA = -4
};

enum vu_morph_op { VU_DILATE = 0, VU_ERODE = 1 };
enum vu_cmp_op { VU_CMP_GE = 0, VU_CMP_GT = 1, VU_CMP_LT = 2, VU_CMP_EQ = 3, VU_CMP_NE = 4 };
enum vu_patch_mode { VU_PATCH_NONE = 0, VU_PATCH_ALPHA_LT128 = 1, VU_PATCH_ALPHA_EQ0 = 2 };
enum vu_blend_mode {
  VU_BLEND_NAIVE = 0,     /* u8(f64(img) * a)                        fgfuncs.py:68-81   */
  VU_BLEND_FUSE = 1,      /* u8(a*fg + (1-a)*bg)                     visualize.py:7-24  */
  VU_BLEND_COMPOSITE = 2, /* a[a>0.9]=1; u8(clip(fg + bg*(1-a)))     fgfuncs.py:201-207 */
  VU_BLEND_REPLACE = 3    /* u8(fg*m + bg*(1-m)), m = mask/255       replace.py:74-76   */
};

int vu_abi_version(void);
const char* vu_status_string(int status);
/* text of the last CUDA error seen by this library on the calling thread */
const char* vu_last_cuda_error(void);
/* number of kernels this library has launched in this process (all threads) */
uint64_t vu_launch_count(void);

/* ---- colour ------------------------------------------------------------ */
/* cv2.cvtColor(BGR2HSV) uint8, H in [0,179]; colorfiltering/agent.py:310,
 * fgfuncs.py:36,39,100,101,129 */
int vu_bgr2hsv_u8(const uint8_t* bgr, uint8_t* hsv, int64_t npix, vu_stream_t stream);
/* cv2.cvtColor(HSV2BGR) uint8 (whole-image = truncating variant);
 * colorfiltering/agent.py:352, fgfuncs.py:109,136 */
int vu_hsv2bgr_u8(const uint8_t* hsv, uint8_t* bgr, int64_t npix, vu_stream_t stream);
/* cv2.cvtColor(BGR2GRAY) uint8; bg.py:86, bg_offline.py:152,155 */
int vu_bgr2gray_u8(const uint8_t* bgr, uint8_t* gray, int64_t npix, vu_stream_t stream);
/* is_pixel_inrange, bg-colour variant (fgfuncs.py:53-64): out = 1 where
 * lo[c] <= HSV(bgr)[c] <= hi[c] for all c, else 0.  lo/hi are HOST arrays. */
int vu_inrange_color(const uint8_t* bgr, int64_t npix, const int32_t lo[3], const int32_t hi[3],
                     uint8_t* mask01, vu_stream_t stream);
/* is_pixel_inrange, bg-image variant (fgfuncs.py:37-52): per-pixel bounds
 * clamp(HSV(bg) -/+ half, 10, 255).  The bg image repeats every bg_npix
 * pixels (bg_npix == npix: one bg per frame; bg_npix == h*w: shared). */
int vu_inrange_image(const uint8_t* bgr, const uint8_t* bgimg, int64_t npix, int64_t bg_npix,
                     const int32_t half[3], uint8_t* mask01, vu_stream_t stream);

/* ---- morphology: dilate_mask / erode_mask, maskprocess.py:7-34 ---------- */
/* grey-scale max/min under cv2 MORPH_ELLIPSE(ksize,ksize), `iters` times,
 * taps outside the image ignored.  ksize 3 runs as ONE pass with the L1
 * diamond of radius `iters`; other sizes ping-pong through `workspace`. */
size_t vu_morph_workspace_bytes(int n, int h, int w, int ksize, int iters);
int vu_morph_u8(const uint8_t* src, uint8_t* dst, int n, int h, int w, int ksize, int iters, int op,
                void* workspace, size_t workspace_bytes, vu_stream_t stream);

/* chains of 3x3-cross passes (== MORPH_ELLIPSE(3,3) with iterations) run in ONE
 * kernel in shared memory: up to 4 segments {ops[i], iters[i]}, <= 12 passes in
 * total, e.g. postprocess' d2,e2,e2,d2 (colorfiltering/agent.py:281-282).  If
 * stats2 != NULL the adaptive threshold of agent.py:277-280 is applied on load
 * (stats2[i] = {sum, count} of frame i, see vu_cf_threshold_stats). */
int vu_cross_chain_u8(const uint8_t* src, uint8_t* dst, int n, int h, int w, int nseg, const int32_t* ops,
                      const int32_t* iters, const uint64_t* stats2, double thr_ratio, vu_stream_t stream);
/* trimap/agent.py:53-58 at working resolution in one kernel:
 * dst = 0 where dilate^iters(src) < 128, 255 where erode^iters(src) > 127, else 128 */
int vu_trimap_core_u8(const uint8_t* src, uint8_t* dst, int n, int h, int w, int iters, vu_stream_t stream);

/* ---- resize: cv2.resize uint8 ------------------------------------------ */
/* default INTER_LINEAR (exact 2x down-scale == rounded 2x2 mean);
 * colorfiltering/agent.py:315-316,342, trimap/agent.py:59 (the "nearest"
 * call that is really bilinear), imgprocess.py:36 */
int vu_resize_linear_u8(const uint8_t* src, int n, int sh, int sw, int channels, uint8_t* dst, int dh, int dw,
                        vu_stream_t stream);
/* INTER_NEAREST; trimap/agent.py:52 */
int vu_resize_nearest_u8(const uint8_t* src, int n, int sh, int sw, int channels, uint8_t* dst, int dh, int dw,
                         vu_stream_t stream);

/* shift_fg: cv2.warpAffine(img, [[1,0,dx],[0,1,dy]], (w,h)) -- fixed-point
 * bilinear translation, taps outside the image read 0 (SURVEY.md A.8).
 * dx / dy are float because the reference stores the matrix as float32.
 * channels is 1 or 3.  unscreen/utils/imgprocess.py:55-64, replace.py:69,71 */
int vu_shift_u8(const uint8_t* src, uint8_t* dst, int n, int h, int w, int channels, float dx, float dy,
                vu_stream_t stream);
/* rescale_fg: cv2.resize(fx=fy=factor, INTER_CUBIC) then the centre crop back
 * to h x w; 1 <= factor <= 16; channels is 1 or 3.
 * unscreen/utils/imgprocess.py:40-52, replace.py:70,72 */
int vu_rescale_cubic_u8(const uint8_t* src, uint8_t* dst, int n, int h, int w, int channels, double factor,
                        vu_stream_t stream);

/* color_correct (unscreen/utils/imgprocess.py:263-300, green.py:120) for a
 * clip, after its two cv2.resize calls: frames_lo [n,th,tw,3] and alpha_lo
 * [n,th,tw] are the frames / alphas resized to the working resolution
 * (vu_resize_linear_u8), alpha [n,h,w] the full-resolution alphas, bg_bgr the
 * background colour (3 bytes, HOST memory), mean_exp the target mean (0.95).
 * out [n,h,w] = uint8(alpha * distance map).  Workspace: device memory. */
size_t vu_color_correct_workspace_bytes(int n, int th, int tw);
int vu_color_correct(const uint8_t* frames_lo, const uint8_t* alpha_lo, const uint8_t* alpha, int n, int h, int w, int th,
                     int tw, const uint8_t* bg_bgr, double mean_exp, uint8_t* out, void* workspace,
                     size_t workspace_bytes, vu_stream_t stream);
/* The same from the full-resolution frames [n,h,w,3], with cv2's down-scale
 * fused in, when the frame is exactly 2x or 4x the working resolution and w is
 * a multiple of 16 (1080p and 4K at target_long_side 960); otherwise
 * VU_ERR_UNSUPPORTED: resize and call vu_color_correct. */
int vu_color_correct_frames(const uint8_t* frames, const uint8_t* alpha, int n, int h, int w, int th, int tw,
                            const uint8_t* bg_bgr, double mean_exp, uint8_t* out, void* workspace,
                            size_t workspace_bytes, vu_stream_t stream);

/* cv2.resize (bilinear) of single-channel maps with the coefficient math hoisted
 * out of the pixel loop.  mode 1 fuses trimap/agent.py:60 (values strictly between
 * 0 and 255 -> 128) and :100 (128 where fuzzy != 0, only for frames with
 * flags[i] == 0).  alt_src / alt_flags (both NULL or both set): frames with
 * alt_flags[i] != 0 are copied from alt_src[n][dh][dw] instead (the early-outs of
 * colorfiltering/agent.py:303-307). */
int vu_resize_up_u8(const uint8_t* src, int n, int sh, int sw, uint8_t* dst, int dh, int dw, int mode,
                    const uint8_t* fuzzy, const uint8_t* flags, const uint8_t* alt_src, const uint8_t* alt_flags,
                    vu_stream_t stream);

/* ---- reductions -------------------------------------------------------- */
/* counts[i] = #{ src[i][j] <op> thr }; exist_foreground (maskprocess.py:56-60),
 * the early-outs of colorfiltering/agent.py:303-307 and trimap/agent.py:88 */
int vu_count_cmp_u8(const uint8_t* src, int n, int64_t per_item, int op, int thr, uint64_t* counts,
                    vu_stream_t stream);
/* counts2[i] = {#{src > thr}, #{src < thr}} in one pass */
int vu_count_gt_lt_u8(const uint8_t* src, int n, int64_t per_item, int thr, uint64_t* counts2, vu_stream_t stream);
/* counts[i][0] = #{a>0 && b>0}, counts[i][1] = #{a>0}; the fuzzy-area ratio
 * of trimap/agent.py:91-94 */
int vu_count_and_u8(const uint8_t* a, const uint8_t* b, int n, int64_t per_item, uint64_t* counts2,
                    vu_stream_t stream);
/* out = a where b == 0 else 0 (trimap/agent.py:97-98: mask[fuzzy] = 0) and
 * out = 128 where b != 0 else a (:100: trimap[fuzzy] = 128) */
int vu_mask_clear_where(const uint8_t* a, const uint8_t* b, uint8_t* out, int64_t count, vu_stream_t stream);
int vu_mask_set128_where(const uint8_t* a, const uint8_t* b, uint8_t* out, int64_t count, vu_stream_t stream);

/* out = 1 where a > 0 && b > 0 else 0 (the fuzzy area itself, :91) */
int vu_mask_and01(const uint8_t* a, const uint8_t* b, uint8_t* out, int64_t count, vu_stream_t stream);
/* trimap/agent.py:90-94 in one pass: fuzzy01 = (alpha > 0) && lo <= HSV(frame) <= hi,
 * counts2[i] = {#fuzzy, #alpha>0} */
int vu_fuzzy_count(const uint8_t* frames, const uint8_t* alpha, int n, int64_t npix, const int32_t lo[3],
                   const int32_t hi[3], uint8_t* fuzzy01, uint64_t* counts2, vu_stream_t stream);
/* trimap/agent.py:52 (INTER_NEAREST down-scale) with :97-98 fused:
 * out[y][x] = (flags[i] == 0 && fuzzy[sy][sx]) ? 0 : mask[sy][sx]; fuzzy/flags may both be NULL */
int vu_trimap_src_lo(const uint8_t* mask, const uint8_t* fuzzy, const uint8_t* flags, int n, int h, int w, int th,
                     int tw, uint8_t* out, vu_stream_t stream);
/* generate_trimap, trimap/agent.py:54-58: out = 0 where dilated < 128, else
 * 255 where eroded > 127, else 128 */
/* The whole trimap tail (trimap/agent.py:52-60 and :97, :100) for frames that are an exact 2x or 4x of the working
 * resolution th x tw, MORPH_ELLIPSE(3,3): nearest down-scale of mask [n,h,w] (fuzzy pixels cleared first in frames
 * with flags[i] == 0), `iters` cross dilations / erosions, classification, bilinear up-scale, snap, fuzzy -> 128,
 * all in bit logic (see vu_trimap_bits.cu).  fuzzy / flags may both be NULL.  workspace: vu_trimap_bits_workspace_bytes.
 * VU_ERR_UNSUPPORTED for other scales, tw % 4 != 0, iters > 12 or pointers that are not 16-byte aligned. */
size_t vu_trimap_bits_workspace_bytes(int n, int th, int tw);
int vu_trimap_bits(const uint8_t* mask, const uint8_t* fuzzy, const uint8_t* flags, int n, int h, int w, int th, int tw,
                   int iters, uint8_t* out, void* workspace, size_t workspace_bytes, vu_stream_t stream);

/* The same tail from bit planes (no full-resolution byte map is read): mask_bits [n][th][tw/8] = (nearest-sampled
 * mask >= 128) at the working resolution, fuzzy_bits [n][h][w/8] = one bit per full-resolution pixel (bit i of byte j =
 * pixel 8j + i), as vu_cf_alpha_up_fuzzy writes them; fuzzy_bits / flags may both be NULL.  tw % 16 == 0.  The
 * reference's iters == 5 at tw % 32 == 0, tw <= 1024 (every input_long_side of the agents) runs the marching kernel, one
 * warp per band of rows; VU_TRIMAP_MARCH=0 in the environment keeps the tile kernel (same bytes). */
int vu_trimap_bits_packed(const uint8_t* mask_bits, const uint8_t* fuzzy_bits, const uint8_t* flags, int n, int h, int w,
                          int th, int tw, int iters, uint8_t* out, void* workspace, size_t workspace_bytes,
                          vu_stream_t stream);

/* The second full-resolution pass of the green-screen loop for frames that are an exact 2x / 4x of the working
 * resolution th x tw (tw % 16 == 0), in one kernel:
 *   alpha      = cv2.resize(alpha_lo, (w, h)), colorfiltering/agent.py:342; frames with alt_flags[i] != 0 (the
 *                early-outs of :303-307) are copied from alt_src [n][h][w] instead (both NULL or both set);
 *   fuzzy_bits = (alpha > 0) && lo <= BGR2HSV(frame) <= hi, trimap/agent.py:84-91 (is_pixel_inrange with a background
 *                colour, utils/fgfuncs.py:55-64), one bit per pixel, [n][h][w/8];
 *   counts2[i] = {#fuzzy, #(alpha > 0)}, trimap/agent.py:92-94;
 *   mask_bits  = alpha[SC*y][SC*x] >= 128, the nearest down-scale of trimap/agent.py:52 as bits, [n][th][tw/8];
 *   fg_out / bg_out (both NULL or both set, with bg_bgr = 3 HOST bytes): tools/unscreen/green.py:125-126,
 *                bgimg = bg colour, bgimg[alpha < 128] = frame[alpha < 128], fg = get_fg(frame, alpha, bgimg)
 *                (utils/fgfuncs.py:84-110).
 * The frame is only read where the matte is non-zero (everywhere when fg_out is set).  Feed mask_bits / fuzzy_bits /
 * ratio flags of counts2 to vu_trimap_bits_packed. */
int vu_cf_alpha_up_fuzzy(const uint8_t* alpha_lo, int n, int th, int tw, int h, int w, const uint8_t* alt_src,
                         const uint8_t* alt_flags, const uint8_t* frames, const int32_t lo[3], const int32_t hi[3],
                         uint8_t* alpha, uint8_t* fuzzy_bits, uint8_t* mask_bits, uint64_t* counts2,
                         const uint8_t* bg_bgr, uint8_t* fg_out, uint8_t* bg_out, vu_stream_t stream);
int vu_trimap_classify(const uint8_t* dilated, const uint8_t* eroded, uint8_t* out, int64_t count,
                       vu_stream_t stream);
/* trimap/agent.py:60: values strictly between 0 and 255 become 128 */
int vu_trimap_snap(const uint8_t* a, int64_t count, uint8_t* out, vu_stream_t stream);

/* per-frame branches taken on the device (batched clips, no host round trip):
 * flags[i] = 2 if counts2[i][1] == 0 (trimap/agent.py:88: mask returned as is),
 * 1 if float(counts2[i][0]) / counts2[i][1] > thr (:94: trust the mask), else 0 */
int vu_ratio_flags(const uint64_t* counts2, int n, double thr, uint8_t* flags, vu_stream_t stream);
/* colorfiltering/agent.py:303-307: flags[i] = 1 if nfg[i] < fg_min, 2 if nbg[i] < bg_min, else 0;
 * nfg / nbg are read with a stride of `stride` uint64 (1: two arrays, 2: the interleaved output of vu_count_gt_lt_u8) */
int vu_cf_degenerate_flags(const uint64_t* nfg, const uint64_t* nbg, int n, int stride, uint64_t fg_min,
                           uint64_t bg_min, uint8_t* flags, vu_stream_t stream);
/* out[i] = flags[i] ? a[i] : b[i] for whole frames of per_item bytes */
int vu_select_frames(const uint8_t* a, const uint8_t* b, const uint8_t* flags, int n, int64_t per_item,
                     uint8_t* out, vu_stream_t stream);
/* out = 128 where flags[i] == 0 && b != 0, else a (trimap/agent.py:100 on the ensemble branch only) */
int vu_set128_unflagged(const uint8_t* a, const uint8_t* b, const uint8_t* flags, int n, int64_t per_item,
                        uint8_t* out, vu_stream_t stream);

/* ---- colour filtering: ColorFilteringAgent, colorfiltering/agent.py ----- */
/* get_alpha_by_gmm (:232-257) with the six 1-D mixtures folded into 256-entry
 * float32 tables (luts = [bg H,S,V, fg H,S,V][256], DEVICE): per pixel
 * bg = (lutH[h]*lutS[s])*lutV[v], same for fg, p = fg^(1/3f) / (bg^(1/3f) +
 * fg^(1/3f) + 1e-6), alpha = u8(clip(p*255)). */
/* The training samples of the mixtures gathered on the device, order-exact (colorfiltering/agent.py:139-141,
 * 165-167, 192-194): samples = channel[selection] in row-major order, every (len // max_samples)-th of them when
 * there are more than max_samples, for the three channels of hsv [h,w,3] under ONE selection
 *   selection = (mask_op == 0 ? mask < 128 : mask > 128) && prior
 *   prior_mode 0: none   1: prior_lo < H < prior_hi   2: !(prior_lo < H < prior_hi)       (get_color_prior's interval)
 * samples: [3][cap] bytes (cap >= 2 * max_samples); meta3 = {selected pixels, stride, samples per channel};
 * hist256 = histogram of the H samples kept (agent.py:142-143).  workspace: vu_cf_samples_workspace_bytes(h). */
size_t vu_cf_samples_workspace_bytes(int h);
int vu_cf_samples(const uint8_t* hsv, const uint8_t* mask, int h, int w, int mask_op, int prior_mode, int prior_lo,
                  int prior_hi, int max_samples, uint8_t* samples, int cap, int32_t* meta3, uint32_t* hist256,
                  void* workspace, size_t workspace_bytes, vu_stream_t stream);
int vu_cf_alpha_u8(const uint8_t* hsv, int64_t npix, const float* luts, uint8_t* alpha, vu_stream_t stream);
/* the same function tabulated over every (h<180, s, v): lut3d[180][256][256] */
int vu_cf_build_lut3d(const float* luts, uint8_t* lut3d, vu_stream_t stream);
int vu_cf_alpha_lut3d_u8(const uint8_t* hsv, int64_t npix, const uint8_t* lut3d, uint8_t* alpha,
                         vu_stream_t stream);
/* one pass over the full-resolution frames: BGR2HSV (:310) + cv2.resize of the
 * HSV image and the mask for exact 2x / 4x down-scales (:315-316) + tabulated
 * get_alpha_by_gmm (:319) + the statistics of postprocess (:277-279).
 * h == s*th, w == s*tw, s in {2,4}; anything else returns VU_ERR_UNSUPPORTED and
 * the caller composes the stage from the primitives above. */
int vu_cf_lowres(const uint8_t* frames, const uint8_t* masks, int n, int h, int w, int th, int tw,
                 const uint8_t* lut3d, uint8_t* alpha_lo, uint64_t* stats2, uint64_t* mask_counts2, vu_stream_t stream);
/* mask_counts2 (nullable): per frame {#(mask > 128), #(mask < 128)}, the early-out counts of agent.py:303-307, taken
 * from the mask bytes this pass reads (at s == 4 it then reads all four rows of the mask); w % 16 == 0 and 16-byte aligned inputs
 * (VU_ERR_UNSUPPORTED otherwise: use vu_count_gt_lt_u8). */
/* postprocess (:259-283) step 1: per frame sum/count of alpha over
 * (alpha>128 && mask>0) -> stats[i] = {sum, count}; step 2 zeroes alpha below
 * 0.8 * sum/count (f64; count==0 leaves alpha untouched).  The d2,e2,e2,d2
 * morphology that follows is four vu_morph_u8 calls. */
int vu_cf_threshold_stats(const uint8_t* alpha, const uint8_t* mask, int n, int64_t per_item, uint64_t* stats2,
                          vu_stream_t stream);
int vu_cf_threshold_apply(const uint8_t* alpha, int n, int64_t per_item, const uint64_t* stats2, double thr_ratio,
                          uint8_t* out, vu_stream_t stream);
/* ---- compositing -------------------------------------------------------- */
/* get_fg, fgfuncs.py:84-110, optionally fused with the predicated background
 * patch of green.py:125 (ALPHA_LT128) or bg.py:99 / bg_offline.py:171
 * (ALPHA_EQ0).  bg repeats every bg_npix pixels.  If bg_out != NULL the
 * patched background is also written (green.py saves it). */
int vu_get_fg(const uint8_t* frame, const uint8_t* alpha, const uint8_t* bg, int64_t npix, int64_t bg_npix,
              int patch_mode, uint8_t* fg_out, uint8_t* bg_out, vu_stream_t stream);
/* get_bg, fgfuncs.py:113-137 */
int vu_get_bg(const uint8_t* alpha, const uint8_t* bg, int64_t npix, uint8_t* out, vu_stream_t stream);
/* float64 blends (see vu_blend_mode).  alpha_channels is 1 (HW mask) or 3
 * (HWC mask, replace.py).  bg repeats every bg_npix pixels; may be NULL for
 * VU_BLEND_NAIVE.  out may be fg (in place).  The bytes are those of the
 * reference's float64 expression in every case; FUSE / REPLACE with one
 * alpha channel, 16-byte aligned buffers, npix % 16 == 0 and an out that
 * overlaps no input take the integer kernel (float64 only where the
 * quotient is exact); VU_BLEND_FP64=1 in the environment keeps the float64
 * kernel for them too. */
int vu_blend(int mode, const uint8_t* fg, const uint8_t* alpha, int alpha_channels, const uint8_t* bg,
             int64_t npix, int64_t bg_npix, uint8_t* out, vu_stream_t stream);
/* bg_offline.py:150-151: u8(f32(bg)*beta + (1-beta)*f32(bg_always)) */
int vu_fuse_bg(const uint8_t* bg, const uint8_t* bg_always, int64_t npix, int64_t always_npix, float beta,
               float one_minus_beta, uint8_t* out, vu_stream_t stream);
/* bg.py:85-88 == bg_offline.py:154-157: g = BGR2GRAY(|frame-bg|); g[g>thr]=255 */
int vu_bgdiff_gray(const uint8_t* frame, const uint8_t* bg, int64_t npix, int64_t bg_npix, int thr, uint8_t* gray,
                   vu_stream_t stream);
/* bg.py:85-92 == bg_offline.py:154-160 in one pass over n frames: out = mask * (dilate_mask(g, 4, 2) // 255) with
 * g = BGR2GRAY(|frame - bg|), g[g > thr] = 255.  bg is one [h,w,3] image (bg_frames == 1) or one per frame
 * (bg_frames == n).  Needs w % 4 == 0 and 4-byte aligned pointers. */
int vu_bgdiff_gate(const uint8_t* frames, const uint8_t* bg, const uint8_t* masks, int n, int h, int w, int bg_frames,
                   int thr, uint8_t* out, vu_stream_t stream);
/* bg.py:92 == bg_offline.py:160: out = mask * (g // 255) (uint8 wrap-free) */
int vu_gate(const uint8_t* mask, const uint8_t* g, int64_t count, uint8_t* out, vu_stream_t stream);
/* bg.py:74-76: >128 -> 255 else 0 */
int vu_binarise(const uint8_t* alpha, int64_t count, int thr, uint8_t* out, vu_stream_t stream);
/* get_outer_boundary tail, maskprocess.py:73: out = a - b (uint8 wrap) */
int vu_sub_wrap_u8(const uint8_t* a, const uint8_t* b, int64_t count, uint8_t* out, vu_stream_t stream);

/* ---- temporal background ------------------------------------------------ */
/* exact per-element median over n frames of m bytes each (NEW SPEC, SURVEY.md
 * section 8 a23; oracle np.median(stack,0).astype(u8)): even n ->
 * (sorted[n/2-1] + sorted[n/2]) >> 1.  1 <= n <= 65535. */
int vu_temporal_median_u8(const uint8_t* frames, int n, int64_t m, uint8_t* out, vu_stream_t stream);
/* the same with caller-provided scratch memory (device, vu_temporal_median_workspace_bytes(n, m) bytes; 0 for
 * n <= 608): clips of more than 608 frames then take the estimate + streaming-refine path instead of histograms */
size_t vu_temporal_median_workspace_bytes(int n, int64_t m);
int vu_temporal_median_u8_ws(const uint8_t* frames, int n, int64_t m, uint8_t* out, void* workspace,
                             size_t workspace_bytes, vu_stream_t stream);
/* masked temporal mean, bg_offline.py:106-125.  masks are the ALREADY DILATED
 * single-channel masks [n][h*w] (dilate_mask(mask,3,2) is a vu_morph_u8 call).
 * bg_out[h*w*3], mask_always_out[h*w] (255 where count <= min_count). */
int vu_masked_temporal_mean(const uint8_t* frames, const uint8_t* masks, int n, int64_t npix, int min_count,
                            uint8_t* bg_out, uint8_t* mask_always_out, vu_stream_t stream);
/* The same from the RAW masks, with dilate_mask(mask, 3, 2) (bg_offline.py:116)
 * fused in as two bit-plane dilations: the dilated masks never exist.
 * w % 16 == 0 and 16-byte aligned pointers, else VU_ERR_UNSUPPORTED (dilate with
 * vu_morph_u8, then vu_masked_temporal_mean). */
int vu_masked_temporal_mean_dilate32(const uint8_t* frames, const uint8_t* masks, int n, int h, int w, int min_count,
                                     uint8_t* bg_out, uint8_t* mask_always_out, vu_stream_t stream);

/* Streamed temporal median: the clip is added in chunks, in any chunking and any order, and the finish writes the
 * bytes vu_temporal_median_u8 writes for the whole clip (np.median(stack, 0).astype(u8)).  The state is
 * vu_median_accum_bytes(m) bytes of device memory (512 per frame byte, rounded up to 128-byte tiles; 3.2 GB at 1080p,
 * 12.7 GB at 4K), 16-byte aligned, whatever the clip length; its layout is private to these calls.
 *   reset:  zero the state (an add with n_before == 0 overwrites it anyway, except an add captured into a CUDA graph,
 *           which always accumulates: its replays add to whatever the state holds, and the caller counts them).
 *   add:    frames [k][m] (any m, any alignment: 4-byte aligned rows with m % 4 == 0 take the vector loads); n_before
 *           = frames added since the reset, tracked by the caller.  VU_ERR_INVALID_ARG, state untouched, when k < 1 or
 *           n_before + k > 65535: the counters are 16 bits, so a state holds at most 65535 frames.
 *   finish: out [m] = the median of the n frames added (1 <= n <= 65535): odd n order statistic (n + 1) / 2, even n
 *           (s[n/2 - 1] + s[n/2]) >> 1.  The state is left as it was.
 * Each add reads and writes the whole state (~1024 * m bytes) besides its k * m bytes of frames: add in chunks of
 * hundreds of frames. */
size_t vu_median_accum_bytes(int64_t m);
int vu_median_accum_reset(void* state, int64_t m, vu_stream_t stream);
int vu_median_accum_add_u8(void* state, int64_t m, const uint8_t* frames, int k, int n_before, vu_stream_t stream);
int vu_median_accum_finish_u8(const void* state, int64_t m, int n, uint8_t* out, vu_stream_t stream);

/* Streamed masked temporal mean, bg_offline.py:106-125 as the script runs it - a sum and a count accumulated frame by
 * frame inside the read loop.  Any chunking and order gives the bytes of vu_masked_temporal_mean[_dilate32] on the
 * whole clip.  State: vu_masked_mean_accum_bytes(h, w) = 16 bytes per pixel (uint32 sums of B, G, R and the count),
 * 16-byte aligned, layout private; at most 16,000,000 frames in all (the sums are 32 bits).
 *   add_dilate32: frames [k][h][w][3] and the RAW masks [k][h][w], dilate_mask(mask, 3, 2) (bg_offline.py:116) fused
 *                 in as in vu_masked_temporal_mean_dilate32; w % 16 == 0 and 16-byte aligned frames / masks, else
 *                 VU_ERR_UNSUPPORTED (dilate with vu_morph_u8, then add).
 *   add:          the ALREADY DILATED masks [k][npix]; any npix and alignment.
 *   finish:       bg_out [npix][3], mask_always_out [npix] as vu_masked_temporal_mean (255 where count <= min_count,
 *                 bg 0 there).  The state is left as it was. */
size_t vu_masked_mean_accum_bytes(int h, int w);
int vu_masked_mean_accum_reset(void* state, int h, int w, vu_stream_t stream);
int vu_masked_mean_accum_add_dilate32(void* state, const uint8_t* frames, const uint8_t* masks, int k, int h, int w,
                                      vu_stream_t stream);
int vu_masked_mean_accum_add(void* state, const uint8_t* frames, const uint8_t* masks_dilated, int k, int64_t npix,
                             vu_stream_t stream);
int vu_masked_mean_accum_finish(const void* state, int64_t npix, int min_count, uint8_t* bg_out, uint8_t* mask_always_out,
                                vu_stream_t stream);

/* One pass per frame of the bg_step live loop, tools/unscreen/bg_offline.py:154-160 + :171-172 (== bg.py:85-92, :99-100):
 * alpha = mask * (dilate_mask(g, 4, 2) // 255) with g = thresholded BGR2GRAY(|frame - bg|) (the difference gate of
 * vu_bgdiff_gate), fg = get_fg(frame, alpha, bgimg) with bgimg[alpha == 0] = frame[alpha == 0] (vu_get_fg with
 * VU_PATCH_ALPHA_EQ0), and - mask_bits != NULL, scale = 2 or 4 - the bits alpha[scale*y][scale*x] >= 128 that
 * vu_trimap_bits_packed turns into the trimap of :166.  frames [n][h][w][3], bg [bg_frames][h][w][3] (1 or n), masks /
 * alpha [n][h][w], fg [n][h][w][3], mask_bits [n][h/scale][w/scale/8].  The frame and the background are fetched
 * once, as TMA tiles with halo.  w % 16 == 0 and 16-byte aligned buffers, else VU_ERR_UNSUPPORTED (use the two
 * separate entry points). */
int vu_bgstep_frames(const uint8_t* frames, const uint8_t* bg, const uint8_t* masks, int n, int h, int w, int bg_frames,
                     int thr, uint8_t* alpha, uint8_t* fg, uint8_t* mask_bits, int scale, vu_stream_t stream);

/* ---- BackgroundAgent (unscreen/bgmodel/agent.py), methods 'mean' and 'pcov' ---- */
/* get_fgbox (utils/maskprocess.py:37-53): out4 = {min row, max row, min column, max column} of mask > 0
 * ({INT_MAX, -1, INT_MAX, -1} for an empty mask) */
int vu_mask_bbox(const uint8_t* mask, int h, int w, int32_t* out4, vu_stream_t stream);
/* get_mean_bg (bgmodel/agent.py:80-88): out4 = {sum ch0, sum ch1, sum ch2, count} of img [npix][3] over mask > 0
 * (mask NULL: all pixels) */
int vu_masked_sum3(const uint8_t* img, const uint8_t* mask, int64_t npix, uint64_t* out4, vu_stream_t stream);
/* one round of get_bg_by_pcov (bgmodel/agent.py:118-129) on the rh x rw box around the hole: normalised ksize x ksize
 * cv2.boxFilter (BORDER_REFLECT_101) of the image and of the validity map, mean / validity where the window saw a
 * valid pixel.  first != 0: img_in / valid_in are the image and the DILATED MASK at the box's origin (row pitch
 * in_pitch_px pixels; mask > 0 = hole: zero, invalid); later rounds read the dense rh x rw outputs of the round before
 * (in_pitch_px = rw).  flags [101] uint32, zeroed by the caller before round 0: round r sets flags[r + 1] when it
 * leaves an invalid pixel and returns at once when flags[r] == 0 (r > 0), so rounds can be enqueued ahead. */
int vu_pcov_round(const uint8_t* img_in, const uint8_t* valid_in, int in_pitch_px, int first, int rh, int rw, int ksize,
                  uint8_t* img_out, uint8_t* valid_out, uint32_t* flags, int round, vu_stream_t stream);

/* ---- remove_invalid_objects (unscreen/utils/maskprocess.py:77-152; green.py:106-109, bg.py:67,93, bg_offline.py:76,165) ----
 * out = alpha with every pixel cleared that no valid contour paints: the contours of cv2.findContours(alpha, RETR_LIST)
 * (outer borders of the 8-connected components of alpha > 0 and the borders of their holes) with contourArea >= 100 whose
 * filled polygon scores saliency = sum(score_map under it) / (h w) and consensus = mean(segmask under it) / 255 with
 * (saliency > saliency_thr && consensus > consensus_thr) || saliency > 10 saliency_thr.  alpha, segmask, out: [n][h][w]
 * (segmask = alpha for the one-argument form of the reference); score_map: [h][w] float64 (get_score_map, :155-178), shared by
 * the frames.  status[i] = number of contours of frame i; a frame with more than max_objects contours has
 * status[i] > max_objects and an undefined output: call again with a larger workspace.  Nesting may be of any depth.  Everything
 * stays on the device.  workspace: vu_remove_objects_workspace_bytes(n, h, w, max_objects), 16-byte aligned. */
size_t vu_remove_objects_workspace_bytes(int n, int h, int w, int max_objects);
int vu_remove_invalid_objects(const uint8_t* alpha, const uint8_t* segmask, const double* score_map, int n, int h, int w,
                              double saliency_thr, double consensus_thr, uint8_t* out, int32_t* status, void* workspace,
                              size_t workspace_bytes, int max_objects, vu_stream_t stream);

/* regionfill (unscreen/utils/region_fill.py:26-63; BackgroundAgent 'rf', bgmodel/agent.py:133-157; bg.py:79): the masked
 * pixels of x [planes][h][w] (float64, in place; the planes share mask [h][w], > 0 = fill) become the solution of the
 * discrete Laplace equation whose boundary data are the pixels outside the mask (every masked pixel = the mean of its
 * in-image 4-neighbours).  The reference builds the sparse matrix and calls scipy's direct solver; this is conjugate
 * gradients in float64, stopped at |r| <= tol |b| or after max_iters iterations: parity is a tolerance (tol 1e-10: ~1e-6
 * grey levels on a 1080p person-sized hole).  snap_eps > 0: filled values within snap_eps of an integer become that integer
 * (the reference truncates the result to uint8, and exact-integer solutions -- isolated pixels, flat boundaries -- come out of
 * the direct solver exactly; 1e-6 with tol 1e-10).  HOST-SYNCHRONOUS on `stream` (the residuals are read every 64 iterations);
 * iters_out / resid_out (host pointers, may be NULL) receive the iterations done and the final max |r| / |b|. */
size_t vu_regionfill_workspace_bytes(int planes, int h, int w);
int vu_regionfill_f64(double* x, const uint8_t* mask, int planes, int h, int w, double tol, int max_iters, double snap_eps, void* workspace,
                      size_t workspace_bytes, int32_t* iters_out, double* resid_out, vu_stream_t stream);
/* cv2.resize of float64 planes with the default INTER_LINEAR (region_fill.py:10-15): scale_x / scale_y are the sampling
 * steps (1 / fx for the `(0, 0), fx=` form, else src / dst size); exactly 2 in both axes = cv2's INTER_AREA shortcut.
 * keep_mask [dh][dw] / keep_src [planes][dh][dw] (both or neither): where keep_mask == 0 the output is keep_src
 * (region_fill.py:16). */
int vu_resize_linear_f64(const double* src, int planes, int sh, int sw, double* dst, int dh, int dw, double scale_x, double scale_y,
                         const uint8_t* keep_mask, const double* keep_src, vu_stream_t stream);

/* ---- frame I/O glue (unscreen/utils/fileio.py:31-62): the JPEG codec itself is nvJPEG (library code); these convert
 * between its planar RGB [3][npix] and the reference's interleaved BGR [npix][3] ---- */
int vu_planar_rgb_to_bgr(const uint8_t* src, uint8_t* dst, int64_t npix, vu_stream_t stream);
int vu_bgr_to_planar_rgb(const uint8_t* src, uint8_t* dst, int64_t npix, vu_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VU_B200_H */
