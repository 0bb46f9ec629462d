// remove_invalid_objects (unscreen/utils/maskprocess.py:77-152; called between colour filtering and the trimap in all
// three pipeline scripts: green.py:106-109, bg.py:67,93, bg_offline.py:76,165) on the device, batched over frames.
//
// The reference walks cv2.findContours(alpha, RETR_LIST), and for every contour with contourArea >= 100 paints it
// FILLED, sums a saliency map and the segmentation mask under the paint, and keeps the paint if the scores pass.  What
// those cv2 calls compute has a closed form (oracle/refport.py:contour_objects, checked against cv2 on thousands of
// shapes): contours = outer borders of the 8-connected foreground components + borders of the holes (4-connected
// background components other than the outside); a filled outer border covers the component and everything it
// encloses; a filled hole border covers the hole, everything inside it and the ring of component pixels 4-adjacent to
// it; contourArea follows from Pick's theorem with the chain length B = L - n1 (outer; L = pixel edges of the filled
// region, n1 = 2x2 windows with one pixel of it) or B = L - n3 (hole).  So the whole function is
//
//   1. connected components of both classes (union-find on one forest: foreground 8-connected, background 4-connected,
//      node 0 = everything outside the image; a set's root is its first pixel in raster order),
//   2. the nesting tree: the parent of a component is the set of the pixel left of its first pixel,
//   3. per-set sums (pixels, saliency, mask) and local boundary counts (L, n1 / n3, ring sums) in one pass,
//   4. subtree totals, areas, scores, validity and "is painted by a valid ancestor" on the (small) tree: one CTA per frame,
//   5. out = alpha where the pixel's component is painted or the pixel sits on the ring of a valid hole, else 0.
//
// Nothing returns to the host.  Sums of the saliency map are float64 atomics: a score within ~1e-12 (relative) of its
// threshold could be decided differently from numpy's pairwise sum; everything else is integer-exact.
#include "vu_common.cuh"

namespace vu {
namespace {

constexpr int OT = 256;

struct ObjWs {   // per-frame slices of the workspace
  int* P;        // [npix + 1] union-find parent, then the label (root) of every node; node = pixel index + 1, node 0 = outside
  int* dense;    // [npix + 1] dense index of a root node
  int* nroots;   // [1]
  int* overflow; // [1]
  // per root, [cap]
  int* node; int* up; unsigned* size; unsigned long long* seg; double* score;
  unsigned* L; unsigned* nw; unsigned* rcnt; unsigned long long* rseg; double* rscore;
  int* depth; unsigned char* keep; unsigned char* vhole;
};

__host__ __device__ inline size_t align_up(size_t v) { return (v + 15) & ~(size_t)15; }
__host__ __device__ inline size_t ws_frame_bytes(int64_t npix, int cap) {
  return 2 * align_up((npix + 1) * sizeof(int)) + align_up(2 * sizeof(int) + 8) +
         align_up((size_t)cap * (sizeof(int) * 3 + sizeof(unsigned) * 4 + sizeof(unsigned long long) * 2 + sizeof(double) * 2 + 2));
}
__host__ __device__ inline ObjWs ws_of(void* base, int frame, int64_t npix, int cap) {
  char* p = static_cast<char*>(base) + (size_t)frame * ws_frame_bytes(npix, cap);
  ObjWs w;
  w.P = reinterpret_cast<int*>(p); p += align_up((npix + 1) * sizeof(int));
  w.dense = reinterpret_cast<int*>(p); p += align_up((npix + 1) * sizeof(int));
  w.nroots = reinterpret_cast<int*>(p); w.overflow = w.nroots + 1; p += align_up(2 * sizeof(int) + 8);
  w.seg = reinterpret_cast<unsigned long long*>(p); p += (size_t)cap * 8;
  w.rseg = reinterpret_cast<unsigned long long*>(p); p += (size_t)cap * 8;
  w.score = reinterpret_cast<double*>(p); p += (size_t)cap * 8;
  w.rscore = reinterpret_cast<double*>(p); p += (size_t)cap * 8;
  w.node = reinterpret_cast<int*>(p); p += (size_t)cap * 4;
  w.up = reinterpret_cast<int*>(p); p += (size_t)cap * 4;
  w.depth = reinterpret_cast<int*>(p); p += (size_t)cap * 4;
  w.size = reinterpret_cast<unsigned*>(p); p += (size_t)cap * 4;
  w.L = reinterpret_cast<unsigned*>(p); p += (size_t)cap * 4;
  w.nw = reinterpret_cast<unsigned*>(p); p += (size_t)cap * 4;
  w.rcnt = reinterpret_cast<unsigned*>(p); p += (size_t)cap * 4;
  w.keep = reinterpret_cast<unsigned char*>(p); p += cap;
  w.vhole = reinterpret_cast<unsigned char*>(p);
  return w;
}

__device__ __forceinline__ int uf_find(int* P, int i) {
  int p = P[i];
  while (p != i) {          // path halving: every write moves a node closer to its root, races are benign
    const int g = P[p];
    if (g != p) P[i] = g;
    i = p;
    p = g;
  }
  return i;
}
__device__ __forceinline__ void uf_unite(int* P, int a, int b) {
  while (true) {
    a = uf_find(P, a);
    b = uf_find(P, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }   // link the larger root under the smaller: a root is its set's first node
    const int old = atomicMin(&P[a], b);
    if (old == a) return;
    a = old;
  }
}

// one CTA per row: every pixel starts as a child of the first pixel of its horizontal run of equal class, so the forest
// is shallow before the vertical links go in
__global__ void __launch_bounds__(OT) obj_init_kernel(const uint8_t* __restrict__ alpha, int h, int w, void* wsbase, int cap) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.y, npix, cap);
  const uint8_t* a = alpha + (int64_t)blockIdx.y * npix;
  const int y = blockIdx.x;
  __shared__ int carry_start, carry_cls;   // the run that reaches the end of the pixels handled so far
  if (threadIdx.x == 0) { carry_start = -1; carry_cls = -1; }
  if (y == 0 && threadIdx.x == 0) {
    ws.P[0] = 0;
    *ws.nroots = 0;
    *ws.overflow = 0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  for (int x0 = 0; x0 < w; x0 += OT) {
    const int x = x0 + threadIdx.x;
    const bool in = x < w;
    const int cls = in ? (int)(a[(int64_t)y * w + x] != 0) : 2 + lane;   // pixels past the row end: classes of their own
    const int prev = __shfl_up_sync(0xffffffffu, cls, 1);
    const bool brk = lane == 0 || prev != cls;                           // a run starts here, as far as the warp can tell
    const unsigned bm = __ballot_sync(0xffffffffu, brk);
    const int s = 31 - __clz(bm & (0xFFFFFFFFu >> (31 - lane)));         // lane where my run starts within the warp
    int start = x0 + wp * 32 + s;
    // the warps take turns: a run that starts at lane 0 may continue the run the previous warp (or segment) ended with
    for (int k = 0; k < OT / 32; ++k) {
      if (wp == k) {
        if (s == 0 && carry_cls == cls) start = carry_start;
        const int last_start = __shfl_sync(0xffffffffu, start, 31), last_cls = __shfl_sync(0xffffffffu, cls, 31);
        __syncwarp();
        if (lane == 0) { carry_start = last_start; carry_cls = last_cls; }
      }
      __syncthreads();
    }
    if (in) ws.P[(int64_t)y * w + x + 1] = y * w + start + 1;
  }
}

// vertical and diagonal links (foreground: N, NW, NE, background: N) between run starts, and the frame: background pixels
// on the image border belong to the outside (node 0)
__global__ void __launch_bounds__(OT) obj_merge_kernel(const uint8_t* __restrict__ alpha, int h, int w, void* wsbase, int cap) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.y, npix, cap);
  const uint8_t* a = alpha + (int64_t)blockIdx.y * npix;
  for (int64_t i = (int64_t)blockIdx.x * OT + threadIdx.x; i < npix; i += (int64_t)gridDim.x * OT) {
    const int y = (int)(i / w), x = (int)(i - (int64_t)y * w);
    const bool fg = a[i] != 0;
    const int me = (int)i + 1;
    if (fg) {
      if (y > 0) {
        const uint8_t* up = a + i - w;
        // a link to N makes the links to NW / NE redundant when those are foreground too (they are joined to N by the run)
        if (up[0]) uf_unite(ws.P, me, me - w);
        else {
          if (x > 0 && up[-1]) uf_unite(ws.P, me, me - w - 1);
          if (x + 1 < w && up[1]) uf_unite(ws.P, me, me - w + 1);
        }
      }
    } else {
      if (y > 0 && a[i - w] == 0) {
        // only one link per pair of runs is needed: link where the run above starts or mine starts
        if (x == 0 || a[i - 1] != 0 || a[i - w - 1] != 0) uf_unite(ws.P, me, me - w);
      }
      if (x == 0 || y == 0 || x == w - 1 || y == h - 1) uf_unite(ws.P, me, 0);
    }
  }
}

// labels (roots) for every node; roots get a dense index and their parent in the nesting tree
__global__ void __launch_bounds__(OT) obj_flatten_kernel(const uint8_t* __restrict__ alpha, int h, int w, void* wsbase, int cap) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.y, npix, cap);
  for (int64_t i = (int64_t)blockIdx.x * OT + threadIdx.x; i < npix; i += (int64_t)gridDim.x * OT) {
    const int me = (int)i + 1;
    // read-only walk: a path-halving find here would let another thread overwrite my final label with a mere ancestor
    // (it writes into the nodes it passes); every entry only ever moves towards the root, so reading while others write
    // their roots is safe
    int r = me;
    for (int p = ws.P[r]; p != r; p = ws.P[r]) r = p;
    ws.P[me] = r;
    if (r == me) {
      const int k = atomicAdd(ws.nroots, 1);
      if (k < cap) {
        ws.dense[me] = k;
        ws.node[k] = me;
        ws.size[k] = 0; ws.seg[k] = 0; ws.score[k] = 0.0; ws.L[k] = 0; ws.nw[k] = 0; ws.rcnt[k] = 0; ws.rseg[k] = 0; ws.rscore[k] = 0.0;
        ws.depth[k] = 0; ws.keep[k] = 0; ws.vhole[k] = 0;
      } else {
        *ws.overflow = 1;
      }
    }
  }
}

// the parent of a root = the set of the pixel left of it (outside the image: node 0); needs every label final
__global__ void __launch_bounds__(OT) obj_parent_kernel(int h, int w, void* wsbase, int cap) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.y, npix, cap);
  const int nr = min(*ws.nroots, cap);
  for (int k = blockIdx.x * OT + threadIdx.x; k < nr; k += gridDim.x * OT) {
    const int me = ws.node[k];
    const int x = (me - 1) % w;
    int parent = 0;
    if (x > 0) parent = ws.P[me - 1];
    ws.up[k] = parent == 0 ? -1 : ws.dense[parent];
  }
}

__device__ __forceinline__ int label_at(const ObjWs& ws, int h, int w, int x, int y) {   // 0 outside the image
  return ((unsigned)x < (unsigned)w && (unsigned)y < (unsigned)h) ? ws.P[y * w + x + 1] : 0;
}

// per-set sums and the local boundary counts.  Thread (x, y), x in -1 .. w-1, y in -1 .. h-1, owns: pixel (x, y)'s own
// sums and ring contributions, the pixel edges to its right and below (and the image's left / top edges), and the 2x2
// window whose top-left corner it is (windows reach one pixel outside the image).
__global__ void __launch_bounds__(OT) obj_stats_kernel(const uint8_t* __restrict__ alpha, const uint8_t* __restrict__ segmask,
                                                       const double* __restrict__ score_map, int h, int w, void* wsbase, int cap) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.y, npix, cap);
  if (*ws.overflow) return;
  const uint8_t* a = alpha + (int64_t)blockIdx.y * npix;
  const uint8_t* sg = segmask + (int64_t)blockIdx.y * npix;
  const int W1 = w + 1;
  const int64_t total = (int64_t)(h + 1) * W1;
  for (int64_t t = (int64_t)blockIdx.x * OT + threadIdx.x; t < total; t += (int64_t)gridDim.x * OT) {
    const int y = (int)(t / W1) - 1, x = (int)(t % W1) - 1;
    // labels of the window (x, y) (x+1, y) (x, y+1) (x+1, y+1); foreground test per pixel
    const int l00 = label_at(ws, h, w, x, y), l10 = label_at(ws, h, w, x + 1, y), l01 = label_at(ws, h, w, x, y + 1),
              l11 = label_at(ws, h, w, x + 1, y + 1);
    auto isfg = [&](int xx, int yy) { return (unsigned)xx < (unsigned)w && (unsigned)yy < (unsigned)h && a[(int64_t)yy * w + xx] != 0; };
    const bool f00 = isfg(x, y), f10 = isfg(x + 1, y), f01 = isfg(x, y + 1), f11 = isfg(x + 1, y + 1);
    // ---- own sums ----
    if (x >= 0 && y >= 0) {
      const int64_t i = (int64_t)y * w + x;
      if (l00 != 0) {
        const int k = ws.dense[l00];
        atomicAdd(&ws.size[k], 1u);
        atomicAdd(&ws.seg[k], (unsigned long long)sg[i]);
        atomicAdd(&ws.score[k], score_map[i]);
      }
      if (f00) {   // ring of every distinct hole among the 4 neighbours (a hole = a background set other than my parent)
        const int k = ws.dense[l00];
        const int par = ws.up[k];
        int nb[4] = {label_at(ws, h, w, x - 1, y), label_at(ws, h, w, x + 1, y), label_at(ws, h, w, x, y - 1), label_at(ws, h, w, x, y + 1)};
        const bool nf[4] = {isfg(x - 1, y), isfg(x + 1, y), isfg(x, y - 1), isfg(x, y + 1)};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (nf[j] || nb[j] == 0) continue;
          const int hk = ws.dense[nb[j]];
          if (hk == par) continue;
          bool seen = false;
#pragma unroll
          for (int q = 0; q < j; ++q) seen = seen || (!nf[q] && nb[q] == nb[j]);
          if (seen) continue;
          atomicAdd(&ws.rcnt[hk], 1u);
          atomicAdd(&ws.rseg[hk], (unsigned long long)sg[i]);
          atomicAdd(&ws.rscore[hk], score_map[i]);
        }
      }
    }
    // ---- pixel edges: (x,y)|(x+1,y) for y >= 0, (x,y)|(x,y+1) for x >= 0 ----
    auto edge = [&](bool fa, int la, bool fb, int lb) {
      if (fa == fb) return;
      const int lf = fa ? la : lb, lbg = fa ? lb : la;
      const int kf = ws.dense[lf];
      const int kb = lbg == 0 ? -1 : ws.dense[lbg];
      if (kb == ws.up[kf]) atomicAdd(&ws.L[kf], 1u);     // the component's outer border
      else atomicAdd(&ws.L[kb], 1u);                      // the border of one of its holes
    };
    if (y >= 0) edge(f00, l00, f10, l10);
    if (x >= 0) edge(f00, l00, f01, l01);
    // ---- the 2x2 window ----
    const int nfg = (int)f00 + (int)f10 + (int)f01 + (int)f11;
    if (nfg == 1) {
      const int lf = f00 ? l00 : (f10 ? l10 : (f01 ? l01 : l11));
      const int kf = ws.dense[lf];
      const int par = ws.up[kf];
      // the other three: background sets; all three the parent -> a convex corner of the filled component (n1);
      // all three one hole -> a concave corner of that hole (n3)
      const int b0 = f00 ? l10 : l00, b1 = (f00 || f10) ? l01 : l10, b2 = f11 ? l01 : l11;
      const int k0 = b0 == 0 ? -1 : ws.dense[b0], k1 = b1 == 0 ? -1 : ws.dense[b1], k2 = b2 == 0 ? -1 : ws.dense[b2];
      if (k0 == k1 && k1 == k2) {
        if (k0 == par) atomicAdd(&ws.nw[kf], 1u);
        else atomicAdd(&ws.nw[k0], 1u);
      }
    }
  }
}

// the tree: depths, subtree totals, areas and scores, validity, "painted".  One CTA per frame.
__global__ void __launch_bounds__(1024) obj_tree_kernel(int h, int w, void* wsbase, int cap, double saliency_thr, double consensus_thr) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.x, npix, cap);
  if (*ws.overflow) return;
  const int nr = *ws.nroots;
  // kind: foreground roots have a foreground pixel: a component's depth is odd (children of the outside), a hole's even
  // depth by relaxation, one level per sweep: sweep s gives depth s + 2 to the children of the nodes of depth s + 1 (a
  // node written in this sweep is not read as a parent in it, so the sweep is race-free).  The tree has nr nodes, so it
  // is at most nr deep and the sweeps stop, at the latest, after nr of them
  for (int k = threadIdx.x; k < nr; k += blockDim.x) ws.depth[k] = ws.up[k] < 0 ? 1 : 0;
  __syncthreads();
  int maxd = 1;
  for (int sweep = 0; sweep < nr; ++sweep) {
    int changed = 0;
    for (int k = threadIdx.x; k < nr; k += blockDim.x) {
      if (ws.depth[k] == 0) {
        const int dp = ws.depth[ws.up[k]];
        if (dp == sweep + 1) { ws.depth[k] = dp + 1; changed = 1; }
      }
    }
    if (!__syncthreads_or(changed)) break;
    maxd = sweep + 2;
  }
  // subtree totals, deepest level first (only the sums a filled contour needs: pixels, mask sum, saliency sum)
  for (int d = maxd; d >= 2; --d) {
    for (int k = threadIdx.x; k < nr; k += blockDim.x) {
      if (ws.depth[k] == d) {
        const int p = ws.up[k];
        atomicAdd(&ws.size[p], ws.size[k]);
        atomicAdd(&ws.seg[p], ws.seg[k]);
        atomicAdd(&ws.score[p], ws.score[k]);
      }
    }
    __syncthreads();
  }
  // validity of every contour (maskprocess.py:130-148)
  const double hw = (double)h * (double)w;
  for (int k = threadIdx.x; k < nr; k += blockDim.x) {
    const bool hole = (ws.depth[k] & 1) == 0;
    const double B = 0.5 * ((double)ws.L[k] - (double)ws.nw[k]);
    double area, cnt, segsum, sal;
    if (!hole) {
      area = (double)ws.size[k] - B - 1.0;
      cnt = (double)ws.size[k]; segsum = (double)ws.seg[k]; sal = ws.score[k];
    } else {
      area = (double)ws.size[k] + B - 1.0;
      cnt = (double)ws.size[k] + (double)ws.rcnt[k]; segsum = (double)(ws.seg[k] + ws.rseg[k]); sal = ws.score[k] + ws.rscore[k];
    }
    bool valid = false;
    if (!(area < 100.0)) {
      const double saliency = sal / hw;
      const double consensus = (segsum / cnt) / 255.0;
      valid = (saliency > saliency_thr && consensus > consensus_thr) || (saliency > saliency_thr * 10);
    }
    ws.vhole[k] = hole && valid;
    ws.keep[k] = valid;   // for now: "this contour is valid"; below: "painted by this contour or an ancestor"
  }
  __syncthreads();
  for (int d = 2; d <= maxd; ++d) {
    for (int k = threadIdx.x; k < nr; k += blockDim.x)
      if (ws.depth[k] == d && ws.keep[ws.up[k]]) ws.keep[k] = 1;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(OT) obj_apply_kernel(const uint8_t* __restrict__ alpha, int h, int w, void* wsbase, int cap,
                                                       uint8_t* __restrict__ out) {
  const int64_t npix = (int64_t)h * w;
  const ObjWs ws = ws_of(wsbase, blockIdx.y, npix, cap);
  if (*ws.overflow) return;
  const uint8_t* a = alpha + (int64_t)blockIdx.y * npix;
  uint8_t* o = out + (int64_t)blockIdx.y * npix;
  for (int64_t i = (int64_t)blockIdx.x * OT + threadIdx.x; i < npix; i += (int64_t)gridDim.x * OT) {
    const int v = a[i];
    int keep = 0;
    if (v) {
      keep = ws.keep[ws.dense[ws.P[i + 1]]];
      if (!keep) {   // on the ring of a valid hole?
        const int y = (int)(i / w), x = (int)(i - (int64_t)y * w);
        const int xs[4] = {x - 1, x + 1, x, x}, ys[4] = {y, y, y - 1, y + 1};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if ((unsigned)xs[j] < (unsigned)w && (unsigned)ys[j] < (unsigned)h && a[(int64_t)ys[j] * w + xs[j]] == 0) {
            const int l = ws.P[ys[j] * w + xs[j] + 1];
            if (l != 0 && ws.vhole[ws.dense[l]]) keep = 1;
          }
        }
      }
    }
    o[i] = keep ? (uint8_t)v : (uint8_t)0;
  }
}

}  // namespace
}  // namespace vu

using namespace vu;

extern "C" size_t vu_remove_objects_workspace_bytes(int n, int h, int w, int max_objects) {
  if (n <= 0 || h <= 0 || w <= 0 || max_objects <= 0) return 0;
  return (size_t)n * ws_frame_bytes((int64_t)h * w, max_objects);
}

extern "C" int vu_remove_invalid_objects(const uint8_t* alpha, const uint8_t* segmask, const double* score_map, int n, int h, int w,
                                         double saliency_thr, double consensus_thr, uint8_t* out, int32_t* status, void* workspace,
                                         size_t workspace_bytes, int max_objects, vu_stream_t stream) {
  VU_REQUIRE(alpha && segmask && score_map && out && status && workspace && n >= 0 && h > 0 && w > 0 && max_objects > 0);
  if ((int64_t)h * w >= (1LL << 31) - 2 || n > 65535) return VU_ERR_UNSUPPORTED;
  if (workspace_bytes < vu_remove_objects_workspace_bytes(n, h, w, max_objects) || (reinterpret_cast<uintptr_t>(workspace) & 15)) return VU_ERR_WORKSPACE;
  if (n == 0) return VU_OK;
  const int64_t npix = (int64_t)h * w;
  cudaStream_t st = S(stream);
  const int gx = grid_for(npix, OT, 8);
  obj_init_kernel<<<dim3(h, n), OT, 0, st>>>(alpha, h, w, workspace, max_objects);
  obj_merge_kernel<<<dim3(gx, n), OT, 0, st>>>(alpha, h, w, workspace, max_objects);
  obj_flatten_kernel<<<dim3(gx, n), OT, 0, st>>>(alpha, h, w, workspace, max_objects);
  obj_parent_kernel<<<dim3((max_objects + OT - 1) / OT, n), OT, 0, st>>>(h, w, workspace, max_objects);
  obj_stats_kernel<<<dim3(gx, n), OT, 0, st>>>(alpha, segmask, score_map, h, w, workspace, max_objects);
  obj_tree_kernel<<<n, 1024, 0, st>>>(h, w, workspace, max_objects, saliency_thr, consensus_thr);
  obj_apply_kernel<<<dim3(gx, n), OT, 0, st>>>(alpha, h, w, workspace, max_objects, out);
  // status[i] = number of contours of frame i; more than max_objects: the frame's output is undefined (the caller redoes
  // it with a larger table)
  for (int i = 0; i < n; ++i) {
    const ObjWs ws = ws_of(workspace, i, npix, max_objects);
    int e = record_cuda(cudaMemcpyAsync(status + i, ws.nroots, sizeof(int), cudaMemcpyDeviceToDevice, st));
    if (e) return e;
  }
  note_launch(7);
  VU_RETURN_LAUNCH();
}
