// regionfill (unscreen/utils/region_fill.py:7-63; BackgroundAgent 'rf', bgmodel/agent.py:133-157; bg.py:79):
// fill the masked pixels of an image plane with the solution of the discrete Laplace equation -- every masked pixel is the
// mean of its in-image 4-neighbours, the pixels outside the mask are the boundary data.
//
// The reference assembles the sparse matrix D = diag(number of in-image neighbours) - adjacency(masked pixels) and hands
// it to scipy's direct solver.  D is symmetric positive definite (a Dirichlet Laplacian), so here it is solved matrix-free
// by conjugate gradients in float64 on the pixel grid: the search direction p is kept zero outside the mask, which makes
// D p a plain 5-point stencil without any mask test on the neighbours.  Two kernels per iteration:
//
//   rf_dir_kernel   p_k = r + beta p_(k-1) (recomputed for the 4 neighbours instead of a third pass), D p_k, <p_k, D p_k>
//   rf_step_kernel  x += alpha p_k, r -= alpha D p_k, <r, r>
//
// alpha / beta are formed on the device from the dot products (float64 atomics, three rotating slots), the host only reads
// the residuals every CHECK iterations.  Several planes that share one mask (the B, G, R planes of bg.py:79) are solved
// together.  Parity with the direct solver is a TOLERANCE: iteration stops at |r| <= tol |b| (default 1e-10: within ~1e-6
// grey levels of spsolve on a 1080p person-sized hole), and the reference truncates the float result to uint8 (hence
// rf_snap_kernel at the end).
//
//   vu_resize_linear_f64   the two cv2.resize calls on float64 data around the solve (region_fill.py:10-15)
#include "vu_common.cuh"

namespace vu {
namespace {

constexpr int RT = 256;     // 32 x 8 threads, RROWS rows each
constexpr int RROWS = 4;
constexpr int CHECK = 64;

// per-plane scalars
struct RfScal {
  double rr[3];      // <r, r> of iterations k-1, k, k+1 (slot = k % 3)
  double pap[2];     // <p, D p> (slot = k & 1)
  double bb;         // <b, b>
  double psum;       // sum / count of the perimeter values: the initial guess
  double pcnt;
};

__device__ __forceinline__ double block_sum(double v, double* sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  if (wid == 0) {
    v = lane < RT / 32 ? sm[lane] : 0.0;
#pragma unroll
    for (int o = RT / 64; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  }
  return v;     // valid in thread 0
}

__device__ __forceinline__ int nn_of(int y, int x, int h, int w) { return (y > 0) + (y < h - 1) + (x > 0) + (x < w - 1); }

// perimeter pixels (outside the mask, a 4-neighbour inside): sum and count per plane
__global__ void __launch_bounds__(RT) rf_perimeter_kernel(const double* __restrict__ x, const uint8_t* __restrict__ mask, int h, int w, RfScal* __restrict__ sc) {
  __shared__ double sm[RT / 32];
  const int c = blockIdx.z;
  const int64_t plane = (int64_t)c * h * w;
  const int px = blockIdx.x * 32 + (threadIdx.x & 31);
  double s = 0.0, n = 0.0;
  for (int j = 0; j < RROWS; ++j) {
    const int py = (blockIdx.y * 8 + (threadIdx.x >> 5)) * RROWS + j;
    if (px >= w || py >= h) continue;
    const int64_t i = (int64_t)py * w + px;
    if (mask[i]) continue;
    const bool per = (py > 0 && mask[i - w]) || (py < h - 1 && mask[i + w]) || (px > 0 && mask[i - 1]) || (px < w - 1 && mask[i + 1]);
    if (per) { s += x[plane + i]; n += 1.0; }
  }
  s = block_sum(s, sm);
  n = block_sum(n, sm);
  if (threadIdx.x == 0 && n > 0.0) { atomicAdd(&sc[c].psum, s); atomicAdd(&sc[c].pcnt, n); }
}

// x = c on the mask; r = p = b - D c; zeros outside the mask
__global__ void __launch_bounds__(RT) rf_init_kernel(double* __restrict__ x, const uint8_t* __restrict__ mask, int h, int w, double* __restrict__ r,
                                                     double* __restrict__ p0, double* __restrict__ p1, double* __restrict__ ap, RfScal* __restrict__ sc) {
  __shared__ double sm[RT / 32];
  const int c = blockIdx.z;
  const int64_t plane = (int64_t)c * h * w;
  const int px = blockIdx.x * 32 + (threadIdx.x & 31);
  const double guess = sc[c].pcnt > 0.0 ? sc[c].psum / sc[c].pcnt : 0.0;
  double rr = 0.0, bb = 0.0;
  bool on[RROWS];
  for (int j = 0; j < RROWS; ++j) {
    const int py = (blockIdx.y * 8 + (threadIdx.x >> 5)) * RROWS + j;
    on[j] = false;
    if (px >= w || py >= h) continue;
    const int64_t i = (int64_t)py * w + px;
    double res = 0.0;
    if (mask[i]) {
      double b = 0.0;
      int nout = 0;
      if (py > 0 && !mask[i - w]) { b += x[plane + i - w]; ++nout; }
      if (py < h - 1 && !mask[i + w]) { b += x[plane + i + w]; ++nout; }
      if (px > 0 && !mask[i - 1]) { b += x[plane + i - 1]; ++nout; }
      if (px < w - 1 && !mask[i + 1]) { b += x[plane + i + 1]; ++nout; }
      res = b - guess * nout;
      rr += res * res;
      bb += b * b;
      on[j] = true;
    }
    r[plane + i] = res;
    p0[plane + i] = res;     // slot of p_(-1): beta is 0 in iteration 0, so only its zeros outside the mask matter
    p1[plane + i] = 0.0;
    ap[plane + i] = 0.0;
  }
  // x is only written inside the mask and the reads above only touch pixels outside it: no ordering needed
  for (int j = 0; j < RROWS; ++j) {
    const int py = (blockIdx.y * 8 + (threadIdx.x >> 5)) * RROWS + j;
    if (on[j]) x[plane + (int64_t)py * w + px] = guess;
  }
  rr = block_sum(rr, sm);
  bb = block_sum(bb, sm);
  if (threadIdx.x == 0) { atomicAdd(&sc[c].rr[0], rr); atomicAdd(&sc[c].bb, bb); }
}

__global__ void __launch_bounds__(RT) rf_dir_kernel(const uint8_t* __restrict__ mask, int h, int w, const double* __restrict__ r, const double* __restrict__ pold,
                                                    double* __restrict__ pnew, double* __restrict__ ap, RfScal* __restrict__ sc, int k) {
  __shared__ double sm[RT / 32];
  const int c = blockIdx.z;
  const int64_t plane = (int64_t)c * h * w;
  const int cur = k % 3, prev = (k + 2) % 3, next = (k + 1) % 3;
  const double rr_prev = sc[c].rr[prev];
  const double beta = (k > 0 && rr_prev > 0.0) ? sc[c].rr[cur] / rr_prev : 0.0;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) sc[c].rr[next] = 0.0;
  const int px = blockIdx.x * 32 + (threadIdx.x & 31);
  double dot = 0.0;
  for (int j = 0; j < RROWS; ++j) {
    const int py = (blockIdx.y * 8 + (threadIdx.x >> 5)) * RROWS + j;
    if (px >= w || py >= h) continue;
    const int64_t i = (int64_t)py * w + px;
    if (!mask[i]) continue;
    const double* rp = r + plane + i;
    const double* pp = pold + plane + i;
    const double pc = rp[0] + beta * pp[0];
    double nb = 0.0;
    if (py > 0) nb += rp[-w] + beta * pp[-w];
    if (py < h - 1) nb += rp[w] + beta * pp[w];
    if (px > 0) nb += rp[-1] + beta * pp[-1];
    if (px < w - 1) nb += rp[1] + beta * pp[1];
    const double a = nn_of(py, px, h, w) * pc - nb;
    pnew[plane + i] = pc;
    ap[plane + i] = a;
    dot += pc * a;
  }
  dot = block_sum(dot, sm);
  if (threadIdx.x == 0) atomicAdd(&sc[c].pap[k & 1], dot);
}

__global__ void __launch_bounds__(RT) rf_step_kernel(double* __restrict__ x, const uint8_t* __restrict__ mask, int h, int w, double* __restrict__ r,
                                                     const double* __restrict__ p, const double* __restrict__ ap, RfScal* __restrict__ sc, int k) {
  __shared__ double sm[RT / 32];
  const int c = blockIdx.z;
  const int64_t plane = (int64_t)c * h * w;
  const double pap = sc[c].pap[k & 1];
  const double alpha = pap > 0.0 ? sc[c].rr[k % 3] / pap : 0.0;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) sc[c].pap[(k + 1) & 1] = 0.0;
  const int px = blockIdx.x * 32 + (threadIdx.x & 31);
  double rr = 0.0;
  for (int j = 0; j < RROWS; ++j) {
    const int py = (blockIdx.y * 8 + (threadIdx.x >> 5)) * RROWS + j;
    if (px >= w || py >= h) continue;
    const int64_t i = plane + (int64_t)py * w + px;
    if (!mask[i - plane]) continue;
    x[i] += alpha * p[i];
    const double res = r[i] - alpha * ap[i];
    r[i] = res;
    rr += res * res;
  }
  rr = block_sum(rr, sm);
  if (threadIdx.x == 0) atomicAdd(&sc[c].rr[(k + 1) % 3], rr);
}

// values within eps of an integer become that integer.  The reference truncates the fill to uint8: where the exact solution
// IS an integer (an isolated masked pixel whose four neighbours sum to a multiple of 4, a flat boundary) the direct solver
// returns it exactly, the iteration returns it -1e-7 half of the time, and the truncation would differ by a whole level.
__global__ void __launch_bounds__(RT) rf_snap_kernel(double* __restrict__ x, const uint8_t* __restrict__ mask, int h, int w, double eps) {
  const int c = blockIdx.z;
  const int64_t plane = (int64_t)c * h * w;
  const int px = blockIdx.x * 32 + (threadIdx.x & 31);
  for (int j = 0; j < RROWS; ++j) {
    const int py = (blockIdx.y * 8 + (threadIdx.x >> 5)) * RROWS + j;
    if (px >= w || py >= h) continue;
    const int64_t i = (int64_t)py * w + px;
    if (!mask[i]) continue;
    const double v = x[plane + i], n = rint(v);
    if (fabs(v - n) <= eps) x[plane + i] = n;
  }
}

// cv2.resize of CV_64F data (INTER_LINEAR, IPP: double weights); AREA: the exact-2x case, which cv2 turns into 2 x 2
// means (the last row / column of an odd source averages what exists, in float32)
template <bool AREA>
__global__ void __launch_bounds__(RT) resize_f64_kernel(const double* __restrict__ src, int sh, int sw, double* __restrict__ dst, int dh, int dw,
                                                        double scale_x, double scale_y, const uint8_t* __restrict__ keep_mask,
                                                        const double* __restrict__ keep_src, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * RT + threadIdx.x; i < total; i += (int64_t)gridDim.x * RT) {
    const int64_t pl = i / ((int64_t)dh * dw);
    const int64_t rem = i - pl * dh * dw;
    const int y = (int)(rem / dw), x = (int)(rem - (int64_t)y * dw);
    if (keep_mask && keep_mask[rem] == 0) { dst[i] = keep_src[i]; continue; }
    const double* s = src + pl * sh * sw;
    double v;
    if (AREA) {
      const int y0 = 2 * y, x0 = 2 * x;
      if (y0 + 1 < sh && x0 + 1 < sw) {
        v = (s[(int64_t)y0 * sw + x0] + s[(int64_t)y0 * sw + x0 + 1] + s[(int64_t)(y0 + 1) * sw + x0] + s[(int64_t)(y0 + 1) * sw + x0 + 1]) * 0.25;
      } else {
        double sum = 0.0;
        int cnt = 0;
        for (int yy = y0; yy < min(y0 + 2, sh); ++yy)
          for (int xx = x0; xx < min(x0 + 2, sw); ++xx) { sum += s[(int64_t)yy * sw + xx]; ++cnt; }
        v = cnt ? (double)__fdiv_rn((float)sum, (float)cnt) : 0.0;
      }
    } else {
      double fx = (x + 0.5) * scale_x - 0.5, fy = (y + 0.5) * scale_y - 0.5;
      int x0 = (int)floor(fx), y0 = (int)floor(fy);
      fx -= x0; fy -= y0;
      if (x0 < 0) { x0 = 0; fx = 0.0; }
      if (x0 >= sw - 1) { x0 = sw - 1; fx = 0.0; }
      if (y0 < 0) { y0 = 0; fy = 0.0; }
      if (y0 >= sh - 1) { y0 = sh - 1; fy = 0.0; }
      const int x1 = min(x0 + 1, sw - 1), y1 = min(y0 + 1, sh - 1);
      const double top = __dadd_rn(__dmul_rn(s[(int64_t)y0 * sw + x0], 1.0 - fx), __dmul_rn(s[(int64_t)y0 * sw + x1], fx));
      const double bot = __dadd_rn(__dmul_rn(s[(int64_t)y1 * sw + x0], 1.0 - fx), __dmul_rn(s[(int64_t)y1 * sw + x1], fx));
      v = __dadd_rn(__dmul_rn(top, 1.0 - fy), __dmul_rn(bot, fy));
    }
    dst[i] = v;
  }
}

}  // namespace
}  // namespace vu

using namespace vu;

extern "C" size_t vu_regionfill_workspace_bytes(int planes, int h, int w) {
  if (planes <= 0 || h <= 0 || w <= 0) return 0;
  return 4 * (size_t)planes * h * w * sizeof(double) + (size_t)planes * sizeof(RfScal);
}

extern "C" int vu_regionfill_f64(double* x, const uint8_t* mask, int planes, int h, int w, double tol, int max_iters, double snap_eps, void* workspace,
                                 size_t workspace_bytes, int32_t* iters_out, double* resid_out, vu_stream_t stream) {
  VU_REQUIRE(x && mask && planes > 0 && planes <= 16 && h > 0 && w > 0 && tol > 0.0 && max_iters >= 0 && snap_eps >= 0.0);
  if (!workspace || workspace_bytes < vu_regionfill_workspace_bytes(planes, h, w)) return VU_ERR_WORKSPACE;
  cudaStream_t st = S(stream);
  const size_t n = (size_t)planes * h * w;
  double* r = static_cast<double*>(workspace);
  double* p[2] = {r + n, r + 2 * n};
  double* ap = r + 3 * n;
  RfScal* sc = reinterpret_cast<RfScal*>(r + 4 * n);
  int e = record_cuda(cudaMemsetAsync(sc, 0, planes * sizeof(RfScal), st));
  if (e) return e;
  const dim3 grid((w + 31) / 32, (h + 8 * RROWS - 1) / (8 * RROWS), planes);
  rf_perimeter_kernel<<<grid, RT, 0, st>>>(x, mask, h, w, sc);
  rf_init_kernel<<<grid, RT, 0, st>>>(x, mask, h, w, r, p[0], p[1], ap, sc);
  note_launch(2);
  RfScal host[16];
  int k = 0;
  bool done = false;
  double worst = 0.0;
  while (!done) {
    // residuals of iteration k (slot k % 3) against |b|
    e = record_cuda(cudaMemcpyAsync(host, sc, planes * sizeof(RfScal), cudaMemcpyDeviceToHost, st));
    if (e) return e;
    e = record_cuda(cudaStreamSynchronize(st));
    if (e) return e;
    done = true;
    worst = 0.0;
    bool nan = false;
    for (int c = 0; c < planes; ++c) {
      const double rr = host[c].rr[k % 3], bb = host[c].bb;
      if (!(rr <= tol * tol * bb)) done = false;
      nan |= rr != rr;
      const double rel = bb > 0.0 ? sqrt(rr / bb) : (rr > 0.0 ? INFINITY : 0.0);
      if (!(rel <= worst)) worst = rel;
    }
    if (done || nan || k >= max_iters) break;      // a NaN (non-finite input) stops at once and is reported as the residual
    const int upto = k + CHECK < max_iters ? k + CHECK : max_iters;
    note_launch(2 * (upto - k));
    for (; k < upto; ++k) {
      // p_(k-1) lives in p[k & 1] (the init wrote r into p[0]), p_k goes to the other buffer
      rf_dir_kernel<<<grid, RT, 0, st>>>(mask, h, w, r, p[k & 1], p[(k + 1) & 1], ap, sc, k);
      rf_step_kernel<<<grid, RT, 0, st>>>(x, mask, h, w, r, p[(k + 1) & 1], ap, sc, k);
    }
    e = record_cuda(cudaGetLastError());
    if (e) return e;
  }
  if (snap_eps > 0.0) {
    rf_snap_kernel<<<grid, RT, 0, st>>>(x, mask, h, w, snap_eps);
    note_launch();
    e = record_cuda(cudaGetLastError());
    if (e) return e;
  }
  if (iters_out) *iters_out = k;
  if (resid_out) *resid_out = worst;     // max over the planes of |r| / |b|: above tol = not converged within max_iters
  return VU_OK;
}

extern "C" int vu_resize_linear_f64(const double* src, int planes, int sh, int sw, double* dst, int dh, int dw, double scale_x, double scale_y,
                                    const uint8_t* keep_mask, const double* keep_src, vu_stream_t stream) {
  VU_REQUIRE(src && dst && planes >= 0 && sh > 0 && sw > 0 && dh > 0 && dw > 0 && scale_x > 0.0 && scale_y > 0.0);
  VU_REQUIRE((keep_mask == nullptr) == (keep_src == nullptr));
  if (planes == 0) return VU_OK;
  const int64_t total = (int64_t)planes * dh * dw;
  const int grid = grid_for(total, RT, 8);
  const bool area = fabs(scale_x - 2.0) < 2.220446049250313e-16 && fabs(scale_y - 2.0) < 2.220446049250313e-16;
  if (area) resize_f64_kernel<true><<<grid, RT, 0, S(stream)>>>(src, sh, sw, dst, dh, dw, scale_x, scale_y, keep_mask, keep_src, total);
  else resize_f64_kernel<false><<<grid, RT, 0, S(stream)>>>(src, sh, sw, dst, dh, dw, scale_x, scale_y, keep_mask, keep_src, total);
  VU_RETURN_LAUNCH();
}
