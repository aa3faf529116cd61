// Text-line crops for OCR: `TextBlock.get_transformed_region(img, idx, textheight)` (reference utils/textblock.py:
// 162-194) for every line of a page in two launches, bit-exact with OpenCV 4.x.
//   ctd_plan_regions (host)  quad expansion / clip, aspect ratio, output size and the failure cases of the reference,
//                            packed output offsets -- the caller sizes its buffer from this before any GPU work.
//   k_region_homography      one thread per line: cv2.findHomography for 4 points (calib3d fundam.cpp,
//                            HomographyEstimatorCallback::runKernel: float32 points, per-axis centroid / mean-abs
//                            normalisation, 9x9 LtL, eigenvector of the smallest eigenvalue by OpenCV's pivoting Jacobi
//                            (core lapack.cpp JacobiImpl_), de-normalised, scaled by 1/H[2][2] unless |H[2][2]| <= FLT_EPSILON) and the inverse
//                            warpPerspective applies (cv::invert DECOMP_LU, 3x3 cofactor formula).
//   k_region_warp            one launch over the packed output of all lines: the fixed-point INTER_LINEAR gather of
//                            warpPerspective (imgwarp.cpp WarpPerspectiveInvoker + remapBilinear), rotation of vertical
//                            lines folded into the index so every line's stores are contiguous.
// All double arithmetic that OpenCV evaluates unfused is written with __dmul_rn / __dadd_rn so nvcc cannot contract it
// into FMAs.  Oracle: oracle/regions_ref.py (pinned against the installed cv2, tests/test_cpu_regions.py).
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "engine.h"

namespace {

constexpr int kWarpThreads = 256;   // output pixels per warp block (a block never spans two lines)
constexpr int kInterBits = 5;
constexpr int kTab = 1 << kInterBits;

// per-line launch record (lines with status CTD_REGION_OK only)
struct RegionLine {
  double M[9];     // forward homography (k_region_homography)
  double Mi[9];    // its inverse, what the warp maps output pixels through
  float src[8];    // the expanded / clipped quad as findHomography sees it (float32)
  int dw, dh;      // the reference's w, h: dst corners (w-1, h-1)
  int ww, wh;      // warpPerspective's output size (the page's size when w or h is 0)
  int vertical, bw0;
  long long offset;   // byte offset in the packed output
  long long tile0;    // first block of k_region_warp that belongs to this line
};

__device__ __forceinline__ double dm(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double da(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double ds(double a, double b) { return __dsub_rn(a, b); }

// lapack.cpp's own hypot (JacobiImpl_ calls it, not libm's): the larger magnitude times sqrt(1 + ratio^2)
__device__ __forceinline__ double cv_hypot(double a, double b) {
  a = fabs(a);
  b = fabs(b);
  if (a > b) {
    b = __ddiv_rn(b, a);
    return dm(a, __dsqrt_rn(da(1.0, dm(b, b))));
  }
  if (b > 0) {
    a = __ddiv_rn(a, b);
    return dm(b, __dsqrt_rn(da(1.0, dm(a, a))));
  }
  return 0.0;
}

// cv::eigen for a symmetric 9x9 (JacobiImpl_): returns in v the eigenvector of the smallest eigenvalue
__device__ void jacobi9_smallest(double* A, double* v) {
  constexpr int n = 9;
  double V[n * n], W[n];
  int indR[n], indC[n];
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) V[i * n + j] = i == j ? 1.0 : 0.0;
  auto row_max = [&](int k) {
    int m = k + 1;
    double mv = fabs(A[n * k + m]);
    for (int i = k + 2; i < n; ++i) {
      const double val = fabs(A[n * k + i]);
      if (mv < val) mv = val, m = i;
    }
    indR[k] = m;
  };
  auto col_max = [&](int k) {
    int m = 0;
    double mv = fabs(A[k]);
    for (int i = 1; i < k; ++i) {
      const double val = fabs(A[n * i + k]);
      if (mv < val) mv = val, m = i;
    }
    indC[k] = m;
  };
  for (int k = 0; k < n; ++k) {
    W[k] = A[(n + 1) * k];
    if (k < n - 1) row_max(k);
    if (k > 0) col_max(k);
  }
  for (int iters = 0; iters < n * n * 30; ++iters) {
    int k = 0;
    double mv = fabs(A[indR[0]]);
    for (int i = 1; i < n - 1; ++i) {
      const double val = fabs(A[n * i + indR[i]]);
      if (mv < val) mv = val, k = i;
    }
    int l = indR[k];
    for (int i = 1; i < n; ++i) {
      const double val = fabs(A[n * indC[i] + i]);
      if (mv < val) mv = val, k = indC[i], l = i;
    }
    const double p = A[n * k + l];
    if (fabs(p) <= DBL_EPSILON) break;
    const double y = dm(ds(W[l], W[k]), 0.5);
    double t = da(fabs(y), cv_hypot(p, y));
    double s = cv_hypot(p, t);
    const double c = t / s;
    s = p / s;
    t = dm(p / t, p);
    if (y < 0) s = -s, t = -t;
    A[n * k + l] = 0;
    W[k] = ds(W[k], t);
    W[l] = da(W[l], t);
    auto rot = [&](double& v0, double& v1) {
      const double a0 = v0, b0 = v1;
      v0 = ds(dm(a0, c), dm(b0, s));
      v1 = da(dm(a0, s), dm(b0, c));
    };
    for (int i = 0; i < k; ++i) rot(A[n * i + k], A[n * i + l]);
    for (int i = k + 1; i < l; ++i) rot(A[n * k + i], A[n * i + l]);
    for (int i = l + 1; i < n; ++i) rot(A[n * k + i], A[n * l + i]);
    for (int i = 0; i < n; ++i) rot(V[n * k + i], V[n * l + i]);
    for (int j = 0; j < 2; ++j) {
      const int idx = j == 0 ? k : l;
      if (idx < n - 1) row_max(idx);
      if (idx > 0) col_max(idx);
    }
  }
  // eigenvalues sorted descending (selection sort with swaps, as OpenCV): the last row is the wanted vector
  int order[n];
  for (int i = 0; i < n; ++i) order[i] = i;
  for (int k = 0; k < n - 1; ++k) {
    int m = k;
    for (int i = k + 1; i < n; ++i)
      if (W[m] < W[i]) m = i;
    if (k != m) {
      const double tw = W[m]; W[m] = W[k]; W[k] = tw;
      const int to = order[m]; order[m] = order[k]; order[k] = to;
    }
  }
  for (int i = 0; i < n; ++i) v[i] = V[n * order[n - 1] + i];
}

// C = A * B for 3x3 row-major, each element summed k = 0, 1, 2 from 0 (cv::gemm)
__device__ void mul3(const double* A, const double* B, double* C) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double s = 0.0;
      for (int k = 0; k < 3; ++k) s = da(s, dm(A[i * 3 + k], B[k * 3 + j]));
      C[i * 3 + j] = s;
    }
}

__global__ void k_region_homography(RegionLine* __restrict__ lines, int n) {
  const int li = blockIdx.x * blockDim.x + threadIdx.x;
  if (li >= n) return;
  RegionLine& L = lines[li];
  double Mx[4], My[4], mx[4], my[4];
  for (int i = 0; i < 4; ++i) { Mx[i] = L.src[2 * i]; My[i] = L.src[2 * i + 1]; }
  const double w1 = float(L.dw - 1), h1 = float(L.dh - 1);
  mx[0] = 0; my[0] = 0; mx[1] = w1; my[1] = 0; mx[2] = w1; my[2] = h1; mx[3] = 0; my[3] = h1;
  double cmx = 0, cmy = 0, cMx = 0, cMy = 0;
  for (int i = 0; i < 4; ++i) { cmx = da(cmx, mx[i]); cmy = da(cmy, my[i]); cMx = da(cMx, Mx[i]); cMy = da(cMy, My[i]); }
  cmx /= 4; cmy /= 4; cMx /= 4; cMy /= 4;
  double smx = 0, smy = 0, sMx = 0, sMy = 0;
  for (int i = 0; i < 4; ++i) {
    smx = da(smx, fabs(ds(mx[i], cmx))); smy = da(smy, fabs(ds(my[i], cmy)));
    sMx = da(sMx, fabs(ds(Mx[i], cMx))); sMy = da(sMy, fabs(ds(My[i], cMy)));
  }
  // the planner only launches lines whose spreads are non-zero (the reference's None case is a status there)
  smx = 4 / smx; smy = 4 / smy; sMx = 4 / sMx; sMy = 4 / sMy;
  double A[81];
  for (int i = 0; i < 81; ++i) A[i] = 0;
  for (int i = 0; i < 4; ++i) {
    const double x = dm(ds(mx[i], cmx), smx), y = dm(ds(my[i], cmy), smy);
    const double X = dm(ds(Mx[i], cMx), sMx), Y = dm(ds(My[i], cMy), sMy);
    const double Lx[9] = {X, Y, 1, 0, 0, 0, dm(-x, X), dm(-x, Y), -x};
    const double Ly[9] = {0, 0, 0, X, Y, 1, dm(-y, X), dm(-y, Y), -y};
    for (int j = 0; j < 9; ++j)
      for (int k = j; k < 9; ++k) A[j * 9 + k] = da(A[j * 9 + k], da(dm(Lx[j], Lx[k]), dm(Ly[j], Ly[k])));
  }
  for (int j = 0; j < 9; ++j)
    for (int k = 0; k < j; ++k) A[j * 9 + k] = A[k * 9 + j];
  double h0[9], t[9], H[9];
  jacobi9_smallest(A, h0);
  const double inv_hnorm[9] = {1. / smx, 0, cmx, 0, 1. / smy, cmy, 0, 0, 1};
  const double hnorm2[9] = {sMx, 0, dm(-cMx, sMx), 0, sMy, dm(-cMy, sMy), 0, 0, 1};
  mul3(inv_hnorm, h0, t);
  mul3(t, hnorm2, H);
  // scaled by 1/H[2][2] only when |H[2][2]| > FLT_EPSILON; a nearly degenerate quad (three corners collinear after
  // the clip) keeps the unscaled matrix, as cv2 returns it
  if (fabs(H[8]) > double(FLT_EPSILON)) {
    const double sc = 1. / H[8];
    for (int i = 0; i < 9; ++i) L.M[i] = dm(H[i], sc);
  } else {
    for (int i = 0; i < 9; ++i) L.M[i] = H[i];
  }
  // cv::invert(M, DECOMP_LU), n == 3: cofactors * (1 / det); a singular M leaves zeros
  const double* S = L.M;
  auto s_ = [&](int r, int c) { return S[r * 3 + c]; };
  const double det = da(ds(dm(s_(0, 0), ds(dm(s_(1, 1), s_(2, 2)), dm(s_(1, 2), s_(2, 1)))),
                           dm(s_(0, 1), ds(dm(s_(1, 0), s_(2, 2)), dm(s_(1, 2), s_(2, 0))))),
                        dm(s_(0, 2), ds(dm(s_(1, 0), s_(2, 1)), dm(s_(1, 1), s_(2, 0)))));
  if (det != 0.) {
    const double d = 1. / det;
    L.Mi[0] = dm(ds(dm(s_(1, 1), s_(2, 2)), dm(s_(1, 2), s_(2, 1))), d);
    L.Mi[1] = dm(ds(dm(s_(0, 2), s_(2, 1)), dm(s_(0, 1), s_(2, 2))), d);
    L.Mi[2] = dm(ds(dm(s_(0, 1), s_(1, 2)), dm(s_(0, 2), s_(1, 1))), d);
    L.Mi[3] = dm(ds(dm(s_(1, 2), s_(2, 0)), dm(s_(1, 0), s_(2, 2))), d);
    L.Mi[4] = dm(ds(dm(s_(0, 0), s_(2, 2)), dm(s_(0, 2), s_(2, 0))), d);
    L.Mi[5] = dm(ds(dm(s_(0, 2), s_(1, 0)), dm(s_(0, 0), s_(1, 2))), d);
    L.Mi[6] = dm(ds(dm(s_(1, 0), s_(2, 1)), dm(s_(1, 1), s_(2, 0))), d);
    L.Mi[7] = dm(ds(dm(s_(0, 1), s_(2, 0)), dm(s_(0, 0), s_(2, 1))), d);
    L.Mi[8] = dm(ds(dm(s_(0, 0), s_(1, 1)), dm(s_(0, 1), s_(1, 0))), d);
  } else {
    for (int i = 0; i < 9; ++i) L.Mi[i] = 0.;
  }
}

template <int C>
__global__ void __launch_bounds__(kWarpThreads) k_region_warp(const RegionLine* __restrict__ lines, int n,
                                                              const uint8_t* __restrict__ img, int ih, int iw,
                                                              uint8_t* __restrict__ out) {
  __shared__ int s_line;
  if (threadIdx.x == 0) {   // last line whose first block is <= this block
    int lo = 0, hi = n - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (lines[mid].tile0 <= (long long)blockIdx.x) lo = mid;
      else hi = mid - 1;
    }
    s_line = lo;
  }
  __syncthreads();
  const RegionLine& L = lines[s_line];
  const long long p = ((long long)blockIdx.x - L.tile0) * kWarpThreads + threadIdx.x;
  const int ww = L.ww, wh = L.wh;
  if (p >= (long long)ww * wh) return;
  int x, y;   // pixel of the warped (un-rotated) image; p indexes the stored (rotated) crop
  if (L.vertical) {   // rot90 CCW: stored (i, j) of the wh-wide crop = warped (y = j, x = ww-1-i)
    const int i = int(p / wh), j = int(p - (long long)i * wh);
    y = j; x = ww - 1 - i;
  } else {
    y = int(p / ww); x = int(p - (long long)y * ww);
  }
  const double* Mi = L.Mi;
  const int xb = (x / L.bw0) * L.bw0, x1 = x - xb;
  const double X0 = da(da(dm(Mi[0], double(xb)), dm(Mi[1], double(y))), Mi[2]);
  const double Y0 = da(da(dm(Mi[3], double(xb)), dm(Mi[4], double(y))), Mi[5]);
  const double W0 = da(da(dm(Mi[6], double(xb)), dm(Mi[7], double(y))), Mi[8]);
  double W = da(W0, dm(Mi[6], double(x1)));
  W = W != 0. ? __ddiv_rn(double(kTab), W) : 0.;
  double fX = dm(da(X0, dm(Mi[0], double(x1))), W);
  double fY = dm(da(Y0, dm(Mi[3], double(x1))), W);
  // std::max(INT_MIN, std::min(INT_MAX, v)) with std::min/max's comparison order (nan -> INT_MAX)
  fX = fX < 2147483647.0 ? fX : 2147483647.0;
  fX = -2147483648.0 < fX ? fX : -2147483648.0;
  fY = fY < 2147483647.0 ? fY : 2147483647.0;
  fY = -2147483648.0 < fY ? fY : -2147483648.0;
  const int X = __double2int_rn(fX), Y = __double2int_rn(fY);   // cvRound: half to even
  const int sx = min(max(X >> kInterBits, -32768), 32767), sy = min(max(Y >> kInterBits, -32768), 32767);
  const int fx = X & (kTab - 1), fy = Y & (kTab - 1);
  // bilinear table entry (fy, fx): (32-fy)(32-fx), (32-fy)fx, fy(32-fx), fy*fx, times 32 (sum 32768)
  const int w00 = (kTab - fy) * (kTab - fx) * 32, w01 = (kTab - fy) * fx * 32;
  const int w10 = fy * (kTab - fx) * 32, w11 = fy * fx * 32;
  const bool x0in = sx >= 0 && sx < iw, x1in = sx + 1 >= 0 && sx + 1 < iw;
  const bool y0in = sy >= 0 && sy < ih, y1in = sy + 1 >= 0 && sy + 1 < ih;
  const uint8_t* r0 = img + ((long long)sy * iw + sx) * C;
  const uint8_t* r1 = r0 + (long long)iw * C;
  uint8_t* o = out + L.offset + p * C;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const int v00 = (y0in && x0in) ? r0[c] : 0, v01 = (y0in && x1in) ? r0[C + c] : 0;
    const int v10 = (y1in && x0in) ? r1[c] : 0, v11 = (y1in && x1in) ? r1[C + c] : 0;
    const int acc = v00 * w00 + v01 * w01 + v10 * w10 + v11 * w11;
    o[c] = uint8_t(min((acc + (1 << 14)) >> 15, 255));
  }
}

// textblock.py:163-186 for one line, in the reference's float64 arithmetic; fills status, w, h, out_h, out_w, bytes and
// (for status OK) the float32 quad and the warp size of the launch record
void plan_line(const double* quad, int32_t flags, double font_size, int im_w, int im_h, int channels, double textheight,
               ctd_region& r, RegionLine& L) {
  double x[4], y[4];
  for (int i = 0; i < 4; ++i) { x[i] = quad[2 * i]; y[i] = quad[2 * i + 1]; }
  if (flags & CTD_REGION_EXPAND) {
    const double e = font_size / 3;
    const double ex[4] = {-e, e, e, -e}, ey[4] = {-e, -e, e, e};
    for (int i = 0; i < 4; ++i) {
      x[i] = x[i] + ex[i];
      y[i] = y[i] + ey[i];
      x[i] = std::min(std::max(x[i], 0.0), double(im_w));   // np.clip (nan stays nan)
      y[i] = std::min(std::max(y[i], 0.0), double(im_h));
    }
  }
  double mx[4], my[4];
  for (int i = 0; i < 4; ++i) { mx[i] = (x[(i + 1) & 3] + x[i]) / 2; my[i] = (y[(i + 1) & 3] + y[i]) / 2; }
  const double vvx = mx[2] - mx[0], vvy = my[2] - my[0], vhx = mx[1] - mx[3], vhy = my[1] - my[3];
  const double ratio = std::sqrt(vvx * vvx + vvy * vvy) / std::sqrt(vhx * vhx + vhy * vhy);
  const bool vertical = flags & CTD_REGION_VERTICAL;
  const double q = vertical ? textheight * ratio : textheight / ratio;
  r = ctd_region{};
  if (!std::isfinite(q) || !std::isfinite(textheight)) { r.status = CTD_REGION_E_RATIO; return; }
  const double qr = std::nearbyint(q), th = std::trunc(textheight);   // round(): half to even; int(): truncation
  if (std::fabs(qr) > 2147483647.0 || std::fabs(th) > 2147483647.0) { r.status = CTD_REGION_E_SIZE; return; }
  const int w = vertical ? int(th) : int(qr), h = vertical ? int(qr) : int(th);
  r.w = w; r.h = h;
  // findHomography's runKernel: float32 points, zero spread along an axis of either side -> None
  float fx[4], fy[4];
  for (int i = 0; i < 4; ++i) { fx[i] = float(x[i]); fy[i] = float(y[i]); }
  double cx = 0, cy = 0;
  for (int i = 0; i < 4; ++i) { cx += fx[i]; cy += fy[i]; }
  cx /= 4; cy /= 4;
  double sx = 0, sy = 0;
  for (int i = 0; i < 4; ++i) { sx += std::fabs(fx[i] - cx); sy += std::fabs(fy[i] - cy); }
  const double dxs = std::fabs(double(float(w - 1))) * 2, dys = std::fabs(double(float(h - 1))) * 2;   // dst spreads
  if (!(std::fabs(sx) >= DBL_EPSILON) || !(std::fabs(sy) >= DBL_EPSILON) || dxs < DBL_EPSILON || dys < DBL_EPSILON) {
    r.status = CTD_REGION_E_HOMOGRAPHY;
    return;
  }
  const int ww = (w <= 0 || h <= 0) ? im_w : w, wh = (w <= 0 || h <= 0) ? im_h : h;   // OpenCV: empty dsize = src size
  const double bytes = double(ww) * wh * channels;
  if (bytes >= 2147483648.0) { r.status = CTD_REGION_E_SIZE; return; }
  r.out_h = vertical ? ww : wh;
  r.out_w = vertical ? wh : ww;
  r.bytes = size_t(ww) * wh * channels;
  for (int i = 0; i < 4; ++i) { L.src[2 * i] = fx[i]; L.src[2 * i + 1] = fy[i]; }
  L.dw = w; L.dh = h; L.ww = ww; L.wh = wh; L.vertical = vertical;
  const int bh0 = std::min(kTab * kTab / 2 / kTab, wh);   // WarpPerspectiveInvoker: min(BLOCK_SZ/2, height)
  L.bw0 = std::min(kTab * kTab / bh0, ww);                 // columns per block (X0 is evaluated at the block start)
}

int plan_all(const double* quads, const int32_t* flags, const double* font_size, int n, int im_w, int im_h, int channels,
             double textheight, ctd_region* regions, std::vector<RegionLine>* launch, size_t* total) {
  size_t off = 0;
  long long tiles = 0;
  for (int i = 0; i < n; ++i) {
    RegionLine L{};
    plan_line(quads + 8 * i, flags[i], font_size[i], im_w, im_h, channels, textheight, regions[i], L);
    regions[i].offset = off;
    off += regions[i].bytes;
    if (regions[i].status == CTD_REGION_OK && launch) {
      L.offset = (long long)regions[i].offset;
      L.tile0 = tiles;
      tiles += ((long long)regions[i].bytes / channels + kWarpThreads - 1) / kWarpThreads;
      launch->push_back(L);
    }
  }
  *total = off;
  return CTD_OK;
}

}  // namespace

#define CK(expr)                                                                                      \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess) return ctd_fail(h, CTD_E_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

extern "C" int ctd_plan_regions(const double* quads, const int32_t* flags, const double* font_size, int32_t n,
                                int32_t im_w, int32_t im_h, int32_t channels, double textheight, ctd_region* regions,
                                size_t* total_bytes) {
  if (n < 0 || !total_bytes || (n > 0 && (!quads || !flags || !font_size || !regions))) return CTD_E_INVALID;
  if ((channels != 1 && channels != 3) || im_w < 1 || im_h < 1) return CTD_E_INVALID;
  return plan_all(quads, flags, font_size, n, im_w, im_h, channels, textheight, regions, nullptr, total_bytes);
}

extern "C" int ctd_transform_regions(ctd_handle* h, const uint8_t* img, int32_t ih, int32_t iw, int32_t channels,
                                     int32_t img_on_device, const double* quads, const int32_t* flags,
                                     const double* font_size, int32_t n, double textheight, ctd_region* regions,
                                     uint8_t* out, int32_t out_on_device, size_t out_bytes) {
  if (!h) return CTD_E_INVALID;
  if (n < 0 || !img || (n > 0 && (!quads || !flags || !font_size || !regions)))
    return ctd_fail(h, CTD_E_INVALID, "ctd_transform_regions: null argument or n < 0");
  if (channels != 1 && channels != 3) return ctd_fail(h, CTD_E_INVALID, "ctd_transform_regions: channels must be 1 or 3, got %d", channels);
  if (ih < 1 || iw < 1 || ih > 32767 || iw > 32767) return ctd_fail(h, CTD_E_INVALID, "ctd_transform_regions: bad page size %dx%d", ih, iw);
  std::vector<RegionLine> lines;
  size_t total = 0;
  plan_all(quads, flags, font_size, n, iw, ih, channels, textheight, regions, &lines, &total);
  if (out_bytes < total || (total > 0 && !out))
    return ctd_fail(h, CTD_E_CAPACITY, "ctd_transform_regions: the crops need %zu bytes, the output holds %zu", total, out_bytes);
  if (lines.empty()) return CTD_OK;
  CK(cudaSetDevice(h->cfg.device));
  // scratch: [page (host pages only)] [line records] [packed crops (host output only)]
  const size_t page_bytes = img_on_device ? 0 : size_t(ih) * iw * channels;
  const size_t rec_off = (page_bytes + 255) / 256 * 256;
  const size_t rec_bytes = lines.size() * sizeof(RegionLine);
  const size_t out_off = (rec_off + rec_bytes + 255) / 256 * 256;
  if (int rc = ensure_io_scratch(h, out_off + (out_on_device ? 0 : total))) return rc;
  const uint8_t* d_img = img;
  if (!img_on_device) {
    CK(cudaMemcpyAsync(h->d_io_scratch, img, page_bytes, cudaMemcpyHostToDevice, h->stream));
    d_img = h->d_io_scratch;
  }
  RegionLine* d_lines = reinterpret_cast<RegionLine*>(h->d_io_scratch + rec_off);
  uint8_t* d_out = out_on_device ? out : h->d_io_scratch + out_off;
  CK(cudaMemcpyAsync(d_lines, lines.data(), rec_bytes, cudaMemcpyHostToDevice, h->stream));
  const int nl = int(lines.size());
  k_region_homography<<<(nl + 63) / 64, 64, 0, h->stream>>>(d_lines, nl);
  CK(cudaGetLastError());
  const RegionLine& last = lines.back();
  const long long tiles = last.tile0 + ((long long)last.ww * last.wh + kWarpThreads - 1) / kWarpThreads;
  if (tiles > 0x7fffffffLL) return ctd_fail(h, CTD_E_CAPACITY, "ctd_transform_regions: %lld blocks", tiles);
  if (channels == 3) k_region_warp<3><<<unsigned(tiles), kWarpThreads, 0, h->stream>>>(d_lines, nl, d_img, ih, iw, d_out);
  else k_region_warp<1><<<unsigned(tiles), kWarpThreads, 0, h->stream>>>(d_lines, nl, d_img, ih, iw, d_out);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(lines.data(), d_lines, rec_bytes, cudaMemcpyDeviceToHost, h->stream));
  if (!out_on_device) CK(cudaMemcpyAsync(out, d_out, total, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  for (int i = 0, j = 0; i < n; ++i)
    if (regions[i].status == CTD_REGION_OK) {
      for (int k = 0; k < 9; ++k) regions[i].M[k] = lines[j].M[k];
      ++j;
    }
  return CTD_OK;
}
