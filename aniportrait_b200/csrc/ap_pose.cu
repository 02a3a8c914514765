// Face-mesh pose maps of audio2vid / vid2vid: head-pose smoothing, landmark projection and the face-mesh rasteriser
// (reference src/utils/pose_util.py and src/utils/draw_util.py FaceMeshVisualizer.draw_landmarks).
//
//   pose_smooth        the sliding-window mean of smooth_pose_seq, summed row after row in the input dtype, no FMA
//   project            perspective projection of [L, N, 3] points in fp64, one CTA per frame
//   facemesh_raster    cv2.line(thickness=2, LINE_8) of every face-mesh edge on a 512 x 512 canvas of colour-group ids,
//                      one CTA per (frame, band of canvas rows), one thread per edge; the highest group wins a pixel
//   facemesh_colour    group ids -> BGR colours, fused with cv2.resize(INTER_LINEAR) to the target size
//
// Every step is order-fixed or an atomicMax over integers: two calls give the same bytes. oracle/cv2_line.py is the
// written specification of the line and resize arithmetic.
#include "ap_host.h"
#include "ap_ptx.cuh"

namespace ap {

// ---------------------------------------------------------------------------------------------------------
// smooth_pose_seq: out[i] = mean(x[max(0, i - w/2) : min(L, i + w/2 + 1)], axis=0) as numpy computes it (the first
// row, then each further row added in the input dtype, then one division by the count).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double div_rn(double a, double b) { return __ddiv_rn(a, b); }

template <typename T>
__global__ void __launch_bounds__(256) pose_smooth_kernel(const T* __restrict__ x, int L, int C, int half, T* __restrict__ out) {
  griddep_launch_dependents();
  griddep_wait();
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)L * C) return;
  const int i = (int)(idx / C), c = (int)(idx % C);
  const int s = max(0, i - half), e = min(L, i + half + 1);
  T acc = x[(long long)s * C + c];
  for (int r = s + 1; r < e; ++r) acc = add_rn(acc, x[(long long)r * C + c]);
  out[idx] = div_rn(acc, (T)(e - s));
}

// ---------------------------------------------------------------------------------------------------------
// Projection. The frame's 4 x 4 model matrix M (trans_mat @ [R | t], or the given per-frame matrix) is built by thread 0
// in fp64; then per point u = M (x, y, z, 1) and, with create_perspective_matrix's P (fp32 entries promoted to fp64):
//   t0 = u0 P00, t1 = u1 P11, t3 = u2 P23 (the only non-zero entries that reach x, y and w),
//   px = (t0 / t3 + 1) 0.5 W,  py = (t1 / t3 + 1) 0.5 H.
// R = Rz Ry Rx is scipy's Rotation.from_euler('xyz', degrees=True) (extrinsic axes).
// ---------------------------------------------------------------------------------------------------------
constexpr double kPerspF = 0x1.a1c1083c23fccp+0;  // 1 / tan(63 degrees / 2), as numpy computes it in fp64

template <typename T>
__device__ __forceinline__ double ld64(const void* p, long long i) { return (double)static_cast<const T*>(p)[i]; }

__device__ __forceinline__ double load_any(const void* p, long long i, int f64) {
  return f64 ? ld64<double>(p, i) : ld64<float>(p, i);
}

__global__ void __launch_bounds__(256)
project_kernel(const void* __restrict__ pts, int pts_f64, int N, const void* __restrict__ trans, int trans_f64,
               const void* __restrict__ pose, int pose_f64, int W, int H, double* __restrict__ out) {
  griddep_launch_dependents();
  griddep_wait();
  __shared__ double M[12];  // rows 0..2 of the model matrix (row 3 reaches only t2, which is unused)
  const int f = blockIdx.x;
  if (threadIdx.x == 0) {
    double T[16];
    if (pose) {
      const double kDeg = 0x1.1df46a2529d39p-6;  // np.pi / 180
      double a[3], s[3], c[3];
      for (int k = 0; k < 3; ++k) {
        a[k] = __dmul_rn(load_any(pose, (long long)f * 6 + k, pose_f64), kDeg);
        sincos(a[k], &s[k], &c[k]);
      }
      const double R[9] = {c[2] * c[1], c[2] * s[1] * s[0] - s[2] * c[0], c[2] * s[1] * c[0] + s[2] * s[0],
                           s[2] * c[1], s[2] * s[1] * s[0] + c[2] * c[0], s[2] * s[1] * c[0] - c[2] * s[0],
                           -s[1],       c[1] * s[0],                      c[1] * c[0]};
      double E[16];
      for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) E[r * 4 + k] = R[r * 3 + k];
        E[r * 4 + 3] = load_any(pose, (long long)f * 6 + 3 + r, pose_f64);
      }
      E[12] = E[13] = E[14] = 0.0;
      E[15] = 1.0;
      double Tm[16];
      for (int k = 0; k < 16; ++k) Tm[k] = load_any(trans, k, trans_f64);
      for (int r = 0; r < 4; ++r)
        for (int k = 0; k < 4; ++k) {
          double acc = 0.0;
          for (int j = 0; j < 4; ++j) acc += Tm[r * 4 + j] * E[j * 4 + k];
          T[r * 4 + k] = acc;
        }
    } else {
      for (int k = 0; k < 16; ++k) T[k] = load_any(trans, (long long)f * 16 + k, trans_f64);
    }
    // rows 0, 1 and 2 of M: x, y and the depth that w is made of
    for (int k = 0; k < 12; ++k) M[k] = T[k];
  }
  __syncthreads();
  const double aspect = __ddiv_rn((double)W, (double)H);
  const double p00 = (double)__double2float_rn(__ddiv_rn(kPerspF, aspect));
  const double p11 = -(double)__double2float_rn(kPerspF);
  const double p23 = (double)__double2float_rn(__dmul_rn(10000.0, __ddiv_rn(1.0, -9999.0)));
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    const long long b = ((long long)f * N + n) * 3;
    const double x = load_any(pts, b, pts_f64), y = load_any(pts, b + 1, pts_f64), z = load_any(pts, b + 2, pts_f64);
    const double u0 = M[0] * x + M[1] * y + M[2] * z + M[3];
    const double u1 = M[4] * x + M[5] * y + M[6] * z + M[7];
    const double u2 = M[8] * x + M[9] * y + M[10] * z + M[11];
    const double w = u2 * p23;
    out[((long long)f * N + n) * 2 + 0] = (u0 * p00 / w + 1.0) * 0.5 * (double)W;
    out[((long long)f * N + n) * 2 + 1] = (u1 * p11 / w + 1.0) * 0.5 * (double)H;
  }
}

// ---------------------------------------------------------------------------------------------------------
// Face-mesh rasteriser (oracle/cv2_line.py step by step). Canvas 512 x 512, 16-bit fixed point (XY_SHIFT = 16).
// ---------------------------------------------------------------------------------------------------------
constexpr int CANVAS = 512;
constexpr int RASTER_BAND = 16;         // canvas rows per CTA
constexpr int RASTER_THREADS = 128;
constexpr int XY_SHIFT = 16;
constexpr long long XY_ONE = 1ll << XY_SHIFT;

struct Band {
  int* grp;  // [RASTER_BAND][CANVAS] highest group id per pixel, -1 = none
  int y0;
  int g;
  __device__ __forceinline__ void put(long long x, long long y) const {
    if (x >= 0 && x < CANVAS && y >= y0 && y < y0 + RASTER_BAND) atomicMax(&grp[(y - y0) * CANVAS + x], g);
  }
};

__device__ __forceinline__ long long cdiv(long long a, long long b) { return a / b; }  // C truncation, as OpenCV

// clipLine on [0, (512 << 16) - 1]^2; false if the segment lies outside.
__device__ bool clip_line(long long& x1, long long& y1, long long& x2, long long& y2) {
  const long long right = ((long long)CANVAS << XY_SHIFT) - 1, bottom = right;
  int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
  int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
  if ((c1 & c2) == 0 && (c1 | c2) != 0) {
    long long a;
    if (c1 & 12) {
      a = c1 < 8 ? 0 : bottom;
      x1 += (long long)__ddiv_rn(__dmul_rn((double)(a - y1), (double)(x2 - x1)), (double)(y2 - y1));
      y1 = a;
      c1 = (x1 < 0) + (x1 > right) * 2;
    }
    if (c2 & 12) {
      a = c2 < 8 ? 0 : bottom;
      x2 += (long long)__ddiv_rn(__dmul_rn((double)(a - y2), (double)(x2 - x1)), (double)(y2 - y1));
      y2 = a;
      c2 = (x2 < 0) + (x2 > right) * 2;
    }
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
      if (c1) {
        a = c1 == 1 ? 0 : right;
        y1 += (long long)__ddiv_rn(__dmul_rn((double)(a - x1), (double)(y2 - y1)), (double)(x2 - x1));
        x1 = a;
        c1 = 0;
      }
      if (c2) {
        a = c2 == 1 ? 0 : right;
        y2 += (long long)__ddiv_rn(__dmul_rn((double)(a - x2), (double)(y2 - y1)), (double)(x2 - x1));
        x2 = a;
        c2 = 0;
      }
    }
  }
  return (c1 | c2) == 0;
}

// Line2: the 8-connected line between two fixed-point points.
__device__ void line2(const Band& band, long long x1, long long y1, long long x2, long long y2) {
  if (!clip_line(x1, y1, x2, y2)) return;
  long long dx = x2 - x1, dy = y2 - y1;
  const long long ax = dx < 0 ? -dx : dx, ay = dy < 0 ? -dy : dy;
  long long x_step = 0, y_step = 0, ecount;
  if (ax > ay) {
    if (dx < 0) {
      dy = -dy;
      long long t = x1; x1 = x2; x2 = t;
      t = y1; y1 = y2; y2 = t;
    }
    y_step = cdiv(dy * XY_ONE, ax | 1);
    ecount = (x2 - x1) >> XY_SHIFT;
  } else {
    if (dy < 0) {
      dx = -dx;
      long long t = x1; x1 = x2; x2 = t;
      t = y1; y1 = y2; y2 = t;
    }
    x_step = cdiv(dx * XY_ONE, ay | 1);
    ecount = (y2 - y1) >> XY_SHIFT;
  }
  x1 += XY_ONE >> 1;
  y1 += XY_ONE >> 1;
  band.put((x2 + (XY_ONE >> 1)) >> XY_SHIFT, (y2 + (XY_ONE >> 1)) >> XY_SHIFT);
  if (ax > ay) {
    x1 >>= XY_SHIFT;
    for (; ecount >= 0; --ecount, ++x1, y1 += y_step) band.put(x1, y1 >> XY_SHIFT);
  } else {
    y1 >>= XY_SHIFT;
    for (; ecount >= 0; --ecount, x1 += x_step, ++y1) band.put(x1 >> XY_SHIFT, y1);
  }
}

// FillConvexPoly of the four corners (shift = XY_SHIFT, LINE_8): outline, then the scanline fill.
__device__ void fill_quad(const Band& band, const long long (&vx)[4], const long long (&vy)[4]) {
  constexpr int npts = 4;
  const long long delta = XY_ONE >> 1;
  long long xmin = vx[0], xmax = vx[0], ymin = vy[0], ymax = vy[0];
  int imin = 0;
  for (int i = 0, prev = npts - 1; i < npts; prev = i++) {
    if (vy[i] < ymin) {
      ymin = vy[i];
      imin = i;
    }
    ymax = max(ymax, vy[i]);
    xmax = max(xmax, vx[i]);
    xmin = min(xmin, vx[i]);
    line2(band, vx[prev], vy[prev], vx[i], vy[i]);
  }
  xmin = (xmin + delta) >> XY_SHIFT;
  xmax = (xmax + delta) >> XY_SHIFT;
  ymin = (ymin + delta) >> XY_SHIFT;
  ymax = (ymax + delta) >> XY_SHIFT;
  if (xmax < 0 || ymax < 0 || xmin >= CANVAS || ymin >= CANVAS) return;
  ymax = min(ymax, (long long)CANVAS - 1);
  int e_idx[2] = {imin, imin};
  const int e_di[2] = {1, npts - 1};
  long long e_x[2] = {-XY_ONE, -XY_ONE}, e_dx[2] = {0, 0}, e_ye[2] = {ymin, ymin};
  int edges = npts;
  long long y = ymin;
  do {
    for (int i = 0; i < 2; ++i) {
      if (y >= e_ye[i]) {
        int idx0 = e_idx[i];
        int idx = idx0 + e_di[i];
        if (idx >= npts) idx -= npts;
        for (; edges-- > 0;) {
          const long long ty = (vy[idx] + delta) >> XY_SHIFT;
          if (ty > y) {
            e_ye[i] = ty;
            e_dx[i] = cdiv((vx[idx] - vx[idx0]) * 2 + (ty - y), 2 * (ty - y));
            e_x[i] = vx[idx0];
            e_idx[i] = idx;
            break;
          }
          idx0 = idx;
          idx += e_di[i];
          if (idx >= npts) idx -= npts;
        }
      }
    }
    if (edges < 0) break;
    if (y >= band.y0 + RASTER_BAND) break;  // the remaining rows lie below this band
    if (y >= band.y0) {
      const int l = e_x[0] > e_x[1] ? 1 : 0;
      long long xx1 = (e_x[l] + delta) >> XY_SHIFT, xx2 = (e_x[1 - l] + delta) >> XY_SHIFT;
      if (xx2 >= 0 && xx1 < CANVAS) {
        xx1 = max(xx1, 0ll);
        xx2 = min(xx2, (long long)CANVAS - 1);
        for (long long x = xx1; x <= xx2; ++x) band.put(x, y);
      }
    }
    e_x[0] += e_dx[0];
    e_x[1] += e_dx[1];
  } while (++y <= ymax);
}

// The landmark's canvas pixel, or false if mediapipe's is_valid_normalized_value rejects it. The normalised value is
// rounded to fp32 (the landmark protobuf's float field); x / size in fp32 for fp32 input (numpy: float32 / int).
__device__ __forceinline__ bool landmark_px(const void* kp, int f64, long long i, int normed, int size, int& px) {
  float v;
  if (f64) {
    const double d = static_cast<const double*>(kp)[i];
    v = __double2float_rn(normed ? d : __ddiv_rn(d, (double)size));
  } else {
    const float s = static_cast<const float*>(kp)[i];
    v = normed ? s : __fdiv_rn(s, (float)size);
  }
  if (!(v >= 0.f && v <= 1.f)) return false;
  px = min((int)floorf(v * (float)CANVAS), CANVAS - 1);
  return true;
}

__global__ void __launch_bounds__(RASTER_THREADS)
facemesh_raster_kernel(const void* __restrict__ kp, int kp_f64, int N, int normed, int W, int H,
                       const int* __restrict__ edges, int E, unsigned char* __restrict__ canvas) {
  griddep_launch_dependents();
  __shared__ int grp[RASTER_BAND * CANVAS];
  const int f = blockIdx.y;
  for (int i = threadIdx.x; i < RASTER_BAND * CANVAS; i += RASTER_THREADS) grp[i] = -1;
  griddep_wait();
  __syncthreads();
  for (int e = threadIdx.x; e < E; e += RASTER_THREADS) {
    const int a = edges[e * 3], b = edges[e * 3 + 1];
    if (a < 0 || b < 0 || a >= N || b >= N) continue;
    Band band{grp, (int)blockIdx.x * RASTER_BAND, edges[e * 3 + 2]};
    const long long base = (long long)f * N;
    int x0, y0, x1, y1;
    if (!(landmark_px(kp, kp_f64, (base + a) * 2, normed, W, x0) &&
          landmark_px(kp, kp_f64, (base + a) * 2 + 1, normed, H, y0) &&
          landmark_px(kp, kp_f64, (base + b) * 2, normed, W, x1) &&
          landmark_px(kp, kp_f64, (base + b) * 2 + 1, normed, H, y1)))
      continue;
    // every pixel of a thickness-2 line lies within one row of its end points' rows
    if (max(y0, y1) + 1 < band.y0 || min(y0, y1) - 1 >= band.y0 + RASTER_BAND) continue;
    const long long p0x = (long long)x0 << XY_SHIFT, p0y = (long long)y0 << XY_SHIFT;
    const long long p1x = (long long)x1 << XY_SHIFT, p1y = (long long)y1 << XY_SHIFT;
    const double ddx = (double)(p0x - p1x) * (1.0 / XY_ONE), ddy = (double)(p1y - p0y) * (1.0 / XY_ONE);
    const double r2 = __dadd_rn(__dmul_rn(ddx, ddx), __dmul_rn(ddy, ddy));
    if (r2 > 0x1p-52) {  // DBL_EPSILON: a zero-length segment draws only the end circles
      const double r = __ddiv_rn((double)XY_ONE, __dsqrt_rn(r2));
      const long long dpx = __double2ll_rn(__dmul_rn(ddy, r)), dpy = __double2ll_rn(__dmul_rn(ddx, r));
      const long long vx[4] = {p0x + dpx, p0x - dpx, p1x - dpx, p1x + dpx};
      const long long vy[4] = {p0y + dpy, p0y - dpy, p1y - dpy, p1y + dpy};
      fill_quad(band, vx, vy);
    }
    const int cx[2] = {x0, x1}, cy[2] = {y0, y1};
    for (int k = 0; k < 2; ++k) {  // filled circle of radius 1
      band.put(cx[k], cy[k]);
      band.put(cx[k] - 1, cy[k]);
      band.put(cx[k] + 1, cy[k]);
      band.put(cx[k], cy[k] - 1);
      band.put(cx[k], cy[k] + 1);
    }
  }
  __syncthreads();
  // group id + 1 per pixel (0 = background), 16 bytes per store
  uint4* dst = reinterpret_cast<uint4*>(canvas + ((long long)f * CANVAS + blockIdx.x * RASTER_BAND) * CANVAS);
  for (int i = threadIdx.x; i < RASTER_BAND * CANVAS / 16; i += RASTER_THREADS) {
    uint32_t w[4];
    for (int q = 0; q < 4; ++q) {
      const int* g = &grp[i * 16 + q * 4];
      w[q] = (uint32_t)(g[0] + 1) | ((uint32_t)(g[1] + 1) << 8) | ((uint32_t)(g[2] + 1) << 16) |
             ((uint32_t)(g[3] + 1) << 24);
    }
    dst[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// cv2.resize INTER_LINEAR taps of destination index d (src = 512): source index, and 11-bit weights c0 + c1.
__device__ __forceinline__ void linear_tap(int d, int dst, int& i0, int& i1, int& c0, int& c1) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn((double)dst, (double)CANVAS));
  float fx = __double2float_rn(__dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5));
  int sx = (int)floorf(fx);
  fx = __fsub_rn(fx, (float)sx);
  if (sx < 0) fx = 0.f, sx = 0;
  if (sx >= CANVAS - 1) fx = 0.f, sx = CANVAS - 1;
  i0 = sx;
  i1 = min(sx + 1, CANVAS - 1);
  c0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, fx), 2048.f));
  c1 = __float2int_rn(__fmul_rn(fx, 2048.f));
}

// One thread = 4 consecutive output pixels (12 bytes, three 32-bit stores). Colour = colours[group id - 1], black for 0.
// Horizontal pass to int (weights sum to 2048), then OpenCV's vectorised vertical rounding
// ((h0 >> 4) * b0 >> 16) + ((h1 >> 4) * b1 >> 16) + 2 >> 2. At 512 x 512 the weights are (2048, 0): a plain copy.
__global__ void __launch_bounds__(256)
facemesh_colour_kernel(const unsigned char* __restrict__ canvas, const unsigned char* __restrict__ colours, int G, int W,
                       int H, long long quads, unsigned char* __restrict__ out) {
  griddep_launch_dependents();
  __shared__ unsigned char lut[256 * 3];
  for (int i = threadIdx.x; i < 256 * 3; i += blockDim.x) lut[i] = (i >= 3 && i < (G + 1) * 3) ? colours[i - 3] : 0;
  griddep_wait();
  __syncthreads();
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= quads) return;
  const int qpr = W / 4;
  const long long row = q / qpr;
  const int f = (int)(row / H), oy = (int)(row % H), ox0 = (int)(q % qpr) * 4;
  int r0, r1, b0, b1;
  linear_tap(oy, H, r0, r1, b0, b1);
  const unsigned char* c0row = canvas + ((long long)f * CANVAS + r0) * CANVAS;
  const unsigned char* c1row = canvas + ((long long)f * CANVAS + r1) * CANVAS;
  uint32_t packed[3] = {0, 0, 0};
  for (int p = 0; p < 4; ++p) {
    int s0, s1, a0, a1;
    linear_tap(ox0 + p, W, s0, s1, a0, a1);
    const unsigned char* k00 = &lut[c0row[s0] * 3];
    const unsigned char* k01 = &lut[c0row[s1] * 3];
    const unsigned char* k10 = &lut[c1row[s0] * 3];
    const unsigned char* k11 = &lut[c1row[s1] * 3];
    for (int ch = 0; ch < 3; ++ch) {
      const int h0 = k00[ch] * a0 + k01[ch] * a1, h1 = k10[ch] * a0 + k11[ch] * a1;
      int v = ((((h0 >> 4) * b0) >> 16) + (((h1 >> 4) * b1) >> 16) + 2) >> 2;
      v = min(max(v, 0), 255);
      const int byte = p * 3 + ch;
      packed[byte >> 2] |= (uint32_t)v << ((byte & 3) * 8);
    }
  }
  uint32_t* dst = reinterpret_cast<uint32_t*>(out + q * 12);
  dst[0] = packed[0];
  dst[1] = packed[1];
  dst[2] = packed[2];
}

}  // namespace ap

using namespace ap;

extern "C" int ap_pose_smooth(const void* x, int L, int window, int f64, void* out, void* stream) {
  AP_REQUIRE(x && out, "pose_smooth: null pointer");
  AP_REQUIRE(L > 0 && window > 0, "pose_smooth: bad shape L=%d window=%d", L, window);
  AP_REQUIRE(x != out, "pose_smooth: out must not alias x");
  const long long n = (long long)L * 6;
  if (f64)
    AP_LAUNCH(pose_smooth_kernel<double>, (unsigned)((n + 255) / 256), 256, 0, stream, (const double*)x, L, 6,
              window / 2, (double*)out);
  else
    AP_LAUNCH(pose_smooth_kernel<float>, (unsigned)((n + 255) / 256), 256, 0, stream, (const float*)x, L, 6,
              window / 2, (float*)out);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}

extern "C" int ap_project_points(const void* points, int points_f64, int L, int N, const void* trans, int trans_f64,
                                 const void* pose, int pose_f64, int W, int H, double* out, void* stream) {
  AP_REQUIRE(points && trans && out, "project_points: null pointer");
  AP_REQUIRE(L > 0 && N > 0 && W > 0 && H > 0, "project_points: bad shape L=%d N=%d W=%d H=%d", L, N, W, H);
  AP_LAUNCH(project_kernel, (unsigned)L, 256, 0, stream, points, points_f64, N, trans, trans_f64, pose, pose_f64, W, H,
            out);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}

extern "C" int ap_facemesh_raster(const void* keypoints, int kp_f64, int L, int N, int normed, int W, int H,
                                  const int* edges, int E, const unsigned char* colours, int G, void* canvas, void* out,
                                  void* stream) {
  AP_REQUIRE(keypoints && edges && colours && canvas && out, "facemesh_raster: null pointer");
  AP_REQUIRE(L > 0 && N > 0 && E > 0, "facemesh_raster: bad shape L=%d N=%d E=%d", L, N, E);
  AP_REQUIRE(G > 0 && G <= 255, "facemesh_raster: %d colour groups (1..255)", G);
  AP_REQUIRE(W > 0 && H > 0 && W % 8 == 0 && H % 8 == 0, "facemesh_raster: W=%d H=%d must be multiples of 8", W, H);
  AP_REQUIRE((reinterpret_cast<uintptr_t>(canvas) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0,
             "facemesh_raster: canvas must be 16-byte and out 4-byte aligned");
  AP_LAUNCH(facemesh_raster_kernel, dim3(CANVAS / RASTER_BAND, (unsigned)L), RASTER_THREADS, 0, stream, keypoints,
            kp_f64, N, normed, W, H, edges, E, (unsigned char*)canvas);
  AP_CHECK_CUDA(cudaGetLastError());
  const long long quads = (long long)L * H * (W / 4);
  AP_LAUNCH(facemesh_colour_kernel, (unsigned)((quads + 255) / 256), 256, 0, stream, (const unsigned char*)canvas,
            colours, G, W, H, quads, (unsigned char*)out);
  AP_CHECK_CUDA(cudaGetLastError());
  return AP_OK;
}
