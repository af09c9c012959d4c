// Post-NMS geometry and CSL targets (HBM-bound elementwise kernels; one thread per box):
//   y5obb_rbox2poly_f32      /root/reference/utils/rboxs_utils.py:106-126  (torch branch of rbox2poly)
//   y5obb_poly2hbb_f32       /root/reference/utils/rboxs_utils.py:147-165  (torch branch of poly2hbb)
//   y5obb_scale_polys_f32    /root/reference/utils/general.py:636-650      (scale_polys, in place)
//   y5obb_gaussian_label     /root/reference/utils/rboxs_utils.py:9-26     (gaussian_label_cpu: 180-bin CSL row)
// Each arithmetic step is a separately rounded fp32 op (no FMA contraction), like the chain of ATen
// elementwise kernels it replaces; the CSL row is evaluated in fp64 like the numpy original.
#include <algorithm>

#include "common.cuh"
#include "rbox_poly.cuh"

namespace y5obb {
namespace {

__global__ void k_rbox2poly(const float* __restrict__ r, float* __restrict__ p, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  rbox_to_poly(r[5 * i], r[5 * i + 1], r[5 * i + 2], r[5 * i + 3], r[5 * i + 4], p + 8 * i);
}

__global__ void k_poly2hbb(const float* __restrict__ p, float* __restrict__ hbb, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* q = p + 8 * i;
  const float xmax = fmaxf(fmaxf(q[0], q[2]), fmaxf(q[4], q[6])), xmin = fminf(fminf(q[0], q[2]), fminf(q[4], q[6]));
  const float ymax = fmaxf(fmaxf(q[1], q[3]), fmaxf(q[5], q[7])), ymin = fminf(fminf(q[1], q[3]), fminf(q[5], q[7]));
  hbb[4 * i] = __fdiv_rn(__fadd_rn(xmax, xmin), 2.0f);
  hbb[4 * i + 1] = __fdiv_rn(__fadd_rn(ymax, ymin), 2.0f);
  hbb[4 * i + 2] = __fsub_rn(xmax, xmin);
  hbb[4 * i + 3] = __fsub_rn(ymax, ymin);
}

__global__ void k_scale_polys(float* __restrict__ p, int64_t n, float padx, float pady, float gain) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * 8) return;
  const float pad = (i & 1) ? pady : padx;
  p[i] = __fdiv_rn(__fsub_rn(p[i], pad), gain);
}

// out[k] = exp(-(x_j)^2 / (2 sigma^2)), j = (k + int(nc/2 - angle)) mod nc, x_j = j - nc/2
__global__ void k_gaussian_label(const double* __restrict__ angle, float* __restrict__ out, int64_t n, int nc, double sig) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * nc) return;
  const int64_t row = i / nc;
  const int k = (int)(i - row * nc);
  const int index = (int)((double)nc / 2.0 - angle[row]);  // int(): truncation toward zero
  int j = (k + index) % nc;
  if (j < 0) j += nc;
  const double x = (double)j - (double)nc / 2.0;
  out[i] = (float)exp(-(x * x) / (2.0 * sig * sig));
}

// poly2rbox (utils/rboxs_utils.py:39-81): the arithmetic of the reference is cv2.minAreaRect on the 4 float32 points
// (opencv-python >= 4.5.4, not vendored).  Published algorithm restated (rotcalipers.cpp): convex hull; the minimum-area
// enclosing rectangle has a side collinear with a hull edge.  One thread per polygon, double precision throughout
// (the long-edge result does not depend on which of cv2's equivalent (w, h, angle) forms is used), then the reference's
// own post-processing verbatim: theta = -angle/180*pi, long-edge swap (+pi/2), wrap to [-pi/2, pi/2) with pi = 3.141592.
__device__ __forceinline__ double cross3(const double* o, const double* a, const double* b) {
  return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0]);
}

__global__ void k_poly2rbox(const float* __restrict__ polys, double* __restrict__ out, long long n, int use_pi) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double PI_REF = 3.141592;
  double p[4][2];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    p[k][0] = (double)polys[i * 8 + 2 * k];
    p[k][1] = (double)polys[i * 8 + 2 * k + 1];
  }
  // sort lexicographically (x, then y), drop duplicates
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3 - a; ++b)
      if (p[b][0] > p[b + 1][0] || (p[b][0] == p[b + 1][0] && p[b][1] > p[b + 1][1])) {
        const double tx = p[b][0], ty = p[b][1];
        p[b][0] = p[b + 1][0];
        p[b][1] = p[b + 1][1];
        p[b + 1][0] = tx;
        p[b + 1][1] = ty;
      }
  int m = 0;
  double q[4][2];
  for (int k = 0; k < 4; ++k)
    if (k == 0 || p[k][0] != p[k - 1][0] || p[k][1] != p[k - 1][1]) {
      q[m][0] = p[k][0];
      q[m][1] = p[k][1];
      ++m;
    }
  double x = q[0][0], y = q[0][1], w = 0.0, h = 0.0, angle = 0.0;
  double hull[8][2];
  int nh = 0;
  if (m >= 3) {  // Andrew's monotone chain
    int lo = 0;
    for (int k = 0; k < m; ++k) {
      while (lo >= 2 && cross3(hull[lo - 2], hull[lo - 1], q[k]) <= 0) --lo;
      hull[lo][0] = q[k][0];
      hull[lo][1] = q[k][1];
      ++lo;
    }
    int up = lo - 1;  // the last lower point is shared
    const int base = up;
    for (int k = m - 1; k >= 0; --k) {
      while (up - base >= 2 && cross3(hull[up - 2], hull[up - 1], q[k]) <= 0) --up;
      hull[up][0] = q[k][0];
      hull[up][1] = q[k][1];
      ++up;
    }
    nh = up - 1;  // the last upper point is the first lower point
  }
  if (m >= 3 && nh >= 3) {
    double best = -1.0, bu0 = 1, bu1 = 0, amin = 0, amax = 0, bmin = 0, bmax = 0;
    for (int e = 0; e < nh; ++e) {
      const double ex = hull[(e + 1) % nh][0] - hull[e][0], ey = hull[(e + 1) % nh][1] - hull[e][1];
      const double len = hypot(ex, ey);
      const double u0 = ex / len, u1 = ey / len;
      double a0 = 1e300, a1 = -1e300, b0 = 1e300, b1 = -1e300;
      for (int k = 0; k < nh; ++k) {
        const double a = __dadd_rn(__dmul_rn(hull[k][0], u0), __dmul_rn(hull[k][1], u1));
        const double b = __dadd_rn(__dmul_rn(hull[k][0], -u1), __dmul_rn(hull[k][1], u0));
        a0 = fmin(a0, a);
        a1 = fmax(a1, a);
        b0 = fmin(b0, b);
        b1 = fmax(b1, b);
      }
      const double area = __dmul_rn(a1 - a0, b1 - b0);
      if (best < 0 || area < best * (1 - 1e-12)) {
        best = area;
        bu0 = u0;
        bu1 = u1;
        amin = a0;
        amax = a1;
        bmin = b0;
        bmax = b1;
      }
    }
    const double ca = (amax + amin) / 2, cb = (bmax + bmin) / 2;
    x = __dadd_rn(__dmul_rn(bu0, ca), __dmul_rn(-bu1, cb));
    y = __dadd_rn(__dmul_rn(bu1, ca), __dmul_rn(bu0, cb));
    const double eu = amax - amin, en = bmax - bmin;
    double alpha = fmod(atan2(bu1, bu0) * (180.0 / 3.14159265358979323846), 180.0);
    if (alpha < 0) alpha += 180.0;
    if (alpha < 1e-9 || alpha > 180.0 - 1e-9) {
      w = en;
      h = eu;
      angle = 90.0;
    } else if (alpha <= 90.0) {
      w = eu;
      h = en;
      angle = alpha;
    } else {
      w = en;
      h = eu;
      angle = alpha - 90.0;
    }
  } else if (m == 2 || (m >= 3 && nh == 2)) {  // a segment: its two extreme points are the first and last sorted ones
    const double x0 = q[0][0], y0 = q[0][1], x1 = q[m - 1][0], y1 = q[m - 1][1];
    x = (x0 + x1) / 2;
    y = (y0 + y1) / 2;
    w = hypot(x1 - x0, y1 - y0);
    h = 0.0;
    angle = atan2(y1 - y0, x1 - x0) * (180.0 / 3.14159265358979323846);
  }
  double theta = -angle / 180 * PI_REF;
  if (w != fmax(w, h)) {
    const double t = w;
    w = h;
    h = t;
    theta += PI_REF / 2;
  }
  const double start = -PI_REF / 2;
  double r = fmod(theta - start, PI_REF);  // python %: result has the sign of the divisor
  if (r < 0) r += PI_REF;
  theta = r + start;
  double* o = out + i * 5;
  o[0] = x;
  o[1] = y;
  o[2] = w;
  o[3] = h;
  o[4] = use_pi ? theta : theta * 180 / PI_REF + 90;
}

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

int y5obb_rbox2poly_f32(const float* rboxes5, float* polys8, int64_t n, void* stream) {
  if (n < 0) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!rboxes5 || !polys8) return Y5OBB_EINVAL;
  k_rbox2poly<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rboxes5, polys8, n);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_poly2hbb_f32(const float* polys8, float* hbb4, int64_t n, void* stream) {
  if (n < 0) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!polys8 || !hbb4) return Y5OBB_EINVAL;
  k_poly2hbb<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(polys8, hbb4, n);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_scale_polys_f32(float* polys8, int64_t n, float pad_x, float pad_y, float gain, void* stream) {
  if (n < 0 || gain == 0.0f) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!polys8) return Y5OBB_EINVAL;
  k_scale_polys<<<(unsigned)((n * 8 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(polys8, n, pad_x, pad_y, gain);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_poly2rbox(const float* polys8, double* rbox5, int64_t n, int use_pi, void* stream) {
  if (n < 0) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!polys8 || !rbox5) return Y5OBB_EINVAL;
  k_poly2rbox<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(polys8, rbox5, n, use_pi);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_gaussian_label(const double* angle_deg, float* csl_out, int64_t n, int num_class, double sigma, void* stream) {
  if (n < 0 || num_class <= 0 || !(sigma > 0)) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!angle_deg || !csl_out) return Y5OBB_EINVAL;
  k_gaussian_label<<<(unsigned)((n * num_class + 255) / 256), 256, 0, (cudaStream_t)stream>>>(angle_deg, csl_out, n,
                                                                                              num_class, sigma);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

}  // extern "C"
