// Tile-merge polygon NMS of the DOTA devkit on the device (SURVEY section 8f rank 4, row A14's CPU form):
//   /root/reference/DOTA_devkit/ResultMerge_multi_process.py:62-123  py_cpu_nms_poly_fast
//   /root/reference/DOTA_devkit/polyiou.cpp:9-128                    iou_poly (double, eps = 1e-8 sign tests)
// Written against the bit-equal CPU restatement (oracle/poly_ref.py, pinned to the reference's polyiou.cpp compiled in
// place); on the B200 tests/test_poly_gpu.py finds the IoUs bit-equal and the keep lists equal to the reference's.
//
// Pipeline: CUB radix sort by descending score (stable, ties -> lower index, as numpy's argsort()[::-1] is NOT: the
// reference's tie order is the reverse index order; callers with tied scores get the documented lower-index-first rule) ->
// k_poly_mask: for every pair i < j of the sorted order the axis-aligned pre-filter and, where it fires, the polygon IoU
// in double precision with explicit round-to-nearest multiplies / adds (no FMA contraction: bit-equal to the reference's
// g++ -O2 build) -> bit r of word (i, j / 64) = "j is suppressed by i" = !(ovr <= thresh) -> k_poly_reduce: greedy scan.
#include <cub/cub.cuh>

#include "common.cuh"
#include "rbox_poly.cuh"

namespace y5obb {
namespace {

constexpr double PEPS = 1e-8;

struct P2 {
  double x, y;
};

__device__ __forceinline__ int psig(double d) { return (d > PEPS) - (d < -PEPS); }
__device__ __forceinline__ double pmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double padd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double psub(double a, double b) { return __dsub_rn(a, b); }
// (a.x-o.x)*(b.y-o.y) - (b.x-o.x)*(a.y-o.y)
__device__ __forceinline__ double pcross(P2 o, P2 a, P2 b) {
  return psub(pmul(psub(a.x, o.x), psub(b.y, o.y)), pmul(psub(b.x, o.x), psub(a.y, o.y)));
}
__device__ double parea(const P2* ps, int n) {
  double res = 0.0;
  for (int i = 0; i < n; ++i) {
    const int j = (i + 1 == n) ? 0 : i + 1;
    res = padd(res, psub(pmul(ps[i].x, ps[j].y), pmul(ps[i].y, ps[j].x)));
  }
  return res / 2.0;
}
__device__ __forceinline__ bool psame(P2 p, P2 q) { return psig(psub(p.x, q.x)) == 0 && psig(psub(p.y, q.y)) == 0; }

// polyiou.cpp:57-70: the part of polygon p (n points, n <= 8) to the left of a->b, in place
__device__ void polygon_cut(P2* p, int& n, P2 a, P2 b) {
  P2 pp[12];
  int m = 0;
  for (int i = 0; i < n; ++i) {
    const P2 pi = p[i], pj = p[(i + 1 == n) ? 0 : i + 1];
    const int si = psig(pcross(a, b, pi)), sj = psig(pcross(a, b, pj));
    if (si > 0) pp[m++] = pi;
    if (si != sj) {
      const double s1 = pcross(a, b, pi), s2 = pcross(a, b, pj);
      P2 x = pi;  // lineCross leaves its output untouched for (anti)parallel lines: cannot happen when the signs differ
      if (!(psig(s1) == 0 && psig(s2) == 0) && psig(psub(s2, s1)) != 0) {
        const double d = psub(s2, s1);
        x.x = psub(pmul(pi.x, s2), pmul(pj.x, s1)) / d;
        x.y = psub(pmul(pi.y, s2), pmul(pj.y, s1)) / d;
      }
      pp[m++] = x;
    }
  }
  n = 0;
  for (int i = 0; i < m; ++i)
    if (i == 0 || !psame(pp[i], pp[i - 1])) p[n++] = pp[i];
  while (n > 1 && psame(p[n - 1], p[0])) --n;
}

// polyiou.cpp:73-88: signed intersection area of the triangles (o, a, b) and (o, c, d), o the origin
__device__ double tri_intersect(P2 a, P2 b, P2 c, P2 d) {
  const P2 o = {0.0, 0.0};
  const int s1 = psig(pcross(o, a, b)), s2 = psig(pcross(o, c, d));
  if (s1 == 0 || s2 == 0) return 0.0;
  if (s1 == -1) {
    const P2 t = a;
    a = b;
    b = t;
  }
  if (s2 == -1) {
    const P2 t = c;
    c = d;
    d = t;
  }
  P2 p[12];
  p[0] = o;
  p[1] = a;
  p[2] = b;
  int n = 3;
  polygon_cut(p, n, o, c);
  polygon_cut(p, n, c, d);
  polygon_cut(p, n, d, o);
  const double res = n > 0 ? fabs(parea(p, n)) : 0.0;
  return (s1 * s2 == -1) ? -res : res;
}

__device__ double iou_poly_dev(const double* p8, const double* q8) {
  P2 a[4], b[4];
  for (int i = 0; i < 4; ++i) {
    a[i].x = p8[2 * i];
    a[i].y = p8[2 * i + 1];
    b[i].x = q8[2 * i];
    b[i].y = q8[2 * i + 1];
  }
  if (parea(a, 4) < 0) {
    P2 t = a[0];
    a[0] = a[3];
    a[3] = t;
    t = a[1];
    a[1] = a[2];
    a[2] = t;
  }
  if (parea(b, 4) < 0) {
    P2 t = b[0];
    b[0] = b[3];
    b[3] = t;
    t = b[1];
    b[1] = b[2];
    b[2] = t;
  }
  double inter = 0.0;
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) inter = padd(inter, tri_intersect(a[i], a[(i + 1) & 3], b[j], b[(j + 1) & 3]));
  const double uni = psub(padd(fabs(parea(a, 4)), fabs(parea(b, 4))), inter);
  return inter / uni;
}

__global__ void k_poly_keys(const double* __restrict__ dets9, long long n, unsigned long long* __restrict__ keys,
                            unsigned int* __restrict__ vals) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long u = (unsigned long long)__double_as_longlong(dets9[i * 9 + 8] + 0.0);
  u ^= (u >> 63) ? ~0ull : 0x8000000000000000ull;  // ascending on unsigned compare
  keys[i] = ~u;                                      // descending score
  vals[i] = (unsigned int)i;
}

__global__ void k_poly_pair_iou(const double* __restrict__ p8, const double* __restrict__ q8, double* __restrict__ out,
                                long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = iou_poly_dev(p8 + 8 * i, q8 + 8 * i);
}

// ResultMerge_multi_process.py:64-70: the axis-aligned hull of a polygon row and its area with the +1 pixel convention
__device__ __forceinline__ void poly_hbb(const double* d, double& x1, double& y1, double& x2, double& y2, double& area) {
  x1 = d[0], x2 = d[0], y1 = d[1], y2 = d[1];
  for (int k = 1; k < 4; ++k) {
    x1 = fmin(x1, d[2 * k]);
    x2 = fmax(x2, d[2 * k]);
    y1 = fmin(y1, d[2 * k + 1]);
    y2 = fmax(y2, d[2 * k + 1]);
  }
  area = pmul(padd(psub(x2, x1), 1.0), padd(psub(y2, y1), 1.0));
}

// ResultMerge_multi_process.py:88-115 for one pair: "j is suppressed by i".  The intersection of the hulls has no +1, the
// polygon IoU runs only where the hulls overlap, and a NaN overlap suppresses (the reference keeps `ovr <= thresh`).
__device__ __forceinline__ bool poly_suppresses(const double* di, double ix1, double iy1, double ix2, double iy2, double ai,
                                                const double* dj, double thresh) {
  double jx1, jy1, jx2, jy2, aj;
  poly_hbb(dj, jx1, jy1, jx2, jy2, aj);
  const double ww = fmax(0.0, psub(fmin(ix2, jx2), fmax(ix1, jx1)));
  const double hh = fmax(0.0, psub(fmin(iy2, jy2), fmax(iy1, jy1)));
  const double hb = pmul(ww, hh);
  double ovr = hb / psub(padd(ai, aj), hb);
  if (ovr > 0) ovr = iou_poly_dev(di, dj);
  return !(ovr <= thresh);
}

// one thread per (row i, 64-column word): bit c = candidate (w * 64 + c) of the sorted order is suppressed by i
__global__ void k_poly_mask(const double* __restrict__ dets9, const unsigned int* __restrict__ order, long long n, double thresh,
                            unsigned long long* __restrict__ mask) {
  const long long words = (n + 63) / 64;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n * words) return;
  const long long i = t / words, w = t - i * words;
  unsigned long long bits = 0ull;
  if ((w + 1) * 64 > i + 1) {
    const double* di = dets9 + (long long)order[i] * 9;
    double ix1, iy1, ix2, iy2, ai;
    poly_hbb(di, ix1, iy1, ix2, iy2, ai);
    for (int c = 0; c < 64; ++c) {
      const long long j = w * 64 + c;
      if (j <= i || j >= n) continue;
      if (poly_suppresses(di, ix1, iy1, ix2, iy2, ai, dets9 + (long long)order[j] * 9, thresh)) bits |= 1ull << c;
    }
  }
  mask[i * words + w] = bits;
}

__global__ void k_poly_reduce(const unsigned long long* __restrict__ mask, const unsigned int* __restrict__ order, long long n,
                              long long* __restrict__ keep, long long* __restrict__ n_keep) {
  extern __shared__ unsigned long long remv[];
  const long long words = (n + 63) / 64;
  for (long long w = threadIdx.x; w < words; w += blockDim.x) remv[w] = 0ull;
  __syncthreads();
  __shared__ long long s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  for (long long i = 0; i < n; ++i) {
    const bool alive = !((remv[i >> 6] >> (i & 63)) & 1ull);  // uniform: every thread reads the same word
    if (alive) {
      if (threadIdx.x == 0) keep[s_cnt++] = (long long)order[i];
      for (long long w = (i >> 6) + threadIdx.x; w < words; w += blockDim.x) remv[w] |= mask[i * words + w];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *n_keep = s_cnt;
}

// ---- whole-scene merge: ResultMerge_multi_process.py:175-236 (poly2origpoly + mergesingle) for every (scene, class) at once ----
// k_tiles_to_scene: tile detections [T, max_det, 7] -> scene-space rows dets9 + segment id (scene * nc + class), compacted by a
// one-CTA prefix sum over the tile counts.  Then y5obb_poly_nms_segmented_f64 runs py_cpu_nms_poly_fast independently on every
// segment: stable radix sort by descending score, stable radix sort by segment (so each segment is contiguous and in score
// order, ties -> lower index), segment extents, the upper triangle of each segment's 64-wide suppression-bit blocks only
// (sum of n_s^2 / 128 words instead of n^2 / 64), one CTA per segment for the greedy scan, and a compaction of the kept rows.
constexpr int SCAN_THREADS = 256;

// exclusive prefix sum of get(0..n) by ONE CTA of SCAN_THREADS threads: out[i] = sum of get(0..i), out[n] = total
template <typename Get>
__device__ void cta_exclusive_scan(long long n, Get get, long long* out) {
  typedef cub::BlockScan<long long, SCAN_THREADS> Scan;
  __shared__ typename Scan::TempStorage tmp;
  __shared__ long long carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (long long base = 0; base < n; base += SCAN_THREADS) {
    const long long i = base + threadIdx.x;
    long long v = i < n ? get(i) : 0, agg;
    Scan(tmp).ExclusiveSum(v, v, agg);
    if (i < n) out[i] = carry + v;
    __syncthreads();
    if (threadIdx.x == 0) carry += agg;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = carry;
}

// Upper-triangle mask layout of one segment of m rows, w = ceil(m / 64) words per full row: row i stores words
// [i / 64, w) only, so row block k (rows 64k .. 64k + 63) holds 64 * (w - k) words.  tri_row_off(i) = first word of row i;
// tri_row_off(m) = words of the whole segment.
__host__ __device__ __forceinline__ long long tri_row_off(long long i, long long w) {
  const long long bi = i >> 6;
  return 64 * (bi * w - bi * (bi - 1) / 2) + (i - 64 * bi) * (w - bi);
}
__host__ __device__ __forceinline__ long long tri_words(long long m) { return tri_row_off(m, (m + 63) >> 6); }

__device__ __forceinline__ long long tile_rows(const long long* counts, const int* scene_of, int t, int max_det) {
  return scene_of[t] < 0 ? 0 : min((long long)max_det, max(0ll, counts[t]));
}

__global__ void __launch_bounds__(SCAN_THREADS) k_tile_offsets(const long long* __restrict__ counts, const int* __restrict__ scene_of,
                                                              int n_tiles, int max_det, long long* __restrict__ off,
                                                              long long* __restrict__ n_out) {
  cta_exclusive_scan(n_tiles, [&](long long t) { return tile_rows(counts, scene_of, (int)t, max_det); }, off);
  __syncthreads();
  if (threadIdx.x == 0) *n_out = off[n_tiles];
}

// one thread per (tile, row slot): rbox2poly in fp32 (rboxs_utils.py:106-126), widened to double and moved by the tile origin
// (poly2origpoly at rate 1: (x + left) / 1.0), score widened to double
__global__ void k_tiles_to_scene(const float* __restrict__ det7, const long long* __restrict__ counts,
                                 const int* __restrict__ origins, const int* __restrict__ scene_of, int n_tiles, int max_det,
                                 int nc, const long long* __restrict__ off, double* __restrict__ dets9, int* __restrict__ seg,
                                 unsigned long long* __restrict__ hist, long long n_hist) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n_tiles * max_det) return;
  const int t = (int)(idx / max_det), r = (int)(idx - (long long)t * max_det);
  if (r >= tile_rows(counts, scene_of, t, max_det)) return;
  const float* d = det7 + idx * 7;
  float p[8];
  rbox_to_poly(d[0], d[1], d[2], d[3], d[4], p);
  const double left = (double)origins[2 * t], up = (double)origins[2 * t + 1];
  const long long o = off[t] + r;
  double* q = dets9 + o * 9;
#pragma unroll
  for (int k = 0; k < 8; ++k) q[k] = padd((double)p[k], (k & 1) ? up : left);
  q[8] = (double)d[5];
  const int cls = min(nc - 1, max(0, (int)d[6]));
  const long long sg = (long long)scene_of[t] * nc + cls;
  seg[o] = (int)sg;
  if (sg < n_hist) atomicAdd(hist + sg, 1ull);
}

__global__ void k_seg_of_sorted(const int* __restrict__ seg, const unsigned int* __restrict__ order, long long n,
                                unsigned int* __restrict__ out) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < n) out[p] = (unsigned int)seg[order[p]];
}

// segment s occupies sorted positions [begin[s], end[s]) (both pre-zeroed: an empty segment stays [0, 0))
__global__ void k_seg_extents(const unsigned int* __restrict__ sseg, long long n, long long n_seg, long long* __restrict__ begin,
                              long long* __restrict__ end) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n || sseg[p] >= n_seg) return;  // (an id outside [0, n_segments) belongs to no segment)
  if (p == 0 || sseg[p] != sseg[p - 1]) begin[sseg[p]] = p;
  if (p == n - 1 || sseg[p] != sseg[p + 1]) end[sseg[p]] = p + 1;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_seg_mask_offsets(const long long* __restrict__ begin,
                                                                  const long long* __restrict__ end, long long n_seg,
                                                                  long long* __restrict__ mask_off) {
  cta_exclusive_scan(n_seg, [&](long long s) { return tri_words(end[s] - begin[s]); }, mask_off);
}

// one thread per stored mask word (segment s, row i, word w >= i / 64): the pair predicate of k_poly_mask within segment s
__global__ void k_seg_mask(const double* __restrict__ dets9, const unsigned int* __restrict__ order,
                           const long long* __restrict__ begin, const long long* __restrict__ end,
                           const long long* __restrict__ mask_off, long long n_seg, long long cap_words, double thresh,
                           unsigned long long* __restrict__ mask) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= min(mask_off[n_seg], cap_words)) return;
  long long lo = 0, hi = n_seg - 1;  // the last segment s with mask_off[s] <= t (empty segments share their offset)
  while (lo < hi) {
    const long long mid = (lo + hi + 1) >> 1;
    if (mask_off[mid] <= t) lo = mid; else hi = mid - 1;
  }
  const long long s = lo, p0 = begin[s], m = end[s] - begin[s], w = (m + 63) >> 6, u = t - mask_off[s];
  long long blo = 0, bhi = w - 1;  // row block: the last k with 64 * (k * w - k (k - 1) / 2) <= u
  while (blo < bhi) {
    const long long mid = (blo + bhi + 1) >> 1;
    if (tri_row_off(mid * 64, w) <= u) blo = mid; else bhi = mid - 1;
  }
  const long long bi = blo, v = u - tri_row_off(bi * 64, w), rw = w - bi;
  const long long i = bi * 64 + v / rw, wd = bi + v % rw;
  unsigned long long bits = 0ull;
  if (i < m) {
    const double* di = dets9 + (long long)order[p0 + i] * 9;
    double ix1, iy1, ix2, iy2, ai;
    poly_hbb(di, ix1, iy1, ix2, iy2, ai);
    for (int c = 0; c < 64; ++c) {
      const long long j = wd * 64 + c;
      if (j <= i || j >= m) continue;
      if (poly_suppresses(di, ix1, iy1, ix2, iy2, ai, dets9 + (long long)order[p0 + j] * 9, thresh)) bits |= 1ull << c;
    }
  }
  mask[t] = bits;
}

// one CTA per segment: the greedy scan of k_poly_reduce over the segment's triangular mask rows
__global__ void k_seg_reduce(const unsigned long long* __restrict__ mask, const unsigned int* __restrict__ order,
                             const long long* __restrict__ begin, const long long* __restrict__ end,
                             const long long* __restrict__ mask_off, long long cap_words, long long* __restrict__ keep_tmp,
                             long long* __restrict__ seg_kept) {
  extern __shared__ unsigned long long remv[];
  const long long s = blockIdx.x, p0 = begin[s], m = end[s] - begin[s], w = (m + 63) >> 6;
  __shared__ long long s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  if (m == 0 || mask_off[s] + tri_words(m) > cap_words) {
    if (threadIdx.x == 0) seg_kept[s] = 0;
    return;
  }
  const unsigned long long* mk = mask + mask_off[s];
  for (long long wd = threadIdx.x; wd < w; wd += blockDim.x) remv[wd] = 0ull;
  __syncthreads();
  for (long long i = 0; i < m; ++i) {
    const bool alive = !((remv[i >> 6] >> (i & 63)) & 1ull);  // uniform: every thread reads the same word
    if (alive) {
      if (threadIdx.x == 0) keep_tmp[p0 + s_cnt++] = (long long)order[p0 + i];
      const long long bi = i >> 6;
      const unsigned long long* row = mk + tri_row_off(i, w) - bi;
      for (long long wd = bi + threadIdx.x; wd < w; wd += blockDim.x) remv[wd] |= row[wd];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) seg_kept[s] = s_cnt;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_seg_keep_offsets(const long long* __restrict__ seg_kept, long long n_seg,
                                                                  long long* __restrict__ seg_offsets) {
  cta_exclusive_scan(n_seg, [&](long long s) { return seg_kept[s]; }, seg_offsets);
}

__global__ void k_seg_compact(const long long* __restrict__ keep_tmp, const unsigned int* __restrict__ sseg,
                              const long long* __restrict__ begin, const long long* __restrict__ seg_kept,
                              const long long* __restrict__ seg_offsets, long long n, long long n_seg,
                              long long* __restrict__ keep) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n || sseg[p] >= n_seg) return;
  const unsigned int s = sseg[p];
  const long long k = p - begin[s];
  if (k < seg_kept[s]) keep[seg_offsets[s] + k] = keep_tmp[p];
}

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

size_t y5obb_poly_nms_workspace_bytes(int64_t n) {
  if (n <= 0) return 256;
  size_t cub_bytes = 0;
  if (cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                      (const unsigned int*)nullptr, (unsigned int*)nullptr, (int)n) != cudaSuccess) {
    (void)cudaGetLastError();
    cub_bytes = (size_t)(32u << 20) + (size_t)n * 16;
  }
  const size_t words = (size_t)((n + 63) / 64);
  return 4096 + cub_bytes + (size_t)n * (8 + 8 + 4 + 4) + (size_t)n * words * 8;
}

int y5obb_poly_iou_pairs_f64(const double* p8, const double* q8, double* iou_out, int64_t n, void* stream) {
  if (n < 0) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!p8 || !q8 || !iou_out) return Y5OBB_EINVAL;
  k_poly_pair_iou<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(p8, q8, iou_out, n);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_poly_nms_f64(const double* dets9, int64_t n, double thresh, int64_t* keep_out, int64_t* n_keep_out, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (n < 0 || !keep_out || !n_keep_out) return Y5OBB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    Y5_CUDA(cudaMemsetAsync(n_keep_out, 0, sizeof(int64_t), st));
    return Y5OBB_OK;
  }
  if (!dets9 || !workspace || n > 200000) return Y5OBB_EINVAL;  // the dense bit matrix is n^2 / 8 bytes
  if (y5obb_poly_nms_workspace_bytes(n) > workspace_bytes) return Y5OBB_EWORKSPACE;
  const size_t words = (size_t)((n + 63) / 64);
  if (words * 8 > 200 * 1024) return Y5OBB_EINVAL;
  Carver c(workspace);
  unsigned long long* keys_a = c.take<unsigned long long>(n);
  unsigned long long* keys_b = c.take<unsigned long long>(n);
  unsigned int* vals_a = c.take<unsigned int>(n);
  unsigned int* vals_b = c.take<unsigned int>(n);
  unsigned long long* mask = c.take<unsigned long long>((size_t)n * words);
  size_t cub_bytes = workspace_bytes - c.used();
  void* cub_tmp = c.take<char>(1);
  k_poly_keys<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dets9, n, keys_a, vals_a);
  Y5_LAUNCH_CHECK();
  Y5_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, keys_a, keys_b, vals_a, vals_b, (int)n, 0, 64, st));
  const long long total = (long long)n * (long long)words;
  k_poly_mask<<<(unsigned)((total + 127) / 128), 128, 0, st>>>(dets9, vals_b, n, thresh, mask);
  Y5_LAUNCH_CHECK();
  static bool attr = false;
  if (!attr) {
    Y5_CUDA(cudaFuncSetAttribute(k_poly_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr = true;
  }
  k_poly_reduce<<<1, 1024, words * 8, st>>>(mask, vals_b, n, reinterpret_cast<long long*>(keep_out),
                                            reinterpret_cast<long long*>(n_keep_out));
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

size_t y5obb_tiles_to_scene_workspace_bytes(int n_tiles) { return 4096 + (size_t)(n_tiles + 1) * 8; }

int y5obb_tiles_to_scene_f64(const float* det7, const int64_t* counts, int n_tiles, int max_det, const int32_t* origins2,
                             const int32_t* scene_of, int n_scenes, int nc, double* dets9_out, int32_t* seg_out,
                             int64_t* n_out, int64_t* seg_hist_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (n_tiles <= 0 || max_det <= 0 || n_scenes <= 0 || nc <= 0 || (long long)n_scenes * nc > 0x7FFFFFFFll) return Y5OBB_EINVAL;
  if (!det7 || !counts || !origins2 || !scene_of || !dets9_out || !seg_out || !n_out || !seg_hist_out || !workspace)
    return Y5OBB_EINVAL;
  if (y5obb_tiles_to_scene_workspace_bytes(n_tiles) > workspace_bytes) return Y5OBB_EWORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  long long* off = static_cast<long long*>(workspace);
  const long long n_hist = (long long)n_scenes * nc;
  Y5_CUDA(cudaMemsetAsync(seg_hist_out, 0, (size_t)n_hist * 8, st));
  k_tile_offsets<<<1, SCAN_THREADS, 0, st>>>(reinterpret_cast<const long long*>(counts), scene_of, n_tiles, max_det, off,
                                              reinterpret_cast<long long*>(n_out));
  Y5_LAUNCH_CHECK();
  const long long slots = (long long)n_tiles * max_det;
  k_tiles_to_scene<<<(unsigned)((slots + 255) / 256), 256, 0, st>>>(det7, reinterpret_cast<const long long*>(counts), origins2,
                                                                     scene_of, n_tiles, max_det, nc, off, dets9_out, seg_out,
                                                                     reinterpret_cast<unsigned long long*>(seg_hist_out), n_hist);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

// the greedy scan keeps one mask row of its segment in shared memory, as y5obb_poly_nms_f64 does for the whole list
static constexpr size_t SEG_SMEM_MAX = 200 * 1024;

static int seg_sizes(const int64_t* seg_counts_host, int64_t n_seg, long long& n, long long& words, long long& max_w) {
  if (n_seg <= 0 || n_seg > 0x7FFFFFFFll || !seg_counts_host) return Y5OBB_EINVAL;
  n = 0, words = 0, max_w = 0;
  for (int64_t s = 0; s < n_seg; ++s) {
    const long long m = seg_counts_host[s];
    if (m < 0) return Y5OBB_EINVAL;
    n += m;
    words += tri_words(m);
    max_w = std::max(max_w, (m + 63) / 64);
  }
  if (n > 0x7FFFFFFFll || (size_t)max_w * 8 > SEG_SMEM_MAX) return Y5OBB_EINVAL;
  return Y5OBB_OK;
}

static size_t seg_cub_bytes(long long n) {
  size_t a = 0, b = 0;
  if (cub::DeviceRadixSort::SortPairs(nullptr, a, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                      (const unsigned int*)nullptr, (unsigned int*)nullptr, (int)n) != cudaSuccess ||
      cub::DeviceRadixSort::SortPairs(nullptr, b, (const unsigned int*)nullptr, (unsigned int*)nullptr,
                                      (const unsigned int*)nullptr, (unsigned int*)nullptr, (int)n) != cudaSuccess) {
    (void)cudaGetLastError();
    return (size_t)(32u << 20) + (size_t)n * 16;
  }
  return std::max(a, b);
}

size_t y5obb_poly_nms_segmented_workspace_bytes(const int64_t* seg_counts_host, int64_t n_segments) {
  long long n, words, max_w;
  if (seg_sizes(seg_counts_host, n_segments, n, words, max_w) != Y5OBB_OK) return 0;
  const size_t nn = (size_t)std::max(n, 1ll), ns = (size_t)n_segments + 1;
  return 8192 + seg_cub_bytes(std::max(n, 1ll)) + nn * (8 + 8 + 4 + 4 + 4 + 4 + 8) + ns * 8 * 4 + (size_t)words * 8;
}

int y5obb_poly_nms_segmented_f64(const double* dets9, const int32_t* seg_id, int64_t n, const int64_t* seg_counts_host,
                                 int64_t n_segments, double thresh, int64_t* keep_out, int64_t* seg_offsets_out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  long long n_chk, words, max_w;
  if (seg_sizes(seg_counts_host, n_segments, n_chk, words, max_w) != Y5OBB_OK || n != n_chk || !seg_offsets_out)
    return Y5OBB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    Y5_CUDA(cudaMemsetAsync(seg_offsets_out, 0, (size_t)(n_segments + 1) * 8, st));
    return Y5OBB_OK;
  }
  if (!dets9 || !seg_id || !keep_out || !workspace) return Y5OBB_EINVAL;
  if (y5obb_poly_nms_segmented_workspace_bytes(seg_counts_host, n_segments) > workspace_bytes) return Y5OBB_EWORKSPACE;
  int seg_bits = 1;
  while (seg_bits < 32 && (1ll << seg_bits) < n_segments) ++seg_bits;
  Carver c(workspace);
  unsigned long long* keys_a = c.take<unsigned long long>(n);
  unsigned long long* keys_b = c.take<unsigned long long>(n);
  unsigned int* vals_a = c.take<unsigned int>(n);
  unsigned int* vals_b = c.take<unsigned int>(n);
  unsigned int* sseg_a = c.take<unsigned int>(n);
  unsigned int* sseg_b = c.take<unsigned int>(n);
  long long* keep_tmp = c.take<long long>(n);
  long long* begin = c.take<long long>(n_segments + 1);
  long long* end = c.take<long long>(n_segments + 1);
  long long* mask_off = c.take<long long>(n_segments + 1);
  long long* seg_kept = c.take<long long>(n_segments + 1);
  unsigned long long* mask = c.take<unsigned long long>((size_t)std::max(words, 1ll));
  size_t cub_bytes = workspace_bytes - c.used();
  void* cub_tmp = c.take<char>(1);
  const unsigned nb = (unsigned)((n + 255) / 256);
  // descending score, ties -> lower index; then by segment, stable, so every segment is contiguous in that order
  k_poly_keys<<<nb, 256, 0, st>>>(dets9, n, keys_a, vals_a);
  Y5_LAUNCH_CHECK();
  Y5_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, keys_a, keys_b, vals_a, vals_b, (int)n, 0, 64, st));
  k_seg_of_sorted<<<nb, 256, 0, st>>>(seg_id, vals_b, n, sseg_a);
  Y5_LAUNCH_CHECK();
  Y5_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cub_bytes, sseg_a, sseg_b, vals_b, vals_a, (int)n, 0, seg_bits, st));
  Y5_CUDA(cudaMemsetAsync(begin, 0, (size_t)n_segments * 8, st));
  Y5_CUDA(cudaMemsetAsync(end, 0, (size_t)n_segments * 8, st));
  k_seg_extents<<<nb, 256, 0, st>>>(sseg_b, n, n_segments, begin, end);
  Y5_LAUNCH_CHECK();
  k_seg_mask_offsets<<<1, SCAN_THREADS, 0, st>>>(begin, end, n_segments, mask_off);
  Y5_LAUNCH_CHECK();
  if (words > 0) {
    k_seg_mask<<<(unsigned)((words + 127) / 128), 128, 0, st>>>(dets9, vals_a, begin, end, mask_off, n_segments, words, thresh,
                                                                 mask);
    Y5_LAUNCH_CHECK();
  }
  static bool attr = false;
  if (!attr) {
    Y5_CUDA(cudaFuncSetAttribute(k_seg_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SEG_SMEM_MAX));
    attr = true;
  }
  k_seg_reduce<<<(unsigned)n_segments, 256, (size_t)max_w * 8, st>>>(mask, vals_a, begin, end, mask_off, words, keep_tmp,
                                                                      seg_kept);
  Y5_LAUNCH_CHECK();
  k_seg_keep_offsets<<<1, SCAN_THREADS, 0, st>>>(seg_kept, n_segments, reinterpret_cast<long long*>(seg_offsets_out));
  Y5_LAUNCH_CHECK();
  k_seg_compact<<<nb, 256, 0, st>>>(keep_tmp, sseg_b, begin, seg_kept, reinterpret_cast<const long long*>(seg_offsets_out), n,
                                    n_segments, reinterpret_cast<long long*>(keep_out));
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

}  // extern "C"
