// Device-resident rotated NMS for sm_100a.
//
// Replaces the reference's sort -> 64x64 IoU bit-matrix -> N^2/8-byte D2H -> serial host scan
// (/root/reference/utils/nms_rotated/src/nms_rotated_cuda.cu:71-134) with five launches that never
// leave the GPU:
//   k_make_keys   64-bit key = (image << 32) | ~orderable(score); value = input index
//   cub radix     one stable sort orders every image's boxes by descending score (ties: lower index)
//   k_segments / k_plan   per-image extents, work-unit and mask offsets (device side, no sync)
//   k_prep        per-box trig/area/circumradius once (the reference recomputes them per pair)
//   k_tiles       persistent CTAs pull (row block, 8 col blocks) units of the UPPER triangle only;
//                 phase 1 = exact far-pair reject into a shared-memory candidate list,
//                 phase 2 = all lanes evaluate candidates with the bit-faithful IoU (rbox_iou.cuh),
//                 phase 3 = one 64-bit mask word per row
//   k_reduce      one CTA per image runs the greedy scan over the bit-matrix in shared memory and
//                 writes the compacted keep list in score order
// Algorithmic bytes per box: 24 in (5 floats + score) + 8 out per kept box; the bit-matrix is
// internal traffic (8 bytes per 64x64 tile row, upper triangle only).
#include <cooperative_groups.h>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "rbox_iou.cuh"

namespace y5obb {

thread_local int g_last_cuda_error = 0;

namespace {

constexpr int TB = 64;            // boxes per block == bits per mask word
constexpr int CHUNK = 8;          // col blocks per work unit
constexpr int TILE_THREADS = 128;
constexpr int REDUCE_THREADS = 1024;
constexpr int MAX_IMAGES = 1 << 20;

struct NmsSeg {
  int64_t unit_off;  // first work unit of this image
  int64_t mask_off;  // first mask word of this image
  int32_t off;       // first sorted position
  int32_t n;         // boxes in this image
  int32_t nblk;      // ceil(n / 64)
  int32_t pad;
};

struct NmsCtrl {
  unsigned long long next_unit;
  long long total_units;
  long long mask_capacity_words;
  int err;
  int pad;
};

__device__ __forceinline__ uint32_t orderable_desc(float s) {
  s = s + 0.0f;  // -0 -> +0
  uint32_t u = __float_as_uint(s);
  u ^= (u >> 31) ? 0xFFFFFFFFu : 0x80000000u;  // ascending order on unsigned compare
  return ~u;                                     // descending
}

// units of an image with nb blocks, rows ordered by m = nb - rb (m = 1 .. nb): row with m blocks of
// columns has ceil(m / CHUNK) units.
__host__ __device__ inline long long units_for(long long nb) {
  long long q = nb / CHUNK, r = nb % CHUNK;
  return (CHUNK / 2) * q * (q + 1) + (q + 1) * r;
}

__global__ void k_make_keys(const float* __restrict__ dets, const float* __restrict__ scores,
                            const int32_t* __restrict__ image_ids, int64_t n, int n_images, int flags,
                            const int64_t* __restrict__ n_valid_dev, uint64_t* __restrict__ keys,
                            uint32_t* __restrict__ vals) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (n_valid_dev && i >= *n_valid_dev) {  // tail of an over-allocated candidate list
    keys[i] = ((uint64_t)(uint32_t)n_images << 32) | 0xFFFFFFFFull;
    vals[i] = (uint32_t)i;
    return;
  }
  int img = image_ids ? image_ids[i] : 0;
  if (img < 0 || img >= n_images) img = n_images;  // dump segment
  if (flags & Y5OBB_NMS_DROP_SMALL) {
    float w = dets[5 * i + 2], h = dets[5 * i + 3];
    if (fminf(w, h) < 0.001f) img = n_images;
  }
  keys[i] = ((uint64_t)(uint32_t)img << 32) | orderable_desc(scores[i]);
  vals[i] = (uint32_t)i;
}

// seg_start[b] = first sorted position whose image id is >= b, for b in [0, n_images]
__global__ void k_segments(const uint64_t* __restrict__ keys, int64_t n, int n_images, int32_t* __restrict__ seg_start) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  int prev = (i == 0) ? -1 : (int)(keys[i - 1] >> 32);
  int cur = (i == n) ? n_images : (int)(keys[i] >> 32);
  for (int b = prev + 1; b <= cur; ++b) seg_start[b] = (int32_t)i;
}

__global__ void k_plan(const int32_t* __restrict__ seg_start, int n_images, long long mask_capacity_words,
                       int per_image_clamp, NmsSeg* __restrict__ seg, NmsCtrl* ctrl) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  long long units = 0, words = 0;
  for (int b = 0; b < n_images; ++b) {
    NmsSeg s;
    s.off = seg_start[b];
    s.n = seg_start[b + 1] - seg_start[b];
    if (per_image_clamp > 0 && s.n > per_image_clamp) s.n = per_image_clamp;  // top-k by score (max_nms)
    s.nblk = (s.n + TB - 1) / TB;
    s.unit_off = units;
    s.mask_off = words;
    s.pad = 0;
    units += units_for(s.nblk);
    words += (long long)s.n * s.nblk;
    seg[b] = s;
  }
  NmsSeg tail;
  tail.off = seg_start[n_images];
  tail.n = 0;
  tail.nblk = 0;
  tail.unit_off = units;
  tail.mask_off = words;
  tail.pad = 0;
  seg[n_images] = tail;
  ctrl->next_unit = 0;
  ctrl->mask_capacity_words = mask_capacity_words;
  if (words > mask_capacity_words) {
    ctrl->err = 1;  // max_per_image was exceeded: refuse rather than overrun the workspace
    ctrl->total_units = 0;
  } else {
    ctrl->err = 0;
    ctrl->total_units = units;
  }
}

__global__ void k_prep(const float* __restrict__ dets, const uint32_t* __restrict__ order, int64_t n,
                       PreBox* __restrict__ pre) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* d = dets + 5 * (int64_t)order[i];
  pre[i] = make_prebox(d[0], d[1], d[2], d[3], d[4]);
}

__device__ __forceinline__ void load_prebox(PreBox* dst, const PreBox* src) {
  const float4* s = reinterpret_cast<const float4*>(src);
  float4* d = reinterpret_cast<float4*>(dst);
  d[0] = s[0];
  d[1] = s[1];
}

// Conservative separating-axis test: true only if the rectangles are apart by more than 1e-3 of their size on one of
// the four edge normals (then the reference finds no intersection point and no contained vertex: IoU == 0).
__device__ __forceinline__ bool sat_separated(const PreBox& A, const PreBox& B) {
  const float dx = B.cx - A.cx, dy = B.cy - A.cy;
  // unit axes of A: u = (cos, -sin) along w, v = (-sin, -cos) along h (box_corners); c2/s2 hold cos/2, sin/2
  const float ac = 2.f * A.c2, as = 2.f * A.s2, bc = 2.f * B.c2, bs = 2.f * B.s2;
  const float ahw = 0.5f * A.w, ahh = 0.5f * A.h, bhw = 0.5f * B.w, bhh = 0.5f * B.h;
  const float cab = fabsf(ac * bc + as * bs);   // |uA.uB| = |vA.vB|
  const float sab = fabsf(ac * bs - as * bc);   // |uA.vB| = |vA.uB|
  const float m = 1e-3f * (ahw + ahh + bhw + bhh) + 1e-3f;
  if (fabsf(dx * ac - dy * as) > ahw + bhw * cab + bhh * sab + m) return true;   // axis uA
  if (fabsf(-dx * as - dy * ac) > ahh + bhw * sab + bhh * cab + m) return true;  // axis vA
  if (fabsf(dx * bc - dy * bs) > bhw + ahw * cab + ahh * sab + m) return true;   // axis uB
  if (fabsf(-dx * bs - dy * bc) > bhh + ahw * sab + ahh * cab + m) return true;  // axis vB
  return false;
}

// Exact upper bound of the IoU from the axis-aligned bounding boxes: intersection <= min(AABB overlap, smaller area), and
// x / (aA + aB - x) grows with x.  True when that bound is below thr_lo (= 0.999 thr: three orders of magnitude above the
// reference's own rounding), i.e. the pair cannot suppress.  Extents are inflated like the circumradius.
__device__ __forceinline__ bool aabb_bound_below(const PreBox& A, const PreBox& B, float thr_lo) {
  const float ax = (fabsf(A.w * A.c2) + fabsf(A.h * A.s2)) * 1.001f + 1e-3f, ay = (fabsf(A.w * A.s2) + fabsf(A.h * A.c2)) * 1.001f + 1e-3f;
  const float bx = (fabsf(B.w * B.c2) + fabsf(B.h * B.s2)) * 1.001f + 1e-3f, by = (fabsf(B.w * B.s2) + fabsf(B.h * B.c2)) * 1.001f + 1e-3f;
  const float ix = fminf(A.cx + ax, B.cx + bx) - fmaxf(A.cx - ax, B.cx - bx);
  const float iy = fminf(A.cy + ay, B.cy + by) - fmaxf(A.cy - ay, B.cy - by);
  if (ix <= 0.f || iy <= 0.f) return true;  // disjoint bounding boxes: IoU == 0
  if (!(A.area >= 0.f) || !(B.area >= 0.f)) return false;
  const float inter = fminf(ix * iy * 1.003f, fminf(A.area, B.area));
  return inter < thr_lo * (A.area + B.area - inter);
}

constexpr int CAND_CAP = 8192;  // candidate pairs buffered per work unit before the IoU phase runs

__global__ void __launch_bounds__(TILE_THREADS)
k_tiles(const PreBox* __restrict__ pre, const NmsSeg* __restrict__ seg, int n_images, NmsCtrl* ctrl,
        unsigned long long* __restrict__ mask, uint8_t* __restrict__ rowflag, float thr, int strict) {
  __shared__ __align__(16) PreBox s_row[TB];
  __shared__ __align__(16) PreBox s_col[TB];
  __shared__ float4 s_colq[TB];  // (cx, cy, rad, area) of the column boxes: what the far-pair test reads
  __shared__ unsigned long long s_mask[TB * CHUNK];  // [row][col block of the unit]
  __shared__ unsigned short s_cand[CAND_CAP];        // row (6 bits) | col block in unit (3) | col (6)
  __shared__ int s_ncand;
  __shared__ long long s_unit;

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const long long total = ctrl->total_units;
  // decision-exact shortcuts need a margin against the ~1e-6 relative error of the reference's own arithmetic;
  // they are only taken for ordinary thresholds
  const float thr_lo = thr >= 0.01f ? thr * 0.999f : -1.0f;

  for (;;) {
    if (tid == 0) s_unit = (long long)atomicAdd(&ctrl->next_unit, 1ull);
    __syncthreads();
    const long long u = s_unit;
    if (u >= total) break;

    // image lookup: last b with unit_off <= u
    int lo = 0, hi = n_images - 1;
    while (lo < hi) {
      int mid = (lo + hi + 1) >> 1;
      if (seg[mid].unit_off <= u) lo = mid; else hi = mid - 1;
    }
    const NmsSeg S = seg[lo];
    const long long lu = u - S.unit_off;
    // decode lu -> (m, k): groups of CHUNK consecutive m share the chunk count q + 1
    long long q = (long long)((sqrt(1.0 + 8.0 * (double)lu / CHUNK) - 1.0) * 0.5);
    if (q < 0) q = 0;
    while ((CHUNK / 2) * (q + 1) * (q + 2) <= lu) ++q;
    while (q > 0 && (CHUNK / 2) * q * (q + 1) > lu) --q;
    const long long rem = lu - (CHUNK / 2) * q * (q + 1);
    const int m = (int)(CHUNK * q + 1 + rem / (q + 1));
    const int k = (int)(rem % (q + 1));
    const int rb = S.nblk - m;
    const int cb0 = rb + CHUNK * k;
    const int cb1 = min(cb0 + CHUNK, S.nblk);
    const int nrow = min(TB, S.n - rb * TB);

    if (tid < nrow) load_prebox(&s_row[tid], &pre[S.off + rb * TB + tid]);
    for (int i = tid; i < TB * CHUNK; i += TILE_THREADS) s_mask[i] = 0ull;
    if (tid == 0) s_ncand = 0;

    // phase 2 (all lanes busy): evaluate the buffered candidates with the bit-faithful IoU
    auto drain = [&]() {
      __syncthreads();
      const int nc = s_ncand;
      for (int c = tid; c < nc; c += TILE_THREADS) {
        const int pr = s_cand[c];
        const int r = pr >> 9, cbl = (pr >> 6) & 7, j = pr & 63;
        PreBox cbx;
        load_prebox(&cbx, &pre[S.off + (cb0 + cbl) * TB + j]);
        if (thr_lo > 0.f && aabb_bound_below(s_row[r], cbx, thr_lo)) continue;  // IoU <= bound < thr (57 % of the candidates of a DOTA-like step)
        if (thr_lo > 0.f && sat_separated(s_row[r], cbx)) continue;              // disjoint rectangles: IoU == 0 < thr
        const float v = rbox_iou(s_row[r], cbx);
        const bool sup = strict ? (v > thr) : (v >= thr);
        if (sup) atomicOr(&s_mask[r * CHUNK + cbl], 1ull << j);
      }
      __syncthreads();
      if (tid == 0) s_ncand = 0;
    };

    for (int cb = cb0; cb < cb1; ++cb) {
      const int ncol = min(TB, S.n - cb * TB);
      __syncthreads();  // s_col free (previous phase 1 done), s_row / s_ncand visible
      if (tid >= TB) {
        const int j = tid - TB;
        if (j < ncol) {
          load_prebox(&s_col[j], &pre[S.off + cb * TB + j]);
          s_colq[j] = make_float4(s_col[j].cx, s_col[j].cy, s_col[j].rad, s_col[j].area);
        } else {
          s_colq[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      __syncthreads();
      {  // phase 1: exact reject of pairs whose circumscribed circles do not touch; four columns per step (one 16-byte
         // shared-memory load each, one vote for the four: most steps find nothing)
        const int r = tid & (TB - 1);
        const int half = tid >> 6;
        const bool rvalid = r < nrow;
        const float rx = s_row[r].cx, ry = s_row[r].cy, rr = s_row[r].rad, ra = s_row[r].area;
        const int tag = (r << 9) | ((cb - cb0) << 6);
        const bool diag = cb == rb;  // on the diagonal block only j > r counts
#pragma unroll 2
        for (int jj = 0; jj < TB / 2; jj += 4) {
          const int j0 = half * (TB / 2) + jj;
          bool c[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            const float4 b = s_colq[j];  // cx, cy, rad, area
            const float dx = rx - b.x, dy = ry - b.y, R = rr + b.z;
            bool cc = rvalid && j < ncol && (!diag || j > r) && (dx * dx + dy * dy) <= R * R;
            // IoU <= min(area) / max(area): boxes of very different size can never reach the threshold
            if (ra >= 0.f && b.w >= 0.f && fminf(ra, b.w) < thr_lo * fmaxf(ra, b.w)) cc = false;
            c[q] = cc;
          }
          if (__ballot_sync(0xffffffffu, c[0] | c[1] | c[2] | c[3])) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const unsigned bal = __ballot_sync(0xffffffffu, c[q]);
              if (bal) {
                int base = 0;
                if (lane == 0) base = atomicAdd(&s_ncand, __popc(bal));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (c[q]) s_cand[base + __popc(bal & ((1u << lane) - 1u))] = (unsigned short)(tag | (j0 + q));
              }
            }
          }
        }
      }
      __syncthreads();
      if (s_ncand > CAND_CAP - TB * TB) drain();  // the next tile could add up to 4096 pairs
    }
    drain();

    // phase 3: the unit's mask words, contiguous along the column blocks of a row
    const int ncb = cb1 - cb0;
    for (int i = tid; i < nrow * ncb; i += TILE_THREADS) {
      const int r = i / ncb, cbl = i - r * ncb;
      const unsigned long long w = s_mask[r * CHUNK + cbl];
      mask[S.mask_off + (long long)(rb * TB + r) * S.nblk + cb0 + cbl] = w;
      if (w) rowflag[S.off + rb * TB + r] = 1;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(REDUCE_THREADS)
k_reduce(const NmsSeg* __restrict__ seg, const NmsCtrl* __restrict__ ctrl,
         const unsigned long long* __restrict__ mask, const uint8_t* __restrict__ rowflag,
         const uint32_t* __restrict__ order, long long max_keep, int n_images,
         int64_t* __restrict__ keep_out, int64_t* __restrict__ n_keep_out, int64_t* __restrict__ seg_off_out,
         const PreBox* __restrict__ pre, int late_drop_small) {
  extern __shared__ unsigned long long remv[];
  __shared__ unsigned long long s_diag[TB];
  __shared__ int s_orrows[TB];
  __shared__ int s_nor;
  __shared__ unsigned long long s_kept;

  const int tid = threadIdx.x;
  const int b = blockIdx.x;
  const NmsSeg S = seg[b];
  if (tid == 0) {
    seg_off_out[b] = S.off;
    if (b == 0) seg_off_out[n_images] = seg[n_images].off;
  }
  if (ctrl->err) {
    if (tid == 0) n_keep_out[b] = -1;
    return;
  }
  for (int w = tid; w < S.nblk; w += REDUCE_THREADS) remv[w] = 0ull;
  if (tid == 0) s_nor = 0;
  __syncthreads();
  if (late_drop_small) {
    // Reference order (general.py:845-846 then nms_rotated_wrapper.py:32-39): the top-max_nms clamp counts degenerate
    // boxes, obb_nms drops them afterwards.  They start out "removed": never kept, their mask rows never applied.
    for (int i = tid; i < S.n; i += REDUCE_THREADS) {
      const PreBox& q = pre[S.off + i];
      if (fminf(q.w, q.h) < 0.001f) atomicOr(&remv[i >> 6], 1ull << (i & 63));
    }
    __syncthreads();
  }

  long long count = 0;
  const unsigned long long* M = mask + S.mask_off;
  for (int blk = 0; blk < S.nblk; ++blk) {
    const int rows = min(TB, S.n - blk * TB);
    unsigned long long cur = remv[blk];
    if (rows < TB) cur |= ~0ull << rows;
    if (cur == ~0ull) continue;  // whole block already suppressed (uniform branch)

    if (tid < TB) s_diag[tid] = (tid < rows) ? M[(long long)(blk * TB + tid) * S.nblk + blk] : 0ull;
    __syncthreads();
    if (tid == 0) {
      unsigned long long kept = 0ull;
#pragma unroll
      for (int i = 0; i < TB; ++i) {
        const unsigned long long bit = 1ull << i;
        if (!(cur & bit)) {
          kept |= bit;
          cur |= s_diag[i];
        }
      }
      if (max_keep > 0) {
        long long room = max_keep - count;
        while ((long long)__popcll(kept) > room) kept &= ~(1ull << (63 - __clzll(kept)));
      }
      s_kept = kept;
    }
    __syncthreads();
    const unsigned long long kept = s_kept;
    if (tid < TB && ((kept >> tid) & 1ull)) {
      const long long pos = count + __popcll(kept & ((1ull << tid) - 1ull));
      const int srow = blk * TB + tid;
      keep_out[S.off + pos] = (int64_t)order[S.off + srow];
      if (rowflag[S.off + srow]) s_orrows[atomicAdd(&s_nor, 1)] = srow;
    }
    count += __popcll(kept);
    __syncthreads();
    const int nor = s_nor;
    if (nor) {
      for (int w = blk + 1 + tid; w < S.nblk; w += REDUCE_THREADS) {
        unsigned long long acc = 0ull;
        for (int r = 0; r < nor; ++r) acc |= M[(long long)s_orrows[r] * S.nblk + w];
        if (acc) remv[w] |= acc;
      }
    }
    __syncthreads();
    if (tid == 0) s_nor = 0;
    if (max_keep > 0 && count >= max_keep) break;
  }
  if (tid == 0) n_keep_out[b] = count;
}

// The same greedy scan by a CLUSTER of RC CTAs per image (large problems: the single CTA above spends its time pulling the
// kept rows' mask words - up to gigabytes at 200 k boxes - through one SM).  CTA `rank` owns the words w with w % RC == rank of
// the removed-set and resolves the 64-row blocks blk with blk % RC == rank: it publishes the block's kept bits in its shared
// memory, ONE cluster barrier later every CTA reads them through distributed shared memory and ORs the kept rows' mask words
// of ITS columns.  The word a block's owner needs next (remv[blk]) is its own, so one barrier per block suffices; a CTA's
// publication slot is rewritten RC blocks (>= 2 barriers) later.  Same keep list, same order as k_reduce.
constexpr int RC = 8;  // portable cluster size

__global__ void __launch_bounds__(REDUCE_THREADS)
k_reduce_cluster(const NmsSeg* __restrict__ seg, const NmsCtrl* __restrict__ ctrl, const unsigned long long* __restrict__ mask,
                 const uint8_t* __restrict__ rowflag, const uint32_t* __restrict__ order, long long max_keep, int n_images,
                 int64_t* __restrict__ keep_out, int64_t* __restrict__ n_keep_out, int64_t* __restrict__ seg_off_out,
                 const PreBox* __restrict__ pre, int late_drop_small) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  extern __shared__ unsigned long long remv[];  // this CTA's words: remv[w / RC] for w % RC == rank
  __shared__ unsigned long long s_diag[TB];
  __shared__ unsigned long long s_pub;          // kept bits of the block this CTA resolved last
  __shared__ int s_orrows[TB];
  __shared__ int s_nor;

  const int tid = threadIdx.x;
  const int rank = (int)cluster.block_rank();
  const int b = blockIdx.x / RC;
  const NmsSeg S = seg[b];
  if (tid == 0 && rank == 0) {
    seg_off_out[b] = S.off;
    if (b == 0) seg_off_out[n_images] = seg[n_images].off;
  }
  if (ctrl->err) {  // uniform across the cluster: nobody reaches a barrier
    if (tid == 0 && rank == 0) n_keep_out[b] = -1;
    return;
  }
  const int my_words = (S.nblk - rank + RC - 1) / RC;
  for (int i = tid; i < my_words; i += REDUCE_THREADS) remv[i] = 0ull;
  if (tid == 0) s_nor = 0;
  __syncthreads();
  if (late_drop_small) {
    for (int i = tid; i < S.n; i += REDUCE_THREADS) {
      const int w = i >> 6;
      if (w % RC != rank) continue;
      const PreBox& q = pre[S.off + i];
      if (fminf(q.w, q.h) < 0.001f) atomicOr(&remv[w / RC], 1ull << (i & 63));
    }
    __syncthreads();
  }

  long long count = 0;
  const unsigned long long* M = mask + S.mask_off;
  for (int blk = 0; blk < S.nblk; ++blk) {
    const int owner = blk % RC;
    const int rows = min(TB, S.n - blk * TB);
    if (owner == rank) {  // resolve the diagonal chain of this block
      if (tid < TB) s_diag[tid] = (tid < rows) ? M[(long long)(blk * TB + tid) * S.nblk + blk] : 0ull;
      __syncthreads();
      if (tid == 0) {
        unsigned long long cur = remv[blk / RC], kept = 0ull;
        if (rows < TB) cur |= ~0ull << rows;
#pragma unroll
        for (int i = 0; i < TB; ++i) {
          const unsigned long long bit = 1ull << i;
          if (!(cur & bit)) {
            kept |= bit;
            cur |= s_diag[i];
          }
        }
        if (max_keep > 0) {
          long long room = max_keep - count;
          while ((long long)__popcll(kept) > room) kept &= ~(1ull << (63 - __clzll(kept)));
        }
        s_pub = kept;
      }
    }
    cluster.sync();  // the owner's s_pub is visible cluster-wide
    const unsigned long long kept = *cluster.map_shared_rank(&s_pub, owner);
    if (tid < TB && ((kept >> tid) & 1ull)) {
      const int srow = blk * TB + tid;
      if (owner == rank) {
        const long long pos = count + __popcll(kept & ((1ull << tid) - 1ull));
        keep_out[S.off + pos] = (int64_t)order[S.off + srow];
      }
      if (rowflag[S.off + srow]) s_orrows[atomicAdd(&s_nor, 1)] = srow;
    }
    count += __popcll(kept);
    __syncthreads();
    const int nor = s_nor;
    if (nor) {  // this CTA's columns beyond blk: w = rank, rank + RC, ... with w > blk
      int w0 = blk + 1;
      w0 += (rank - w0 % RC + RC) % RC;
      for (int w = w0 + tid * RC; w < S.nblk; w += REDUCE_THREADS * RC) {
        unsigned long long acc = 0ull;
        for (int r = 0; r < nor; ++r) acc |= M[(long long)s_orrows[r] * S.nblk + w];
        if (acc) remv[w / RC] |= acc;
      }
    }
    __syncthreads();
    if (tid == 0) s_nor = 0;
    if (max_keep > 0 && count >= max_keep) break;  // uniform: every CTA counts the same bits
  }
  cluster.sync();  // nobody exits while a peer may still read its s_pub
  if (tid == 0 && rank == 0) n_keep_out[b] = count;
}

__global__ void k_zero_outputs(int n_images, int64_t* n_keep_out, int64_t* seg_off_out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_images) n_keep_out[i] = 0;
  if (i <= n_images) seg_off_out[i] = 0;
}

__global__ void k_iou_pairs(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, int64_t n) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  PreBox A = make_prebox(a[5 * i], a[5 * i + 1], a[5 * i + 2], a[5 * i + 3], a[5 * i + 4]);
  PreBox B = make_prebox(b[5 * i], b[5 * i + 1], b[5 * i + 2], b[5 * i + 3], b[5 * i + 4]);
  out[i] = rbox_iou(A, B);
}

struct NmsWs {
  uint64_t *keys_a, *keys_b;
  uint32_t *vals_a, *vals_b;
  PreBox* pre;
  uint8_t* rowflag;
  int32_t* seg_start;
  NmsSeg* seg;
  NmsCtrl* ctrl;
  void* cub_tmp;
  size_t cub_bytes;
  unsigned long long* mask;
  long long mask_words;
  size_t total;
};

size_t cub_sort_bytes(int64_t n) {
  size_t bytes = 0;
  cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, bytes, (const uint64_t*)nullptr, (uint64_t*)nullptr,
                                                  (const uint32_t*)nullptr, (uint32_t*)nullptr, (int)n, 0, 64, 0);
  if (e != cudaSuccess || bytes == 0) {
    (void)cudaGetLastError();
    bytes = (size_t)(32u << 20) + (size_t)n * 4;  // generous bound when no device can be queried
  }
  return bytes;
}

NmsWs carve_nms(void* base, int64_t n, int64_t n_images, int64_t max_per_image) {
  NmsWs w;
  Carver c(base);
  if (max_per_image <= 0 || max_per_image > n) max_per_image = n;
  w.keys_a = c.take<uint64_t>(n);
  w.keys_b = c.take<uint64_t>(n);
  w.vals_a = c.take<uint32_t>(n);
  w.vals_b = c.take<uint32_t>(n);
  w.pre = c.take<PreBox>(n);
  w.rowflag = c.take<uint8_t>(n);
  w.seg_start = c.take<int32_t>(n_images + 2);
  w.seg = c.take<NmsSeg>(n_images + 2);
  w.ctrl = c.take<NmsCtrl>(1);
  w.cub_bytes = cub_sort_bytes(n);
  w.cub_tmp = c.take<char>(w.cub_bytes);
  long long nb = (max_per_image + TB - 1) / TB;
  long long mask_rows = n;
  if ((long long)n_images * max_per_image < mask_rows) mask_rows = (long long)n_images * max_per_image;
  w.mask_words = mask_rows * nb;
  w.mask = c.take<unsigned long long>((size_t)w.mask_words);
  w.total = c.used();
  return w;
}

// profiling aid (y5obb_nms_debug_stage_timing): CUDA events between the stages of nms_impl on the caller's stream
struct StageTimer {
  cudaEvent_t ev[5];
  bool made = false, on = false;
  int n = 0;
};
StageTimer g_stage;
inline void stage_mark(cudaStream_t st) {
  if (g_stage.on && g_stage.n < 5) cudaEventRecord(g_stage.ev[g_stage.n++], st);
}

int nms_impl(const float* dets, const float* scores, const int32_t* image_ids, int64_t n, int64_t n_images,
             int64_t max_per_image, float thr, int flags, int64_t max_keep, int64_t* keep_out, int64_t* n_keep_out,
             int64_t* seg_off_out, void* workspace, size_t ws_bytes, cudaStream_t st,
             const int64_t* n_valid_dev = nullptr, int per_image_clamp = 0) {
  if (n < 0 || n_images < 1 || n_images > MAX_IMAGES || n > 0x7FFFFFF0ll) return Y5OBB_EINVAL;
  if (!keep_out || !n_keep_out || !seg_off_out) return Y5OBB_EINVAL;
  if (n == 0) {
    k_zero_outputs<<<(unsigned)((n_images + 1 + 255) / 256), 256, 0, st>>>((int)n_images, n_keep_out, seg_off_out);
    Y5_LAUNCH_CHECK();
    return Y5OBB_OK;
  }
  if (!dets || !scores || !workspace) return Y5OBB_EINVAL;
  if (max_per_image <= 0 || max_per_image > n) max_per_image = n;
  NmsWs w = carve_nms(workspace, n, n_images, max_per_image);
  if (w.total > ws_bytes) return Y5OBB_EWORKSPACE;

  const unsigned g = (unsigned)((n + 255) / 256);
  g_stage.n = 0;
  stage_mark(st);
  // with a top-k clamp the degenerate boxes keep their rank (reference order: clamp first, too-small filter second)
  const int late_drop = ((flags & Y5OBB_NMS_DROP_SMALL) && per_image_clamp > 0) ? 1 : 0;
  k_make_keys<<<g, 256, 0, st>>>(dets, scores, image_ids, n, (int)n_images, late_drop ? (flags & ~Y5OBB_NMS_DROP_SMALL) : flags,
                                 n_valid_dev, w.keys_a, w.vals_a);
  Y5_LAUNCH_CHECK();
  int img_bits = 1;
  while ((1ll << img_bits) <= n_images) ++img_bits;
  size_t cub_bytes = w.cub_bytes;
  Y5_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, cub_bytes, w.keys_a, w.keys_b, w.vals_a, w.vals_b, (int)n, 0,
                                          32 + img_bits, st));
  stage_mark(st);
  Y5_CUDA(cudaMemsetAsync(w.rowflag, 0, (size_t)n, st));
  k_segments<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(w.keys_b, n, (int)n_images, w.seg_start);
  Y5_LAUNCH_CHECK();
  k_plan<<<1, 32, 0, st>>>(w.seg_start, (int)n_images, w.mask_words, per_image_clamp, w.seg, w.ctrl);
  Y5_LAUNCH_CHECK();
  k_prep<<<g, 256, 0, st>>>(dets, w.vals_b, n, w.pre);
  Y5_LAUNCH_CHECK();

  // persistent tile kernel: a few CTAs per SM, bounded by the number of units that can exist
  long long max_units = 0;
  {
    long long nb = (max_per_image + TB - 1) / TB;
    long long imgs_full = n / max_per_image + 1;
    max_units = units_for(nb) * imgs_full;
  }
  long long grid = (long long)sm_count() * 8;
  if (grid > max_units) grid = max_units;
  if (grid < 1) grid = 1;
  stage_mark(st);
  k_tiles<<<(unsigned)grid, TILE_THREADS, 0, st>>>(w.pre, w.seg, (int)n_images, w.ctrl, w.mask, w.rowflag, thr,
                                                   (flags & Y5OBB_NMS_STRICT_GT) ? 1 : 0);
  Y5_LAUNCH_CHECK();
  stage_mark(st);

  const size_t smem = (size_t)((max_per_image + TB - 1) / TB) * sizeof(unsigned long long);
  if (smem > 200 * 1024) return Y5OBB_EINVAL;  // > 1.6 M boxes in one image
  static size_t smem_set = 0;
  if (smem > 32 * 1024 && smem > smem_set) {
    Y5_CUDA(cudaFuncSetAttribute(k_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    smem_set = 200 * 1024;
  }
  // >= 640 blocks of 64 boxes in an image: a cluster of RC CTAs shares the scan
  if ((max_per_image + TB - 1) / TB >= 640) {  // measured break-even ~40 k boxes (one barrier per 64-row block)
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)n_images * RC);
    cfg.blockDim = dim3(REDUCE_THREADS);
    cfg.dynamicSmemBytes = smem / RC + 64;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = RC;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    Y5_CUDA(cudaLaunchKernelEx(&cfg, k_reduce_cluster, (const NmsSeg*)w.seg, (const NmsCtrl*)w.ctrl,
                               (const unsigned long long*)w.mask, (const uint8_t*)w.rowflag, (const uint32_t*)w.vals_b,
                               (long long)max_keep, (int)n_images, keep_out, n_keep_out, seg_off_out, (const PreBox*)w.pre,
                               late_drop));
  } else {
    k_reduce<<<(unsigned)n_images, REDUCE_THREADS, smem, st>>>(w.seg, w.ctrl, w.mask, w.rowflag, w.vals_b,
                                                              (long long)max_keep, (int)n_images, keep_out, n_keep_out,
                                                              seg_off_out, w.pre, late_drop);
    Y5_LAUNCH_CHECK();
  }
  stage_mark(st);
  return Y5OBB_OK;
}


// ---------------------------------------------------------------------------------------------
// non_max_suppression_obb on the device (/root/reference/utils/general.py:772-862)
//   k_pp_count   one warp per anchor row: obj > conf (:781,:804), conf = cls * obj (:820), per-class
//                candidates when multi_label (:826-828) or the best class (:830-832), class filter (:835)
//   cub scan     deterministic candidate offsets in (image, anchor, class) order == the reference's order
//   k_pp_emit    theta = (argmax(180) - 90) / 180 * 3.141592 (:822-823), class offset cls * 4096 on the
//                centre (:849-851), un-offset 7-float row for the output
//   nms_impl     batched NMS with the max_nms top-k clamp (:845-846) and max_det (:854-855)
//   k_pp_gather  output rows [cx, cy, l, s, theta, conf, cls] in score order
// ---------------------------------------------------------------------------------------------
struct PPArgs {
  const float* pred;
  long long rows;  // B * A
  int A, no, nc;
  float conf;
  int multi_label, agnostic;
  unsigned long long class_mask;  // bit j set = class j allowed
  float max_wh;
  int* far_flag;  // set when a box is so large / far out that boxes of different classes could touch despite the offset
  int row_w;      // floats per row of `pred`: no (the Detect tensor) or the compact record width (Y5OBB_NMS_COMPACT_PRED)
  int compact;    // 1: rows are (cx, cy, w, h, obj, cls[nc], theta index) records written by the Detect epilogue
};

__global__ void k_pp_count(PPArgs a, int* __restrict__ cnt) {
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= a.rows) return;
  const float* p = a.pred + row * a.row_w;
  const float obj = p[4];
  int n = 0;
  if (obj > a.conf) {
    if (a.multi_label) {
      for (int j0 = 0; j0 < a.nc; j0 += 32) {
        const int j = j0 + lane;
        bool ok = false;
        if (j < a.nc) ok = (__fmul_rn(p[5 + j], obj) > a.conf) && ((a.class_mask >> (j & 63)) & 1ull);
        n += __popc(__ballot_sync(0xffffffffu, ok));
      }
    } else {
      float bv = -INFINITY;
      int bj = 0x7fffffff;
      for (int j = lane; j < a.nc; j += 32) {
        const float v = __fmul_rn(p[5 + j], obj);
        if (v > bv) {
          bv = v;
          bj = j;
        }
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
        if (ov > bv || (ov == bv && oj < bj)) {
          bv = ov;
          bj = oj;
        }
      }
      n = (bv > a.conf && bj < a.nc && ((a.class_mask >> (bj & 63)) & 1ull)) ? 1 : 0;
    }
  }
  if (lane == 0) cnt[row] = n;
}

__global__ void k_pp_emit(PPArgs a, const int* __restrict__ cnt, const int* __restrict__ off, long long capacity,
                          float* __restrict__ dets5, float* __restrict__ scores, int32_t* __restrict__ image_ids,
                          float* __restrict__ out7, int64_t* __restrict__ n_valid) {
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= a.rows) return;
  if (row == 0 && lane == 0) {
    const long long total = (long long)off[a.rows - 1] + cnt[a.rows - 1];
    n_valid[0] = total < capacity ? total : capacity;  // entries the NMS may look at
    n_valid[1] = total;                                // what the host checks against capacity
  }
  if (cnt[row] == 0) return;
  const float* p = a.pred + row * a.row_w;
  const float obj = p[4];
  // theta = first argmax over the 180 angle bins (compact records carry it already)
  float bv = -INFINITY;
  int bk = 0x7fffffff;
  const int cidx = 5 + a.nc;
  for (int k = lane; k < (a.compact ? 0 : 180); k += 32) {
    const float v = p[cidx + k];
    if (v > bv) {
      bv = v;
      bk = k;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int ok = __shfl_xor_sync(0xffffffffu, bk, o);
    if (ov > bv || (ov == bv && ok < bk)) {
      bv = ov;
      bk = ok;
    }
  }
  if (a.compact) bk = (int)p[cidx];
  if (bk > 179 || bk < 0) bk = 0;  // all-NaN row: torch.max returns index 0
  const float theta = __fmul_rn(__fdiv_rn((float)(bk - 90), 180.0f), 3.141592f);
  const float cx = p[0], cy = p[1], w = p[2], h = p[3];
  const int img = (int)(row / a.A);
  long long base = off[row];
  // class-split NMS is exact only if boxes of different classes cannot overlap: with r + max(|cx|, |cy|) < max_wh / 2
  // for every box, two offset centres are further apart than the two circumradii (NaN fails the test)
  if (lane == 0 && a.far_flag && !(0.5f * sqrtf(w * w + h * h) + fmaxf(fabsf(cx), fabsf(cy)) < 0.5f * a.max_wh - 8.0f))
    atomicOr(a.far_flag, 1);

  auto put = [&](long long slot, int cls, float sc) {
    if (slot >= capacity) return;
    const float c = a.agnostic ? 0.0f : __fmul_rn((float)cls, a.max_wh);
    float* d = dets5 + slot * 5;
    d[0] = __fadd_rn(cx, c);
    d[1] = __fadd_rn(cy, c);
    d[2] = w;
    d[3] = h;
    d[4] = theta;
    scores[slot] = sc;
    image_ids[slot] = img;
    float* o = out7 + slot * 7;
    o[0] = cx;
    o[1] = cy;
    o[2] = w;
    o[3] = h;
    o[4] = theta;
    o[5] = sc;
    o[6] = (float)cls;
  };

  if (a.multi_label) {
    for (int j0 = 0; j0 < a.nc; j0 += 32) {
      const int j = j0 + lane;
      bool ok = false;
      float sc = 0.f;
      if (j < a.nc) {
        sc = __fmul_rn(p[5 + j], obj);
        ok = (sc > a.conf) && ((a.class_mask >> (j & 63)) & 1ull);
      }
      const unsigned bal = __ballot_sync(0xffffffffu, ok);
      if (ok) put(base + __popc(bal & ((1u << lane) - 1u)), j, sc);
      base += __popc(bal);
    }
  } else {
    float cv = -INFINITY;
    int cj = 0x7fffffff;
    for (int j = lane; j < a.nc; j += 32) {
      const float v = __fmul_rn(p[5 + j], obj);
      if (v > cv) {
        cv = v;
        cj = j;
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, cv, o);
      const int oj = __shfl_xor_sync(0xffffffffu, cj, o);
      if (ov > cv || (ov == cv && oj < cj)) {
        cv = ov;
        cj = oj;
      }
    }
    if (lane == 0) put(base, cj, cv);
  }
}

// ---- compact records (Y5OBB_NMS_COMPACT_PRED): one THREAD per anchor row.  A row is 96 B and almost every row fails the
// objectness test on its first read, so a warp per row (the layout the 800-byte tensor rows want) would only schedule warps.
// Same arithmetic, same candidate order (ascending class inside a row) as k_pp_count / k_pp_emit above.
__global__ void k_pp_count_rec(PPArgs a, int* __restrict__ cnt) {
  const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= a.rows) return;
  const float* p = a.pred + row * a.row_w;
  const float obj = p[4];
  int n = 0;
  if (obj > a.conf) {
    if (a.multi_label) {
      for (int j = 0; j < a.nc; ++j)
        n += ((__fmul_rn(p[5 + j], obj) > a.conf) && ((a.class_mask >> (j & 63)) & 1ull)) ? 1 : 0;
    } else {
      float bv = -INFINITY;
      int bj = 0x7fffffff;
      for (int j = 0; j < a.nc; ++j) {
        const float v = __fmul_rn(p[5 + j], obj);
        if (v > bv) {
          bv = v;
          bj = j;
        }
      }
      n = (bv > a.conf && bj < a.nc && ((a.class_mask >> (bj & 63)) & 1ull)) ? 1 : 0;
    }
  }
  cnt[row] = n;
}

__global__ void k_pp_emit_rec(PPArgs a, const int* __restrict__ cnt, const int* __restrict__ off, long long capacity,
                              float* __restrict__ dets5, float* __restrict__ scores, int32_t* __restrict__ image_ids,
                              float* __restrict__ out7, int64_t* __restrict__ n_valid) {
  const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= a.rows) return;
  if (row == 0) {
    const long long total = (long long)off[a.rows - 1] + cnt[a.rows - 1];
    n_valid[0] = total < capacity ? total : capacity;
    n_valid[1] = total;
  }
  if (cnt[row] == 0) return;
  const float* p = a.pred + row * a.row_w;
  const float obj = p[4];
  int bk = (int)p[5 + a.nc];
  if (bk > 179 || bk < 0) bk = 0;
  const float theta = __fmul_rn(__fdiv_rn((float)(bk - 90), 180.0f), 3.141592f);
  const float cx = p[0], cy = p[1], w = p[2], h = p[3];
  const int img = (int)(row / a.A);
  long long slot = off[row];
  if (a.far_flag && !(0.5f * sqrtf(w * w + h * h) + fmaxf(fabsf(cx), fabsf(cy)) < 0.5f * a.max_wh - 8.0f)) atomicOr(a.far_flag, 1);
  auto put = [&](int cls, float sc) {
    if (slot < capacity) {
      const float c = a.agnostic ? 0.0f : __fmul_rn((float)cls, a.max_wh);
      float* d = dets5 + slot * 5;
      d[0] = __fadd_rn(cx, c);
      d[1] = __fadd_rn(cy, c);
      d[2] = w;
      d[3] = h;
      d[4] = theta;
      scores[slot] = sc;
      image_ids[slot] = img;
      float* o = out7 + slot * 7;
      o[0] = cx;
      o[1] = cy;
      o[2] = w;
      o[3] = h;
      o[4] = theta;
      o[5] = sc;
      o[6] = (float)cls;
    }
    ++slot;
  };
  if (a.multi_label) {
    for (int j = 0; j < a.nc; ++j) {
      const float sc = __fmul_rn(p[5 + j], obj);
      if ((sc > a.conf) && ((a.class_mask >> (j & 63)) & 1ull)) put(j, sc);
    }
  } else {
    float cv = -INFINITY;
    int cj = 0x7fffffff;
    for (int j = 0; j < a.nc; ++j) {
      const float v = __fmul_rn(p[5 + j], obj);
      if (v > cv) {
        cv = v;
        cj = j;
      }
    }
    put(cj, cv);
  }
}

__global__ void k_pp_gather(const float* __restrict__ out7, const int64_t* __restrict__ keep,
                            const int64_t* __restrict__ n_keep, const int64_t* __restrict__ seg_off, int n_images,
                            int max_det, float* __restrict__ dst, int64_t* __restrict__ counts,
                            const int64_t* __restrict__ n_valid, const int* __restrict__ far_flag) {
  const int b = blockIdx.y;
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long nk = n_keep[b];
  if (k == 0) {
    counts[b] = nk;
    // total candidates before the capacity clamp; -2 = the class-split shortcut was not applicable (a box large or far
    // enough to reach another class's offset copy): the caller re-runs with Y5OBB_NMS_NO_CLASS_SPLIT
    if (b == 0) counts[n_images] = (far_flag && *far_flag) ? -2 : n_valid[1];
  }
  if (k >= nk || k >= max_det) return;
  const float* s = out7 + keep[seg_off[b] + k] * 7;
  float* d = dst + ((long long)b * max_det + k) * 7;
#pragma unroll
  for (int e = 0; e < 7; ++e) d[e] = s[e];
}

// ---- class-split NMS (the reference separates classes by adding cls * max_wh to the centres, general.py:849-851:
// boxes of different classes never overlap, so the greedy pass decomposes into independent (image, class) problems:
// sum_c n_c^2 pair tests instead of (sum_c n_c)^2) ---------------------------------------------------------------
// key2 of the candidate at score-sorted position pos: ((image * nc + cls) << 32), or the dump segment when the image's
// top-max_nms clamp (general.py:845-846) or the dump image excludes it.  A stable sort on these bits keeps the score order.
__global__ void k_class_keys(const uint64_t* __restrict__ keys1, const uint32_t* __restrict__ order1,
                             const int32_t* __restrict__ seg1_start, const float* __restrict__ out7, int64_t n,
                             int n_images, int nc, int max_nms, int drop_small, uint64_t* __restrict__ keys2) {
  const int64_t pos = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (pos >= n) return;
  const int img = (int)(keys1[pos] >> 32);
  uint32_t seg = (uint32_t)(n_images * nc);
  if (img < n_images) {
    const long long r = pos - seg1_start[img];
    if (max_nms <= 0 || r < max_nms) {
      const float* o = out7 + (long long)order1[pos] * 7;
      int cls = (int)o[6];
      cls = min(max(cls, 0), nc - 1);
      // reference order: the top-max_nms clamp above counted this box; obb_nms then drops it if it is degenerate
      // (nms_rotated_wrapper.py:32-39)
      if (!(drop_small && fminf(o[2], o[3]) < 0.001f)) seg = (uint32_t)(img * nc + cls);
    }
  }
  keys2[pos] = (uint64_t)seg << 32;
}

__global__ void k_flag_kept(const int64_t* __restrict__ keep, const int64_t* __restrict__ n_keep,
                            const int64_t* __restrict__ seg_off, uint8_t* __restrict__ flag) {
  const int s = blockIdx.y;
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n_keep[s]) flag[keep[seg_off[s] + k]] = 1;
}

// one CTA per image: the kept candidates of all its classes, in the image's score order, first max_det of them
__global__ void __launch_bounds__(1024) k_merge_classes(const uint32_t* __restrict__ order1,
                                                        const int32_t* __restrict__ seg1_start,
                                                        const uint8_t* __restrict__ flag, const NmsCtrl* __restrict__ ctrl,
                                                        int n_images, int max_nms, long long max_keep,
                                                        int64_t* __restrict__ keep_out, int64_t* __restrict__ n_keep_out,
                                                        int64_t* __restrict__ seg_off_out) {
  __shared__ int s_warp[32];
  __shared__ long long s_count;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const long long off = seg1_start[b];
  long long nb = (long long)seg1_start[b + 1] - off;
  if (max_nms > 0 && nb > max_nms) nb = max_nms;
  if (tid == 0) {
    seg_off_out[b] = off;
    if (b == 0) seg_off_out[n_images] = seg1_start[n_images];
    s_count = 0;
  }
  if (ctrl->err) {
    if (tid == 0) n_keep_out[b] = -1;
    return;
  }
  __syncthreads();
  for (long long base = 0; base < nb; base += 1024) {
    const long long p = base + tid;
    const uint32_t cand = p < nb ? order1[off + p] : 0u;
    const bool kept = p < nb && flag[cand];
    const unsigned bal = __ballot_sync(0xffffffffu, kept);
    if (lane == 0) s_warp[wid] = __popc(bal);
    __syncthreads();
    long long before = s_count;
    for (int w2 = 0; w2 < wid; ++w2) before += s_warp[w2];
    const long long idx = before + __popc(bal & ((1u << lane) - 1u));
    if (kept && (max_keep <= 0 || idx < max_keep)) keep_out[off + idx] = (int64_t)cand;
    __syncthreads();
    if (tid == 0) {
      long long t = s_count;
      for (int w2 = 0; w2 < 32; ++w2) t += s_warp[w2];
      s_count = t;
    }
    __syncthreads();
    if (max_keep > 0 && s_count >= max_keep) break;
  }
  if (tid == 0) n_keep_out[b] = (max_keep > 0 && s_count > max_keep) ? max_keep : s_count;
}

struct PPWs {
  int *cnt, *off;
  void* scan_tmp;
  size_t scan_bytes;
  float *dets5, *scores, *out7;
  int32_t* image_ids;
  int64_t *n_valid, *keep, *n_keep, *seg_off;
  void* nms_ws;
  size_t nms_bytes;
  // class-split path
  uint64_t *keys2_a, *keys2_b;
  uint32_t *vals2_a, *order2;
  int32_t* seg1_start;
  uint8_t* keepflag;
  int64_t *keepC, *n_keepC, *seg_offC;
  int* far_flag;
  size_t total;
};

size_t scan_bytes_for(long long rows) {
  size_t bytes = 0;
  cudaError_t e = cub::DeviceScan::ExclusiveSum(nullptr, bytes, (const int*)nullptr, (int*)nullptr, (int)rows, 0);
  if (e != cudaSuccess || bytes == 0) {
    (void)cudaGetLastError();
    bytes = (size_t)(1u << 20) + (size_t)rows / 64;
  }
  return bytes;
}

PPWs carve_pp(void* base, long long rows, int n_images, long long capacity, int max_nms, int nc) {
  PPWs w;
  Carver c(base);
  w.cnt = c.take<int>(rows);
  w.off = c.take<int>(rows);
  w.scan_bytes = scan_bytes_for(rows);
  w.scan_tmp = c.take<char>(w.scan_bytes);
  w.dets5 = c.take<float>(capacity * 5);
  w.scores = c.take<float>(capacity);
  w.out7 = c.take<float>(capacity * 7);
  w.image_ids = c.take<int32_t>(capacity);
  w.n_valid = c.take<int64_t>(2);
  w.keep = c.take<int64_t>(capacity);
  w.n_keep = c.take<int64_t>(n_images);
  w.seg_off = c.take<int64_t>(n_images + 1);
  long long mpi = max_nms > 0 && max_nms < capacity ? max_nms : capacity;
  const long long n_seg = (long long)n_images * nc;
  NmsWs nw = carve_nms(nullptr, capacity, n_seg, mpi);  // the (image, class) segmentation needs the larger tables
  w.nms_bytes = nw.total + 256;
  w.nms_ws = c.take<char>(w.nms_bytes);
  w.keys2_a = c.take<uint64_t>(capacity);
  w.keys2_b = c.take<uint64_t>(capacity);
  w.vals2_a = c.take<uint32_t>(capacity);
  w.order2 = c.take<uint32_t>(capacity);
  w.seg1_start = c.take<int32_t>(n_images + 2);
  w.keepflag = c.take<uint8_t>(capacity);
  w.keepC = c.take<int64_t>(capacity);
  w.n_keepC = c.take<int64_t>(n_seg + 1);
  w.seg_offC = c.take<int64_t>(n_seg + 2);
  w.far_flag = c.take<int>(4);
  w.total = c.used();
  return w;
}

// Class-split variant of nms_impl for the post-process path (every candidate carries its class in out7[6]).
// Same outputs as nms_impl: keep_out[seg_off_out[b] + k], k < n_keep_out[b], in descending score order per image.
int nms_classes(const PPWs& w, const float* out7, int64_t n, int n_images, int nc, int64_t max_per_image, float thr, int flags,
                int64_t max_keep, int max_nms, cudaStream_t st) {
  const int n_seg = n_images * nc;
  if (n_seg < 1 || n_seg >= MAX_IMAGES) return Y5OBB_EINVAL;
  if (max_per_image <= 0 || max_per_image > n) max_per_image = n;
  NmsWs ws = carve_nms(w.nms_ws, n, n_seg, max_per_image);
  if (ws.total > w.nms_bytes) return Y5OBB_EWORKSPACE;
  const unsigned g = (unsigned)((n + 255) / 256);
  // 1. every image's candidates by descending score (ties: lower index), as the reference's argsort
  k_make_keys<<<g, 256, 0, st>>>(w.dets5, w.scores, w.image_ids, n, n_images, flags & ~Y5OBB_NMS_DROP_SMALL, w.n_valid,
                                 ws.keys_a, ws.vals_a);
  Y5_LAUNCH_CHECK();
  int img_bits = 1;
  while ((1ll << img_bits) <= n_images) ++img_bits;
  size_t cub_bytes = ws.cub_bytes;
  Y5_CUDA(cub::DeviceRadixSort::SortPairs(ws.cub_tmp, cub_bytes, ws.keys_a, ws.keys_b, ws.vals_a, ws.vals_b, (int)n, 0,
                                          32 + img_bits, st));
  k_segments<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(ws.keys_b, n, n_images, w.seg1_start);
  Y5_LAUNCH_CHECK();
  // 2. stable re-grouping by (image, class) of the top-max_nms of every image: score order survives inside a class
  k_class_keys<<<g, 256, 0, st>>>(ws.keys_b, ws.vals_b, w.seg1_start, out7, n, n_images, nc, max_nms,
                                  (flags & Y5OBB_NMS_DROP_SMALL) ? 1 : 0, w.keys2_a);
  Y5_LAUNCH_CHECK();
  int seg_bits = 1;
  while ((1ll << seg_bits) <= n_seg) ++seg_bits;
  cub_bytes = ws.cub_bytes;
  Y5_CUDA(cub::DeviceRadixSort::SortPairs(ws.cub_tmp, cub_bytes, w.keys2_a, w.keys2_b, ws.vals_b, w.order2, (int)n, 32,
                                          32 + seg_bits, st));
  Y5_CUDA(cudaMemsetAsync(ws.rowflag, 0, (size_t)n, st));
  Y5_CUDA(cudaMemsetAsync(w.keepflag, 0, (size_t)n, st));
  k_segments<<<(unsigned)((n + 1 + 255) / 256), 256, 0, st>>>(w.keys2_b, n, n_seg, ws.seg_start);
  Y5_LAUNCH_CHECK();
  k_plan<<<1, 32, 0, st>>>(ws.seg_start, n_seg, ws.mask_words, 0, ws.seg, ws.ctrl);
  Y5_LAUNCH_CHECK();
  k_prep<<<g, 256, 0, st>>>(w.dets5, w.order2, n, ws.pre);
  Y5_LAUNCH_CHECK();
  // 3. independent greedy passes per (image, class)
  long long grid = (long long)sm_count() * 8;
  {
    const long long nb = (max_per_image + TB - 1) / TB;
    const long long max_units = units_for(nb) * (n / max_per_image + 1) + n_seg;
    if (grid > max_units) grid = max_units;
    if (grid < 1) grid = 1;
  }
  k_tiles<<<(unsigned)grid, TILE_THREADS, 0, st>>>(ws.pre, ws.seg, n_seg, ws.ctrl, ws.mask, ws.rowflag, thr,
                                                   (flags & Y5OBB_NMS_STRICT_GT) ? 1 : 0);
  Y5_LAUNCH_CHECK();
  const size_t smem = (size_t)((max_per_image + TB - 1) / TB) * sizeof(unsigned long long);
  if (smem > 200 * 1024) return Y5OBB_EINVAL;
  static size_t smem_set = 0;
  if (smem > 32 * 1024 && smem > smem_set) {
    Y5_CUDA(cudaFuncSetAttribute(k_reduce, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(200 * 1024)));
    smem_set = 200 * 1024;
  }
  k_reduce<<<(unsigned)n_seg, REDUCE_THREADS, smem, st>>>(ws.seg, ws.ctrl, ws.mask, ws.rowflag, w.order2, (long long)max_keep,
                                                         n_seg, w.keepC, w.n_keepC, w.seg_offC, ws.pre, 0);
  Y5_LAUNCH_CHECK();
  // 4. merge: kept flags, then every image's keepers in its own score order, first max_keep of them
  const long long per_seg = max_keep > 0 ? max_keep : max_per_image;
  dim3 gf((unsigned)((per_seg + 255) / 256), (unsigned)n_seg);
  k_flag_kept<<<gf, 256, 0, st>>>(w.keepC, w.n_keepC, w.seg_offC, w.keepflag);
  Y5_LAUNCH_CHECK();
  k_merge_classes<<<(unsigned)n_images, 1024, 0, st>>>(ws.vals_b, w.seg1_start, w.keepflag, ws.ctrl, n_images, max_nms,
                                                      (long long)max_keep, w.keep, w.n_keep, w.seg_off);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

int y5obb_abi_version(void) { return 2; }
int y5obb_last_cuda_error(void) { return g_last_cuda_error; }
const char* y5obb_build_info(void) { return "liby5obb sm_100a " __DATE__ " " __TIME__; }

size_t y5obb_nms_workspace_bytes(int64_t n_total, int64_t n_images, int64_t max_per_image) {
  if (n_total <= 0) return 256;
  if (n_images < 1) n_images = 1;
  NmsWs w = carve_nms(nullptr, n_total, n_images, max_per_image);
  return w.total + 256;
}

int y5obb_nms_rotated_f32(const float* dets5, const float* scores, int64_t n, float iou_thr, int flags,
                          int64_t* keep_out, int64_t* n_keep_out, void* workspace, size_t workspace_bytes,
                          void* stream) {
  // the two-entry seg_off output lives at the head of the workspace
  if (n > 0 && (!workspace || workspace_bytes < 512)) return Y5OBB_EWORKSPACE;
  if (n == 0) {
    if (!n_keep_out) return Y5OBB_EINVAL;
    Y5_CUDA(cudaMemsetAsync(n_keep_out, 0, sizeof(int64_t), (cudaStream_t)stream));
    return Y5OBB_OK;
  }
  int64_t* seg_off = static_cast<int64_t*>(workspace);
  return nms_impl(dets5, scores, nullptr, n, 1, n, iou_thr, flags, 0, keep_out, n_keep_out, seg_off,
                  static_cast<char*>(workspace) + 256, workspace_bytes - 256, (cudaStream_t)stream);
}

int y5obb_nms_rotated_batched_f32(const float* dets5, const float* scores, const int32_t* image_ids,
                                  int64_t n_total, int64_t n_images, int64_t max_per_image, float iou_thr, int flags,
                                  int64_t max_keep, int64_t* keep_out, int64_t* n_keep_out, int64_t* seg_off_out,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  return nms_impl(dets5, scores, image_ids, n_total, n_images, max_per_image, iou_thr, flags, max_keep, keep_out,
                  n_keep_out, seg_off_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

size_t y5obb_nms_obb_workspace_bytes(int64_t batch, int64_t anchors, int64_t max_candidates, int64_t max_nms) {
  if (batch <= 0 || anchors <= 0 || max_candidates <= 0) return 256;
  PPWs w = carve_pp(nullptr, batch * anchors, (int)batch, max_candidates, (int)max_nms, 64);
  return w.total + 256;
}

int y5obb_nms_obb_f32(const float* pred, int64_t batch, int64_t anchors, int no, int nc, float conf_thres,
                      float iou_thres, uint64_t class_mask, int agnostic, int multi_label, int max_det, int max_nms,
                      float max_wh, int flags, int64_t max_candidates, float* out7, int64_t* counts, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (!pred || !out7 || !counts || !workspace) return Y5OBB_EINVAL;
  if (batch <= 0 || anchors <= 0 || nc <= 0 || nc > 64 || no != nc + 5 + 180 || max_det <= 0 || max_candidates <= 0)
    return Y5OBB_EINVAL;
  const long long rows = batch * anchors;
  if (rows > 0x7FFFFFF0ll || max_candidates > 0x7FFFFFF0ll) return Y5OBB_EINVAL;
  cudaStream_t st = (cudaStream_t)stream;
  PPWs w = carve_pp(workspace, rows, (int)batch, max_candidates, max_nms, nc);
  if (w.total > workspace_bytes) return Y5OBB_EWORKSPACE;
  PPArgs a;
  a.compact = (flags & Y5OBB_NMS_COMPACT_PRED) ? 1 : 0;
  a.row_w = a.compact ? ((nc + 6) + 3) / 4 * 4 : no;
  a.pred = pred;
  a.rows = rows;
  a.A = (int)anchors;
  a.no = no;
  a.nc = nc;
  a.conf = conf_thres;
  a.multi_label = (multi_label && nc > 1) ? 1 : 0;  // general.py:797
  a.agnostic = agnostic;
  a.class_mask = class_mask;
  a.max_wh = max_wh;
  // class-split NMS when the class offset separates the classes (not agnostic, > 1 class) and the caller did not veto it
  const bool split = !agnostic && nc > 1 && !(flags & Y5OBB_NMS_NO_CLASS_SPLIT) && batch * (long long)nc < (1 << 16);
  a.far_flag = split ? w.far_flag : nullptr;
  if (split) Y5_CUDA(cudaMemsetAsync(w.far_flag, 0, sizeof(int), st));
  const unsigned g = (unsigned)((rows * 32 + 255) / 256);
  const unsigned g1 = (unsigned)((rows + 255) / 256);
  if (a.compact) k_pp_count_rec<<<g1, 256, 0, st>>>(a, w.cnt);
  else k_pp_count<<<g, 256, 0, st>>>(a, w.cnt);
  Y5_LAUNCH_CHECK();
  size_t sb = w.scan_bytes;
  Y5_CUDA(cub::DeviceScan::ExclusiveSum(w.scan_tmp, sb, w.cnt, w.off, (int)rows, st));
  if (a.compact)
    k_pp_emit_rec<<<g1, 256, 0, st>>>(a, w.cnt, w.off, max_candidates, w.dets5, w.scores, w.image_ids, w.out7, w.n_valid);
  else
    k_pp_emit<<<g, 256, 0, st>>>(a, w.cnt, w.off, max_candidates, w.dets5, w.scores, w.image_ids, w.out7, w.n_valid);
  Y5_LAUNCH_CHECK();
  long long mpi = max_nms > 0 && max_nms < max_candidates ? max_nms : max_candidates;
  int rc;
  if (split)
    rc = nms_classes(w, w.out7, max_candidates, (int)batch, nc, mpi, iou_thres, flags | Y5OBB_NMS_DROP_SMALL, max_det, max_nms, st);
  else
    rc = nms_impl(w.dets5, w.scores, w.image_ids, max_candidates, batch, mpi, iou_thres, flags | Y5OBB_NMS_DROP_SMALL,
                  max_det, w.keep, w.n_keep, w.seg_off, w.nms_ws, w.nms_bytes, st, w.n_valid, max_nms);
  if (rc) return rc;
  dim3 gg((unsigned)((max_det + 127) / 128), (unsigned)batch);
  k_pp_gather<<<gg, 128, 0, st>>>(w.out7, w.keep, w.n_keep, w.seg_off, (int)batch, max_det, out7, counts, w.n_valid,
                                  split ? w.far_flag : nullptr);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_nms_debug_stage_timing(int on) {
  if (on && !g_stage.made) {
    for (int i = 0; i < 5; ++i) Y5_CUDA(cudaEventCreate(&g_stage.ev[i]));
    g_stage.made = true;
  }
  g_stage.on = on != 0;
  g_stage.n = 0;
  return Y5OBB_OK;
}

int y5obb_nms_debug_stage_ms(float* ms4) {
  if (!ms4 || !g_stage.on || g_stage.n != 5) return Y5OBB_EINVAL;
  Y5_CUDA(cudaEventSynchronize(g_stage.ev[4]));
  for (int i = 0; i < 4; ++i) Y5_CUDA(cudaEventElapsedTime(&ms4[i], g_stage.ev[i], g_stage.ev[i + 1]));
  return Y5OBB_OK;
}

int y5obb_rbox_iou_pairs_f32(const float* a5, const float* b5, float* iou_out, int64_t n, void* stream) {
  if (n < 0) return Y5OBB_EINVAL;
  if (n == 0) return Y5OBB_OK;
  if (!a5 || !b5 || !iou_out) return Y5OBB_EINVAL;
  k_iou_pairs<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a5, b5, iou_out, n);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

}  // extern "C"
