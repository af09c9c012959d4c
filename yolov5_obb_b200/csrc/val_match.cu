// Post-NMS geometry + validation matching of one batch in ONE launch (SURVEY section 8f rank 3):
//   /root/reference/val.py:226-250 per image:  rbox2poly -> scale_polys -> poly2hbb -> xywh2xyxy for the detections,
//       rbox2poly -> poly2hbb -> xywh2xyxy -> scale_coords (+ clip) for the labels, then
//   /root/reference/val.py:69-92 process_batch:  HBB box_iou (utils/metrics.py:246-268), class match, IoU >= iouv[0]; every
//       detection keeps its highest-IoU label, every label keeps its lowest-index (= most confident) detection among those;
//       correct[d, :] = iou >= iouv for the surviving pairs.
// The reference runs ~40 small ATen kernels, two host round trips (numpy argsort / unique) and a Python loop per image.
// Every arithmetic step below is a separately rounded fp32 op in the reference's order (no FMA contraction), so the boxes
// are bit-identical to the ATen chain ON A GPU (where val.py runs it) and the IoUs decide the same thresholds.  One ATen
// detail matters for that: a CUDA tensor divided by a Python scalar is multiplied by the scalar's fp32 reciprocal
// (BinaryDivTrueKernel.cu), so `/= gain` below is `* (1.0f / gain)`; divisions by 2 are exact either way.  Ties (two labels with exactly the same IoU for
// one detection) go to the lower label index; the reference's numpy quicksort leaves them unspecified.
// HBM-bound: 28 B read + (niou + 48) B written per detection; the label list of an image lives in shared memory.
#include "common.cuh"
#include "rbox_poly.cuh"  // rbox_to_poly: utils/rboxs_utils.py:106-126 (torch branch)

namespace y5obb {
namespace {

constexpr int VM_THREADS = 256;
constexpr int VM_MAX_LABELS = 1536;  // per image, in shared memory

struct VmArgs {
  const float* pred7;      // [B, max_det, 7] rows (cx, cy, l, s, theta, conf, cls), counts[b] valid rows per image
  const long long* counts;
  int B, max_det;
  const float* labels;     // [nl, 7] rows (image, cls, cx, cy, l, s, theta), pixel units of the network input, grouped or not
  int nl;
  const float* scale;      // [B, 5]: gain, pad_x, pad_y, raw_h, raw_w   (shapes[si][1] and shapes[si][0] of val.py:213,233)
  const float* iouv;       // [niou] ascending
  int niou;
  unsigned char* correct;  // [B, max_det, niou]
  float* polyn;            // [B, max_det, 8] native-space polygons (pred_polyn) or null
  float* hbbn;             // [B, max_det, 4] native-space xyxy boxes (pred_hbbn) or null
  int* overflow;           // set to 1 if an image has more than VM_MAX_LABELS labels
};

// poly2hbb (utils/rboxs_utils.py:147-165) then xywh2xyxy (utils/general.py:555-562): note x1 = xc - w/2, not x_min
__device__ __forceinline__ void poly_to_xyxy(const float* p, float* b) {
  const float x_max = fmaxf(fmaxf(p[0], p[2]), fmaxf(p[4], p[6])), x_min = fminf(fminf(p[0], p[2]), fminf(p[4], p[6]));
  const float y_max = fmaxf(fmaxf(p[1], p[3]), fmaxf(p[5], p[7])), y_min = fminf(fminf(p[1], p[3]), fminf(p[5], p[7]));
  const float xc = __fdiv_rn(__fadd_rn(x_max, x_min), 2.0f), yc = __fdiv_rn(__fadd_rn(y_max, y_min), 2.0f);
  const float w = __fsub_rn(x_max, x_min), h = __fsub_rn(y_max, y_min);
  b[0] = __fsub_rn(xc, __fdiv_rn(w, 2.0f));
  b[1] = __fsub_rn(yc, __fdiv_rn(h, 2.0f));
  b[2] = __fadd_rn(xc, __fdiv_rn(w, 2.0f));
  b[3] = __fadd_rn(yc, __fdiv_rn(h, 2.0f));
}

__global__ void __launch_bounds__(VM_THREADS) k_val_match(VmArgs a) {
  __shared__ float s_lab[VM_MAX_LABELS * 5];  // cls, x1, y1, x2, y2 (native space)
  __shared__ float s_area[VM_MAX_LABELS];
  __shared__ int s_win[VM_MAX_LABELS];        // lowest detection index whose best label this is
  __shared__ int s_n;
  __shared__ int s_warp[VM_THREADS / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float gain = a.scale[b * 5 + 0], pad_x = a.scale[b * 5 + 1], pad_y = a.scale[b * 5 + 2];
  const float raw_h = a.scale[b * 5 + 3], raw_w = a.scale[b * 5 + 4];
  const float inv_gain = __fdiv_rn(1.0f, gain);
  if (tid == 0) s_n = 0;
  __syncthreads();
  // ---- labels of image b, in their order of appearance (val.py:214 `targets[targets[:, 0] == si, 1:7]`)
  for (int base = 0; base < a.nl; base += VM_THREADS) {
    const int i = base + tid;
    const bool mine = i < a.nl && (int)a.labels[(long long)i * 7] == b;
    const unsigned bal = __ballot_sync(0xffffffffu, mine);
    if (lane == 0) s_warp[wid] = __popc(bal);
    __syncthreads();
    int before = s_n;
    for (int w = 0; w < wid; ++w) before += s_warp[w];
    const int slot = before + __popc(bal & ((1u << lane) - 1u));
    if (mine && slot < VM_MAX_LABELS) {
      const float* L = a.labels + (long long)i * 7;
      float poly[8], box[4];
      rbox_to_poly(L[2], L[3], L[4], L[5], L[6], poly);   // tpoly = rbox2poly(labels[:, 1:6])
      poly_to_xyxy(poly, box);                            // tbox = xywh2xyxy(poly2hbb(tpoly))
      // scale_coords (utils/general.py:621-634): subtract the padding, divide by the gain, clip to the raw image
      box[0] = __fmul_rn(__fsub_rn(box[0], pad_x), inv_gain);
      box[2] = __fmul_rn(__fsub_rn(box[2], pad_x), inv_gain);
      box[1] = __fmul_rn(__fsub_rn(box[1], pad_y), inv_gain);
      box[3] = __fmul_rn(__fsub_rn(box[3], pad_y), inv_gain);
      box[0] = fminf(fmaxf(box[0], 0.f), raw_w);
      box[2] = fminf(fmaxf(box[2], 0.f), raw_w);
      box[1] = fminf(fmaxf(box[1], 0.f), raw_h);
      box[3] = fminf(fmaxf(box[3], 0.f), raw_h);
      s_lab[slot * 5 + 0] = L[1];
      s_lab[slot * 5 + 1] = box[0];
      s_lab[slot * 5 + 2] = box[1];
      s_lab[slot * 5 + 3] = box[2];
      s_lab[slot * 5 + 4] = box[3];
      s_area[slot] = __fmul_rn(__fsub_rn(box[2], box[0]), __fsub_rn(box[3], box[1]));  // box_area (metrics.py:259-261)
      s_win[slot] = 0x7fffffff;
    }
    __syncthreads();
    if (tid == 0) {
      int t = s_n;
      for (int w = 0; w < VM_THREADS / 32; ++w) t += s_warp[w];
      s_n = t;
    }
    __syncthreads();
  }
  int nlab = s_n;
  if (nlab > VM_MAX_LABELS) {
    if (tid == 0) *a.overflow = 1;
    nlab = VM_MAX_LABELS;
  }
  const int nd = (int)min((long long)a.max_det, max(0ll, a.counts[b]));
  const float thr0 = a.iouv[0];
  // ---- pass 1: geometry of every detection, its best label, the label's lowest such detection
  for (int d0 = 0; d0 < nd; d0 += VM_THREADS) {
    const int d = d0 + tid;
    if (d < nd) {
      const float* P = a.pred7 + ((long long)b * a.max_det + d) * 7;
      float poly[8], box[4];
      rbox_to_poly(P[0], P[1], P[2], P[3], P[4], poly);
#pragma unroll
      for (int k = 0; k < 8; k += 2) {  // scale_polys (utils/general.py:636-650), no clipping
        poly[k] = __fmul_rn(__fsub_rn(poly[k], pad_x), inv_gain);
        poly[k + 1] = __fmul_rn(__fsub_rn(poly[k + 1], pad_y), inv_gain);
      }
      poly_to_xyxy(poly, box);
      if (a.polyn) {
        float* o = a.polyn + ((long long)b * a.max_det + d) * 8;
#pragma unroll
        for (int k = 0; k < 8; ++k) o[k] = poly[k];
      }
      if (a.hbbn) {
        float* o = a.hbbn + ((long long)b * a.max_det + d) * 4;
#pragma unroll
        for (int k = 0; k < 4; ++k) o[k] = box[k];
      }
      const float area_d = __fmul_rn(__fsub_rn(box[2], box[0]), __fsub_rn(box[3], box[1]));
      const float cls = P[6];
      int best = -1;
      float best_iou = -1.f;
      for (int l = 0; l < nlab; ++l) {
        if (s_lab[l * 5] != cls) continue;
        const float iw = fmaxf(__fsub_rn(fminf(s_lab[l * 5 + 3], box[2]), fmaxf(s_lab[l * 5 + 1], box[0])), 0.f);
        const float ih = fmaxf(__fsub_rn(fminf(s_lab[l * 5 + 4], box[3]), fmaxf(s_lab[l * 5 + 2], box[1])), 0.f);
        const float inter = __fmul_rn(iw, ih);
        const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(s_area[l], area_d), inter));
        if (iou >= thr0 && iou > best_iou) {
          best_iou = iou;
          best = l;
        }
      }
      if (best >= 0) atomicMin(&s_win[best], d);
    }
  }
  __syncthreads();
  // ---- pass 2: correct[d, :] for the surviving (label, detection) pairs; the IoU is recomputed (same bits)
  for (int d0 = 0; d0 < a.max_det; d0 += VM_THREADS) {
    const int d = d0 + tid;
    if (d >= a.max_det) continue;
    unsigned char* out = a.correct + ((long long)b * a.max_det + d) * a.niou;
    float iou_keep = -1.f;
    if (d < nd) {
      const float* P = a.pred7 + ((long long)b * a.max_det + d) * 7;
      float poly[8], box[4];
      rbox_to_poly(P[0], P[1], P[2], P[3], P[4], poly);
#pragma unroll
      for (int k = 0; k < 8; k += 2) {
        poly[k] = __fmul_rn(__fsub_rn(poly[k], pad_x), inv_gain);
        poly[k + 1] = __fmul_rn(__fsub_rn(poly[k + 1], pad_y), inv_gain);
      }
      poly_to_xyxy(poly, box);
      const float area_d = __fmul_rn(__fsub_rn(box[2], box[0]), __fsub_rn(box[3], box[1]));
      const float cls = P[6];
      int best = -1;
      float best_iou = -1.f;
      for (int l = 0; l < nlab; ++l) {
        if (s_lab[l * 5] != cls) continue;
        const float iw = fmaxf(__fsub_rn(fminf(s_lab[l * 5 + 3], box[2]), fmaxf(s_lab[l * 5 + 1], box[0])), 0.f);
        const float ih = fmaxf(__fsub_rn(fminf(s_lab[l * 5 + 4], box[3]), fmaxf(s_lab[l * 5 + 2], box[1])), 0.f);
        const float inter = __fmul_rn(iw, ih);
        const float iou = __fdiv_rn(inter, __fsub_rn(__fadd_rn(s_area[l], area_d), inter));
        if (iou >= thr0 && iou > best_iou) {
          best_iou = iou;
          best = l;
        }
      }
      if (best >= 0 && s_win[best] == d) iou_keep = best_iou;
    }
    for (int k = 0; k < a.niou; ++k) out[k] = (iou_keep >= a.iouv[k]) ? 1 : 0;
  }
}

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

int y5obb_val_match_f32(const float* pred7, const int64_t* counts, int batch, int max_det, const float* labels7, int n_labels,
                        const float* scale5, const float* iouv, int niou, uint8_t* correct, float* polyn8, float* hbbn4,
                        int* overflow_flag, void* stream) {
  if (batch <= 0 || max_det <= 0 || n_labels < 0 || niou <= 0 || niou > 64) return Y5OBB_EINVAL;
  if (!pred7 || !counts || !scale5 || !iouv || !correct || !overflow_flag || (n_labels > 0 && !labels7)) return Y5OBB_EINVAL;
  VmArgs a;
  a.pred7 = pred7;
  a.counts = reinterpret_cast<const long long*>(counts);
  a.B = batch;
  a.max_det = max_det;
  a.labels = labels7;
  a.nl = n_labels;
  a.scale = scale5;
  a.iouv = iouv;
  a.niou = niou;
  a.correct = correct;
  a.polyn = polyn8;
  a.hbbn = hbbn4;
  a.overflow = overflow_flag;
  cudaStream_t st = (cudaStream_t)stream;
  Y5_CUDA(cudaMemsetAsync(overflow_flag, 0, sizeof(int), st));
  k_val_match<<<(unsigned)batch, VM_THREADS, 0, st>>>(a);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

}  // extern "C"
