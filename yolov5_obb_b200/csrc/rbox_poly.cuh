// rbox2poly of one box, shared by every kernel that turns (cx, cy, l, s, theta) rows into corner polygons:
//   csrc/rbox_utils.cu k_rbox2poly, csrc/val_match.cu k_val_match, csrc/poly_nms.cu k_tiles_to_scene.
// /root/reference/utils/rboxs_utils.py:106-126 (torch branch): each arithmetic step is a separately rounded fp32 op (no FMA
// contraction), like the chain of ATen elementwise kernels it replaces.
#pragma once

namespace y5obb {

__device__ __forceinline__ void rbox_to_poly(float cx, float cy, float w, float h, float th, float* o) {
  const float c = cosf(th), s = sinf(th);
  const float w2 = __fdiv_rn(w, 2.0f), h2 = __fdiv_rn(h, 2.0f);
  const float v1x = __fmul_rn(w2, c), v1y = __fmul_rn(-w2, s);   // vector1 = (w/2 * Cos, -w/2 * Sin)
  const float v2x = __fmul_rn(-h2, s), v2y = __fmul_rn(-h2, c);  // vector2 = (-h/2 * Sin, -h/2 * Cos)
  o[0] = __fadd_rn(__fadd_rn(cx, v1x), v2x);  // point1 = center + vector1 + vector2
  o[1] = __fadd_rn(__fadd_rn(cy, v1y), v2y);
  o[2] = __fsub_rn(__fadd_rn(cx, v1x), v2x);  // point2 = center + vector1 - vector2
  o[3] = __fsub_rn(__fadd_rn(cy, v1y), v2y);
  o[4] = __fsub_rn(__fsub_rn(cx, v1x), v2x);  // point3 = center - vector1 - vector2
  o[5] = __fsub_rn(__fsub_rn(cy, v1y), v2y);
  o[6] = __fadd_rn(__fsub_rn(cx, v1x), v2x);  // point4 = center - vector1 + vector2
  o[7] = __fadd_rn(__fsub_rn(cy, v1y), v2y);
}

}  // namespace y5obb
