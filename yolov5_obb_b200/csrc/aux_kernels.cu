// HBM-bound helpers around the conv stack (NHWC bf16):
//   y5obb_stem_s2d     NCHW fp32 image -> 2x2 space-to-depth NHWC bf16 [B, H/2, W/2, 16] (12 real + 4 zero
//                      channels), which turns the 6x6/s2/p2 stem conv (models/yolov5*.yaml layer 0,
//                      models/common.py:37-49) into a 3x3/s1/p1 conv with K = 9 x 16 that the tcgen05
//                      kernel runs with 32-byte swizzled tiles.
//   y5obb_sppf_pool    the three chained 5x5/s1/p2 max-pools of SPPF (models/common.py:181-196) in one
//                      pass: y1 = 5x5, y2 = 9x9, y3 = 13x13 windows of x (max-pool composition), written
//                      at channel offsets C, 2C, 3C of the same buffer (the torch.cat disappears).
//   y5obb_stem_s2d_scene_u8  the same layout pass for tiles cropped from a whole HWC BGR uint8 scene (channel flip, zero
//                      padding outside the scene and for invalid tiles), so a DOTA scene never goes through host crops.
// Algorithmic bytes: stem_s2d reads 12*H*W fp32 and writes H*W/4 * 32 B per image; stem_s2d_scene_u8 reads 3 B and writes
// 8 B per tile pixel; sppf_pool reads H*W*C*2 and writes 3x that.  All three are HBM-bound.
#include <cuda_bf16.h>

#include <algorithm>

#include "common.cuh"

namespace y5obb {
namespace {

// The pack-and-store tail of every stem layout pass: the 12 space-to-depth values of output pixel (row r = b * Ho + ho,
// column wo) plus 4 zero channels -> 16 bf16 (round to nearest), one 32-byte store.  Destination rows carry pad_cols zero
// pixels on each side (written once at allocation, never here).
__device__ __forceinline__ void s2d_store(float (&v)[16], __nv_bfloat16* __restrict__ out, long long r, int Wo, int wo,
                                          int pad_cols) {
  v[12] = v[13] = v[14] = v[15] = 0.f;
  uint4 o[2];
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(o);
#pragma unroll
  for (int e = 0; e < 8; ++e) h[e] = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
  uint4* dst = reinterpret_cast<uint4*>(out + ((r * (Wo + 2 * pad_cols)) + wo + pad_cols) * 16);
  dst[0] = o[0];
  dst[1] = o[1];
}

__global__ void k_stem_s2d(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                           int pad_cols) {
  const int Ho = H >> 1, Wo = W >> 1;
  const long long total = (long long)B * Ho * Wo;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int wo = (int)(i % Wo);
    const long long r = i / Wo;
    const int ho = (int)(r % Ho);
    const int b = (int)(r / Ho);
    float v[16];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* p = x + (((long long)b * 3 + c) * H + 2 * ho) * W + 2 * wo;
      const float2 top = *reinterpret_cast<const float2*>(p);
      const float2 bot = *reinterpret_cast<const float2*>(p + W);
      v[0 * 3 + c] = top.x;  // (dy=0, dx=0)
      v[1 * 3 + c] = top.y;  // (dy=0, dx=1)
      v[2 * 3 + c] = bot.x;  // (dy=1, dx=0)
      v[3 * 3 + c] = bot.y;  // (dy=1, dx=1)
    }
    s2d_store(v, out, r, Wo, wo, pad_cols);
  }
}

// uint8 NCHW image: the caller-side `imgs.float() / 255` (train.py:299, val.py:187-188, detect.py:108-109)
// folded into the same pass
__global__ void k_stem_s2d_u8(const uint8_t* __restrict__ x, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                              int pad_cols) {
  const int Ho = H >> 1, Wo = W >> 1;
  const long long total = (long long)B * Ho * Wo;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int wo = (int)(i % Wo);
    const long long r = i / Wo;
    const int ho = (int)(r % Ho);
    const int b = (int)(r / Ho);
    float v[16];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const uint8_t* p = x + (((long long)b * 3 + c) * H + 2 * ho) * W + 2 * wo;
      const uchar2 top = *reinterpret_cast<const uchar2*>(p);
      const uchar2 bot = *reinterpret_cast<const uchar2*>(p + W);
      v[0 * 3 + c] = (float)top.x / 255.0f;
      v[1 * 3 + c] = (float)top.y / 255.0f;
      v[2 * 3 + c] = (float)bot.x / 255.0f;
      v[3 * 3 + c] = (float)bot.y / 255.0f;
    }
    s2d_store(v, out, r, Wo, wo, pad_cols);
  }
}

// Whole-scene form (DOTA_devkit/ImgSplit_multi_process.py:122-132 saveimagepatches at rate 1, then the caller-side `/ 255`):
// tile b of the batch is the tile x tile window at origins[b] = (left, up) of an HWC BGR uint8 scene, as cv2.imread returns
// it; model channel c is scene channel 2 - c; pixels outside the scene (the devkit's zero padding at the bottom and right)
// and every tile b >= n_valid are zero.  Bit-identical to cropping on the host and running k_stem_s2d_u8.
__global__ void k_stem_s2d_scene_u8(const uint8_t* __restrict__ scene, int H, int W, const int* __restrict__ origins, int B,
                                    int n_valid, int tile, __nv_bfloat16* __restrict__ out, int pad_cols) {
  const int Ho = tile >> 1, Wo = tile >> 1;
  const long long total = (long long)B * Ho * Wo;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int wo = (int)(i % Wo);
    const long long r = i / Wo;
    const int ho = (int)(r % Ho);
    const int b = (int)(r / Ho);
    float v[16];
    const bool valid = b < n_valid;
    const int left = valid ? origins[2 * b] : 0, up = valid ? origins[2 * b + 1] : 0;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int y = up + 2 * ho + dy;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int x = left + 2 * wo + dx;
        const bool in = valid && y >= 0 && y < H && x >= 0 && x < W;
        const uint8_t* p = scene + ((long long)y * W + x) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) v[(dy * 2 + dx) * 3 + c] = (float)(in ? p[2 - c] : (uint8_t)0) / 255.0f;
      }
    }
    s2d_store(v, out, r, Wo, wo, pad_cols);
  }
}

__device__ __forceinline__ void vmax8(uint4& a, const uint4& b) {
  __nv_bfloat162* x = reinterpret_cast<__nv_bfloat162*>(&a);
  const __nv_bfloat162* y = reinterpret_cast<const __nv_bfloat162*>(&b);
#pragma unroll
  for (int i = 0; i < 4; ++i) x[i] = __hmax2(x[i], y[i]);
}

// One CTA = one image x 8 channels x one 32x32 spatial tile (+6 halo).  Separable: a horizontal pass builds the
// 5/9/13-wide row maxima in shared memory, a vertical pass the 5/9/13-tall column maxima of those (max-pool pads
// with -inf, so clipped windows are exact).  13 + 27 shared-memory reads per pixel instead of 169 global ones.
constexpr int PT = 32, PH = 6, PIN = PT + 2 * PH;
__global__ void __launch_bounds__(256) k_sppf_pool(__nv_bfloat16* __restrict__ buf, long long pix_stride, int B, int H,
                                                    int W, int C, int tiles_w, int tiles_h) {
  extern __shared__ __align__(16) uint4 sm[];
  uint4* in = sm;                       // [PIN][PIN]
  uint4* r5 = in + PIN * PIN;           // [PIN][PT]
  uint4* r9 = r5 + PIN * PT;
  uint4* r13 = r9 + PIN * PT;
  const int vec = C >> 3;
  int bid = blockIdx.x;
  const int cv = bid % vec;
  bid /= vec;
  const int tw = bid % tiles_w;
  bid /= tiles_w;
  const int th = bid % tiles_h;
  const int b = bid / tiles_h;
  const int h0 = th * PT, w0 = tw * PT;
  const uint4 ninf = make_uint4(0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u, 0xFF80FF80u);
  const __nv_bfloat16* base = buf + (long long)b * H * W * pix_stride + cv * 8;
  for (int i = threadIdx.x; i < PIN * PIN; i += 256) {
    const int y = i / PIN, x = i - y * PIN;
    const int hh = h0 + y - PH, ww = w0 + x - PH;
    uint4 v = ninf;
    if (hh >= 0 && hh < H && ww >= 0 && ww < W) v = *reinterpret_cast<const uint4*>(base + ((long long)hh * W + ww) * pix_stride);
    in[i] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < PIN * PT; i += 256) {
    const int y = i / PT, x = i - y * PT;
    const uint4* row = in + y * PIN + x + PH;
    uint4 a5 = row[0];
    vmax8(a5, row[-1]);
    vmax8(a5, row[1]);
    vmax8(a5, row[-2]);
    vmax8(a5, row[2]);
    uint4 a9 = a5;
    vmax8(a9, row[-3]);
    vmax8(a9, row[3]);
    vmax8(a9, row[-4]);
    vmax8(a9, row[4]);
    uint4 a13 = a9;
    vmax8(a13, row[-5]);
    vmax8(a13, row[5]);
    vmax8(a13, row[-6]);
    vmax8(a13, row[6]);
    r5[i] = a5;
    r9[i] = a9;
    r13[i] = a13;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < PT * PT; i += 256) {
    const int y = i / PT, x = i - y * PT;
    const int hh = h0 + y, ww = w0 + x;
    if (hh >= H || ww >= W) continue;
    const int c = (y + PH) * PT + x;
    uint4 m5 = r5[c];
    for (int d = 1; d <= 2; ++d) {
      vmax8(m5, r5[c - d * PT]);
      vmax8(m5, r5[c + d * PT]);
    }
    uint4 m9 = r9[c];
    for (int d = 1; d <= 4; ++d) {
      vmax8(m9, r9[c - d * PT]);
      vmax8(m9, r9[c + d * PT]);
    }
    uint4 m13 = r13[c];
    for (int d = 1; d <= 6; ++d) {
      vmax8(m13, r13[c - d * PT]);
      vmax8(m13, r13[c + d * PT]);
    }
    __nv_bfloat16* o = buf + (((long long)b * H + hh) * W + ww) * pix_stride + cv * 8;
    *reinterpret_cast<uint4*>(o + C) = m5;
    *reinterpret_cast<uint4*>(o + 2 * C) = m9;
    *reinterpret_cast<uint4*>(o + 3 * C) = m13;
  }
}

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

int y5obb_stem_s2d(const float* x_nchw, void* out_nhwc16, int B, int H, int W, int pad_cols, void* stream) {
  if (!x_nchw || !out_nhwc16 || B <= 0 || H <= 0 || W <= 0 || (H & 1) || (W & 1) || pad_cols < 0) return Y5OBB_EINVAL;
  if ((reinterpret_cast<uintptr_t>(x_nchw) & 7) || (reinterpret_cast<uintptr_t>(out_nhwc16) & 15)) return Y5OBB_EINVAL;
  const long long total = (long long)B * (H / 2) * (W / 2);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
  k_stem_s2d<<<grid, 256, 0, (cudaStream_t)stream>>>(x_nchw, static_cast<__nv_bfloat16*>(out_nhwc16), B, H, W, pad_cols);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_stem_s2d_u8(const uint8_t* x_nchw, void* out_nhwc16, int B, int H, int W, int pad_cols, void* stream) {
  if (!x_nchw || !out_nhwc16 || B <= 0 || H <= 0 || W <= 0 || (H & 1) || (W & 1) || pad_cols < 0) return Y5OBB_EINVAL;
  if ((reinterpret_cast<uintptr_t>(x_nchw) & 1) || (reinterpret_cast<uintptr_t>(out_nhwc16) & 15)) return Y5OBB_EINVAL;
  const long long total = (long long)B * (H / 2) * (W / 2);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
  k_stem_s2d_u8<<<grid, 256, 0, (cudaStream_t)stream>>>(x_nchw, static_cast<__nv_bfloat16*>(out_nhwc16), B, H, W, pad_cols);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_stem_s2d_scene_u8(const uint8_t* scene_hwc, int H, int W, const int32_t* origins2, int B, int n_valid, int tile,
                            void* out_nhwc16, int pad_cols, void* stream) {
  if (!scene_hwc || !out_nhwc16 || H <= 0 || W <= 0 || B <= 0 || n_valid < 0 || n_valid > B || tile <= 0 || (tile & 1) ||
      pad_cols < 0 || (n_valid > 0 && !origins2))
    return Y5OBB_EINVAL;
  if ((reinterpret_cast<uintptr_t>(origins2) & 7) || (reinterpret_cast<uintptr_t>(out_nhwc16) & 15)) return Y5OBB_EINVAL;
  const long long total = (long long)B * (tile / 2) * (tile / 2);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)sm_count() * 16);
  k_stem_s2d_scene_u8<<<grid, 256, 0, (cudaStream_t)stream>>>(scene_hwc, H, W, origins2, B, n_valid, tile,
                                                              static_cast<__nv_bfloat16*>(out_nhwc16), pad_cols);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

int y5obb_sppf_pool(void* buf, int64_t pix_stride, int B, int H, int W, int C, void* stream) {
  if (!buf || B <= 0 || H <= 0 || W <= 0 || C <= 0 || (C & 7) || (pix_stride & 7) || pix_stride < 4 * (int64_t)C)
    return Y5OBB_EINVAL;
  if (reinterpret_cast<uintptr_t>(buf) & 15) return Y5OBB_EINVAL;
  const int tiles_w = (W + PT - 1) / PT, tiles_h = (H + PT - 1) / PT;
  const long long grid = (long long)B * (C / 8) * tiles_w * tiles_h;
  if (grid > 0x7FFFFFFFll) return Y5OBB_EINVAL;
  const size_t smem = (size_t)(PIN * PIN + 3 * PIN * PT) * sizeof(uint4);
  static bool attr_set = false;
  if (!attr_set) {
    Y5_CUDA(cudaFuncSetAttribute(k_sppf_pool, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  k_sppf_pool<<<(unsigned)grid, 256, smem, (cudaStream_t)stream>>>(static_cast<__nv_bfloat16*>(buf), pix_stride, B, H, W,
                                                                  C, tiles_w, tiles_h);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

}  // extern "C"
