// Weight gradient of a convolution on the tensor cores (sm_100a): for every tap (kh, kw)
//   dW[tap][co][ci] = sum over (b, ho, wo) of dz[b, ho, wo, co] * x[b, s*ho + kh - ph, s*wo + kw - pw, ci]
// i.e. a GEMM with M = Cout, N = Cin and K = all output pixels.  Both operands are read straight from the NHWC bf16
// activations / gradients (channel slices allowed): a 4-D TMA box {64 channels, kwp, khp, 1} lands in shared memory
// as [64 pixels][128 B of channels], 128B-swizzled, which is the MN-major canonical layout of tcgen05.mma (the
// reduction axis K = pixel rows).  The tap is a shift of the x box's origin (zero padding = TMA out-of-bounds fill,
// stride 2 = tensor-map element strides on W and H, exactly as the forward kernel reads its input).  The pixel axis
// is split over CTAs (split-K); every CTA accumulates its slice in TMEM (fp32) and adds it into dW with fp32 atomics.
// Replaces the cuDNN wgrad call autograd makes for /root/reference/models/common.py:37-46 in train.py:333.
// Tensor-bound for wide layers (2 * pixels * Cout * Cin * taps flop), L2-bound for narrow ones.
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "ptx.cuh"

namespace y5obb {
namespace {

constexpr int WG_THREADS = 192;
constexpr int WG_MAX_STAGES = 8;
constexpr int WG_SMEM = 200 * 1024;
// a pixel block (= one TMA box per 64-channel chunk) has bk = 64, 128 or 256 pixels; a chunk is [bk pixels][128 B]

struct WgradK {
  CUtensorMap tmA;  // dz NHWC slice: (Cout, Wo, Ho, B), box {64, kwp, khp, 1}
  CUtensorMap tmB;  // x NHWC slice: (Cin, Wi, Hi, B), box {64, kwp*s, khp*s, 1}, element strides {1, s, s, 1}
  int B, Ho, Wo, Cout, Cin;
  int KH, KW, stride, pad_h, pad_w;
  int kwp, khp, BN;         // pixel block kwp x khp = bk pixels; N tile (input channels, multiple of 16)
  int bk;                   // pixels per block (64 / 128 / 256)
  uint32_t chunk;           // bk * 128 bytes
  int tiles_w, tiles_h;     // pixel blocks per image
  int nblocks;              // B * tiles_h * tiles_w
  int T, ngroups;           // taps handled by one CTA (they share the dz tile), tap groups
  int PB;                   // pixel blocks per pipeline stage
  int steps;                // ceil(nblocks / PB) pipeline steps over the whole pixel axis
  int ksplit, co_blks, ci_blks;
  int stages, a_chunks, b_chunks;
  uint32_t idesc, tmem_cols, stage_bytes;  // idesc without the N field (set per instruction)
  float* dW;                // element (tap, co, ci) at dW[tap * s_tap + row(co) * s_co + ci * s_ci]
  long long s_tap, s_co, s_ci;
  int co_group, co_group_pad;
};

// MN-major, 128B-swizzled operand: 64-channel chunks of [pixels][128 B]; 8-pixel groups 1024 B apart (SBO), chunks
// `chunk` bytes apart (LBO).  (cute/atom/mma_traits_sm100.hpp: Swizzle<3,4,3> o ((8,n),(8,k)):((1,LBO),(8,SBO)).)
__device__ __forceinline__ uint64_t make_mnmajor_desc(uint32_t smem_addr, uint32_t chunk) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(chunk >> 4) << 16;      // LBO
  d |= (uint64_t)(1024u >> 4) << 32;      // SBO
  d |= (uint64_t)1 << 46;                 // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                 // SWIZZLE_128B
  return d;
}

// One pipeline stage holds PB pixel blocks; per block: the dz tile (a_chunks chunks) followed by the x tiles of the T
// taps this CTA accumulates (b_chunks chunks each).  The taps' tiles are consecutive 64-channel chunks, i.e. ONE N axis
// of T * b_chunks * 64 columns: an instruction covers up to 4 chunks (N = 256), so the dz tile - which tcgen05.mma
// re-reads from shared memory for every instruction - is fetched once per 4 chunks, and one mbarrier round trip
// (~0.2 us) is amortised over the whole stage.
__global__ void __launch_bounds__(WG_THREADS, 1) wgrad_kernel(const __grid_constant__ WgradK p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[WG_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[WG_MAX_STAGES];
  __shared__ __align__(8) uint64_t done_bar;
  __shared__ uint32_t tmem_base_smem;
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t WG_CHUNK = p.chunk;
  const uint32_t a_bytes = (uint32_t)p.a_chunks * WG_CHUNK, b_bytes = (uint32_t)p.b_chunks * WG_CHUNK;
  const uint32_t blk_bytes = a_bytes + (uint32_t)p.T * b_bytes;

  // work item: (tap group, co block, ci block, k split)
  int item = blockIdx.x;
  const int ks = item % p.ksplit;
  item /= p.ksplit;
  const int cib = item % p.ci_blks;
  item /= p.ci_blks;
  const int cob = item % p.co_blks;
  const int grp = item / p.co_blks;
  const int tap0 = grp * p.T;
  const int ntap = min(p.T, p.KH * p.KW - tap0);
  const int s0 = (int)(((long long)p.steps * ks) / p.ksplit), s1 = (int)(((long long)p.steps * (ks + 1)) / p.ksplit);
  // 64-channel chunks of A this block really has (rows of D beyond Cout are never stored)
  const int a_chunks = min(p.a_chunks, (p.Cout - cob * 128 + 63) >> 6);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&p.tmA);
    ptx::prefetch_tmap(&p.tmB);
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(&done_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&tmem_base_smem, p.tmem_cols);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  const int per_img = p.tiles_h * p.tiles_w;

  if (warp == 0) {
    // elect.sync, not `lane == 0`: ptxas then issues UTMALDG / UTCHMMA straight from uniform registers instead of wrapping each
    // one in a per-lane serialisation loop (see conv_sm100.cu)
    if (ptx::elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t tx = (uint32_t)p.PB * (uint32_t)(a_chunks + ntap * p.b_chunks) * WG_CHUNK;
      for (int st = s0; st < s1; ++st) {
        ptx::mbar_wait(&empty_bar[s], ph ^ 1u);
        uint8_t* sbase = smem + (size_t)s * p.stage_bytes;
        ptx::mbar_expect_tx(&full_bar[s], tx);
        for (int pb = 0; pb < p.PB; ++pb) {
          const int k = st * p.PB + pb;        // pixel block; blocks past the end decode to b >= B: all zero fill
          const int b = k / per_img;
          const int r = k - b * per_img;
          const int th = r / p.tiles_w;
          const int ho0 = th * p.khp, wo0 = (r - th * p.tiles_w) * p.kwp;
          uint8_t* sa = sbase + (size_t)pb * blk_bytes;
          for (int c = 0; c < a_chunks; ++c)
            ptx::tma_load_4d(sa + (size_t)c * WG_CHUNK, &p.tmA, &full_bar[s], cob * 128 + c * 64, wo0, ho0, b);
          for (int t = 0; t < ntap; ++t) {
            const int tap = tap0 + t;
            const int kh = tap / p.KW, kw = tap - kh * p.KW;
            const int wi0 = wo0 * p.stride + kw - p.pad_w, hi0 = ho0 * p.stride + kh - p.pad_h;
            uint8_t* sb = sa + a_bytes + (size_t)t * b_bytes;
            for (int c = 0; c < p.b_chunks; ++c)
              ptx::tma_load_4d(sb + (size_t)c * WG_CHUNK, &p.tmB, &full_bar[s], cib * p.BN + c * 64, wi0, hi0, b);
          }
        }
        if (++s == p.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    if (ptx::elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      const uint64_t desc_hi = make_mnmajor_desc(0u, WG_CHUNK);
      const int nk = p.bk >> 4;
      const uint32_t ring = ptx::smem_u32(smem);
      uint32_t started = 0u;  // bit g: accumulator group g holds a partial sum already
      const int nchunks = ntap * p.b_chunks;  // the taps' x tiles are consecutive 64-channel chunks: ONE N axis
      for (int st = s0; st < s1; ++st) {
        ptx::mbar_wait(&full_bar[s], ph);
        ptx::tc_fence_after();
        for (int pb = 0; pb < p.PB; ++pb) {
          const uint32_t sa = ring + (uint32_t)s * p.stage_bytes + (uint32_t)pb * blk_bytes;
          const uint64_t da = desc_hi | (uint64_t)((sa & 0x3FFFFu) >> 4);
          // up to 4 chunks (N = 256) per instruction: the dz tile (A) is fetched once for all of them
          for (int c0 = 0, g = 0; c0 < nchunks; c0 += 4, ++g) {
            const int nn = min(4, nchunks - c0);
            const uint32_t sb = sa + a_bytes + (uint32_t)c0 * WG_CHUNK;
            const uint64_t db = desc_hi | (uint64_t)((sb & 0x3FFFFu) >> 4);
            const uint32_t d_tmem = tmem_base + (uint32_t)(c0 * 64);
            const uint32_t idesc = p.idesc | ((uint32_t)(nn * 8) << 17);
            uint32_t accumulate = (started >> g) & 1u;
#pragma unroll 4
            for (int j = 0; j < nk; ++j) {  // 16 pixel rows = 2048 B per MMA
              ptx::umma_bf16(d_tmem, da + (uint64_t)(128 * j), db + (uint64_t)(128 * j), idesc, accumulate);
              accumulate = 1u;
            }
            started |= 1u << g;
          }
        }
        ptx::umma_commit(&empty_bar[s]);
        if (++s == p.stages) {
          s = 0;
          ph ^= 1u;
        }
      }
      ptx::umma_commit(&done_bar);
    }
  } else {
    // epilogue: TMEM lane = output channel (row of dW), columns = tap-major, then input channels
    const int q = warp & 3;
    const int co = cob * 128 + q * 32 + lane;
    int co_row = co;
    bool co_ok = co < p.Cout;
    if (p.co_group_pad) {
      const int a = co / p.co_group_pad, c = co - a * p.co_group_pad;
      co_ok = co_ok && c < p.co_group;
      co_row = a * p.co_group + c;
    }
    if (s1 > s0) {
      ptx::mbar_wait(&done_bar, 0u);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
      const int ncols = min(p.BN, p.Cin - cib * p.BN);
      if (cob * 128 + q * 32 < p.Cout) {  // warp-uniform
        for (int t = 0; t < ntap; ++t) {
          float* row = p.dW + (long long)(tap0 + t) * p.s_tap + (long long)co_row * p.s_co + (long long)(cib * p.BN) * p.s_ci;
          for (int c0 = 0; c0 < ncols; c0 += 16) {  // chunk (c0 / 64) of tap t starts at TMEM column (t * b_chunks) * 64
            uint32_t r[16];
            ptx::tmem_ld_32x32b_x16(taddr + (uint32_t)(t * p.b_chunks * 64 + c0), r);
            ptx::tmem_ld_wait();
            if (co_ok) {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (c0 + j < ncols) atomicAdd(row + (long long)(c0 + j) * p.s_ci, __uint_as_float(r[j]));
            }
          }
        }
      }
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, p.tmem_cols);
  }
}

typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
PFN_tmapEncodeTiled wg_get_encode() {
  static PFN_tmapEncodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  });
  return fn;
}

struct WgradObj {
  WgradK k;
  int grid;
  size_t smem;
  double flops;
};

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

int y5obb_wgrad_create(const y5obb_wgrad_desc* d, y5obb_wgrad_t** out) {
  if (!d || !out || !d->dz || !d->x || !d->dw) return Y5OBB_EINVAL;
  if (d->stride != 1 && d->stride != 2) return Y5OBB_EINVAL;
  if (d->B < 1 || d->Cout < 1 || d->Cin < 1 || d->KH < 1 || d->KW < 1 || d->Ho < 1 || d->Wo < 1) return Y5OBB_EINVAL;
  if ((d->dz_pix_stride & 7) || (d->x_pix_stride & 7) || (d->x_row_stride & 7) || (d->x_img_stride & 7) ||
      d->dz_pix_stride < d->Cout)
    return Y5OBB_EINVAL;
  if ((d->x_row_stride == 0) != (d->x_img_stride == 0)) return Y5OBB_EINVAL;
  if (!d->x_row_stride && d->x_pix_stride < d->Cin) return Y5OBB_EINVAL;  // overlapping windows need explicit strides
  if ((reinterpret_cast<uintptr_t>(d->dz) | reinterpret_cast<uintptr_t>(d->x)) & 15) return Y5OBB_EINVAL;
  PFN_tmapEncodeTiled enc = wg_get_encode();
  if (!enc) return Y5OBB_ECUDA;
  WgradObj* o = new WgradObj();
  WgradK& k = o->k;
  memset(&k, 0, sizeof(k));
  k.B = d->B;
  k.Ho = d->Ho;
  k.Wo = d->Wo;
  k.Cout = d->Cout;
  k.Cin = d->Cin;
  k.KH = d->KH;
  k.KW = d->KW;
  k.stride = d->stride;
  k.pad_h = d->pad_h;
  k.pad_w = d->pad_w;
  k.dW = d->dw;
  if (d->dw_tap_stride || d->dw_co_stride || d->dw_ci_stride) {
    k.s_tap = d->dw_tap_stride;
    k.s_co = d->dw_co_stride;
    k.s_ci = d->dw_ci_stride;
  } else {
    k.s_tap = (long long)d->Cout * d->Cin;
    k.s_co = d->Cin;
    k.s_ci = 1;
  }
  if (d->co_group_pad < 0 || d->co_group < 0 || d->co_group > d->co_group_pad) {
    delete o;
    return Y5OBB_EINVAL;
  }
  k.co_group = d->co_group;
  k.co_group_pad = d->co_group_pad;
  k.ci_blks = (d->Cin + 255) / 256;
  k.BN = ((d->Cin + k.ci_blks - 1) / k.ci_blks + 15) / 16 * 16;
  k.b_chunks = (k.BN + 63) / 64;
  k.co_blks = (d->Cout + 127) / 128;
  k.a_chunks = d->Cout > 64 ? 2 : 1;
  const int ntaps = d->KH * d->KW;
  // Block size bk (pixels per TMA box) and taps per CTA T.  Every cp.async.bulk.tensor instruction costs the TMA unit a
  // few hundred cycles whatever its size: measured on B200, 64-pixel boxes deliver ~12 B/clk/SM and 128-pixel boxes
  // 1.3-1.8x that (48->48 3x3 at 256^2: 189 -> 106 us; 192->192 3x3 at 64^2: 80 -> 51 us), while trading taps per CTA for
  // 256-pixel boxes loses again (the dz tile is re-read once per tap group).  So: 128-pixel blocks, as many taps per CTA
  // as fit two pipeline stages and the 8 TMEM chunk slots.
  const long long npx = (long long)d->B * d->Ho * d->Wo;
  int best_bk = npx >= 512 ? 128 : 64;
  int best_T = std::min(ntaps, 8 / k.b_chunks);
  while (best_T > 1 && (uint32_t)(k.a_chunks + best_T * k.b_chunks) * (uint32_t)best_bk * 128 > WG_SMEM / 2) --best_T;
  if ((uint32_t)(k.a_chunks + best_T * k.b_chunks) * (uint32_t)best_bk * 128 > WG_SMEM / 2) best_bk = 64;
  k.bk = best_bk;
  k.chunk = (uint32_t)best_bk * 128;
  // pixel block kwp x khp = bk output pixels: the shape that covers the map with the fewest blocks (ties: widest rows)
  long long best = -1;
  for (int kwp = 1; kwp <= std::min(k.bk, 256); kwp <<= 1) {
    const int khp = k.bk / kwp;
    if (khp * d->stride > 256 || kwp * d->stride > 256) continue;  // TMA box extents (input pixels) are at most 256
    const long long cost = (long long)((d->Wo + kwp - 1) / kwp) * ((d->Ho + khp - 1) / khp);
    if (best < 0 || cost <= best) {
      best = cost;
      k.kwp = kwp;
      k.khp = khp;
    }
  }
  k.tiles_w = (d->Wo + k.kwp - 1) / k.kwp;
  k.tiles_h = (d->Ho + k.khp - 1) / k.khp;
  k.nblocks = d->B * k.tiles_w * k.tiles_h;
  const uint32_t a_bytes = (uint32_t)k.a_chunks * k.chunk, b_bytes = (uint32_t)k.b_chunks * k.chunk;
  k.ngroups = (ntaps + best_T - 1) / best_T;
  k.T = (ntaps + k.ngroups - 1) / k.ngroups;  // balanced groups
  const uint32_t blk_bytes = a_bytes + (uint32_t)k.T * b_bytes;
  if (blk_bytes > WG_SMEM / 2) {
    delete o;
    return Y5OBB_EINVAL;
  }
  k.PB = 1;
  k.stage_bytes = blk_bytes;
  k.stages = (int)std::min<size_t>(WG_MAX_STAGES, WG_SMEM / k.stage_bytes);
  k.steps = k.nblocks;
  k.tmem_cols = 64;
  while (k.tmem_cols < (uint32_t)(k.T * k.b_chunks * 64)) k.tmem_cols <<= 1;
  const int items = k.ngroups * k.co_blks * k.ci_blks;
  {  // split-K: minimise (waves) x (steps per CTA + the fixed cost of a CTA: TMEM alloc, pipeline fill, fp32 atomic
     // epilogue - about 512 pixels' worth of pipeline steps); 1 CTA per SM
    const int sms = sm_count();  // CTAs in flight
    const int fixed = std::max(1, 512 / k.bk);
    long long best_cost2 = -1;
    int bestk = 1;
    for (int ksp = 1; ksp <= std::min(k.steps, 4 * sms); ++ksp) {
      const long long waves = ((long long)items * ksp + sms - 1) / sms;
      const long long cost = waves * ((k.steps + ksp - 1) / ksp + fixed);
      if (best_cost2 < 0 || cost < best_cost2) {
        best_cost2 = cost;
        bestk = ksp;
      }
    }
    k.ksplit = bestk;
  }
  k.idesc = ptx::make_idesc_bf16(128, 0) | (1u << 15) | (1u << 16);  // A and B MN-major; N is set per instruction
  {
    cuuint64_t dims[4] = {(cuuint64_t)d->Cout, (cuuint64_t)d->Wo, (cuuint64_t)d->Ho, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->dz_pix_stride * 2, (cuuint64_t)d->dz_pix_stride * d->Wo * 2,
                             (cuuint64_t)d->dz_pix_stride * d->Wo * d->Ho * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)k.kwp, (cuuint32_t)k.khp, 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&k.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(d->dz), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  {
    const cuuint32_t s = (cuuint32_t)d->stride;
    cuuint64_t dims[4] = {(cuuint64_t)d->Cin, (cuuint64_t)d->Wi, (cuuint64_t)d->Hi, (cuuint64_t)d->B};
    const cuuint64_t row = d->x_row_stride ? (cuuint64_t)d->x_row_stride : (cuuint64_t)d->x_pix_stride * d->Wi;
    const cuuint64_t img = d->x_img_stride ? (cuuint64_t)d->x_img_stride : row * d->Hi;
    cuuint64_t strides[3] = {(cuuint64_t)d->x_pix_stride * 2, row * 2, img * 2};
    cuuint32_t box[4] = {64, (cuuint32_t)k.kwp * s, (cuuint32_t)k.khp * s, 1};
    cuuint32_t es[4] = {1, s, s, 1};
    CUresult r = enc(&k.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(d->x), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  o->grid = items * k.ksplit;
  o->smem = std::max<size_t>((size_t)k.stages * k.stage_bytes + 1024, 116 * 1024);  // one CTA per SM: it may own all 512 TMEM columns
  o->flops = 2.0 * d->B * d->Ho * d->Wo * (double)d->Cout * d->Cin * d->KH * d->KW;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, WG_SMEM + 2048);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(wgrad_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e != cudaSuccess) {
      delete o;
      return cuda_fail(e);
    }
    attr_set = true;
  }
  *out = reinterpret_cast<y5obb_wgrad_t*>(o);
  return Y5OBB_OK;
}

int y5obb_wgrad_run(const y5obb_wgrad_t* w, void* stream) {
  if (!w) return Y5OBB_EINVAL;
  const WgradObj* o = reinterpret_cast<const WgradObj*>(w);
  wgrad_kernel<<<o->grid, WG_THREADS, o->smem, (cudaStream_t)stream>>>(o->k);
  Y5_LAUNCH_CHECK();
  return Y5OBB_OK;
}

void y5obb_wgrad_destroy(y5obb_wgrad_t* w) { delete reinterpret_cast<WgradObj*>(w); }

}  // extern "C"
