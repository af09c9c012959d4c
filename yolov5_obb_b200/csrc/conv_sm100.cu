// Implicit-GEMM NHWC bf16 convolution for sm_100a: TMA -> shared memory -> tcgen05.mma -> TMEM ->
// fused epilogue (folded-BN bias, SiLU, residual add, concat-offset store, 2x nearest up-sample copy,
// or the Detect head's permute + sigmoid + grid/anchor decode).
//
// Replaces, for the layers of models/yolov5{n,s,m,l,x}.yaml, the cuDNN/ATen calls behind
//   /root/reference/models/common.py:37-49   (Conv.forward_fuse: conv + bias + SiLU)
//   /root/reference/models/common.py:94-104  (Bottleneck: x + cv2(cv1(x)))   -> residual epilogue
//   /root/reference/models/common.py:267-274 (Concat)                          -> channel-offset store
//   /root/reference/models/yolo.py:49-81     (Detect: 1x1 conv, view/permute, sigmoid, decode)
//
// GEMM view: D[128 output pixels, BN channels] = sum over (tap, 64-channel chunk) A_tap[128, BK] * W_tap[BN, BK]^T
//   A tile  = one 4-D TMA box {BK ch, Wt, Ht, 1} of the NHWC input at the tap's shifted origin; zero
//             padding, ragged channel counts and ragged image edges are TMA out-of-bounds zero fill;
//             stride-2 convs use the tensor map's element strides.
//   W tile  = 2-D TMA box {BK, BN} of weights packed [tap][Cout_pad][Cin_pad] (K-major).
//   Both land in 32/64/128-byte swizzled K-major layouts that tcgen05.mma consumes directly.
// One persistent CTA per SM, 10 warps: TMA producer, MMA issuer (+TMEM owner), 8 epilogue warps;
// up to 8 TMEM accumulator stages so the epilogue of tile i overlaps the MMAs of the tiles after it.
//
// Roofline: tensor pipe for the wide layers (2*128*BN*K flop per tile), HBM for the narrow ones
// (algorithmic bytes = input pixels*Cin*2 + output pixels*Cout*2 [+ residual] per image).
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"
#include "ptx.cuh"

namespace y5obb {
namespace {

constexpr int BM = 128;  // output pixels per tile == TMEM lanes
constexpr int MAX_STAGES = 16;
constexpr int MAX_ACC = 8;                // TMEM accumulator stages: 512 columns / accumulator stride
constexpr int NUM_THREADS = 320;          // TMA producer, MMA issuer, 8 epilogue warps
constexpr int EPI_WARPS = 8;
constexpr int TMEM_COLS = 512;            // the CTA owns all of the SM's tensor memory
// Staging buffers per epilogue warp, used alternately: in-kernel stamps show ~100 cycles between "accumulator loaded" and
// "staging buffer free" with two, i.e. the TMA stores are not what the epilogue waits for (four measured slower: they cost
// operand-ring depth)
constexpr int EPI_BUFS = 2;
constexpr int EPI_STAGE_CONV = 32 * 64;    // 32 pixels x 32 bf16 channels, 64-byte swizzled
constexpr int EPI_STAGE_DET = 32 * 128;    // 32 pixels x 32 fp32 outputs, 128-byte swizzled
constexpr int SMEM_TOTAL = 224 * 1024;    // dynamic shared memory we ask for at most (227 KB is the hardware cap)

enum Mode : int { MODE_CONV = 0, MODE_DETECT = 1 };

// division by a launch-time constant without the ~100-cycle integer divide (x < 2^31): q = (umulhi(x, m) + x) >> s
struct FastDiv {
  uint32_t d, m, s;
};
inline FastDiv make_fastdiv(uint32_t d) {
  FastDiv f;
  f.d = d;
  uint32_t s = 0;
  while ((1u << s) < d) ++s;
  f.s = s;
  f.m = (uint32_t)((((uint64_t)1 << 32) * (((uint64_t)1 << s) - d)) / d + 1);
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t x, const FastDiv& f) { return (__umulhi(x, f.m) + x) >> f.s; }

struct ConvK {
  CUtensorMap tmA;
  CUtensorMap tmB;
  CUtensorMap tmO;  // output slice, box {32 ch, min(Wt,32), 32/min(Wt,32), 1}, 64-byte swizzle (MODE_CONV)
  CUtensorMap tmU;  // the 2x nearest up-sampled copy viewed as (C, dx, W, dy, B*H): the staged tile is stored four times
  int up_tma;       // 1: up-sampled copy through tmU (needs Hout % tile height == 0: B and H share a dimension); 0: per-thread stores
  // geometry
  int B, Hout, Wout;
  int Wt, Ht, tiles_w, tiles_h;
  int n_tiles_m, n_tiles_n;
  FastDiv fd_ntn, fd_per_img, fd_tiles_w, fd_wt;
  int BN, BK;
  int Cout, cout_pad;
  int Cin, kchunks, KH, KW, stride, pad_h, pad_w;
  int stages;
  int n_acc, acc_shift, acc_stride;  // TMEM accumulator stages (power of two), log2, columns between them
  int m_sub;           // 128-pixel sub-tiles per tile (1, 2 or 4), stacked along H: one barrier round trip, one weight
                       // load and one epilogue hand-over serve m_sub * 128 pixels (sub-tile m: accumulator columns
                       // [m * sub_cols, ...), A rows [m * 128, (m + 1) * 128) of the stage)
  int sub_cols;        // TMEM columns per sub-tile accumulator (acc_stride = m_sub * sub_cols)
  uint32_t a_sub16;    // (128 rows * row bytes) >> 4: descriptor distance between the sub-tiles' A rows
  int pairw;           // 1: stride-2 conv whose input is viewed as horizontal pixel PAIRS (2*pix_stride channels per
                       // position): the column phase of a tap is a channel offset, so TMA reads contiguous rows
  int in_pix_stride;
  int res_red;         // 1: the residual IS the output buffer (in-place Bottleneck add) and the tile leaves as a TMA reduce-add: no
                       // residual loads in the epilogue (the kernel then runs its no-residual flavour)
  int epi_tile_split;  // 1: epilogue warp group g handles the tiles whose accumulator is g (all columns); 0: both
                       // groups work on every tile and split its columns (few tiles per CTA)
  int rowshift;    // 1: one A stage holds Ht + KH - 1 image rows; the KH taps of a column read it at row offsets
  int b_resident;  // 1: every weight tile stays in shared memory for the whole kernel (loaded once)
  int b_per_stage; // weight tiles streamed with each A unit (0 when resident)
  int group;       // (tap, K-chunk) units per pipeline stage: one mbarrier round trip serves `group` TMA boxes
  int n_units;     // units per tile = (rowshift ? KW : KH*KW) * kchunks
  uint32_t a_bytes, a_tx_bytes, b_bytes, b_stage_bytes, b_res_bytes, row_shift_bytes, epi_stage_bytes;
  uint32_t idesc;
  // epilogue
  int mode, act;
  const float* bias;
  __nv_bfloat16* out;
  long long out_pix_stride;
  const __nv_bfloat16* res;
  long long res_pix_stride, res_row_stride, res_img_stride;
  __nv_bfloat16* out2x;
  long long out2x_pix_stride;
  // detect
  float* det_out;
  long long det_rows_per_image, det_row_off;
  int det_no, det_decode;  // det_decode: 0 raw logits, 1 sigmoid + grid/anchor decode, 2 = 1 as compact records (see the epilogue)
  int det_rec_w;           // floats per compact record: (5 + nc + 1) rounded up to 4
  float det_stride;
  float det_anchor[6];
  unsigned long long* ts;  // debug: clock64 stamps of CTA ts_cta, [role 3][tile & 31][slot 8] (y5obb_conv_debug_timestamps):
  int ts_cta;              // the LAST 32 tiles of that CTA survive; slot 7 holds the tile's ordinal + 1
};

#define Y5_TS(role, it, slot)                                                                  \
  do {                                                                                         \
    if (p.ts && (int)blockIdx.x == p.ts_cta) {                                                 \
      p.ts[((role)*32 + ((it) & 31)) * 8 + (slot)] = clock64();                                \
      p.ts[((role)*32 + ((it) & 31)) * 8 + 7] = (unsigned long long)(it) + 1ull;               \
    }                                                                                          \
  } while (0)

struct TileCoord {
  int b, h0, w0, n0, nt;
};

__device__ __forceinline__ TileCoord decode_tile(const ConvK& p, int t) {
  TileCoord c;
  const int mt = (int)fdiv((uint32_t)t, p.fd_ntn);
  c.nt = t - mt * p.n_tiles_n;
  const int per_img = p.tiles_h * p.tiles_w;
  c.b = (int)fdiv((uint32_t)mt, p.fd_per_img);
  const int r = mt - c.b * per_img;
  const int th = (int)fdiv((uint32_t)r, p.fd_tiles_w);
  c.h0 = th * p.Ht * p.m_sub;
  c.w0 = (r - th * p.tiles_w) * p.Wt;
  c.n0 = c.nt * p.BN;
  return c;
}

// x * sigmoid(x) = h + h * tanh(h), h = x / 2: one MUFU op (tanh.approx, rel. error ~2^-11) instead of ex2 + rcp
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float sigmoid_fast(float v) { return fmaf(0.5f, tanh_fast(0.5f * v), 0.5f); }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}



// One (tap, K-chunk) unit: KSUB vertical taps x NK sub-blocks of 16 channels, fully unrolled
template <int KSUB, int NK>
__device__ __forceinline__ void issue_unit(uint32_t d_tmem, uint64_t da0, uint64_t db0, uint32_t a_step, uint32_t b_step,
                                           uint32_t idesc, uint32_t accumulate) {
#pragma unroll
  for (int u = 0; u < KSUB; ++u) {
#pragma unroll
    for (int j = 0; j < NK; ++j) {
      ptx::umma_bf16(d_tmem, da0 + (uint64_t)(u * a_step + 2 * j), db0 + (uint64_t)(u * b_step + 2 * j), idesc,
                     (u | j) ? 1u : accumulate);
    }
  }
}

// The same with the descriptors' low words (address >> 4 | LBO) advanced by 32-bit adds and the constant high word attached by a
// register-pair move: no 64-bit arithmetic between the MMAs (the issuing thread is instruction bound: ncu source view, r2)
__device__ __forceinline__ uint64_t desc_from(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm volatile("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}
template <int KSUB, int NK>
__device__ __forceinline__ void issue_unit_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t a_step, uint32_t b_step,
                                              uint32_t idesc, uint32_t accumulate) {
#pragma unroll
  for (int u = 0; u < KSUB; ++u) {
#pragma unroll
    for (int j = 0; j < NK; ++j) {
      ptx::umma_bf16(d_tmem, desc_from(a_lo + (uint32_t)u * a_step + 2u * j, hi), desc_from(b_lo + (uint32_t)u * b_step + 2u * j, hi), idesc,
                     (u | j) ? 1u : accumulate);
    }
  }
}

struct MmaCtx {
  uint64_t *full_bar, *empty_bar, *tmem_full, *tmem_empty;
  uint32_t tmem_base, ring_lo, res_lo, hi;  // descriptor low words of the operand ring / the resident weights, common high word
  uint32_t stage16, unit16;                 // pipeline stage / unit size in 16-byte units
  int total_tiles, ksub;
};

// The MMA issuer's whole tile loop, specialised on the unit shape (KSUB vertical taps x NK 16-channel sub-blocks of a full K
// chunk; 0, 0 = any shape through runtime loops).  Everything loop invariant sits in registers, the ring position and the resident
// weight tile advance incrementally, and the ragged last K chunk (Cin not a multiple of BK) takes the runtime loop.
template <int KSUB, int NK>
__device__ __forceinline__ void mma_role(const ConvK& p, const MmaCtx& x) {
  const uint32_t a_step = p.row_shift_bytes >> 4;  // per vertical tap: one image row of the tile ...
  const uint32_t bst16 = p.b_stage_bytes >> 4;
  const uint32_t b_step = p.b_resident ? (uint32_t)(p.KW * p.kchunks) * bst16 : bst16;  // ... and KW weight tiles (resident) or one
  const uint32_t a_bytes16 = p.a_bytes >> 4, a_sub16 = p.a_sub16, idesc = p.idesc, hi = x.hi;
  const int n_units = p.n_units, group = p.group, kchunks = p.kchunks, m_sub = p.m_sub, sub_cols = p.sub_cols, stages = p.stages;
  const int nk_last = ((p.Cin - (kchunks - 1) * p.BK) + 15) >> 4;  // MMAs per tap of the last (possibly ragged) K chunk
  const bool resident = p.b_resident != 0;
  int s = 0, it = 0;
  uint32_t ph = 0, s_lo = x.ring_lo;
  for (int t = blockIdx.x; t < x.total_tiles; t += gridDim.x, ++it) {
    const int acc = it & (p.n_acc - 1);
    const uint32_t acc_ph = (uint32_t)(it >> p.acc_shift) & 1u;
    Y5_TS(1, it, 0);
    ptx::mbar_wait(&x.tmem_empty[acc], acc_ph ^ 1u);
    ptx::tc_fence_after();
    Y5_TS(1, it, 1);
    const uint32_t d_tmem = x.tmem_base + (uint32_t)(acc * p.acc_stride);
    uint32_t accumulate = 0u, bres_lo = x.res_lo;
    int kc = 0;
    for (int u0 = 0; u0 < n_units; u0 += group) {
      const int ng = min(group, n_units - u0);
      ptx::mbar_wait(&x.full_bar[s], ph);
      // tcgen05.fence::after_thread_sync orders the MMAs below after this wait (leaving it out measured no faster)
      ptx::tc_fence_after();
      if (u0 == 0) Y5_TS(1, it, 2);
      uint32_t a_lo = s_lo;
      for (int g = 0; g < ng; ++g) {
        const uint32_t b_lo = resident ? bres_lo : a_lo + a_bytes16;
        const bool last = kc + 1 == kchunks;
        if (NK > 0 && (!last || nk_last == NK)) {
          for (int m = 0; m < m_sub; ++m)  // the m_sub sub-tiles of the tile share this unit's weights
            issue_unit_lo<KSUB, NK>(d_tmem + (uint32_t)(m * sub_cols), a_lo + (uint32_t)m * a_sub16, b_lo, hi, a_step, b_step, idesc, accumulate);
        } else {
          const int nk = last ? nk_last : (p.BK >> 4);
          for (int m = 0; m < m_sub; ++m) {
            uint32_t acc_m = accumulate;
            for (int u = 0; u < x.ksub; ++u)
              for (int j = 0; j < nk; ++j) {
                ptx::umma_bf16(d_tmem + (uint32_t)(m * sub_cols), desc_from(a_lo + (uint32_t)m * a_sub16 + (uint32_t)u * a_step + 2u * j, hi),
                               desc_from(b_lo + (uint32_t)u * b_step + 2u * j, hi), idesc, acc_m);
                acc_m = 1u;
              }
          }
        }
        accumulate = 1u;
        a_lo += x.unit16;
        bres_lo += bst16;
        kc = last ? 0 : kc + 1;
      }
      ptx::umma_commit(&x.empty_bar[s]);
      s_lo += x.stage16;
      if (++s == stages) {
        s = 0;
        ph ^= 1u;
        s_lo = x.ring_lo;
      }
    }
    Y5_TS(1, it, 3);
    ptx::umma_commit(&x.tmem_full[acc]);
    Y5_TS(1, it, 4);
  }
}

// ---- epilogue of one MODE_CONV tile for one warp -----------------------------------------------------
struct EpiTile {
  uint32_t taddr;     // TMEM address of this warp's lane quarter, column 0 of the accumulator
  uint8_t* stage;     // two swizzled staging buffers of this warp
  uint32_t stage_bytes;
  uint32_t swz;       // (lane >> 1) & 3
  int lane;
  bool leader;        // the warp's elected thread (elect.sync once per kernel): issues and tracks the TMA stores
  uint32_t bias;      // shared-memory address of the bias (+ n0); holds 0.5 * bias when the layer has SiLU (Y5OBB_CONV_BIAS_HALVED)
  const __nv_bfloat16* rrow;  // residual row of this thread's pixel (+ n0) or null
  const __nv_bfloat16* rrow_next;  // the same for the tile's next sub-tile (null after the last): its first chunk is fetched one step ahead
  __nv_bfloat16* urow;        // up-sampled destination of this thread's pixel (+ n0) or null
  long long up_pix, up_row;
  int nvalid, col_first, col_step;
  const CUtensorMap* tm;
  int cn0, cw, chh, cb;
  const CUtensorMap* tmu;  // up-sampled copy by TMA (null: per-thread stores through urow)
  int ubh;                 // cb * Hout + chh
  unsigned long long* ts;  // debug stamps of this tile's first chunk (slots 4..6 of the epilogue row) or null
  bool red;                // the staged tile is ADDED to the destination (in-place residual) instead of stored
};

// rvn: this thread's residual values of the NEXT chunk to be processed (16-byte loads issued one chunk ahead - across
// sub-tiles too, and for a tile's first chunk before the wait on its accumulator - so the L2 / HBM latency of the residual
// (~1-3k cycles per chunk in the in-kernel timelines) is off the epilogue's critical path)
template <bool ACT, bool RES, bool UP>
__device__ __forceinline__ void conv_epi_tile(const EpiTile& e, int& sbuf, uint4 (&rvn)[4]) {
  for (int c0 = e.col_first; c0 < e.nvalid; c0 += e.col_step) {
    uint32_t r[32];
    if (e.ts && c0 == e.col_first) e.ts[4] = clock64();
    ptx::tmem_ld_32x32b_x32(e.taddr + (uint32_t)c0, r);
    uint4 rv[4];
    if (RES) {
#pragma unroll
      for (int g = 0; g < 4; ++g) rv[g] = rvn[g];
      const int cn = c0 + e.col_step;
      const bool same = cn < e.nvalid;
      const __nv_bfloat16* nx = same ? e.rrow : e.rrow_next;
      const int cc = same ? cn : e.col_first;
#pragma unroll
      for (int g = 0; g < 4; ++g)
        rvn[g] = (nx && cc + g * 8 < e.nvalid) ? *reinterpret_cast<const uint4*>(nx + cc + g * 8) : make_uint4(0, 0, 0, 0);
    }
    const uint32_t b4 = e.bias + (uint32_t)c0 * 4u;  // shared memory, the same address in every lane (a broadcast)
    ptx::tmem_ld_wait();
    if (e.ts && c0 == e.col_first) e.ts[5] = clock64();
    // the staging buffer about to be overwritten must have been read by its TMA store
    if (e.leader) ptx::tma_store_wait_read<1>();
    __syncwarp();
    uint8_t* sb = e.stage + sbuf * e.stage_bytes + e.lane * 64;
#pragma unroll
    for (int g = 0; g < 4; ++g) {  // 8 channels = one 16-byte chunk
      float v[8];
      const float4 bv0 = ptx::ld_shared_v4(b4 + 32u * g), bv1 = ptx::ld_shared_v4(b4 + 32u * g + 16u);
      const float bb[8] = {bv0.x, bv0.y, bv0.z, bv0.w, bv1.x, bv1.y, bv1.z, bv1.w};
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float acc = __uint_as_float(r[g * 8 + k]);
        if (ACT) {  // SiLU(x) = h + h * tanh(h), h = x / 2 = 0.5 * acc + (0.5 * bias)
          const float hh = fmaf(acc, 0.5f, bb[k]);
          v[k] = fmaf(hh, tanh_fast(hh), hh);
        } else {
          v[k] = acc + bb[k];
        }
      }
      if (RES) {
        const __nv_bfloat162* rh = reinterpret_cast<const __nv_bfloat162*>(&rv[g]);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 f = __bfloat1622float2(rh[k]);
          v[2 * k] += f.x;
          v[2 * k + 1] += f.y;
        }
      }
      uint4 o;
      o.x = pack_bf16(v[0], v[1]);
      o.y = pack_bf16(v[2], v[3]);
      o.z = pack_bf16(v[4], v[5]);
      o.w = pack_bf16(v[6], v[7]);
      // 64-byte swizzle (Swizzle<2,4,3>): 16-byte chunk index ^= (row >> 1) & 3
      *reinterpret_cast<uint4*>(sb + (((uint32_t)g ^ e.swz) << 4)) = o;
      if (UP && !e.tmu) {
        const int cg = c0 + g * 8;
        if (e.urow && cg < e.nvalid) {
          *reinterpret_cast<uint4*>(e.urow + cg) = o;
          *reinterpret_cast<uint4*>(e.urow + e.up_pix + cg) = o;
          *reinterpret_cast<uint4*>(e.urow + e.up_row + cg) = o;
          *reinterpret_cast<uint4*>(e.urow + e.up_row + e.up_pix + cg) = o;
        }
      }
    }
    if (e.ts && c0 == e.col_first) e.ts[6] = clock64();
    ptx::fence_proxy_async();
    __syncwarp();
    if (e.leader) {
      // rows beyond the image and channels beyond Cout are clipped by the tensor map
      if (e.red) ptx::tma_reduce_add_4d(e.tm, e.stage + sbuf * e.stage_bytes, e.cn0 + c0, e.cw, e.chh, e.cb);
      else ptx::tma_store_4d(e.tm, e.stage + sbuf * e.stage_bytes, e.cn0 + c0, e.cw, e.chh, e.cb);
      if (UP && e.tmu) {  // nn.Upsample(2x nearest): the same staged tile lands on the four (dy, dx) phases
#pragma unroll
        for (int ph = 0; ph < 4; ++ph)
          ptx::tma_store_5d(e.tmu, e.stage + sbuf * e.stage_bytes, e.cn0 + c0, ph & 1, e.cw, ph >> 1, e.ubh);
      }
      ptx::tma_store_commit();
    }
    sbuf ^= 1;
  }
}

struct EpiCtx {
  uint64_t *tmem_full, *tmem_empty;
  uint32_t tmem_base;
  uint8_t* stage;    // this warp's staging buffers
  uint32_t bias_s;   // shared-memory address of the layer's bias
  int lane, e, q, half, hl, wl, box_w0, box_h0, col_first, col_step, total_tiles;
  bool leader;
};

// The MODE_CONV epilogue's whole tile loop, specialised on the layer flavour (activation, residual, 2x up-sampled copy): the
// flavour is chosen once per kernel instead of through an indirect branch per sub-tile, what is constant over a tile is set up
// once per tile, and per sub-tile only the accumulator columns, the output row and the residual / up-sampling rows move.
template <bool ACT, bool RES, bool UP>
__device__ __forceinline__ void epi_role_conv(const ConvK& p, const EpiCtx& x) {
  int sbuf = 0, it = 0;
  EpiTile et;
  et.stage = x.stage;
  et.stage_bytes = p.epi_stage_bytes;
  et.swz = (uint32_t)((x.lane >> 1) & 3);
  et.lane = x.lane;
  et.leader = x.leader;
  et.up_pix = p.out2x_pix_stride;
  et.up_row = (long long)(2 * p.Wout) * p.out2x_pix_stride;
  et.col_first = x.col_first;
  et.col_step = x.col_step;
  et.tm = &p.tmO;
  et.tmu = (UP && p.up_tma) ? &p.tmU : nullptr;
  et.red = p.res_red != 0;
  const long long rstep = (long long)p.Ht * p.res_row_stride;                                 // residual: one sub-tile down
  const long long ustep = (long long)(2 * p.Ht) * (2 * p.Wout) * p.out2x_pix_stride;           // up-sampled copy: one sub-tile down
  const uint32_t lane_quarter = (uint32_t)(x.q * 32) << 16;
  for (int t = blockIdx.x; t < x.total_tiles; t += gridDim.x, ++it) {
    const int acc = it & (p.n_acc - 1);
    if (p.epi_tile_split && (it & 1) != x.half) continue;  // the other warp group owns this tile
    const TileCoord c = decode_tile(p, t);
    const uint32_t acc_ph = (uint32_t)(it >> p.acc_shift) & 1u;
    const bool ts_on = x.leader && (x.e & 3) == 0 && (p.epi_tile_split || x.e == 0);
    const int h0 = c.h0 + x.hl, w = c.w0 + x.wl;
    const bool wvalid = w < p.Wout;
    const int nvalid = min(p.BN, p.Cout - c.n0);
    // this thread's pixel in sub-tile 0: residual row and up-sampled destination (sub-tile m: + m * rstep / ustep)
    const __nv_bfloat16* rbase =
        RES ? p.res + (long long)c.b * p.res_img_stride + (long long)h0 * p.res_row_stride + (long long)w * p.res_pix_stride + c.n0 : nullptr;
    __nv_bfloat16* ubase =
        (UP && !et.tmu) ? p.out2x + (((long long)c.b * 2 * p.Hout + 2 * h0) * (2 * p.Wout) + 2 * w) * p.out2x_pix_stride + c.n0 : nullptr;
    auto res_row = [&](int m) -> const __nv_bfloat16* {
      return (RES && p.res && m < p.m_sub && wvalid && h0 + m * p.Ht < p.Hout) ? rbase + m * rstep : nullptr;
    };
    uint4 rvn[4];
    if (RES) {  // the tile's first residual chunk is in flight while we wait for the accumulator
      const __nv_bfloat16* r0 = res_row(0);
#pragma unroll
      for (int g = 0; g < 4; ++g)
        rvn[g] = (r0 && x.col_first + g * 8 < nvalid) ? *reinterpret_cast<const uint4*>(r0 + x.col_first + g * 8) : make_uint4(0, 0, 0, 0);
    }
    et.bias = x.bias_s + (uint32_t)c.n0 * 4u;
    et.nvalid = nvalid;
    et.cn0 = c.n0;
    et.cw = c.w0 + x.box_w0;
    et.cb = c.b;
    if (ts_on) Y5_TS(2, it, 0);
    ptx::mbar_wait_suspend(&x.tmem_full[acc], acc_ph);
    ptx::tc_fence_after();
    if (ts_on) Y5_TS(2, it, 1);
    uint32_t taddr = x.tmem_base + (uint32_t)(acc * p.acc_stride) + lane_quarter;
    int chh = c.h0 + x.box_h0;
    for (int m = 0; m < p.m_sub; ++m) {  // the tile's 128-pixel sub-tiles, stacked along H
      et.taddr = taddr;
      et.chh = chh;
      et.ubh = c.b * p.Hout + chh;
      et.rrow = res_row(m);
      et.rrow_next = res_row(m + 1);
      et.urow = (UP && !et.tmu && wvalid && h0 + m * p.Ht < p.Hout) ? ubase + m * ustep : nullptr;
      et.ts = (ts_on && m == 0 && p.ts && (int)blockIdx.x == p.ts_cta) ? p.ts + (2 * 32 + (it & 31)) * 8 : nullptr;
      conv_epi_tile<ACT, RES, UP>(et, sbuf, rvn);
      taddr += (uint32_t)p.sub_cols;
      chh += p.Ht;
    }
    if (ts_on) Y5_TS(2, it, 2);
    ptx::tc_fence_before();
    ptx::mbar_arrive(&x.tmem_empty[acc]);
    if (ts_on) Y5_TS(2, it, 3);
  }
}

__global__ void __launch_bounds__(NUM_THREADS) conv_tc_kernel(const __grid_constant__ ConvK p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full[MAX_ACC];
  __shared__ __align__(8) uint64_t tmem_empty[MAX_ACC];
  __shared__ __align__(8) uint64_t wres_bar;
  __shared__ uint32_t tmem_base_smem;

  // 1024-byte aligned: [resident weights][operand ring][epilogue staging] (swizzle patterns repeat every 8 rows)
  uint8_t* smem_res = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem = smem_res + p.b_res_bytes;
  const uint32_t unit_bytes = p.a_bytes + (uint32_t)p.b_per_stage * p.b_stage_bytes;
  const uint32_t stage_bytes = unit_bytes * (uint32_t)p.group;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.n_tiles_m * p.n_tiles_n;
  const int ksub = p.rowshift ? p.KH : 1;                                  // taps served by one A stage

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&p.tmA);
    ptx::prefetch_tmap(&p.tmB);
    ptx::prefetch_tmap(&p.tmO);
    if (p.out2x && p.up_tma) ptx::prefetch_tmap(&p.tmU);
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < p.n_acc; ++a) {
      ptx::mbar_init(&tmem_full[a], 1);
      ptx::mbar_init(&tmem_empty[a], p.epi_tile_split ? 128 : EPI_WARPS * 32);
    }
    ptx::mbar_init(&wres_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&tmem_base_smem, (uint32_t)TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;
  // Programmatic dependent launch: everything above (barriers, TMEM, descriptor prefetch) overlapped the previous kernel's
  // tail; from here on global memory is touched, so the previous grid must have completed and flushed.  Only then may the
  // NEXT kernel start its own prologue (its pre-wait phase never touches memory, and it finds kernel N-1's inputs final).
  ptx::griddep_wait();
  ptx::griddep_launch_dependents();

  if (warp == 0) {
    // ===================== TMA producer =====================
    // elect.sync (not `lane == 0`): ptxas then knows a single thread runs the region and issues UTMALDG / UTCHMMA straight from
    // uniform registers; under a lane test every such instruction is wrapped in a per-lane serialisation loop (~60 cycles each)
    if (ptx::elect_one()) {
      if (p.b_resident) {  // all weight tiles, once: tile (tap, kc) at smem_res + (tap * kchunks + kc) * b_stage_bytes
        const int ntile = p.KH * p.KW * p.kchunks;
        ptx::mbar_expect_tx(&wres_bar, (uint32_t)ntile * p.b_bytes);
        for (int tap = 0; tap < p.KH * p.KW; ++tap)
          for (int kc = 0; kc < p.kchunks; ++kc)
            ptx::tma_load_2d(smem_res + (size_t)(tap * p.kchunks + kc) * p.b_stage_bytes, &p.tmB, &wres_bar, kc * p.BK,
                             tap * p.cout_pad + (int)(blockIdx.x % (unsigned)p.n_tiles_n) * p.BN);  // this CTA's N tile (see the host plan)
      }
      int s = 0;
      uint32_t ph = 0;
      const uint32_t unit_tx = p.a_tx_bytes + (uint32_t)p.b_per_stage * p.b_bytes;
      int pit = 0;
      for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++pit) {
        const TileCoord c = decode_tile(p, t);
        int kh = 0, kw = 0, kc = 0;  // unit = (tap, kc), kc fastest; rowshift: taps = kw only (kh stays 0), else kh * KW + kw
        for (int u0 = 0; u0 < p.n_units; u0 += p.group) {
          const int ng = min(p.group, p.n_units - u0);
          if (u0 == 0) Y5_TS(0, pit, 0);
          ptx::mbar_wait(&empty_bar[s], ph ^ 1u);
          if (u0 == 0) Y5_TS(0, pit, 1);
          uint8_t* sbase = smem + (size_t)s * stage_bytes;
          ptx::mbar_expect_tx(&full_bar[s], unit_tx * (uint32_t)ng);
          for (int g = 0; g < ng; ++g) {
            int wi = c.w0 * p.stride + kw - p.pad_w;
            const int hi = c.h0 * p.stride + kh - p.pad_h;
            int cbase = 0;
            if (p.pairw) {  // input column 2*wo + (kw - pad): pair index wo + floor(off / 2), phase off & 1
              const int off = kw - p.pad_w;
              const int phase = off & 1;
              wi = c.w0 + ((off - phase) >> 1);
              cbase = phase * p.in_pix_stride;
            }
            uint8_t* sa = sbase + (size_t)g * unit_bytes;
            uint8_t* sb = sa + p.a_bytes;
            ptx::tma_load_4d(sa, &p.tmA, &full_bar[s], cbase + kc * p.BK, wi, hi, c.b);
            for (int j = 0; j < p.b_per_stage; ++j) {
              const int tap = (p.rowshift ? j : kh) * p.KW + kw;
              ptx::tma_load_2d(sb + (size_t)j * p.b_stage_bytes, &p.tmB, &full_bar[s], kc * p.BK,
                               tap * p.cout_pad + c.n0);
            }
            if (++kc == p.kchunks) {
              kc = 0;
              if (++kw == p.KW) {
                kw = 0;
                ++kh;
              }
            }
          }
          if (++s == p.stages) {
            s = 0;
            ph ^= 1u;
          }
        }
        Y5_TS(0, pit, 2);
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (ptx::elect_one()) {
      if (p.b_resident) {
        ptx::mbar_wait(&wres_bar, 0u);
        ptx::tc_fence_after();
      }
      MmaCtx x;
      x.full_bar = full_bar;
      x.empty_bar = empty_bar;
      x.tmem_full = tmem_full;
      x.tmem_empty = tmem_empty;
      x.tmem_base = tmem_base;
      // descriptors differ only in the 14-bit (address >> 4) field of the low word; K-major, SBO = 8 rows
      const uint64_t desc0 = ptx::make_kmajor_desc(0u, (uint32_t)p.BK * 2u);
      x.hi = (uint32_t)(desc0 >> 32);
      x.ring_lo = (uint32_t)desc0 | ((ptx::smem_u32(smem) & 0x3FFFFu) >> 4);
      x.res_lo = (uint32_t)desc0 | ((ptx::smem_u32(smem_res) & 0x3FFFFu) >> 4);
      x.stage16 = stage_bytes >> 4;
      x.unit16 = unit_bytes >> 4;
      x.total_tiles = total_tiles;
      x.ksub = ksub;
      const int nkf = (min(p.BK, p.Cin) + 15) >> 4;  // MMAs per tap of a full K chunk
      if (ksub == 3) {
        switch (nkf) {
          case 1: mma_role<3, 1>(p, x); break;
          case 2: mma_role<3, 2>(p, x); break;
          case 3: mma_role<3, 3>(p, x); break;
          default: mma_role<3, 4>(p, x); break;
        }
      } else if (ksub == 1) {
        switch (nkf) {
          case 1: mma_role<1, 1>(p, x); break;
          case 2: mma_role<1, 2>(p, x); break;
          case 3: mma_role<1, 3>(p, x); break;
          default: mma_role<1, 4>(p, x); break;
        }
      } else {
        mma_role<0, 0>(p, x);
      }
    }
  } else {
    // ===================== epilogue: 8 warps =====================
    // warp e = warp - 2; TMEM lane quarter q = warp & 3 (hardware rule: a warp reads lanes 32*(warp%4)..+31);
    // the two warps sharing a quarter split the columns: 32-column chunks with (chunk & 1) == half.
    const int e = warp - 2;
    const bool leader = ptx::elect_one();  // one fixed thread per warp owns the bulk-store groups (per-thread state)
    const int q = warp & 3;
    const int half = e >> 2;
    const int row = q * 32 + lane;
    const int hl = (int)fdiv((uint32_t)row, p.fd_wt);
    const int wl = row - hl * p.Wt;
    // this warp's 32 pixels as a TMA box: {32 ch, bw, 32 / bw, 1}
    const int bw = min(p.Wt, 32);
    const int box_h0 = (q * 32) / p.Wt, box_w0 = (q * 32) % p.Wt;
    uint8_t* stage = smem + (size_t)p.stages * stage_bytes + (size_t)e * ((size_t)EPI_BUFS * p.epi_stage_bytes);
    // the layer's bias in shared memory: with 224 KB of the SM configured as shared memory the L1 that is left is a few KB, the
    // residual stream evicts the bias line at every chunk and each 32-column chunk then waited an L2 round trip (~700+ cycles
    // in the in-kernel stamps) for the SAME 128 bytes
    float* bias_s = reinterpret_cast<float*>(smem + (size_t)p.stages * stage_bytes + (size_t)EPI_WARPS * EPI_BUFS * p.epi_stage_bytes);
    for (int i = (int)threadIdx.x - 64; i < p.cout_pad + 32; i += 32 * EPI_WARPS) bias_s[i] = __ldg(p.bias + i);
    asm volatile("bar.sync 1, %0;" ::"r"(32 * EPI_WARPS) : "memory");
    int sbuf = 0;
    int it = 0;
    const int col_first = p.epi_tile_split ? 0 : half * 32;  // first 32-column chunk of this warp
    const int col_step = p.epi_tile_split ? 32 : 64;
    if (p.mode == MODE_CONV) {  // one specialised instantiation of the whole loop per layer flavour
      EpiCtx x;
      x.tmem_full = tmem_full;
      x.tmem_empty = tmem_empty;
      x.tmem_base = tmem_base;
      x.stage = stage;
      x.bias_s = ptx::smem_u32(bias_s);
      x.lane = lane;
      x.e = e;
      x.q = q;
      x.half = half;
      x.hl = hl;
      x.wl = wl;
      x.box_w0 = box_w0;
      x.box_h0 = box_h0;
      x.col_first = col_first;
      x.col_step = col_step;
      x.total_tiles = total_tiles;
      x.leader = leader;
      const int flavour = (p.act ? 1 : 0) | ((p.res && !p.res_red) ? 2 : 0) | (p.out2x ? 4 : 0);
      switch (flavour) {
        case 0: epi_role_conv<false, false, false>(p, x); break;
        case 1: epi_role_conv<true, false, false>(p, x); break;
        case 2: epi_role_conv<false, true, false>(p, x); break;
        case 3: epi_role_conv<true, true, false>(p, x); break;
        case 5: epi_role_conv<true, false, true>(p, x); break;
        case 4:
        case 6: epi_role_conv<false, true, true>(p, x); break;  // generic paths tolerate null rrow / urow
        default: epi_role_conv<true, true, true>(p, x); break;
      }
    } else
    for (int t = blockIdx.x; t < total_tiles; t += gridDim.x, ++it) {
      const int acc = it & (p.n_acc - 1);
      if (p.epi_tile_split && (it & 1) != half) continue;  // the other warp group owns this tile
      const TileCoord c = decode_tile(p, t);
      const uint32_t acc_ph = (uint32_t)(it >> p.acc_shift) & 1u;

      const bool ts_on = leader && (e & 3) == 0 && (p.epi_tile_split || e == 0);
      if (ts_on) Y5_TS(2, it, 0);
      ptx::mbar_wait_suspend(&tmem_full[acc], acc_ph);
      ptx::tc_fence_after();
      if (ts_on) Y5_TS(2, it, 1);
      for (int m = 0; m < p.m_sub; ++m) {  // the tile's 128-pixel sub-tiles, stacked along H
      const int hsub = c.h0 + m * p.Ht;
      const int h = hsub + hl, w = c.w0 + wl;
      const uint32_t taddr = tmem_base + (uint32_t)(acc * p.acc_stride + m * p.sub_cols) + ((uint32_t)(q * 32) << 16);

      if (p.det_decode == 2) {
        // Detect, compact records for the fused post-process (the [B, A, no] tensor is never written): per anchor row
        // rec_w floats = (cx, cy, w, h, obj, cls[nc], theta index) - everything non_max_suppression_obb reads of a row
        // (utils/general.py:781-832).  Box / obj / class columns: same sigmoid and decode arithmetic as the full-tensor mode
        // below.  The theta index is the first maximum of the 180 LOGITS (accumulator + bias): the sigmoid is monotone, so this
        // is the index torch.max returns on the activated values (:822) whenever those are distinct - and the 180 MUFU ops and
        // their arithmetic per row, which bounded this epilogue, are not needed.  (On the tanh.approx sigmoid of the
        // full-tensor mode two logits closer than its 2^-11 error can order differently; the tests bound that.)
        // Every warp owns whole tiles here.  The warp's 32 records are staged densely ([32][rec_w] fp32) and leave through
        // ONE TMA store whose tensor map views the record buffer as (rec_w, W, H, anchor, image).
        const int a = c.nt;
        const int nfix = p.det_no - 180;                    // 5 + nc leading columns
        if (leader) ptx::tma_store_wait_read<1>();
        __syncwarp();
        const uint32_t rec_s = ptx::smem_u32(stage + sbuf * p.epi_stage_bytes) + (uint32_t)(lane * p.det_rec_w) * 4u;
        float best = -INFINITY;
        int bk = 0;
        for (int c0 = 0; c0 < p.det_no; c0 += 32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(taddr + (uint32_t)c0, r);
          ptx::tmem_ld_wait();
          const uint32_t b4 = ptx::smem_u32(bias_s + c.n0 + c0);
          float v[32];
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 bv = ptx::ld_shared_v4(b4 + 16u * g);
            v[4 * g + 0] = __uint_as_float(r[g * 4 + 0]) + bv.x;
            v[4 * g + 1] = __uint_as_float(r[g * 4 + 1]) + bv.y;
            v[4 * g + 2] = __uint_as_float(r[g * 4 + 2]) + bv.z;
            v[4 * g + 3] = __uint_as_float(r[g * 4 + 3]) + bv.w;
          }
          const int lo = nfix - c0;          // entries [lo, hi) of this chunk are theta bins
          const int hi = p.det_no - c0;
          if (lo > 0) {  // (warp-uniform) the chunk holds box / obj / class columns: activate, decode, stage them
#pragma unroll
            for (int g = 0; g < 8; ++g) {
              if (4 * g < lo) {
                float s0 = sigmoid_fast(v[4 * g]), s1 = sigmoid_fast(v[4 * g + 1]);
                float s2 = sigmoid_fast(v[4 * g + 2]), s3 = sigmoid_fast(v[4 * g + 3]);
                if (c0 == 0 && g == 0) {  // xy, wh (models/yolo.py:73-74)
                  s0 = (s0 * 2.0f - 0.5f + (float)w) * p.det_stride;
                  s1 = (s1 * 2.0f - 0.5f + (float)h) * p.det_stride;
                  s2 = (s2 * 2.0f) * (s2 * 2.0f) * p.det_anchor[2 * a];
                  s3 = (s3 * 2.0f) * (s3 * 2.0f) * p.det_anchor[2 * a + 1];
                }
                const uint32_t dst = rec_s + (uint32_t)(c0 + 4 * g) * 4u;
                if (4 * g + 3 < lo) {
                  ptx::st_shared_v4(dst, s0, s1, s2, s3);
                } else {  // the group straddles the first theta bin
                  ptx::st_shared_f32(dst, s0);
                  if (4 * g + 1 < lo) ptx::st_shared_f32(dst + 4, s1);
                  if (4 * g + 2 < lo) ptx::st_shared_f32(dst + 8, s2);
                }
              }
            }
          }
          if (lo > 0 || hi < 32) {  // (warp-uniform) first / last chunk: entries that are not theta bins never win
#pragma unroll
            for (int k = 0; k < 32; ++k)
              if (k < lo || k >= hi) v[k] = -INFINITY;
          }
          // a 5-level tournament over the chunk (the first maximum wins ties: the higher index replaces the lower only if
          // strictly greater), then ONE comparison against the running best - a 180-step dependent chain otherwise
          int id[16];
#pragma unroll
          for (int k = 0; k < 16; ++k) {
            const bool take = v[2 * k + 1] > v[2 * k];
            v[k] = take ? v[2 * k + 1] : v[2 * k];
            id[k] = 2 * k + (take ? 1 : 0);
          }
#pragma unroll
          for (int half = 8; half >= 1; half >>= 1) {
#pragma unroll
            for (int k = 0; k < half; ++k) {
              const bool take = v[2 * k + 1] > v[2 * k];
              v[k] = take ? v[2 * k + 1] : v[2 * k];
              id[k] = take ? id[2 * k + 1] : id[2 * k];
            }
          }
          if (v[0] > best) {
            best = v[0];
            bk = c0 + id[0] - nfix;
          }
        }
        ptx::st_shared_f32(rec_s + (uint32_t)nfix * 4u, (float)bk);
        for (int cc = nfix + 1; cc < p.det_rec_w; ++cc) ptx::st_shared_f32(rec_s + (uint32_t)cc * 4u, 0.0f);  // padding columns
        ptx::fence_proxy_async();
        __syncwarp();
        if (leader) {  // rows beyond the image are clipped by the tensor map
          ptx::tma_store_5d(&p.tmO, stage + sbuf * p.epi_stage_bytes, 0, c.w0 + box_w0, hsub + box_h0, a, c.b);
          ptx::tma_store_commit();
        }
        sbuf ^= 1;
      } else {
        // Detect: N tile nt == anchor nt; columns [0, det_no) are that anchor's outputs.
        // out row = b * rows_per_image + row_off + (a * H + h) * W + w   (models/yolo.py:65,81): the tensor map
        // views the output as (no, W, H, anchor, image), so the permute is the store's addressing.
        const int a = c.nt;
        const float aw = p.det_anchor[2 * a], ah = p.det_anchor[2 * a + 1];
        for (int c0 = col_first; c0 < p.det_no; c0 += col_step) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(taddr + (uint32_t)c0, r);
          ptx::tmem_ld_wait();
          if (leader) ptx::tma_store_wait_read<1>();
          __syncwarp();
          uint8_t* sb = stage + sbuf * p.epi_stage_bytes;
          const uint32_t b4 = ptx::smem_u32(bias_s + c.n0 + c0);
#pragma unroll
          for (int g = 0; g < 8; ++g) {  // 4 floats = one 16-byte chunk
            const float4 bv = ptx::ld_shared_v4(b4 + 16u * g);
            float v[4];
            v[0] = __uint_as_float(r[g * 4 + 0]) + bv.x;
            v[1] = __uint_as_float(r[g * 4 + 1]) + bv.y;
            v[2] = __uint_as_float(r[g * 4 + 2]) + bv.z;
            v[3] = __uint_as_float(r[g * 4 + 3]) + bv.w;
            if (p.det_decode) {
#pragma unroll
              for (int k = 0; k < 4; ++k) v[k] = sigmoid_fast(v[k]);
              if (c0 == 0 && g == 0) {  // xy, wh (models/yolo.py:73-74)
                v[0] = (v[0] * 2.0f - 0.5f + (float)w) * p.det_stride;
                v[1] = (v[1] * 2.0f - 0.5f + (float)h) * p.det_stride;
                v[2] = (v[2] * 2.0f) * (v[2] * 2.0f) * aw;
                v[3] = (v[3] * 2.0f) * (v[3] * 2.0f) * ah;
              }
            }
            // 128-byte swizzle (Swizzle<3,4,3>): 16-byte chunk index ^= row & 7
            *reinterpret_cast<float4*>(sb + lane * 128 + ((g ^ (lane & 7)) << 4)) = make_float4(v[0], v[1], v[2], v[3]);
          }
          ptx::fence_proxy_async();
          __syncwarp();
          if (leader) {
            ptx::tma_store_5d(&p.tmO, sb, c0, c.w0 + box_w0, hsub + box_h0, a, c.b);
            ptx::tma_store_commit();
          }
          sbuf ^= 1;
        }
      }
      }  // sub-tiles
      if (ts_on) Y5_TS(2, it, 2);
      ptx::tc_fence_before();
      ptx::mbar_arrive(&tmem_empty[acc]);
      if (ts_on) Y5_TS(2, it, 3);
    }
    if (leader) ptx::tma_store_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, (uint32_t)TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_tmapEncodeTiled get_encode() {
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

CUtensorMapSwizzle swizzle_for(int bk) {
  return bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (bk == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

struct ConvObj {
  ConvK k;
  int grid;
  size_t smem;
  double flops;      // algorithmic 2*MACs
  double hbm_bytes;  // algorithmic in + out (+ residual) bytes
};

}  // namespace
}  // namespace y5obb

using namespace y5obb;

extern "C" {

int y5obb_conv_tiling(int cin, int cout, int mode, int det_no, int* block_k, int* block_n, int* cin_pad,
                      int* cout_pad, int* n_tiles_n) {
  if (cin <= 0 || cout <= 0 || !block_k || !block_n || !cin_pad || !cout_pad || !n_tiles_n) return Y5OBB_EINVAL;
  int bk = cin > 32 ? 64 : (cin > 16 ? 32 : 16);
  int bn, nt;
  if (mode == MODE_DETECT) {
    if (det_no <= 0 || cout % det_no) return Y5OBB_EINVAL;
    nt = cout / det_no;
    bn = (det_no + 15) / 16 * 16;
    if (bn > 256) return Y5OBB_EINVAL;
  } else {
    int best_nt = 0, best_bn = 0;
    long best_cost = -1;
    for (nt = (cout + 255) / 256; nt <= (cout + 255) / 256 + 3; ++nt) {
      bn = ((cout + nt - 1) / nt + 15) / 16 * 16;
      if (bn > 256) continue;
      long cost = (long)bn * nt * 16 + nt;  // padded width first, then fewer tiles
      if (best_cost < 0 || cost < best_cost) {
        best_cost = cost;
        best_nt = nt;
        best_bn = bn;
      }
    }
    nt = best_nt;
    bn = best_bn;
  }
  *block_k = bk;
  *block_n = bn;
  *cin_pad = (cin + 7) / 8 * 8;
  *cout_pad = bn * nt;
  *n_tiles_n = nt;
  return Y5OBB_OK;
}

int y5obb_conv_create(const y5obb_conv_desc* d, y5obb_conv_t** out) {
  if (!d || !out) return Y5OBB_EINVAL;
  if (!d->in || !d->w || !d->bias) return Y5OBB_EINVAL;
  if (d->stride != 1 && d->stride != 2) return Y5OBB_EINVAL;
  if (d->in_pix_stride % 8 || (reinterpret_cast<uintptr_t>(d->in) & 15)) return Y5OBB_EINVAL;
  if (d->KH < 1 || d->KW < 1 || d->pad_h < 0 || d->pad_w < 0) return Y5OBB_EINVAL;
  if (d->mode == MODE_CONV && d->act && !(d->flags & Y5OBB_CONV_BIAS_HALVED)) return Y5OBB_EINVAL;
  constexpr int known_flags = Y5OBB_CONV_NO_ROWSHIFT | Y5OBB_CONV_NO_RESIDENT | Y5OBB_CONV_NO_PAIRW | Y5OBB_CONV_BIAS_HALVED |
                              Y5OBB_CONV_NO_UP_TMA | Y5OBB_CONV_NO_RES_RED;
  if (d->flags & ~known_flags) return Y5OBB_EINVAL;
  const int64_t in_row_stride = d->in_row_stride ? d->in_row_stride : d->in_pix_stride * d->Win;
  const int64_t in_img_stride = d->in_img_stride ? d->in_img_stride : in_row_stride * d->Hin;
  if (in_row_stride % 8 || in_img_stride % 8) return Y5OBB_EINVAL;
  PFN_tmapEncodeTiled enc = get_encode();
  if (!enc) return Y5OBB_ECUDA;

  int bk, bn, cin_pad, cout_pad, nt;
  int rc = y5obb_conv_tiling(d->Cin, d->Cout, d->mode, d->det_no, &bk, &bn, &cin_pad, &cout_pad, &nt);
  if (rc) return rc;

  ConvObj* o = new ConvObj();
  ConvK& k = o->k;
  memset(&k, 0, sizeof(k));
  const bool geom = d->out_h > 0 || d->out_w > 0 || d->out_row_stride || d->out_img_stride || d->res_row_stride || d->res_img_stride;
  if (geom && (d->mode != MODE_CONV || d->out2x || d->out_h <= 0 || d->out_w <= 0 || !d->out_row_stride || !d->out_img_stride ||
               (d->res && (!d->res_row_stride || !d->res_img_stride)) || (d->out_row_stride & 7) || (d->out_img_stride & 7) ||
               (d->res_row_stride & 7) || (d->res_img_stride & 7))) {
    delete o;
    return Y5OBB_EINVAL;
  }
  const int Hout = geom ? d->out_h : (d->Hin + 2 * d->pad_h - d->KH) / d->stride + 1;
  const int Wout = geom ? d->out_w : (d->Win + 2 * d->pad_w - d->KW) / d->stride + 1;
  k.B = d->B;
  k.Hout = Hout;
  k.Wout = Wout;
  k.n_tiles_n = nt;
  k.BN = bn;
  k.BK = bk;
  k.Cout = d->Cout;
  k.cout_pad = cout_pad;
  k.Cin = d->Cin;
  k.kchunks = (d->Cin + bk - 1) / bk;
  k.KH = d->KH;
  k.KW = d->KW;
  k.stride = d->stride;
  k.pad_h = d->pad_h;
  k.pad_w = d->pad_w;
  k.b_bytes = (uint32_t)bn * bk * 2;
  k.b_stage_bytes = (uint32_t)align_up(k.b_bytes, 1024);
  int a_rows = 0;
  size_t stage_bytes = 0;
  k.epi_stage_bytes = d->mode == MODE_DETECT ? EPI_STAGE_DET : EPI_STAGE_CONV;
  const int det_rec_w = ((d->det_no - 180 + 1) + 3) / 4 * 4;  // compact record: (5 + nc + 1) floats rounded up to 4
  if (d->mode == MODE_DETECT && d->det_decode == 2)
    k.epi_stage_bytes = std::max<uint32_t>(EPI_STAGE_DET, (uint32_t)align_up((size_t)32 * det_rec_w * 4, 128));
  const size_t bias_bytes = align_up((size_t)(cout_pad + 32) * 4, 128);  // the bias lives in shared memory behind the staging buffers
  // operand ring (+ resident weights): everything but the epilogue staging and the bias
  const size_t SMEM_BUDGET = (size_t)SMEM_TOTAL - 1024 - (size_t)EPI_WARPS * EPI_BUFS * k.epi_stage_bytes - bias_bytes;
  // Row-shift mode (stride-1 convs with KH > 1): an 8 x 16 pixel tile whose A stage holds Ht + KH - 1 image
  // rows; the KH vertical taps read the same stage at row offsets that are whole 8-row swizzle groups, so each
  // input row crosses L2 -> shared memory (Ht + KH - 1) / Ht times per kw instead of KH times.  Taken when the
  // weights are resident or at least 3 pipeline stages still fit; otherwise one load per tap (classic).
  // A tile is m_sub 128-pixel sub-tiles stacked along H (Wt x Ht*m_sub pixels): they share the weight tiles of every unit and
  // one trip through the producer -> MMA -> epilogue hand-shakes (about 1000 cycles of single-thread latencies per tile,
  // profiles/r2_conv_timeline*.txt), so narrow layers (few MMAs per 128 pixels) and weight-streaming layers both gain.
  auto plan = [&](bool rowshift, int m_sub) -> bool {
    int best_wt = 128;
    if (rowshift) {
      best_wt = 8;
    } else {  // Wt x Ht = 128 pixels, Wt the power of two (<=128) that wastes the fewest edge pixels
      double best_eff = -1;
      for (int wt = 128; wt >= 8; wt >>= 1) {
        int ht = BM / wt * m_sub;
        if (wt * d->stride > 256 || ht * d->stride > 256) continue;
        double eff = (double)Wout * Hout / ((double)((Wout + wt - 1) / wt * wt) * ((Hout + ht - 1) / ht * ht));
        if (eff > best_eff + 1e-9) {
          best_eff = eff;
          best_wt = wt;
        }
      }
    }
    k.Wt = best_wt;
    k.Ht = BM / best_wt;
    k.m_sub = m_sub;
    const int tile_h = k.Ht * m_sub;
    k.tiles_w = (Wout + k.Wt - 1) / k.Wt;
    k.tiles_h = (Hout + tile_h - 1) / tile_h;
    k.n_tiles_m = d->B * k.tiles_w * k.tiles_h;
    k.rowshift = rowshift ? 1 : 0;
    a_rows = rowshift ? tile_h + d->KH - 1 : tile_h;  // image rows per A stage
    if (a_rows * d->stride > 256) return false;          // TMA box dimension limit
    k.a_tx_bytes = (uint32_t)a_rows * k.Wt * bk * 2;
    k.row_shift_bytes = (uint32_t)k.Wt * bk * 2;
    const size_t a_stage = align_up(k.a_tx_bytes, 1024);
    k.a_bytes = (uint32_t)a_stage;  // ring slots are 1024-aligned; the TMA box fills the first a_rows * Wt rows
    const size_t b_all = (size_t)d->KH * d->KW * k.kchunks * k.b_stage_bytes;
    // weights stay resident when every tile uses the same ones (one N tile) and they leave room for >= 3 A stages
    // (several N tiles: the grid is made a multiple of their count, so that tile t = blockIdx.x + i * gridDim.x keeps ONE N tile
    // per CTA - the Detect head's three anchors - and that tile's weights are the resident ones)
    k.b_resident =
        ((nt == 1 || nt <= 4) && b_all + 3 * a_stage <= SMEM_BUDGET && !(d->flags & Y5OBB_CONV_NO_RESIDENT)) ? 1 : 0;
    k.b_res_bytes = k.b_resident ? (uint32_t)b_all : 0u;
    k.b_per_stage = k.b_resident ? 0 : (rowshift ? d->KH : 1);
    const size_t unit_bytes = a_stage + (size_t)k.b_per_stage * k.b_stage_bytes;
    k.n_units = (rowshift ? d->KW : d->KH * d->KW) * k.kchunks;
    // small units share a stage: every mbarrier round trip (~300-500 cycles in the two single-thread loops)
    // then moves >= ~24 KB
    int group = 1;
    while (group < k.n_units && group < 4 && (size_t)(group + 1) * unit_bytes <= 40 * 1024 &&
           (SMEM_BUDGET - k.b_res_bytes) / ((size_t)(group + 1) * unit_bytes) >= 3)
      ++group;
    k.group = group;
    stage_bytes = unit_bytes * group;
    k.stages = (int)std::min<size_t>(MAX_STAGES, (SMEM_BUDGET - k.b_res_bytes) / stage_bytes);
    return k.stages >= (rowshift ? 3 : 2);
  };
  const bool want_rowshift = d->stride == 1 && d->KH > 1 && Wout >= 8 && !(d->flags & Y5OBB_CONV_NO_ROWSHIFT);
  const int sub_cols = bn <= 32 ? 32 : (bn <= 64 ? 64 : (bn <= 128 ? 128 : 256));
  {
    // Configuration search: the largest m_sub whose two accumulator stages fit the TMEM columns, that keeps every SM busy and
    // adds no edge waste along H (m_sub = 1 only has to fit); row-shift before one load per tap.
    bool ok = false;
    for (int m = 4; m >= 1 && !ok; m >>= 1) {
      if (m * sub_cols * 2 > TMEM_COLS) continue;
      for (int rs = want_rowshift ? 1 : 0; rs >= 0 && !ok; --rs) {
        if (!plan(rs == 1, m)) continue;
        const long long tiles = (long long)k.n_tiles_m * nt;
        ok = m == 1 || (tiles >= sm_count() && Hout % (k.Ht * m) == 0 && k.stages >= 3);
      }
    }
    if (!ok) {
      delete o;
      return Y5OBB_EINVAL;
    }
  }
  // TMEM accumulator stages: the MMA issuer may run that many tiles ahead of the epilogue warps
  k.sub_cols = sub_cols;
  k.acc_stride = sub_cols * k.m_sub;
  k.a_sub16 = (uint32_t)(BM * bk * 2) >> 4;
  k.n_acc = std::min(MAX_ACC, TMEM_COLS / k.acc_stride);
  k.acc_shift = 0;
  while ((1 << k.acc_shift) < k.n_acc) ++k.acc_shift;
  k.fd_ntn = make_fastdiv((uint32_t)k.n_tiles_n);
  k.fd_per_img = make_fastdiv((uint32_t)(k.tiles_h * k.tiles_w));
  k.fd_tiles_w = make_fastdiv((uint32_t)k.tiles_w);
  k.fd_wt = make_fastdiv((uint32_t)k.Wt);
  k.idesc = ptx::make_idesc_bf16(BM, bn);
  k.mode = d->mode;
  k.act = d->act;
  k.bias = d->bias;
  k.out = static_cast<__nv_bfloat16*>(d->out);
  k.out_pix_stride = d->out_pix_stride;
  k.res = static_cast<const __nv_bfloat16*>(d->res);
  k.res_pix_stride = d->res_pix_stride;
  k.res_row_stride = geom ? d->res_row_stride : d->res_pix_stride * Wout;
  k.res_img_stride = geom ? d->res_img_stride : d->res_pix_stride * Wout * Hout;
  // In-place residual (the Bottleneck chain: out = chain = res): the add can be done by the TMA store itself (a bf16 reduce-add at
  // L2), which removes the epilogue's residual loads - they queue behind the producer's outstanding TMA loads (2-3 k cycles) and
  // bounded the residual layers.  The sum is then rounded twice (conv + SiLU to bf16, then the bf16 add) instead of once.
  // (the flag Y5OBB_CONV_NO_RES_RED: the epilogue loads the residual and adds in fp32, one rounding)
  k.res_red = (d->res && d->res == d->out && d->res_pix_stride == d->out_pix_stride && !d->out2x && !(d->flags & Y5OBB_CONV_NO_RES_RED) &&
               (!geom || (d->res_row_stride == d->out_row_stride && d->res_img_stride == d->out_img_stride)))
                  ? 1
                  : 0;
  k.out2x = static_cast<__nv_bfloat16*>(d->out2x);
  k.out2x_pix_stride = d->out2x_pix_stride;
  k.det_out = d->det_out;
  k.det_rows_per_image = d->det_rows_per_image;
  k.det_row_off = d->det_row_off;
  k.det_no = d->det_no;
  k.det_decode = d->det_decode;
  k.det_rec_w = ((d->det_no - 180 + 1) + 3) / 4 * 4;
  k.det_stride = d->det_stride;
  for (int i = 0; i < 6; ++i) k.det_anchor[i] = d->det_anchor[i];
  if (d->mode == MODE_CONV) {
    if (!d->out || d->out_pix_stride % 8 || (reinterpret_cast<uintptr_t>(d->out) & 15) || d->Cout % 8) {
      delete o;
      return Y5OBB_EINVAL;
    }
  } else if (!d->det_out || d->det_no % 4) {
    delete o;
    return Y5OBB_EINVAL;
  }

  // stride-2 convs over dense rows: view the input as horizontal pixel pairs so that no element stride is needed
  // along W (channels beyond the slice are finite activations of the same buffer and meet zero weights)
  k.pairw = (d->stride == 2 && !(d->Win & 1) && in_row_stride == d->in_pix_stride * d->Win &&
             !(d->flags & Y5OBB_CONV_NO_PAIRW)) ? 1 : 0;
  k.in_pix_stride = (int)d->in_pix_stride;
  {  // activations: (C, W, H, B), element strides (1, s, s, 1)
    cuuint64_t dims[4] = {(cuuint64_t)d->Cin, (cuuint64_t)d->Win, (cuuint64_t)d->Hin, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->in_pix_stride * 2, (cuuint64_t)in_row_stride * 2,
                             (cuuint64_t)in_img_stride * 2};
    cuuint32_t box[4] = {(cuuint32_t)bk, (cuuint32_t)(k.Wt * d->stride), (cuuint32_t)(a_rows * d->stride), 1};
    cuuint32_t es[4] = {1, (cuuint32_t)d->stride, (cuuint32_t)d->stride, 1};
    if (k.pairw) {
      dims[0] = (cuuint64_t)d->in_pix_stride + d->Cin;
      dims[1] = (cuuint64_t)d->Win / 2;
      strides[0] = (cuuint64_t)d->in_pix_stride * 4;
      box[1] = (cuuint32_t)k.Wt;
      es[1] = 1;
    }
    CUresult r = enc(&k.tmA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(d->in), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  {  // weights: (Cin, taps * Cout_pad)
    cuuint64_t dims[2] = {(cuuint64_t)d->Cin, (cuuint64_t)d->KH * d->KW * cout_pad};
    cuuint64_t strides[1] = {(cuuint64_t)cin_pad * 2};
    cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)bn};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(&k.tmB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(d->w), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  if (d->mode == MODE_CONV) {  // output: (C, W, H, B); each epilogue warp stores its 32 pixels x 32 channels
    const int bw = std::min(k.Wt, 32);
    cuuint64_t dims[4] = {(cuuint64_t)d->Cout, (cuuint64_t)Wout, (cuuint64_t)Hout, (cuuint64_t)d->B};
    cuuint64_t strides[3] = {(cuuint64_t)d->out_pix_stride * 2, (cuuint64_t)d->out_pix_stride * 2 * Wout,
                             (cuuint64_t)d->out_pix_stride * 2 * Wout * Hout};
    if (geom) {
      strides[1] = (cuuint64_t)d->out_row_stride * 2;
      strides[2] = (cuuint64_t)d->out_img_stride * 2;
    }
    cuuint32_t box[4] = {32, (cuuint32_t)bw, (cuuint32_t)(32 / bw), 1};
    cuuint32_t es[4] = {1, 1, 1, 1};
    CUresult r = enc(&k.tmO, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, d->out, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  k.up_tma = 0;
  if (d->mode == MODE_CONV && d->out2x && Hout % (k.Ht * k.m_sub) == 0 && !(d->out2x_pix_stride % 8) &&
      !(reinterpret_cast<uintptr_t>(d->out2x) & 15)) {
    // out2x[b, 2h + dy, 2w + dx, c] as a 5-D tensor (c, dx, w, dy, b * H + h): images are contiguous, so b and h share one
    // dimension - which is why the tile rows must not run past the image (no per-image clipping along that dimension)
    const int bw = std::min(k.Wt, 32);
    const cuuint64_t pix = (cuuint64_t)d->out2x_pix_stride * 2, row = pix * 2 * Wout;
    cuuint64_t dims[5] = {(cuuint64_t)d->Cout, 2, (cuuint64_t)Wout, 2, (cuuint64_t)d->B * Hout};
    cuuint64_t strides[4] = {pix, 2 * pix, row, 2 * row};
    cuuint32_t box[5] = {32, 1, (cuuint32_t)bw, 1, (cuuint32_t)(32 / bw)};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(&k.tmU, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, d->out2x, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r == CUDA_SUCCESS && !(d->flags & Y5OBB_CONV_NO_UP_TMA)) k.up_tma = 1;
  }
  if (d->mode == MODE_DETECT && d->det_decode == 2) {  // records as (rec_w, W, H, anchor, image) fp32; a warp stores 32 records
    const int bw = std::min(k.Wt, 32);
    const cuuint64_t rowb = (cuuint64_t)det_rec_w * 4;
    cuuint64_t dims[5] = {(cuuint64_t)det_rec_w, (cuuint64_t)Wout, (cuuint64_t)Hout, (cuuint64_t)nt, (cuuint64_t)d->B};
    cuuint64_t strides[4] = {rowb, rowb * Wout, rowb * Wout * Hout, rowb * (cuuint64_t)d->det_rows_per_image};
    cuuint32_t box[5] = {(cuuint32_t)det_rec_w, (cuuint32_t)bw, (cuuint32_t)(32 / bw), 1, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    float* base = d->det_out + (size_t)d->det_row_off * det_rec_w;
    CUresult r = (reinterpret_cast<uintptr_t>(base) & 15)
                     ? CUDA_ERROR_INVALID_VALUE
                     : enc(&k.tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  if (d->mode == MODE_DETECT && d->det_decode != 2) {  // output rows as (no, W, H, anchor, image) fp32; each warp stores 32 pixels x 32 floats
    const int bw = std::min(k.Wt, 32);
    cuuint64_t dims[5] = {(cuuint64_t)d->det_no, (cuuint64_t)Wout, (cuuint64_t)Hout, (cuuint64_t)nt, (cuuint64_t)d->B};
    const cuuint64_t rowb = (cuuint64_t)d->det_no * 4;
    cuuint64_t strides[4] = {rowb, rowb * Wout, rowb * Wout * Hout, rowb * (cuuint64_t)d->det_rows_per_image};
    cuuint32_t box[5] = {32, (cuuint32_t)bw, (cuuint32_t)(32 / bw), 1, 1};
    cuuint32_t es[5] = {1, 1, 1, 1, 1};
    float* base = d->det_out + (size_t)d->det_row_off * d->det_no;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (rowb & 15)) {
      delete o;
      return Y5OBB_EINVAL;
    }
    CUresult r = enc(&k.tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, base, dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      g_last_cuda_error = (int)r;
      delete o;
      return Y5OBB_ECUDA;
    }
  }
  const int total = k.n_tiles_m * k.n_tiles_n;
  o->grid = std::min(total, sm_count());
  if (k.b_resident && k.n_tiles_n > 1) o->grid = o->grid / k.n_tiles_n * k.n_tiles_n;  // one N tile per CTA (resident weights)
  // many tiles per CTA: the two epilogue groups alternate tiles (two epilogues in flight, any BN);
  // few tiles per CTA: they split the columns of each tile (shortest single-tile latency)
  k.epi_tile_split = total >= 4 * o->grid ? 1 : 0;
  if (d->mode == MODE_DETECT && d->det_decode == 2) k.epi_tile_split = 1;  // a record is assembled by one thread over all columns
  // >= 116 KB so that two CTAs (each owning all 512 TMEM columns) can never share an SM
  o->smem = k.b_res_bytes + (size_t)k.stages * stage_bytes + (size_t)EPI_WARPS * EPI_BUFS * k.epi_stage_bytes + bias_bytes + 1024;
  o->smem = std::max<size_t>(o->smem, 116 * 1024);
  o->flops = 2.0 * d->B * Hout * Wout * (double)d->Cout * d->Cin * d->KH * d->KW;
  o->hbm_bytes = 2.0 * d->B * ((double)d->Hin * d->Win * (d->hbm_cin ? d->hbm_cin : d->Cin) + (double)Hout * Wout * d->Cout * (d->res ? 2 : 1));
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_TOTAL);
    if (e != cudaSuccess) {
      delete o;
      return cuda_fail(e);
    }
    attr_set = true;
  }
  *out = reinterpret_cast<y5obb_conv_t*>(o);
  return Y5OBB_OK;
}

int y5obb_conv_run(const y5obb_conv_t* conv, void* stream) {
  if (!conv) return Y5OBB_EINVAL;
  const ConvObj* o = reinterpret_cast<const ConvObj*>(conv);
  // programmatic dependent launch: the kernel's prologue overlaps the previous kernel's tail (griddepcontrol.wait in the kernel)
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)o->grid);
  cfg.blockDim = dim3((unsigned)NUM_THREADS);
  cfg.dynamicSmemBytes = o->smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, conv_tc_kernel, o->k);
  if (e != cudaSuccess) return cuda_fail(e);
  return Y5OBB_OK;
}

int y5obb_conv_info(const y5obb_conv_t* conv, double* flops, double* hbm_bytes, int* grid, int* block_n, int* block_k,
                    int* stages) {
  if (!conv) return Y5OBB_EINVAL;
  const ConvObj* o = reinterpret_cast<const ConvObj*>(conv);
  if (flops) *flops = o->flops;
  if (hbm_bytes) *hbm_bytes = o->hbm_bytes;
  if (grid) *grid = o->grid;
  if (block_n) *block_n = o->k.BN;
  if (block_k) *block_k = o->k.BK;
  if (stages) *stages = o->k.stages;
  return Y5OBB_OK;
}

void y5obb_conv_destroy(y5obb_conv_t* conv) { delete reinterpret_cast<ConvObj*>(conv); }

int y5obb_conv_debug_timestamps(y5obb_conv_t* conv, unsigned long long* dev_buf_768) {
  if (!conv) return Y5OBB_EINVAL;
  reinterpret_cast<ConvObj*>(conv)->k.ts = dev_buf_768;
  const char* c = getenv("Y5OBB_TS_CTA");  // which CTA stamps (default 0)
  reinterpret_cast<ConvObj*>(conv)->k.ts_cta = c ? atoi(c) : 0;
  return Y5OBB_OK;
}

}  // extern "C"
