// Tensor-core implicit-GEMM convolution for sm_100a: TMA -> shared memory (128B swizzle) ->
// tcgen05.mma (bf16 x bf16 -> fp32 in TMEM) -> epilogue (bias, residual, activation) -> global.
//
// Replaces, for the smp 0.3.3 graphs the reference runs (src/models/smp/model.py:70,192):
// conv2d / conv_transpose2d(k4,s2,p1) + eval-mode batch_norm (folded) + relu|swish +
// F.interpolate(scale_factor=2, mode="nearest") + torch.cat + residual add.
//
// Layout: activations NHWC bf16.  A-operand tiles are TH x TW output pixels (<=128 rows) by 64
// input channels, fetched per filter tap as one shifted 4-D TMA box (zero fill outside the image
// = conv padding).  B tiles are BN x 64 slices of the packed weight matrix.  The K loop runs over
// (source tensor of the fused concat) x (tap) x (64-channel chunk).
//
// Nearest-x2 upsample + 3x3 conv and ConvTranspose(k4,s2,p1) are executed as four output-phase
// sub-problems on the half-resolution grid (weights pre-combined per phase on the host).
//
// Halo-tile mode (narrow single-source k x k convs): 16 x 8 pixel tiles, ONE halo box of A per channel
// chunk whose kh*kw taps are shifted views (UMMA group stride = halo row pitch), weights resident in
// shared memory.  Row tiles (TH = 1) reuse one wide box per tap row the same way.
//
// One persistent CTA per SM, 18 warps: warp 0 = TMA producer, warp 1 = MMA issuer + TMEM owner (both run
// converged and predicate only the issuing instruction on an elected lane, so their address arithmetic
// stays on the uniform datapath), warps 2-17 = epilogue (4 per TMEM lane quarter, two chunk-alternating
// groups of 8: the epilogue is instruction-latency bound, so it needs several warps per scheduler).
// Accumulators form a ring of min(8, 512/BN) tiles in TMEM, so the epilogue of tile i overlaps the MMAs of
// the following tiles.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include <cstring>
#include <new>

#include "common.h"
#include "ptx_sm100.h"

namespace octseg {

constexpr int kMaxStages = 8;
constexpr int kMaxAcc = 8;  // TMEM accumulator ring: min(8, 512 / BN) tiles between the MMA warp and the epilogue
constexpr int kABytes = 128 * 128;      // A stage: 128 rows x 64 bf16 ...
constexpr int kABytesWide = 136 * 128;  // ... or 136 rows when a segment loads wide boxes (8 halo pixels)
constexpr int kEpiWarps = 16;                 // 4 per TMEM lane quarter -> 4 warps per SM sub-partition
constexpr int kEpiSplit = kEpiWarps / 4;      // column parts per 64-channel chunk
constexpr int kEpiPart = 64 / kEpiSplit;      // columns per warp per chunk (16)
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kStoreWarp = 2 + kEpiWarps;     // warp 18: issues the epilogue's TMA stores (off the math warps' critical path)
constexpr int kThreads = 64 + kEpiThreads + 32;
constexpr int kOutBufs = 4;                   // staging buffers: 2 per epilogue group
constexpr uint32_t kTmemCols = 512;
constexpr int kOutBytes = 128 * 128;  // one 128-row x 64-channel bf16 staging buffer

struct SegK {
  int C, kh, kw, mul;
  int off_h[2], off_w[2];
  int c_per_tile, cchunks;
  int kc;  // chunk width (16/32/64 channels): swizzle 32B/64B/128B, 64/kc sub-blocks per stage
  int wide;  // 1: one (TW + kw - 1)-pixel box per tap ROW; the kw taps are shifted views of it
  int last_steps;  // K = 16 MMA steps of the LAST chunk that hold real channels (the rest of it is zero padding: skipped)
};

constexpr int kHeadMaxC = 64;  // channels per pixel a fused 1x1 head can read

struct __align__(64) ConvKParams {
  CUtensorMap tmA[OCTSEG_MAX_SEG];
  CUtensorMap tmB[3];  // weight boxes (kc x BN) for kc = 16, 32, 64
  CUtensorMap tmOut;  // bf16 NHWC output (4-D; 5-D phase-strided view in 4-phase mode)
  SegK seg[OCTSEG_MAX_SEG];
  int nseg, phases, N, Hq, Wq, TH, TW, tiles_h, tiles_w;
  int BN, n_tiles_n, cout_per_tile, Cout;
  int per_image_weights, act, res_mode, out_mode;
  int k_iters, nstages, total_tiles;
  int use_tma_store;
  int out_grouped;    // grouped conv with < 64 channels per group: 5-D output map (c in group, group, w, h, n), one chunk per tile
  int bias_floats;    // n_tiles_n * BN + 64 bias values staged in shared memory (rounded up to 4)
  int b_stage_bytes;  // bytes of one B stage (kw weight tiles for wide segments)
  int a_stage_bytes;  // kABytes, kABytesWide, or the halo tile (rounded up to 1 KB) in halo mode
  int d2s_tma;        // depth-to-space output through TMA: 64 % d2s == 0, one store per 2x2 sub-pixel of a 64-column chunk
  int own_spatial;    // 1: a CTA takes whole spatial tiles (all their channel tiles, back to back) -- see tile_at()
  int n_acc;          // accumulators in the TMEM ring (2 for BN = 256 ... 8 for BN <= 64)
  int halo;           // halo-tile mode: TH=16, TW=8, one halo box per channel chunk, resident weights
  int b_res_bytes;    // halo mode: bytes of one channel tile's weights (kh*kw*cchunks tiles of BN x 64)
  const float* bias;
  const __nv_bfloat16* res;
  int res_ldc;
  void* out;
  int out_H, out_W, out_ldc, out_c_off, out_pack, d2s;
  // fused 1x1 head (octseg.h): per packed pixel, head_classes dot products over its head_cmid activated channels
  // The head's operands live HERE, in the kernel-parameter constant bank: every FFMA of the epilogue reads its weight
  // as a constant operand (no shared-memory load, and the FMA pipe's two-register form: tools/ab/ffma_rate.cu).
  int head_classes, head_cmid;
  float head_w[4 * kHeadMaxC];  // [class][channel], zero padded
  float head_b[4];
  float head_cbias[kHeadMaxC];  // the conv's own per-channel bias (the same for every packed pixel)
  FastDiv fd_ntn, fd_phases, fd_tw, fd_th, fd_TW, fd_n, fd_ldc;
};

// ----------------------------------------------------------------------------- tcgen05 wrappers
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t leader, uint32_t bar) {
  asm volatile(
      "{\n.reg .pred q;\nsetp.ne.b32 q, %1, 0;\n"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n}" ::"r"(bar),
      "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t leader, uint32_t d_tmem, uint64_t adesc, uint64_t bdesc,
                                            uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n.reg .pred p, q;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "setp.ne.b32 q, %5, 0;\n"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major swizzled shared-memory matrix descriptor.  Rows are kc*2 bytes (32/64/128 = the swizzle
// span), 8-row groups are 8*kc*2 bytes apart (SBO).  layout_type: 2 = SWIZZLE_128B, 4 = 64B, 6 = 32B.
__device__ __forceinline__ uint64_t make_kmajor_desc(uint32_t saddr, int kc) {
  const uint32_t sbo = static_cast<uint32_t>(kc) * 16u;  // 8 rows * kc * 2 B
  const uint64_t layout = kc == 64 ? 2 : (kc == 32 ? 4 : 6);
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);  // start address
  d |= static_cast<uint64_t>(1) << 16;                 // leading byte offset (unused for swizzled K-major)
  d |= static_cast<uint64_t>(sbo >> 4) << 32;          // stride byte offset
  d |= static_cast<uint64_t>(1) << 46;                 // descriptor version (sm_100)
  d |= layout << 61;
  return d;
}
__device__ __forceinline__ int kc_index(int kc) { return kc == 64 ? 2 : (kc == 32 ? 1 : 0); }

__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// one MUFU per element: sigmoid(x) = 0.5*tanh(x/2) + 0.5, swish(x) = x*sigmoid(x) = h*tanh(h) + h with h = x/2
// (tanh.approx abs error ~5e-4 of full scale, below the bf16 output rounding)
__device__ __forceinline__ float apply_act(float x, int act) {
  if (act == OCTSEG_ACT_RELU) return fmaxf(x, 0.f);
  if (act == OCTSEG_ACT_SWISH) {
    const float h = 0.5f * x;
    return fmaf(h, fast_tanh(h), h);
  }
  if (act == OCTSEG_ACT_SIGMOID) return fmaf(0.5f, fast_tanh(0.5f * x), 0.5f);
  return x;
}

__device__ __forceinline__ void group_bar_sync(int group) {
  asm volatile("bar.sync %0, %1;" ::"r"(1 + group), "n"(kEpiThreads / 2) : "memory");
}

// bias + residual + activation of 8 consecutive channels of one pixel -> 8 packed bf16.
// The epilogue of the output-bound layers is issue-bound, so the per-element code is specialised at
// compile time on (activation, residual mode) and uses packed fp32x2 math (add/mul/fma.f32x2):
//   relu            : FADD2 + cvt.rn.relu.bf16x2            (1 issue slot per element)
//   swish           : FADD2, FMUL2, 2 MUFU.TANH, FFMA2, cvt  (3 per element)
//   residual (bf16) : + 2 unpack + FADD2 per pair
__device__ __forceinline__ uint32_t cvt_bf16x2(float2 x) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(x.y), "f"(x.x));
  return d;
}
__device__ __forceinline__ uint32_t cvt_bf16x2_relu(float2 x) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(x.y), "f"(x.x));
  return d;
}
__device__ __forceinline__ float2 bf16x2_to_f32x2(uint32_t w) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}

template <int ACT, int RES>
__device__ __forceinline__ uint4 epi8(const uint32_t* v, const float* bias8, const __nv_bfloat16* r8) {
  const float4 b0 = *reinterpret_cast<const float4*>(bias8);  // shared memory (staged once per CTA)
  const float4 b1 = *reinterpret_cast<const float4*>(bias8 + 4);
  float2 x[4];
  x[0] = __fadd2_rn(make_float2(__uint_as_float(v[0]), __uint_as_float(v[1])), make_float2(b0.x, b0.y));
  x[1] = __fadd2_rn(make_float2(__uint_as_float(v[2]), __uint_as_float(v[3])), make_float2(b0.z, b0.w));
  x[2] = __fadd2_rn(make_float2(__uint_as_float(v[4]), __uint_as_float(v[5])), make_float2(b1.x, b1.y));
  x[3] = __fadd2_rn(make_float2(__uint_as_float(v[6]), __uint_as_float(v[7])), make_float2(b1.z, b1.w));
  float2 r[4];
  if (RES != OCTSEG_RES_NONE) {
    uint4 rv = make_uint4(0u, 0u, 0u, 0u);
    if (r8) rv = __ldg(reinterpret_cast<const uint4*>(r8));
    r[0] = bf16x2_to_f32x2(rv.x);
    r[1] = bf16x2_to_f32x2(rv.y);
    r[2] = bf16x2_to_f32x2(rv.z);
    r[3] = bf16x2_to_f32x2(rv.w);
  }
  if (RES == OCTSEG_RES_BEFORE_ACT) {
#pragma unroll
    for (int e = 0; e < 4; ++e) x[e] = __fadd2_rn(x[e], r[e]);
  }
  if (ACT == OCTSEG_ACT_SWISH) {  // x*sigmoid(x) = h*tanh(h) + h, h = x/2
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 h = __fmul2_rn(x[e], make_float2(0.5f, 0.5f));
      x[e] = __ffma2_rn(h, make_float2(fast_tanh(h.x), fast_tanh(h.y)), h);
    }
  }
  uint4 ov;
  if (RES == OCTSEG_RES_AFTER_ACT) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (ACT == OCTSEG_ACT_RELU) x[e] = make_float2(fmaxf(x[e].x, 0.f), fmaxf(x[e].y, 0.f));
      x[e] = __fadd2_rn(x[e], r[e]);
    }
    ov = make_uint4(cvt_bf16x2(x[0]), cvt_bf16x2(x[1]), cvt_bf16x2(x[2]), cvt_bf16x2(x[3]));
  } else if (ACT == OCTSEG_ACT_RELU) {
    ov = make_uint4(cvt_bf16x2_relu(x[0]), cvt_bf16x2_relu(x[1]), cvt_bf16x2_relu(x[2]), cvt_bf16x2_relu(x[3]));
  } else {
    ov = make_uint4(cvt_bf16x2(x[0]), cvt_bf16x2(x[1]), cvt_bf16x2(x[2]), cvt_bf16x2(x[3]));
  }
  return ov;
}

#ifdef OCTSEG_TRACE
// Debug build only (tools/trace_conv.py): per-tile clock64 stamps of CTA 0's pipeline roles.
constexpr int kTraceTiles = 256, kTraceEvents = 16;
__device__ unsigned long long g_trace[kTraceEvents][kTraceTiles];
#define OCTSEG_STAMP(ev, it) \
  do { if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (it) < kTraceTiles) g_trace[ev][it] = clock64(); } while (0)
// per-chunk phases of epilogue group 0's first warp: 0 start, 1 TMEM loaded, 2 math done, 3 staging buffer free,
// 4 past barrier 1, 5 tile written + fenced + barrier 2, 6 store issued
__device__ unsigned long long g_trace_chunk[8][kTraceTiles];
__device__ int g_trace_chunk_n;
#define OCTSEG_CSTAMP(ev, k) \
  do { if (blockIdx.x == 0 && threadIdx.x == 64 && (k) < kTraceTiles) g_trace_chunk[ev][k] = clock64(); } while (0)
#else
#define OCTSEG_STAMP(ev, it) do { } while (0)
#define OCTSEG_CSTAMP(ev, k) do { } while (0)
#endif

struct TileCoord {
  int n_tile, tw, th, n, ph, pw, phase;
};
// Tile order: channel tile fastest (CTAs running together share the A tile in L2), then the four
// output phases of one spatial tile (they read the same input pixels), then space, then image.
__device__ __forceinline__ TileCoord decode_tile(const ConvKParams& p, int tile) {
  TileCoord c;
  uint32_t t = static_cast<uint32_t>(tile), q;
  if (p.halo) {  // channel tile slowest: its weights stay resident in shared memory across a CTA's tiles
    q = fd_div(t, p.fd_tw);
    c.tw = static_cast<int>(t - q * p.fd_tw.d);
    t = q;
    q = fd_div(t, p.fd_th);
    c.th = static_cast<int>(t - q * p.fd_th.d);
    t = q;
    q = fd_div(t, p.fd_n);
    c.n = static_cast<int>(t - q * p.fd_n.d);
    c.n_tile = static_cast<int>(q);
    c.phase = c.ph = c.pw = 0;
    return c;
  }
  q = fd_div(t, p.fd_ntn);
  c.n_tile = static_cast<int>(t - q * p.fd_ntn.d);
  t = q;
  q = fd_div(t, p.fd_phases);
  c.phase = static_cast<int>(t - q * p.fd_phases.d);
  t = q;
  q = fd_div(t, p.fd_tw);
  c.tw = static_cast<int>(t - q * p.fd_tw.d);
  t = q;
  q = fd_div(t, p.fd_th);
  c.th = static_cast<int>(t - q * p.fd_th.d);
  c.n = static_cast<int>(q);
  c.ph = c.phase >> 1;
  c.pw = c.phase & 1;
  return c;
}

// i-th tile of this CTA.  Default: tiles blockIdx, blockIdx + grid, ... (channel tile fastest, so CTAs running
// together share the A tile in L2).  With several channel tiles of UNEQUAL width per spatial tile that deal gives
// every CTA the same channel tile each time whenever grid % n_tiles_n == 0 (148 CTAs, 2 or 4 channel tiles): the
// CTAs holding the wide tile set the pace (288 channels = 192 + 96: 25 % lost).  own_spatial deals whole spatial
// tiles instead; the CTA runs their channel tiles back to back (its second A load is an L2 hit).
__device__ __forceinline__ int tile_at(const ConvKParams& p, int i) {
  if (!p.own_spatial) return static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
  const uint32_t q = fd_div(static_cast<uint32_t>(i), p.fd_ntn);
  const int r = i - static_cast<int>(q) * p.n_tiles_n;
  return (static_cast<int>(blockIdx.x) + static_cast<int>(q) * static_cast<int>(gridDim.x)) * p.n_tiles_n + r;
}

// Fused 1x1 segmentation head (octseg.h `head_classes`): a thread's accumulator row holds `out_pack` packed pixels x
// `head_cmid` channels, and each of the 4 warps of a lane quarter takes ONE of those pixels (with fewer packed pixels
// the warps take tiles in rotation).  Activate the pixel's channels (bias + ACT, fp32), fold them into its NC logits
// and store only those (fp32 logits, or the thresholded mask y > 0) into NCHW planes.  The epilogue is bound by
// instruction issue (4 warps per scheduler), so: NC is a template parameter (no predicated-off FMAs), channels go
// two at a time through FADD2 / FFMA2, and all indices into the parameter block are compile-time constants -- the
// weights are 64-bit constant-bank operands, never loaded into registers.
template <int ACT, int NC>
__device__ __forceinline__ void epilogue_head(const ConvKParams& p, uint32_t taddr, size_t idx0, size_t plane, bool valid) {
  float2 a2[NC];
#pragma unroll
  for (int jc = 0; jc < NC; ++jc) a2[jc] = make_float2(p.head_b[jc], 0.f);
  const float2* cb2 = reinterpret_cast<const float2*>(p.head_cbias);
  const float2* w2 = reinterpret_cast<const float2*>(p.head_w);
#pragma unroll
  for (int cb = 0; cb < kHeadMaxC; cb += 32) {
    if (cb < p.head_cmid) {  // warp-uniform
      uint32_t v[32];
      __syncwarp();  // tcgen05.ld is warp-collective
      if (p.head_cmid - cb >= 32) {
        tmem_ld32(taddr + cb, v);
      } else {
        uint32_t v16[16];
        tmem_ld16(taddr + cb, v16);
#pragma unroll
        for (int e = 0; e < 16; ++e) v[e] = v16[e];
#pragma unroll
        for (int e = 16; e < 32; ++e) v[e] = 0u;  // (zero bias and zero weights there in the parameter block)
      }
      tmem_ld_wait();
#pragma unroll
      for (int e = 0; e < 32; e += 2) {
        float2 y = __fadd2_rn(make_float2(__uint_as_float(v[e]), __uint_as_float(v[e + 1])), cb2[(cb + e) >> 1]);
        y.x = apply_act(y.x, ACT);
        y.y = apply_act(y.y, ACT);
#pragma unroll
        for (int jc = 0; jc < NC; ++jc) a2[jc] = __ffma2_rn(y, w2[(jc * kHeadMaxC + cb + e) >> 1], a2[jc]);
      }
    }
  }
  if (!valid) return;
#pragma unroll
  for (int jc = 0; jc < NC; ++jc) {
    if (jc >= p.head_classes) break;  // (NC = 4 also serves 3 classes)
    const float y = a2[jc].x + a2[jc].y;
    const size_t idx = idx0 + static_cast<size_t>(jc) * plane;
    if (p.out_mode == OCTSEG_OUT_F32_NCHW)
      reinterpret_cast<float*>(p.out)[idx] = y;
    else
      reinterpret_cast<uint8_t*>(p.out)[idx] = y > 0.f ? 1 : 0;
  }
}

template <int ACT, int RES, bool HEAD = false>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ ConvKParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int nst = p.nstages;
  const uint32_t b_bytes = static_cast<uint32_t>(p.b_stage_bytes);
  const uint32_t smemA = smem0;
  const uint32_t a_bytes = static_cast<uint32_t>(p.a_stage_bytes);
  const uint32_t smemB = smem0 + nst * a_bytes;
  // 2 x 16 KB epilogue staging (1 KB aligned: its 128B swizzle is address based)
  const uint32_t smemOut = smemB + (p.halo ? ((static_cast<uint32_t>(p.b_res_bytes) + 1023u) & ~1023u) : nst * b_bytes);
  const uint32_t smemBias = smemOut + kOutBufs * kOutBytes;  // fp32 bias of every channel tile
  const uint32_t bars = smemBias + p.bias_floats * 4;    // full[8] empty[8] tfull[2] tempty[2] tmem_ptr
  const uint32_t bar_full = bars, bar_empty = bars + 8 * kMaxStages;
  const uint32_t bar_tfull = bars + 16 * kMaxStages, bar_tempty = bar_tfull + 8 * kMaxAcc;
  const uint32_t bar_bres = bar_tempty + 8 * kMaxAcc;  // halo mode: resident weights landed
  const uint32_t bar_sfull = bar_bres + 8;              // [4] staging buffer written (256 arrivals of its group)
  const uint32_t bar_sfree = bar_sfull + 8 * kOutBufs;  // [4] its TMA store has read it (store warp)
  const uint32_t tmem_slot = bar_sfree + 8 * kOutBufs;
  uint8_t* smem_gen = smem_raw + (smem0 - smem_u32(smem_raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < nst; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < p.n_acc; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, kEpiWarps);  // one arrival per epilogue WARP (512 per-thread arrivals on one
                                              // barrier serialise: ~1000 cycles per tile, the floor of every small tile)
    }
    mbar_init(bar_bres, 1);
    for (int b = 0; b < kOutBufs; ++b) {
      mbar_init(bar_sfull + 8 * b, kEpiWarps / 2);
      mbar_init(bar_sfree + 8 * b, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {
    float* bs = reinterpret_cast<float*>(smem_gen + (smemBias - smem0));
    for (int i = threadIdx.x; i < p.bias_floats; i += kThreads) bs[i] = __ldg(p.bias + i);
  }
  if (p.TH * p.TW < 128) {
    // rows the TMA box never writes must still hold finite values for the MMA
    uint4* z = reinterpret_cast<uint4*>(smem_gen);
    const int n16 = nst * p.a_stage_bytes / 16;
    for (int i = threadIdx.x; i < n16; i += kThreads) z[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nseg; ++s) prefetch_tmap(&p.tmA[s]);
    for (int s = 0; s < 3; ++s) prefetch_tmap(&p.tmB[s]);
    if (p.use_tma_store) prefetch_tmap(&p.tmOut);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  uint32_t tmem_base;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot));

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (converged warp, elected issuer)
    {
      const uint32_t leader = elect_one_sync();
      int stage = 0;
      uint32_t phase = 0;
      int halo_nt = -1;  // halo mode: channel tile whose weights are resident
      // fast path for single-source 1x1 convs (the output-bound layers, one stage per tile): their per-tile
      // cost is this warp's serial setup, so the segment constants live in registers
      const bool simple = p.nseg == 1 && !p.halo && !p.seg[0].wide && p.seg[0].kh == 1 && p.seg[0].kw == 1 && p.phases == 1;
      const int s_kc = p.seg[0].kc, s_cch = p.seg[0].cchunks, s_mul = p.seg[0].mul, s_cpt = p.seg[0].c_per_tile;
      const int s_offh = p.seg[0].off_h[0], s_offw = p.seg[0].off_w[0], s_subs = 64 / s_kc;
      const uint32_t s_asub = 128u * s_kc * 2u, s_bsub = static_cast<uint32_t>(p.BN) * s_kc * 2u;
      const uint32_t s_tx = static_cast<uint32_t>(p.TH * p.TW + p.BN) * s_kc * 2u;
      const CUtensorMap* s_mb = &p.tmB[kc_index(s_kc)];
      for (int it = 0, tile; (tile = tile_at(p, it)) < p.total_tiles; ++it) {
        OCTSEG_STAMP(0, it);  // producer starts issuing this tile
        const TileCoord tc = decode_tile(p, tile);
        const int brow = tc.n_tile * p.BN;
        const int bz = tc.phase + p.phases * (p.per_image_weights ? tc.n : 0);
        int kofs = 0;
        if (simple) {
          // single-source 1x1 conv: everything but the tile origin was hoisted out of the tile loop
          const int h0 = s_mul * tc.th * p.TH + s_offh, w0 = s_mul * tc.tw * p.TW + s_offw;
          const int cbase = s_cpt * tc.n_tile;
          for (int cc = 0; cc < s_cch; cc += s_subs) {
            const int n = s_cch - cc < s_subs ? s_cch - cc : s_subs;
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            mbar_arrive_expect_tx_if(leader, bar_full + 8 * stage, s_tx * n);
            for (int j = 0; j < n; ++j) {
              tma_load_4d_if(leader, smemA + stage * a_bytes + j * s_asub, &p.tmA[0], bar_full + 8 * stage,
                             cbase + (cc + j) * s_kc, w0, h0, tc.n);
              tma_load_3d_if(leader, smemB + stage * b_bytes + j * s_bsub, s_mb, bar_full + 8 * stage, (cc + j) * s_kc, brow, bz);
            }
            if (++stage == nst) {
              stage = 0;
              phase ^= 1;
            }
          }
          continue;
        }
        if (p.halo) {
          const SegK& sg = p.seg[0];
          if (tc.n_tile != halo_nt) {
            // new channel tile: drain the ring (every MMA that reads the old weights has completed), then
            // load its kh*kw*cchunks weight tiles into the resident region
            if (halo_nt >= 0)
              for (int i = 0; i < nst; ++i) {
                const int st = stage + i < nst ? stage + i : stage + i - nst;
                mbar_wait(bar_empty + 8 * st, (stage + i < nst ? phase : phase ^ 1) ^ 1);
              }
            halo_nt = tc.n_tile;
            const int nb = sg.kh * sg.kw * sg.cchunks;
            mbar_arrive_expect_tx_if(leader, bar_bres, static_cast<uint32_t>(p.b_res_bytes));
            for (int i = 0; i < nb; ++i)
              tma_load_3d_if(leader, smemB + static_cast<uint32_t>(i * p.BN * sg.kc * 2), &p.tmB[kc_index(sg.kc)], bar_bres,
                             i * sg.kc, brow, 0);
          }
          const int h0 = tc.th * p.TH + sg.off_h[0], w0 = tc.tw * p.TW + sg.off_w[0];
          const int cbase = sg.c_per_tile * tc.n_tile;
          const uint32_t tx_bytes = static_cast<uint32_t>((p.TH + sg.kh - 1) * (p.TW + sg.kw - 1) * sg.kc * 2);
          for (int cc = 0; cc < sg.cchunks; ++cc) {
            OCTSEG_STAMP(10, it);
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            OCTSEG_STAMP(11, it);
            mbar_arrive_expect_tx_if(leader, bar_full + 8 * stage, tx_bytes);
            tma_load_4d_if(leader, smemA + stage * a_bytes, &p.tmA[0], bar_full + 8 * stage, cbase + cc * sg.kc, w0, h0, tc.n);
            OCTSEG_STAMP(12, it);
            if (++stage == nst) {
              stage = 0;
              phase ^= 1;
            }
          }
          continue;
        }
        for (int s = 0; s < p.nseg; ++s) {
          const SegK& sg = p.seg[s];
          const int h0 = sg.mul * tc.th * p.TH + sg.off_h[tc.ph];
          const int w0 = sg.mul * tc.tw * p.TW + sg.off_w[tc.pw];
          const int cbase = sg.c_per_tile * tc.n_tile;
          const int subs = 64 / sg.kc;                                   // sub-blocks per stage
          const uint32_t a_sub = 128u * sg.kc * 2u, b_sub = static_cast<uint32_t>(p.BN) * sg.kc * 2u;
          const uint32_t tx_sub = static_cast<uint32_t>(p.TH * p.TW + p.BN) * sg.kc * 2u;
          const CUtensorMap* mb = &p.tmB[kc_index(sg.kc)];
          if (sg.wide) {
            // one wide box per (tap row, chunk): the kw taps read it at pixel offsets 0..kw-1
            const CUtensorMap* ma = &p.tmA[s];
            const uint32_t tile_bytes = static_cast<uint32_t>(p.BN) * 128u;
            const uint32_t tx_bytes = static_cast<uint32_t>(p.TW + sg.kw - 1) * 128u + sg.kw * tile_bytes;
            for (int ty = 0; ty < sg.kh; ++ty) {
              for (int cc = 0; cc < sg.cchunks; ++cc) {
                mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                mbar_arrive_expect_tx_if(leader, bar_full + 8 * stage, tx_bytes);
                tma_load_4d_if(leader, smemA + stage * a_bytes, ma, bar_full + 8 * stage, cbase + cc * 64, w0, h0 + ty, tc.n);
                for (int tx = 0; tx < sg.kw; ++tx)
                  tma_load_3d_if(leader, smemB + stage * b_bytes + tx * tile_bytes, mb, bar_full + 8 * stage,
                              kofs + ((ty * sg.kw + tx) * sg.cchunks + cc) * 64, brow, bz);
                if (++stage == nst) {
                  stage = 0;
                  phase ^= 1;
                }
              }
            }
            kofs += sg.kh * sg.kw * sg.cchunks * 64;
            continue;
          }
          if (sg.kc == 64) {
            // hot path: one 64-channel box pair per stage
            const CUtensorMap* ma = &p.tmA[s];
            for (int ty = 0; ty < sg.kh; ++ty) {
              for (int tx = 0; tx < sg.kw; ++tx) {
                for (int cc = 0; cc < sg.cchunks; ++cc) {
                  OCTSEG_STAMP(10, it);  // decode + segment setup done
                  mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                  OCTSEG_STAMP(11, it);  // stage free
                  mbar_arrive_expect_tx_if(leader, bar_full + 8 * stage, tx_sub);
                  tma_load_4d_if(leader, smemA + stage * a_bytes, ma, bar_full + 8 * stage, cbase + cc * 64, w0 + tx, h0 + ty, tc.n);
                  tma_load_3d_if(leader, smemB + stage * b_bytes, mb, bar_full + 8 * stage, kofs, brow, bz);
                  OCTSEG_STAMP(12, it);  // loads issued
                  kofs += 64;
                  if (++stage == nst) {
                    stage = 0;
                    phase ^= 1;
                  }
                }
              }
            }
            continue;
          }
          int nsub = sg.kh * sg.kw * sg.cchunks;
          int ty = 0, tx = 0, cc = 0;
          while (nsub > 0) {
            const int n = nsub < subs ? nsub : subs;
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            mbar_arrive_expect_tx_if(leader, bar_full + 8 * stage, tx_sub * n);
            for (int j = 0; j < n; ++j) {
              tma_load_4d_if(leader, smemA + stage * a_bytes + j * a_sub, &p.tmA[s], bar_full + 8 * stage, cbase + cc * sg.kc,
                          w0 + tx, h0 + ty, tc.n);
              tma_load_3d_if(leader, smemB + stage * b_bytes + j * b_sub, mb, bar_full + 8 * stage, kofs, brow, bz);
              kofs += sg.kc;
              if (++cc == sg.cchunks) {
                cc = 0;
                if (++tx == sg.kw) {
                  tx = 0;
                  ++ty;
                }
              }
            }
            if (++stage == nst) {
              stage = 0;
              phase ^= 1;
            }
            nsub -= n;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (converged warp, elected issuer)
    {
      const uint32_t leader = elect_one_sync();
      // instruction descriptor: D=f32, A=B=bf16, both K-major, N=BN, M=128
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(p.BN >> 3) << 17) |
                             (static_cast<uint32_t>(128 >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int halo_nt = -1;
      uint32_t bres_phase = 0;
      const bool simple = p.nseg == 1 && !p.halo && !p.seg[0].wide && p.seg[0].kh == 1 && p.seg[0].kw == 1 && p.phases == 1;
      const int s_kc = p.seg[0].kc, s_cch = p.seg[0].cchunks, s_subs = 64 / s_kc, s_steps = s_kc / 16, s_last = p.seg[0].last_steps;
      const uint32_t s_asub = 128u * s_kc * 2u, s_bsub = static_cast<uint32_t>(p.BN) * s_kc * 2u;
      const uint64_t s_desc = make_kmajor_desc(0, s_kc);
      // halo mode: loop-invariant geometry of the single segment, hoisted out of the tile loop
      const uint32_t h_kh = p.seg[0].kh, h_kw = p.seg[0].kw, h_cch = p.seg[0].cchunks, h_pw = p.TW + p.seg[0].kw - 1;
      const uint32_t h_rb = p.seg[0].kc * 2;  // bytes per pixel of a chunk = the swizzle span (32 / 64 / 128)
      const uint32_t h_tile_bytes = static_cast<uint32_t>(p.BN) * h_rb;
      const int h_full = p.seg[0].kc / 16, h_last = p.seg[0].last_steps;
      // A: 8-pixel tile rows are the 8-row groups; group stride = one halo row (h_pw * h_rb bytes)
      const uint64_t h_desc_b = make_kmajor_desc(0, p.seg[0].kc);
      const uint64_t h_desc_a = (h_desc_b & ~(0x3FFFull << 32)) | (static_cast<uint64_t>((h_pw * h_rb) >> 4) << 32);
      for (int it = 0, tile; (tile = tile_at(p, it)) < p.total_tiles; ++it) {
        OCTSEG_STAMP(1, it);  // MMA warp ready for this tile
        mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
        tc_fence_after();
        OCTSEG_STAMP(2, it);  // accumulator free
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * p.BN);
        uint32_t accum = 0;  // 0 only for the very first MMA of the tile
        if (simple) {
          for (int cc = 0; cc < s_cch; cc += s_subs) {
            const int n = s_cch - cc < s_subs ? s_cch - cc : s_subs;
            mbar_wait(bar_full + 8 * stage, phase);
            tc_fence_after();
            for (int j = 0; j < n; ++j) {
              const uint64_t adesc = s_desc | ((smemA + stage * a_bytes + j * s_asub) >> 4);
              const uint64_t bdesc = s_desc | ((smemB + stage * b_bytes + j * s_bsub) >> 4);
              const int nsteps = cc + j == s_cch - 1 ? s_last : s_steps;
              for (int t = 0; t < nsteps; ++t) {  // K=16 per MMA: +32 B inside the swizzle span
                tc_mma_bf16(leader, d_tmem, adesc + 2 * t, bdesc + 2 * t, idesc, accum);
                accum = 1;
              }
            }
            tc_commit(leader, bar_empty + 8 * stage);
            if (++stage == nst) {
              stage = 0;
              phase ^= 1;
            }
          }
        } else if (p.halo) {
          const SegK& sg = p.seg[0];
          const int nt = static_cast<int>(fd_div(fd_div(fd_div(static_cast<uint32_t>(tile), p.fd_tw), p.fd_th), p.fd_n));
          if (nt != halo_nt) {  // this channel tile's weights: wait for the producer's resident load
            halo_nt = nt;
            mbar_wait(bar_bres, bres_phase);
            bres_phase ^= 1;
          }
          // Per-tap descriptors advance by ADDITIONS of loop-invariant strides kept in registers: with one K = 16 step
          // per tap (16-channel sources) the issue loop itself was the bottleneck (~240 cycles per tap with the
          // multiplies, parameter loads and vector->uniform moves of the first version; tools/trace_conv.py d2s16).
          const uint32_t a_tap = h_rb, a_row = (h_pw - h_kw) * h_rb, b_tap = h_cch * h_tile_bytes;
          for (int cc = 0; cc < h_cch; ++cc) {
            const int steps = cc == h_cch - 1 ? h_last : h_full;
            OCTSEG_STAMP(13, it);
            mbar_wait(bar_full + 8 * stage, phase);
            tc_fence_after();
            OCTSEG_STAMP(14, it);
            uint32_t a_addr = smemA + stage * a_bytes;
            uint32_t b_addr = smemB + static_cast<uint32_t>(cc) * h_tile_bytes;
            for (int ty = 0; ty < h_kh; ++ty) {
              for (int tx = 0; tx < h_kw; ++tx) {
                const uint64_t adesc = h_desc_a | (a_addr >> 4);
                const uint64_t bdesc = h_desc_b | (b_addr >> 4);
                for (int t = 0; t < steps; ++t) {  // K=16 per MMA: +32 B inside the swizzle span
                  tc_mma_bf16(leader, d_tmem, adesc + 2 * t, bdesc + 2 * t, idesc, accum);
                  accum = 1;
                }
                a_addr += a_tap;
                b_addr += b_tap;
              }
              a_addr += a_row;
            }
            tc_commit(leader, bar_empty + 8 * stage);
            OCTSEG_STAMP(15, it);
            if (++stage == nst) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
        for (int s = 0; s < ((p.halo || simple) ? 0 : p.nseg); ++s) {
          const int kc = p.seg[s].kc;
          int nsub = p.seg[s].kh * p.seg[s].kw * p.seg[s].cchunks;
          const uint64_t desc_hi = make_kmajor_desc(0, kc);
          if (p.seg[s].wide) {
            // tap tx = the same A stage read from pixel row tx on (128 B further).  The 128B swizzle is a
            // function of the absolute shared-memory address (measured: base-offset field must stay 0),
            // so a start address that is only 128-byte aligned still decodes what TMA wrote.
            const int kw = p.seg[s].kw;
            const uint32_t tile_bytes = static_cast<uint32_t>(p.BN) * 128u;
            const int cch = p.seg[s].cchunks, lsteps = p.seg[s].last_steps;
            int ccw = 0;  // chunk index of the current stage (stages run tap row major, chunk fastest)
            for (int st = p.seg[s].kh * cch; st > 0; --st) {
              mbar_wait(bar_full + 8 * stage, phase);
              tc_fence_after();
              const int nsteps = ccw == cch - 1 ? lsteps : 4;
              if (++ccw == cch) ccw = 0;
              for (int tx = 0; tx < kw; ++tx) {
                const uint64_t adesc = desc_hi | ((smemA + stage * a_bytes + tx * 128u) >> 4);
                const uint64_t bdesc = desc_hi | ((smemB + stage * b_bytes + tx * tile_bytes) >> 4);
                for (int t = 0; t < nsteps; ++t) {
                  tc_mma_bf16(leader, d_tmem, adesc + 2 * t, bdesc + 2 * t, idesc, accum);
                  accum = 1;
                }
              }
              tc_commit(leader, bar_empty + 8 * stage);
              if (++stage == nst) {
                stage = 0;
                phase ^= 1;
              }
            }
          } else if (kc == 64) {
            // hot path: one 64-channel sub-block per stage, four back-to-back MMAs
            const int cch = p.seg[s].cchunks, lsteps = p.seg[s].last_steps;
            int cck = 0;  // chunk index of the current sub-block (chunk fastest within a tap)
            for (; nsub > 0; --nsub) {
              OCTSEG_STAMP(13, it);
              mbar_wait(bar_full + 8 * stage, phase);
              tc_fence_after();
              OCTSEG_STAMP(14, it);  // operands landed
              const uint64_t adesc = desc_hi | ((smemA + stage * a_bytes) >> 4);
              const uint64_t bdesc = desc_hi | ((smemB + stage * b_bytes) >> 4);
              const bool full_chunk = lsteps == 4 || cck != cch - 1;
              if (++cck == cch) cck = 0;
              if (full_chunk) {
                tc_mma_bf16(leader, d_tmem, adesc, bdesc, idesc, accum);
                tc_mma_bf16(leader, d_tmem, adesc + 2, bdesc + 2, idesc, 1u);
                tc_mma_bf16(leader, d_tmem, adesc + 4, bdesc + 4, idesc, 1u);
                tc_mma_bf16(leader, d_tmem, adesc + 6, bdesc + 6, idesc, 1u);
              } else {  // the last chunk's K = 16 steps that are all zero padding are skipped
                for (int t = 0; t < lsteps; ++t) tc_mma_bf16(leader, d_tmem, adesc + 2 * t, bdesc + 2 * t, idesc, t ? 1u : accum);
              }
              accum = 1;
              tc_commit(leader, bar_empty + 8 * stage);
              OCTSEG_STAMP(15, it);  // MMAs issued, stage committed
              if (++stage == nst) {
                stage = 0;
                phase ^= 1;
              }
            }
          } else {
            const int subs = 64 / kc, steps = kc / 16;
            const uint32_t a_sub = 128u * kc * 2u, b_sub = static_cast<uint32_t>(p.BN) * kc * 2u;
            while (nsub > 0) {
              const int n = nsub < subs ? nsub : subs;
              mbar_wait(bar_full + 8 * stage, phase);
              tc_fence_after();
              for (int j = 0; j < n; ++j) {
                const uint64_t adesc = desc_hi | ((smemA + stage * a_bytes + j * a_sub) >> 4);
                const uint64_t bdesc = desc_hi | ((smemB + stage * b_bytes + j * b_sub) >> 4);
                for (int t = 0; t < steps; ++t) {  // K=16 per MMA: +32 B inside the swizzle span
                  tc_mma_bf16(leader, d_tmem, adesc + 2 * t, bdesc + 2 * t, idesc, accum);
                  accum = 1;
                }
              }
              tc_commit(leader, bar_empty + 8 * stage);
              if (++stage == nst) {
                stage = 0;
                phase ^= 1;
              }
              nsub -= n;
            }
          }
        }
        tc_commit(leader, bar_tfull + 8 * acc);
        OCTSEG_STAMP(3, it);  // all MMAs of the tile issued + committed
        if (++acc == p.n_acc) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp == kStoreWarp) {
    // ------------------------------------------------------------------ TMA-store issuer (one lane)
    // Replays the epilogue's (tile, chunk) sequence: waits until a group has written a staging buffer, stores it,
    // and hands the buffer back once the store has read it.  Issuing a tensor store costs its thread ~300 cycles
    // (measured, tools/trace_conv.py); on a math warp that sat on the critical path of every 64-channel chunk.
    if (lane == 0 && p.use_tma_store) {
      uint32_t chunk_ctr = 0, cnt0 = 0, cnt1 = 0;  // (two scalars, not an array: a dynamically indexed array lives in local memory)
      int pending = -1;  // buffer whose store was issued last (its read may still be in flight)
      for (int it = 0, tile; (tile = tile_at(p, it)) < p.total_tiles; ++it) {
        const TileCoord tc = decode_tile(p, tile);
        const int ch0 = tc.n_tile * p.cout_per_tile;
        const int nvalid = min(p.cout_per_tile, p.Cout - ch0);
        const int n_tma = p.out_grouped ? 1 : ((nvalid >> 6) + (((nvalid & 63) && ch0 + nvalid == p.Cout) ? 1 : 0));
        for (int ck = 0; ck < n_tma; ++ck) {
          const uint32_t g = (chunk_ctr + ck) & 1u;
          const uint32_t kg = g ? cnt1 : cnt0;
          cnt0 += g ^ 1u;
          cnt1 += g;
          const int buf = static_cast<int>(g * 2 + (kg & 1u));
          mbar_wait(bar_sfull + 8 * buf, (kg >> 1) & 1u);
          const uint32_t sbuf = smemOut + buf * kOutBytes;
          const int cch = p.out_c_off + ch0 + ck * 64;
          if (p.d2s_tma) {  // one box per 2x2 sub-pixel held by this chunk: (channels, pw, j, ph, n*Hq + i)
            const int nsub = 64 / p.d2s;
            for (int sl = 0; sl < nsub; ++sl) {
              const int sub = ck * nsub + sl;
              tma_store_5d(&p.tmOut, sbuf + static_cast<uint32_t>(sl * 128 * p.d2s * 2), 0, sub & 1, tc.tw * p.TW, sub >> 1,
                           tc.n * p.Hq + tc.th * p.TH);
            }
          } else if (p.out_grouped)
            tma_store_5d(&p.tmOut, sbuf, 0, tc.n_tile, tc.tw * p.TW, tc.th * p.TH, tc.n);
          else if (p.phases == 4)
            tma_store_5d(&p.tmOut, sbuf, cch, tc.pw, tc.tw * p.TW, tc.ph, tc.n * p.Hq + tc.th * p.TH);
          else
            tma_store_4d(&p.tmOut, sbuf, cch, tc.tw * p.TW, tc.th * p.TH, tc.n);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          if (pending >= 0) {
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");  // every store but the newest has read its buffer
            mbar_arrive(bar_sfree + 8 * pending);
          }
          pending = buf;
        }
        chunk_ctr += n_tma;
      }
      if (pending >= 0) {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        mbar_arrive(bar_sfree + 8 * pending);
      }
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores landed before exit
    }
  } else {
    // ------------------------------------------------------------------ epilogue
    const int q = warp & 3;             // TMEM lane quarter this warp may access (hardware: warp id % 4)
    const int part = (warp - 2) >> 2;   // direct-store path: which kEpiPart-column slice of every 64-column block
    const int group = (warp - 2) >> 3;  // TMA-store path: chunk-alternating group (8 warps each)
    const int half = part & 1;          //                 32-column half of the group's chunk
    const int gtid = (static_cast<int>(threadIdx.x) - 64) & 255;
    const int row = q * 32 + lane;
    const int th_l = static_cast<int>(fd_div(static_cast<uint32_t>(row), p.fd_TW)), tw_l = row - th_l * p.TW;
    // this thread's staging row; its four 16-byte slots are chunk (half*4 + g) ^ (row & 7) (128B swizzle)
    // (depth-to-space through TMA: a chunk holds 64 / d2s sub-pixels, each its own [128 rows][d2s channels] region
    //  with the 32 / 64 / 128-byte swizzle of its row length)
    const uint32_t sts_base0 = smemOut + group * 2 * kOutBytes;
    uint32_t grp_chunks = 0;  // chunks this group has staged so far (buffer = grp_chunks & 1)
    uint32_t sts_off[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (p.d2s_tma) {
        const int cs = p.d2s, cl = half * 32 + g * 8, sl = cl / cs, co = cl - sl * cs;
        const int swz = cs == 64 ? (row & 7) : (cs == 32 ? ((row >> 1) & 3) : ((row >> 2) & 1));
        sts_off[g] = static_cast<uint32_t>(sl * 128 * cs * 2 + row * cs * 2 + (((co >> 3) ^ swz) << 4));
      } else {
        sts_off[g] = static_cast<uint32_t>(row * 128 + (((half * 4 + g) ^ (row & 7)) << 4));
      }
    }
    int acc = 0;
    uint32_t acc_phase = 0, chunk_ctr = 0;
    int it = 0;
    [[maybe_unused]] const bool tracer = (threadIdx.x == 64) || (threadIdx.x == 64 + 256);  // first thread of each group
    [[maybe_unused]] const int tev = 4 + 3 * group;
    // With one channel tile the chunk layout is the same for every tile, so a group knows from the chunk
    // counter alone whether it owns a chunk of the next tile.  If it does not (single-chunk tiles: every
    // other tile) it only keeps its place in the accumulator ring -- no decode, no per-tile setup.
    const int nvalid1 = min(p.cout_per_tile, p.Cout);
    const int n_tma1 = p.use_tma_store ? ((nvalid1 >> 6) + ((nvalid1 & 63) ? 1 : 0)) : 0;
    const bool can_skip = (p.n_tiles_n == 1 || p.out_grouped) && n_tma1 * 64 >= nvalid1;
    // Narrow direct-store tiles (the NCHW heads: <= 32 output columns): one or two warps per lane quarter
    // cover a tile, so the 4 warps of a quarter take tiles in rotation instead of all walking every tile.
    // (fused-head tiles: one warp per lane quarter and packed pixel -- epilogue_head)
    constexpr bool headm = HEAD;                // (its own instantiation: the common epilogue keeps its register budget)
    const bool rot = p.n_tiles_n == 1 && n_tma1 == 0 && (headm || nvalid1 <= 2 * kEpiPart);
    const int rot_np = headm ? p.out_pack : (nvalid1 <= kEpiPart ? 1 : 2), rot_sets = kEpiSplit / rot_np;
    const int rot_set = part / rot_np, rot_slice = part - rot_set * rot_np;
    for (int tile; (tile = tile_at(p, it)) < p.total_tiles; ++it) {
      if (tracer) OCTSEG_STAMP(tev, it);  // epilogue group ready for this tile
      if ((can_skip && static_cast<int>((group ^ chunk_ctr) & 1u) >= n_tma1) || (rot && (it % rot_sets) != rot_set)) {
        mbar_wait(bar_tfull + 8 * acc, acc_phase);  // stay within the ring: arrivals must land in this tile's phase
        if (tracer) OCTSEG_STAMP(tev + 1, it);
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
        if (tracer) OCTSEG_STAMP(tev + 2, it);
        chunk_ctr += n_tma1;
        if (++acc == p.n_acc) {
          acc = 0;
          acc_phase ^= 1;
        }
        continue;
      }
      const TileCoord tc = decode_tile(p, tile);
      const int i = tc.th * p.TH + th_l, j = tc.tw * p.TW + tw_l;
      const bool valid = (row < p.TH * p.TW) && (i < p.Hq) && (j < p.Wq);
      const int oh = (p.phases == 4) ? 2 * i + tc.ph : i;
      const int ow = (p.phases == 4) ? 2 * j + tc.pw : j;
      const int ch0 = tc.n_tile * p.cout_per_tile;  // first real channel of this tile
      const int nvalid = min(p.cout_per_tile, p.Cout - ch0);
      const size_t pix = (static_cast<size_t>(tc.n) * p.out_H + oh) * p.out_W + ow;
      const float* bias = reinterpret_cast<const float*>(smem_gen + (smemBias - smem0)) + tc.n_tile * p.BN;
      const __nv_bfloat16* rrow = nullptr;
      if (RES != OCTSEG_RES_NONE && valid) rrow = p.res + pix * p.res_ldc + ch0;

      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tc_fence_after();
      if (tracer) OCTSEG_STAMP(tev + 1, it);  // accumulator full seen
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(acc * p.BN);

      // 64-channel chunks: registers -> swizzled shared tile -> one TMA store per chunk.  A partial last
      // chunk also goes this way when the tile ends at the tensor's channel extent (TMA clips it).
      // The 16 warps form two independent groups (own staging buffer, own named barrier) that take
      // alternate chunks, so one group's barrier / TMEM / store latency overlaps the other's math.
      // The math runs BEFORE the wait for the staging buffer, so the previous TMA store drains under it.
      const int n_tma =
          p.out_grouped ? 1
                        : (p.use_tma_store ? ((nvalid >> 6) + (((nvalid & 63) && ch0 + nvalid == p.Cout) ? 1 : 0)) : 0);
      for (int ck = 0; ck < n_tma; ++ck) {
        if (((chunk_ctr + ck) & 1) != static_cast<uint32_t>(group)) continue;  // warp-uniform
        const int cp = ck * 64 + half * 32;
        uint32_t v[32];
        [[maybe_unused]] const int ckey = static_cast<int>((chunk_ctr + ck) >> 1);
        OCTSEG_CSTAMP(0, ckey);
        tmem_ld32(taddr + cp, v);
        tmem_ld_wait();
        OCTSEG_CSTAMP(1, ckey);
        uint4 ov[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const int cc = cp + 8 * g;
          const __nv_bfloat16* r8 = (RES != OCTSEG_RES_NONE && rrow && cc < nvalid) ? rrow + cc : nullptr;
          ov[g] = epi8<ACT, RES>(v + 8 * g, bias + cc, r8);
        }
        OCTSEG_CSTAMP(2, ckey);
        const uint32_t sbi = static_cast<uint32_t>(group * 2) + (grp_chunks & 1u);
        mbar_wait(bar_sfree + 8 * sbi, ((grp_chunks >> 1) & 1u) ^ 1u);  // the store of this buffer's previous chunk has read it
        OCTSEG_CSTAMP(3, ckey);
        const uint32_t sts_base = sts_base0 + (grp_chunks & 1u) * kOutBytes;
#pragma unroll
        for (int g = 0; g < 4; ++g)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(sts_base + sts_off[g]), "r"(ov[g].x), "r"(ov[g].y),
                       "r"(ov[g].z), "r"(ov[g].w)
                       : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();                                       // every lane's rows written and fenced ...
        if (lane == 0) mbar_arrive(bar_sfull + 8 * sbi);    // ... 8 warp arrivals: the store warp issues the TMA store
        ++grp_chunks;
        OCTSEG_CSTAMP(4, ckey);
      }
      chunk_ctr += n_tma;

      if (headm) {
        const int wfull = p.out_W * p.out_pack;
        const size_t plane = static_cast<size_t>(p.out_H) * wfull;
        const size_t base = static_cast<size_t>(tc.n) * p.out_ldc * plane + static_cast<size_t>(oh) * wfull +
                            static_cast<size_t>(ow) * p.out_pack;
        OCTSEG_CSTAMP(0, it);
        OCTSEG_CSTAMP(1, it);
        OCTSEG_CSTAMP(2, it);
        const uint32_t ta = taddr + rot_slice * p.head_cmid;
        if (p.head_classes == 1)  // warp-uniform
          epilogue_head<ACT, 1>(p, ta, base + rot_slice, plane, valid);
        else if (p.head_classes == 2)
          epilogue_head<ACT, 2>(p, ta, base + rot_slice, plane, valid);
        else
          epilogue_head<ACT, 4>(p, ta, base + rot_slice, plane, valid);
        OCTSEG_CSTAMP(3, it);  // (trace columns: "wait_store" = the whole head epilogue of this tile)
        OCTSEG_CSTAMP(4, it);
        OCTSEG_CSTAMP(5, it);
        OCTSEG_CSTAMP(6, it);
      }
      // remaining channels (and every non-bf16 output): direct stores from registers
      for (int c0 = n_tma * 64; c0 < (headm ? 0 : nvalid); c0 += 64) {
        const int cp = rot ? rot_slice * kEpiPart : c0 + part * kEpiPart;
        if (cp >= nvalid) continue;  // warp-uniform
        uint32_t v[kEpiPart];
        __syncwarp();  // tcgen05.ld is warp-collective: reconverge after the predicated stores
        tmem_ld16(taddr + cp, v);
        tmem_ld_wait();
        if (!valid) {
          // row outside the image / tile: nothing to store
        } else if (p.out_mode == OCTSEG_OUT_BF16_NHWC) {
          __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(p.out) + pix * p.out_ldc + p.out_c_off + ch0 + cp;
#pragma unroll
          for (int g = 0; g < kEpiPart / 8; ++g) {
            if (cp + g * 8 < nvalid) {
              const __nv_bfloat16* r8 = (RES != OCTSEG_RES_NONE && rrow) ? rrow + cp + 8 * g : nullptr;
              __nv_bfloat16* og = o + g * 8;
              if (p.d2s) {  // depth-to-space: column -> (2x2 sub-pixel, channel) of a tensor twice the tile grid
                const int col = ch0 + cp + g * 8, sub = col / p.d2s, co = col - sub * p.d2s;
                const size_t opix = (static_cast<size_t>(tc.n) * 2 * p.out_H + 2 * oh + (sub >> 1)) * (2 * p.out_W) +
                                    2 * ow + (sub & 1);
                og = reinterpret_cast<__nv_bfloat16*>(p.out) + opix * p.out_ldc + p.out_c_off + co;
              }
              *reinterpret_cast<uint4*>(og) = epi8<ACT, RES>(v + 8 * g, bias + cp + 8 * g, r8);
            }
          }
        } else {
          // NCHW planes: lanes of a warp are consecutive pixels -> coalesced per channel plane
          // (pixel-packed problems: column c = plane c % out_ldc of pixel ow*out_pack + c / out_ldc)
          const int wfull = p.out_W * p.out_pack;
          const size_t plane = static_cast<size_t>(p.out_H) * wfull;
          const size_t base = static_cast<size_t>(tc.n) * p.out_ldc * plane + static_cast<size_t>(oh) * wfull +
                              static_cast<size_t>(ow) * p.out_pack;
#pragma unroll
          for (int e = 0; e < kEpiPart; ++e) {
            if (cp + e < nvalid) {
              const float y = apply_act(__uint_as_float(v[e]) + bias[cp + e], p.act);
              const int c = p.out_c_off + ch0 + cp + e;
              const int sub = static_cast<int>(fd_div(static_cast<uint32_t>(c), p.fd_ldc));  // c / out_ldc
              const size_t idx = base + static_cast<size_t>(c - sub * p.out_ldc) * plane + sub;
              if (p.out_mode == OCTSEG_OUT_F32_NCHW)
                reinterpret_cast<float*>(p.out)[idx] = y;
              else
                reinterpret_cast<uint8_t*>(p.out)[idx] = y > 0.f ? 1 : 0;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();  // every lane's TMEM reads are complete (tcgen05.wait::ld) before the warp's one arrival
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
      if (tracer) OCTSEG_STAMP(tev + 2, it);  // accumulator released
      if (++acc == p.n_acc) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols)
                 : "memory");
  }
}

// ----------------------------------------------------------------------------- host side
static int encode_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                      const uint64_t* strides_bytes, const uint32_t* box, const uint32_t* estr,
                      const char* what, int kc = 64) {
  return encode_tensor_map_bf16(map, base, rank, dims, strides_bytes, box, estr, kc * 2, 256, what);
}

}  // namespace octseg

struct octseg_conv_plan {
  octseg::ConvKParams kp;
  int grid;
  size_t smem;
};

using namespace octseg;

// epilogue specialisations: [activation none|relu|swish][residual none|before|after]
typedef void (*ConvKernelFn)(const ConvKParams);
static const ConvKernelFn kConvKernels[3][3] = {
    {conv_tc_kernel<OCTSEG_ACT_NONE, OCTSEG_RES_NONE>, conv_tc_kernel<OCTSEG_ACT_NONE, OCTSEG_RES_BEFORE_ACT>,
     conv_tc_kernel<OCTSEG_ACT_NONE, OCTSEG_RES_AFTER_ACT>},
    {conv_tc_kernel<OCTSEG_ACT_RELU, OCTSEG_RES_NONE>, conv_tc_kernel<OCTSEG_ACT_RELU, OCTSEG_RES_BEFORE_ACT>,
     conv_tc_kernel<OCTSEG_ACT_RELU, OCTSEG_RES_AFTER_ACT>},
    {conv_tc_kernel<OCTSEG_ACT_SWISH, OCTSEG_RES_NONE>, conv_tc_kernel<OCTSEG_ACT_SWISH, OCTSEG_RES_BEFORE_ACT>,
     conv_tc_kernel<OCTSEG_ACT_SWISH, OCTSEG_RES_AFTER_ACT>}};
// fused 1x1 head (no residual): [activation]
static const ConvKernelFn kConvHeadKernels[3] = {conv_tc_kernel<OCTSEG_ACT_NONE, OCTSEG_RES_NONE, true>,
                                                 conv_tc_kernel<OCTSEG_ACT_RELU, OCTSEG_RES_NONE, true>,
                                                 conv_tc_kernel<OCTSEG_ACT_SWISH, OCTSEG_RES_NONE, true>};

extern "C" int octseg_conv_plan_create(const octseg_conv_desc* d, octseg_conv_plan** out_plan) {
  if (!d || !out_plan) return fail(OCTSEG_EINVAL, "null argument");
  if (d->nseg < 1 || d->nseg > OCTSEG_MAX_SEG) return fail(OCTSEG_EINVAL, "nseg=%d out of range", d->nseg);
  if (d->phases != 1 && d->phases != 4) return fail(OCTSEG_EINVAL, "phases must be 1 or 4");
  if (d->BN < 16 || d->BN > 256 || d->BN % 16) return fail(OCTSEG_EINVAL, "BN=%d must be a multiple of 16 in [16,256]", d->BN);
  if (d->TH < 1 || d->TW < 1 || d->TH * d->TW > 128) return fail(OCTSEG_EINVAL, "tile %dx%d exceeds 128 pixels", d->TH, d->TW);
  if (d->cout_per_tile < 1 || d->cout_per_tile > d->BN) return fail(OCTSEG_EINVAL, "cout_per_tile=%d vs BN=%d", d->cout_per_tile, d->BN);
  if (d->out_mode == OCTSEG_OUT_BF16_NHWC &&
      (d->cout_per_tile % 8 || d->out_ldc % 8 || d->out_c_off % 8 || d->Cout % 8))
    return fail(OCTSEG_EINVAL, "bf16 NHWC output needs channel counts/pitches that are multiples of 8");
  if (d->res && (d->res_ldc % 8 || d->out_mode != OCTSEG_OUT_BF16_NHWC))
    return fail(OCTSEG_EINVAL, "residual needs bf16 NHWC output and a pitch that is a multiple of 8");
  if ((reinterpret_cast<uintptr_t>(d->weight) & 15) || (reinterpret_cast<uintptr_t>(d->out) & 15) ||
      (reinterpret_cast<uintptr_t>(d->bias) & 15) || (reinterpret_cast<uintptr_t>(d->res) & 15))
    return fail(OCTSEG_EINVAL, "weight/out/bias/res pointers must be 16-byte aligned");

  octseg_conv_plan* pl = new (std::nothrow) octseg_conv_plan;
  if (!pl) return fail(OCTSEG_EINVAL, "out of host memory");
  std::memset(pl, 0, sizeof(*pl));
  ConvKParams& kp = pl->kp;

  int k_iters = 0, k_total = 0, b_tiles = 1;
  bool any_wide = false;
  bool kc_used[3] = {false, false, false};
  for (int s = 0; s < d->nseg; ++s) {
    const octseg_conv_seg& sg = d->seg[s];
    if (sg.kc != 16 && sg.kc != 32 && sg.kc != 64) {
      delete pl;
      return fail(OCTSEG_EINVAL, "segment %d: kc=%d must be 16, 32 or 64", s, sg.kc);
    }
    if (sg.mul < 1 || sg.mul > 2 || sg.kh < 1 || sg.kw < 1 || sg.cchunks < 1 || sg.ldc % 8 ||
        (reinterpret_cast<uintptr_t>(sg.ptr) & 15) || sg.N != d->N) {
      delete pl;
      return fail(OCTSEG_EINVAL, "segment %d: bad geometry (mul=%d kh=%d kw=%d cchunks=%d ldc=%d N=%d)", s, sg.mul,
                  sg.kh, sg.kw, sg.cchunks, sg.ldc, sg.N);
    }
    const uint64_t dims[4] = {static_cast<uint64_t>(sg.C), static_cast<uint64_t>(sg.W), static_cast<uint64_t>(sg.H),
                              static_cast<uint64_t>(sg.N)};
    const uint64_t strides[3] = {static_cast<uint64_t>(sg.ldc) * 2, static_cast<uint64_t>(sg.W) * sg.ldc * 2,
                                 static_cast<uint64_t>(sg.H) * sg.W * sg.ldc * 2};
    if (sg.wide && (sg.kc != 64 || sg.mul != 1 || d->TH != 1 || sg.kw < 2 || d->TW + sg.kw - 1 > 136 ||
                    sg.c_per_tile != 0 && sg.cchunks != 1)) {
      delete pl;
      return fail(OCTSEG_EINVAL, "segment %d: wide boxes need kc=64, mul=1, TH=1, kw>=2 and TW+kw-1<=136", s);
    }
    if (d->halo && (d->nseg != 1 || d->phases != 1 || sg.mul != 1 || sg.wide || d->TH != 16 || d->TW != 8 ||
                    d->per_image_weights || sg.kh > 8 || sg.kw > 8)) {
      delete pl;
      return fail(OCTSEG_EINVAL, "halo mode needs nseg=1, phases=1, mul=1, TH=16, TW=8, shared weights");
    }
    const uint32_t box[4] = {static_cast<uint32_t>(sg.kc),
                             static_cast<uint32_t>(d->halo ? d->TW + sg.kw - 1 : (sg.wide ? d->TW + sg.kw - 1 : d->TW * sg.mul)),
                             static_cast<uint32_t>(d->halo ? d->TH + sg.kh - 1 : d->TH * sg.mul), 1u};
    const uint32_t estr[4] = {1u, static_cast<uint32_t>(sg.mul), static_cast<uint32_t>(sg.mul), 1u};
    int rc = encode_map(&kp.tmA[s], sg.ptr, 4, dims, strides, box, estr, "A", sg.kc);
    if (rc) {
      delete pl;
      return rc;
    }
    SegK& k = kp.seg[s];
    k.C = sg.C;
    k.kh = sg.kh;
    k.kw = sg.kw;
    k.mul = sg.mul;
    k.off_h[0] = sg.off_h[0];
    k.off_h[1] = sg.off_h[1];
    k.off_w[0] = sg.off_w[0];
    k.off_w[1] = sg.off_w[1];
    k.c_per_tile = sg.c_per_tile;
    k.cchunks = sg.cchunks;
    k.kc = sg.kc;
    k.wide = sg.wide ? 1 : 0;
    {
      const int c_eff = sg.c_per_tile > 0 ? sg.c_per_tile : sg.C;
      const int rem = c_eff - (sg.cchunks - 1) * sg.kc;
      const int ls = (rem + 15) / 16;
      k.last_steps = ls < 1 ? 1 : (ls > sg.kc / 16 ? sg.kc / 16 : ls);
    }
    if (sg.wide && sg.kw > b_tiles) b_tiles = sg.kw;
    if (sg.wide) any_wide = true;
    const int nsub = sg.kh * sg.kw * sg.cchunks, subs = 64 / sg.kc;
    k_iters += d->halo ? sg.cchunks : (sg.wide ? sg.kh * sg.cchunks : (nsub + subs - 1) / subs);
    k_total += nsub * sg.kc;
    kc_used[sg.kc == 64 ? 2 : (sg.kc == 32 ? 1 : 0)] = true;
  }
  if (k_total != d->Ktot) {
    delete pl;
    return fail(OCTSEG_EINVAL, "Ktot=%d does not match the segments' sum of kh*kw*cchunks*kc (%d)", d->Ktot, k_total);
  }
  {
    const uint64_t rows = static_cast<uint64_t>(d->n_tiles_n) * d->BN;
    const uint64_t Z = static_cast<uint64_t>(d->phases) * (d->per_image_weights ? d->N : 1);
    const uint64_t dims[3] = {static_cast<uint64_t>(d->Ktot), rows, Z};
    const uint64_t strides[2] = {static_cast<uint64_t>(d->Ktot) * 2, rows * d->Ktot * 2};
    const uint32_t estr[3] = {1u, 1u, 1u};
    for (int i = 0; i < 3; ++i) {
      const int kc = 16 << i;
      if (!kc_used[i]) {
        kp.tmB[i] = kp.tmA[0];  // never dereferenced; keeps the parameter block initialised
        continue;
      }
      const uint32_t box[3] = {static_cast<uint32_t>(kc), static_cast<uint32_t>(d->BN), 1u};
      int rc = encode_map(&kp.tmB[i], d->weight, 3, dims, strides, box, estr, "B", kc);
      if (rc) {
        delete pl;
        return rc;
      }
    }
  }
  kp.nseg = d->nseg;
  kp.phases = d->phases;
  kp.N = d->N;
  kp.Hq = d->Hq;
  kp.Wq = d->Wq;
  kp.TH = d->TH;
  kp.TW = d->TW;
  kp.tiles_h = cdiv(d->Hq, d->TH);
  kp.tiles_w = cdiv(d->Wq, d->TW);
  kp.BN = d->BN;
  kp.n_tiles_n = d->n_tiles_n;
  kp.cout_per_tile = d->cout_per_tile;
  kp.Cout = d->Cout;
  kp.per_image_weights = d->per_image_weights;
  kp.act = d->act;
  kp.res_mode = d->res ? d->res_mode : OCTSEG_RES_NONE;
  kp.out_mode = d->out_mode;
  kp.k_iters = k_iters;
  kp.bias = d->bias;
  kp.res = static_cast<const __nv_bfloat16*>(d->res);
  kp.res_ldc = d->res_ldc;
  kp.out = d->out;
  kp.out_H = d->out_H;
  kp.out_W = d->out_W;
  kp.out_ldc = d->out_ldc;
  kp.out_c_off = d->out_c_off;
  kp.out_pack = d->out_pack > 1 ? d->out_pack : 1;
  kp.d2s = d->d2s;
  if (d->d2s && (d->d2s % 8 || d->phases != 1 || d->res || d->out_mode != OCTSEG_OUT_BF16_NHWC)) {
    delete pl;
    return fail(OCTSEG_EINVAL, "d2s output needs bf16 NHWC, one phase, no residual and d2s %% 8 == 0");
  }
  kp.head_classes = kp.head_cmid = 0;
  memset(kp.head_w, 0, sizeof(kp.head_w));
  memset(kp.head_b, 0, sizeof(kp.head_b));
  memset(kp.head_cbias, 0, sizeof(kp.head_cbias));
  if (d->head_classes) {
    const int pk = kp.out_pack;
    if (d->head_classes < 1 || d->head_classes > 4 || d->head_cmid < 16 || d->head_cmid % 16 || d->head_cmid > kHeadMaxC ||
        !d->head_weight || !d->head_bias || !d->head_conv_bias || (pk != 1 && pk != 2 && pk != 4) || d->n_tiles_n != 1 ||
        d->phases != 1 || d->res || d->d2s || d->out_mode == OCTSEG_OUT_BF16_NHWC || d->Cout != pk * d->head_cmid ||
        d->BN < d->Cout || d->out_ldc != d->head_classes || d->out_c_off != 0) {
      delete pl;
      return fail(OCTSEG_EINVAL,
                  "fused head needs 1..4 classes, head_cmid in {16,32,48,64}, an NCHW out_mode with out_ldc = head_classes, "
                  "one channel tile of out_pack (1|2|4) x head_cmid columns, one phase, no residual");
    }
    kp.head_classes = d->head_classes;
    kp.head_cmid = d->head_cmid;
    for (int j = 0; j < d->head_classes; ++j) {
      kp.head_b[j] = d->head_bias[j];
      for (int c = 0; c < d->head_cmid; ++c) kp.head_w[j * kHeadMaxC + c] = d->head_weight[j * d->head_cmid + c];
    }
    for (int c = 0; c < d->head_cmid; ++c) kp.head_cbias[c] = d->head_conv_bias[c];
  }
  kp.total_tiles = d->phases * d->N * kp.tiles_h * kp.tiles_w * d->n_tiles_n;
  kp.fd_ntn = make_fastdiv(static_cast<uint32_t>(d->n_tiles_n));
  kp.fd_phases = make_fastdiv(static_cast<uint32_t>(d->phases));
  kp.fd_tw = make_fastdiv(static_cast<uint32_t>(kp.tiles_w));
  kp.fd_th = make_fastdiv(static_cast<uint32_t>(kp.tiles_h));
  kp.fd_TW = make_fastdiv(static_cast<uint32_t>(d->TW));
  kp.fd_n = make_fastdiv(static_cast<uint32_t>(d->N));
  kp.fd_ldc = make_fastdiv(static_cast<uint32_t>(d->out_ldc > 0 ? d->out_ldc : 1));
  {
    const long long lim = 1ll << 32;
    const long long t = kp.total_tiles;
    if (t * d->n_tiles_n >= lim || t * kp.tiles_w >= lim || t * kp.tiles_h >= lim || t * d->N >= lim) {
      delete pl;
      return fail(OCTSEG_EINVAL, "too many tiles (%lld) for the 32-bit tile decoder", t);
    }
  }
  if (d->act == OCTSEG_ACT_SIGMOID && d->out_mode == OCTSEG_OUT_BF16_NHWC) {
    delete pl;
    return fail(OCTSEG_EINVAL, "sigmoid is only available with the NCHW head outputs");
  }

  // narrow single-tile outputs (Cout < 64) also leave through one TMA chunk: the box is 64 channels wide
  // and TMA clips it at the tensor map's channel extent
  // channel tiles narrower than a chunk (grouped convs, e.g. 56 channels per group): the output is viewed
  // as (channel in group, group, w, h, n); the 64-wide store box is clipped at the group's extent
  kp.out_grouped = (d->out_mode == OCTSEG_OUT_BF16_NHWC && d->n_tiles_n > 1 && d->cout_per_tile < 64 && d->phases == 1 &&
                    d->d2s == 0 && d->Cout == d->n_tiles_n * d->cout_per_tile && (d->cout_per_tile * 2) % 16 == 0)
                       ? 1
                       : 0;
  kp.d2s_tma = (d->d2s && 64 % d->d2s == 0 && d->Hq % d->TH == 0 && d->BN == 4 * d->d2s && d->n_tiles_n == 1 && d->out_c_off == 0 &&
                d->out_ldc == d->d2s && d->Cout == 4 * d->d2s)
                   ? 1
                   : 0;
  kp.use_tma_store = (d->out_mode == OCTSEG_OUT_BF16_NHWC &&
                      (d->cout_per_tile >= 64 || d->n_tiles_n == 1 || kp.out_grouped) && (d->d2s == 0 || kp.d2s_tma) &&
                      (d->phases == 1 || (d->Hq % d->TH == 0 && d->out_H == 2 * d->Hq && d->out_W == 2 * d->Wq)))
                         ? 1
                         : 0;
  if (kp.out_grouped) {
    const uint64_t ld = static_cast<uint64_t>(d->out_ldc) * 2;
    const uint64_t dims[5] = {static_cast<uint64_t>(d->cout_per_tile), static_cast<uint64_t>(d->n_tiles_n),
                              static_cast<uint64_t>(d->out_W), static_cast<uint64_t>(d->out_H), static_cast<uint64_t>(d->N)};
    const uint64_t strides[4] = {static_cast<uint64_t>(d->cout_per_tile) * 2, ld, ld * d->out_W, ld * d->out_W * d->out_H};
    const uint32_t box[5] = {64u, 1u, static_cast<uint32_t>(d->TW), static_cast<uint32_t>(d->TH), 1u};
    const uint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
    const int rc = encode_map(&kp.tmOut, static_cast<const __nv_bfloat16*>(d->out) + d->out_c_off, 5, dims, strides, box, estr,
                              "out(grouped)");
    if (rc) {
      delete pl;
      return rc;
    }
  } else if (kp.d2s_tma) {
    // low-res pixel (i, j) of image n, sub-pixel (ph, pw): dims (c, pw, j, ph, n*Hq + i) of the 2x larger output
    const uint64_t ld = static_cast<uint64_t>(d->out_ldc) * 2, wout = 2ull * d->Wq;
    const uint64_t dims[5] = {static_cast<uint64_t>(d->d2s), 2u, static_cast<uint64_t>(d->Wq), 2u, static_cast<uint64_t>(d->N) * d->Hq};
    const uint64_t strides[4] = {ld, 2 * ld, ld * wout, 2 * ld * wout};
    const uint32_t box[5] = {static_cast<uint32_t>(d->d2s), 1u, static_cast<uint32_t>(d->TW), 1u, static_cast<uint32_t>(d->TH)};
    const uint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
    const int rc = encode_map(&kp.tmOut, d->out, 5, dims, strides, box, estr, "out(d2s)", d->d2s);
    if (rc) {
      delete pl;
      return rc;
    }
  } else if (kp.use_tma_store) {
    const uint64_t ld = static_cast<uint64_t>(d->out_ldc) * 2;
    const uint64_t cext = static_cast<uint64_t>(d->out_c_off + d->Cout);
    int rc;
    if (d->phases == 1) {
      const uint64_t dims[4] = {cext, static_cast<uint64_t>(d->out_W), static_cast<uint64_t>(d->out_H),
                                static_cast<uint64_t>(d->N)};
      const uint64_t strides[3] = {ld, ld * d->out_W, ld * d->out_W * d->out_H};
      const uint32_t box[4] = {64u, static_cast<uint32_t>(d->TW), static_cast<uint32_t>(d->TH), 1u};
      const uint32_t estr[4] = {1u, 1u, 1u, 1u};
      rc = encode_map(&kp.tmOut, d->out, 4, dims, strides, box, estr, "out");
    } else {
      // pixel (2i+ph, 2j+pw) of image n: dims (c, pw, j, ph, n*Hq + i)
      const uint64_t dims[5] = {cext, 2u, static_cast<uint64_t>(d->Wq), 2u, static_cast<uint64_t>(d->N) * d->Hq};
      const uint64_t strides[4] = {ld, 2 * ld, ld * d->out_W, 2 * ld * d->out_W};
      const uint32_t box[5] = {64u, 1u, static_cast<uint32_t>(d->TW), 1u, static_cast<uint32_t>(d->TH)};
      const uint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
      rc = encode_map(&kp.tmOut, d->out, 5, dims, strides, box, estr, "out(phase)");
    }
    if (rc) {
      delete pl;
      return rc;
    }
  }

  kp.n_acc = 512 / d->BN < kMaxAcc ? 512 / d->BN : kMaxAcc;
  kp.halo = d->halo ? 1 : 0;
  kp.b_res_bytes = 0;
  kp.b_stage_bytes = b_tiles * d->BN * 128;
  kp.a_stage_bytes = any_wide ? kABytesWide : kABytes;
  if (kp.halo) {
    const octseg_conv_seg& sg = d->seg[0];
    kp.b_res_bytes = sg.kh * sg.kw * sg.cchunks * d->BN * sg.kc * 2;
    kp.b_stage_bytes = 0;  // the stages hold halo tiles only
    kp.a_stage_bytes = ((d->TH + sg.kh - 1) * (d->TW + sg.kw - 1) * sg.kc * 2 + 1023) & ~1023;
  }
  const int stage_bytes = kp.a_stage_bytes + kp.b_stage_bytes;
  kp.bias_floats = (d->n_tiles_n * d->BN + 64 + 3) & ~3;
  const int b_res_region = (kp.b_res_bytes + 1023) & ~1023;
  const int budget = 227 * 1024 - 1024 - 512 - kOutBufs * kOutBytes - kp.bias_floats * 4 - b_res_region;
  int nst = budget / stage_bytes;
  if (nst > kMaxStages) nst = kMaxStages;
  if (nst < 2) {
    delete pl;
    return fail(OCTSEG_EINVAL, "tile does not fit shared memory");
  }
  kp.nstages = nst;
  pl->smem = static_cast<size_t>(nst) * stage_bytes + b_res_region + kOutBufs * kOutBytes + kp.bias_floats * 4 + 1024 + 512;
  int sms = octseg_sm_count();
  if (sms <= 0) {
    delete pl;
    return sms;
  }
  pl->grid = kp.total_tiles < sms ? kp.total_tiles : sms;
  // unequal channel tiles + plenty of spatial tiles: deal whole spatial tiles (tile_at)
  kp.own_spatial = (!kp.halo && d->n_tiles_n > 1 && d->Cout % d->cout_per_tile != 0 && pl->grid % d->n_tiles_n == 0 &&
                    kp.total_tiles / d->n_tiles_n >= 4 * sms)
                       ? 1
                       : 0;

  static bool attr_set = false;
  if (!attr_set) {
    for (int a = 0; a < 3; ++a)
      for (int r = 0; r < 4; ++r) {
        cudaError_t e = cudaFuncSetAttribute(r < 3 ? kConvKernels[a][r] : kConvHeadKernels[a],
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) {
          delete pl;
          return fail(OCTSEG_ECUDA, "cudaFuncSetAttribute(conv_tc_kernel): %s", cudaGetErrorString(e));
        }
      }
    attr_set = true;
  }
  *out_plan = pl;
  return OCTSEG_OK;
}

extern "C" int octseg_conv_plan_destroy(octseg_conv_plan* plan) {
  delete plan;
  return OCTSEG_OK;
}

extern "C" int octseg_conv_plan_info(const octseg_conv_plan* plan, struct octseg_conv_plan_info* info) {
  if (!plan || !info) return fail(OCTSEG_EINVAL, "null argument");
  const ConvKParams& kp = plan->kp;
  info->grid = plan->grid;
  info->total_tiles = kp.total_tiles;
  info->n_acc = kp.n_acc;
  info->nstages = kp.nstages;
  info->use_tma_store = kp.use_tma_store;
  info->out_grouped = kp.out_grouped;
  info->d2s_tma = kp.d2s_tma;
  info->own_spatial = kp.own_spatial;
  info->halo = kp.halo;
  info->wide = 0;
  for (int s = 0; s < kp.nseg; ++s) info->wide |= kp.seg[s].wide;
  return OCTSEG_OK;
}

#ifdef OCTSEG_TRACE
extern "C" int octseg_debug_trace(unsigned long long* h_out) {
  OCTSEG_CUDA(cudaMemcpyFromSymbol(h_out, octseg::g_trace, sizeof(unsigned long long) * kTraceEvents * kTraceTiles));
  return OCTSEG_OK;
}
extern "C" int octseg_debug_trace_chunks(unsigned long long* h_out) {
  OCTSEG_CUDA(cudaMemcpyFromSymbol(h_out, octseg::g_trace_chunk, sizeof(unsigned long long) * 8 * kTraceTiles));
  return OCTSEG_OK;
}
#endif

extern "C" int octseg_conv_run(const octseg_conv_plan* plan, void* stream) {
  if (!plan) return fail(OCTSEG_EINVAL, "null plan");
  if (plan->kp.total_tiles <= 0) return OCTSEG_OK;
  // sigmoid exists only on the NCHW head paths, which read p.act at run time
  const int a = plan->kp.act == OCTSEG_ACT_RELU ? 1 : (plan->kp.act == OCTSEG_ACT_SWISH ? 2 : 0);
  const ConvKernelFn fn = plan->kp.head_classes ? kConvHeadKernels[a] : kConvKernels[a][plan->kp.res_mode];
  fn<<<plan->grid, kThreads, plan->smem, static_cast<cudaStream_t>(stream)>>>(plan->kp);
  return check_launch("conv_tc_kernel");
}
