// Depthwise k x k convolution (+ folded BN bias, swish, squeeze-excite channel sums) for the
// EfficientNet MBConv blocks (efficientnet_pytorch MBConvBlock._depthwise_conv with static "same"
// padding).  NHWC bf16 in and out, fp32 math.
//
// HBM-bound by nature (one read + one write per element, 9 or 25 FMAs), issue-bound in practice, so
// the design removes every instruction that is not an FMA, a conversion or the activation:
//   * persistent CTAs walk a contiguous range of (channel block, image, spatial tile) items; the
//     input tile WITH its halo is fetched by ONE TMA box per item into a 2-3 stage shared-memory
//     ring (zero fill outside the image = the conv padding, so there are no border branches and no
//     per-thread global address arithmetic); the next tiles' loads fly under the current tile's math;
//   * a thread owns 4 channels of a 2 x 4 output patch: every shared-memory read uses a compile-time
//     offset from one per-thread base, each input vector is converted bf16->fp32 once and feeds up to
//     min(2,K/S) x K taps (vertical + horizontal register reuse); math is fp32x2 pairs (FFMA2 for k = 3);
//   * fp32 filters of the CTA's channel block sit in shared memory, reloaded only when the block changes;
//   * squeeze-excite sums (of the fp32 activation, before the bf16 rounding) stay in registers across tiles and leave the CTA as one global atomic per
//     channel when the (image, channel block) changes.
//   (round 2: the sums leave as plain stores into one slot per (image, row group of tiles) -- summed in a fixed
//    order by octseg_se_hidden -- instead of fp32 atomics: bit-reproducible, and no buffer to re-zero.)
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

#include "common.h"
#include "ptx_sm100.h"

namespace octseg {

constexpr int kDwR = 2, kDwP = 4;  // output rows x pixels per thread

// Packed FFMA2 or two scalar FFMAs per channel pair.  Measured on B200 (tools/ab/ffma_rate.cu): FFMA2 with three
// register-pair operands sustains 43-56 FMA lanes/clk/SM, scalar three-register FFMA 73-83, so FFMA2 only pays where the
// kernel is bound by issue slots (k = 3), not by the FMA pipe (k = 5).
template <bool PACKED>
__device__ __forceinline__ float2 dw_fma2(float2 a, float2 b, float2 c) {
  if (PACKED) return __ffma2_rn(a, b, c);
  return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
}

// bf16 pair -> fp32 pair on the ALU pipe only (PRMT + LOP3): the compiler would turn `w << 16` into
// IMAD.U32, which competes with the FFMA2s for the FMA pipe this kernel is bound by
__device__ __forceinline__ float2 dw_bf16x2_to_f32x2(uint32_t w) {
  uint32_t lo;
  asm("prmt.b32 %0, %1, 0, 0x1044;" : "=r"(lo) : "r"(w));
  return make_float2(__uint_as_float(lo), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ uint32_t dw_cvt_bf16x2(float2 x) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(x.y), "f"(x.x));
  return d;
}
__device__ __forceinline__ float dw_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// acc[r][q][0..1] = bias + sum over the K x K taps for the thread's 2 x 4 patch x 4 channels, then the activation.
//   base : shared-memory address of the thread's window origin (its first row / pixel / channel quad)
//   w_off: shared-memory address of the thread's 4 channels in the fp32 filter table [K*K][CB] (16-byte aligned)
// With act == swish the filters and bias are pre-halved by the caller, so the accumulators hold h = x/2 and
// swish(x) = h*tanh(h) + h costs one FFMA2 + two MUFU per pair.
template <int K, int S, int CB, int IW, int PIX>
__device__ __forceinline__ void dw_patch(uint32_t base, uint32_t w_off, const float2 (&bias2)[2], int act,
                                         float2 (&acc)[kDwR][kDwP][2]) {
  constexpr int R = kDwR, P = kDwP;
  constexpr bool PK = K == 3;
  constexpr int RH = (R - 1) * S + K, RW = (P - 1) * S + K;  // a thread's input window
#pragma unroll
  for (int r = 0; r < R; ++r)
#pragma unroll
    for (int q = 0; q < P; ++q) {
      acc[r][q][0] = bias2[0];
      acc[r][q][1] = bias2[1];
    }
#pragma unroll
  for (int iy = 0; iy < RH; ++iy) {
    float2 w[R][K][2];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int ky = iy - r * S;
      if (ky >= 0 && ky < K) {
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
          float4 ww;
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                       : "=f"(ww.x), "=f"(ww.y), "=f"(ww.z), "=f"(ww.w)
                       : "r"(w_off + static_cast<uint32_t>((ky * K + kx) * CB * 4)));
          w[r][kx][0] = make_float2(ww.x, ww.y);
          w[r][kx][1] = make_float2(ww.z, ww.w);
        }
      }
    }
#pragma unroll
    for (int dx = 0; dx < RW; ++dx) {
      uint32_t r0, r1;
      asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];"
                   : "=r"(r0), "=r"(r1)
                   : "r"(base + static_cast<uint32_t>((iy * IW + dx) * PIX)));
      const float2 f0 = dw_bf16x2_to_f32x2(r0), f1 = dw_bf16x2_to_f32x2(r1);
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int ky = iy - r * S;
        if (ky >= 0 && ky < K) {
#pragma unroll
          for (int q = 0; q < P; ++q) {
            const int kx = dx - q * S;
            if (kx >= 0 && kx < K) {
              acc[r][q][0] = dw_fma2<PK>(f0, w[r][kx][0], acc[r][q][0]);
              acc[r][q][1] = dw_fma2<PK>(f1, w[r][kx][1], acc[r][q][1]);
            }
          }
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
#pragma unroll
    for (int q = 0; q < P; ++q) {
      float2 y0 = acc[r][q][0], y1 = acc[r][q][1];
      if (act == OCTSEG_ACT_SWISH) {  // the accumulators hold h = x/2
        y0 = __ffma2_rn(y0, make_float2(dw_tanh(y0.x), dw_tanh(y0.y)), y0);
        y1 = __ffma2_rn(y1, make_float2(dw_tanh(y1.x), dw_tanh(y1.y)), y1);
      } else if (act == OCTSEG_ACT_RELU) {
        y0 = make_float2(fmaxf(y0.x, 0.f), fmaxf(y0.y, 0.f));
        y1 = make_float2(fmaxf(y1.x, 0.f), fmaxf(y1.y, 0.f));
      }
      acc[r][q][0] = y0;
      acc[r][q][1] = y1;
    }
  }
}

constexpr int kDwThreads = 256;

struct DwParams {
  const __nv_bfloat16* weight;  // [K*K][C]
  const float* bias;            // [C]
  __nv_bfloat16* out;           // [N][Ho][Wo][C]
  float* pool_sum;              // [N][pool_slots][C] partial sums (slot = row group of tiles) or null
  int pool_slots;
  int C, Ho, Wo, pad_t, pad_l, act;
  // Work order.  A chunk = `chunk_tiles` consecutive tiles of one (image, channel block): one row of
  // tiles, or the whole plane on small maps.  Chunks are dealt round-robin to the persistent CTAs with
  // the channel block as the fastest chunk coordinate, so at any time the machine works on a thin band
  // of the input and consumes all channel blocks of its pixels together: halo rows and the other
  // channel blocks' bytes of every DRAM burst are still in L2 when the neighbouring CTA asks for them.
  int n_chunks, chunk_tiles, tiles_w;
  FastDiv fd_chunk_tiles, fd_tw, fd_cb, fd_rg;  // local index -> chunk; in-chunk index -> (row, tw); chunk -> (cb, row group, n)
  int chunk_rows;
};

template <int K, int S, int CB, int SH, int SW>
struct DwCfg {
  static constexpr int LANES = CB / 4;                         // threads per pixel (4 channels each)
  static_assert(LANES * SH * SW == kDwThreads, "thread layout");
  static constexpr int TH = SH * kDwR, TW = SW * kDwP;         // output tile
  static constexpr int IH = (TH - 1) * S + K, IW = (TW - 1) * S + K;  // input tile incl. halo
  static constexpr int PIX = CB * 2;                           // bytes per pixel in the tile
  static constexpr int STAGE = (IH * IW * PIX + 127) / 128 * 128;
  static constexpr int CTAS = S == 1 ? 2 : 1;  // resident CTAs per SM (registers + shared memory; 3 for k = 3 fits in 80 registers but measured 2 % slower)
  static constexpr int NST = S == 1 ? 3 : 2;   // (a 4-stage ring for k = 3 measured the same 4.0 TB/s)
  static constexpr int WSM = K * K * CB * 4;                   // fp32 filters
  static constexpr int PART = (kDwThreads / 32) * CB * 4;      // per-warp SE partial sums
  static constexpr int SMEM = NST * STAGE + WSM + PART + 64 + 128;  // + barriers + alignment slack
};

template <int K, int S, int CB, int SH, int SW>
__global__ void __launch_bounds__(kDwThreads, DwCfg<K, S, CB, SH, SW>::CTAS)
    dwconv_tma_kernel(const __grid_constant__ CUtensorMap tm_in, const DwParams p) {
  using Cfg = DwCfg<K, S, CB, SH, SW>;
  constexpr int R = kDwR, P = kDwP, LANES = Cfg::LANES, IW = Cfg::IW, PIX = Cfg::PIX, NST = Cfg::NST;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem0 = (smem_u32(smem_raw) + 127u) & ~127u;
  uint8_t* smem_gen = smem_raw + (smem0 - smem_u32(smem_raw));
  const uint32_t s_stage = smem0;
  const uint32_t s_w = smem0 + NST * Cfg::STAGE;
  float* wsm = reinterpret_cast<float*>(smem_gen + NST * Cfg::STAGE);           // [K*K][CB]
  float* part = reinterpret_cast<float*>(smem_gen + NST * Cfg::STAGE + Cfg::WSM);  // [8 warps][CB]
  const uint32_t s_bar = s_w + Cfg::WSM + Cfg::PART;

  const int tid = threadIdx.x, lane_c = tid % LANES, slot = tid / LANES;
  const int sy = slot / SW, sx = slot - sy * SW;
  const uint32_t in_off = static_cast<uint32_t>(((sy * R * S) * IW + sx * P * S) * PIX + lane_c * 8);
  const uint32_t w_off = s_w + static_cast<uint32_t>(lane_c * 16);

  // this CTA's work: chunks blockIdx.x, blockIdx.x + gridDim.x, ...; `n_local` tiles in all
  const int my_chunks = (p.n_chunks - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
  const int n_local = my_chunks * p.chunk_tiles;
  if (n_local <= 0) return;

  if (tid == 0) {
    for (int s = 0; s < NST; ++s) mbar_init(s_bar + 8 * s, 1);
    mbar_fence_init();
    prefetch_tmap(&tm_in);
  }
  __syncthreads();

  auto decode = [&](int i, int& cb, int& n, int& th, int& tw, int& rg) {  // i = local tile index
    const uint32_t ci = fd_div(static_cast<uint32_t>(i), p.fd_chunk_tiles);
    const uint32_t j = static_cast<uint32_t>(i) - ci * p.fd_chunk_tiles.d;
    const uint32_t chunk = blockIdx.x + ci * gridDim.x;
    const uint32_t jr = fd_div(j, p.fd_tw);
    tw = static_cast<int>(j - jr * p.fd_tw.d);
    uint32_t q = fd_div(chunk, p.fd_cb);
    cb = static_cast<int>(chunk - q * p.fd_cb.d);
    const uint32_t nn = fd_div(q, p.fd_rg);
    rg = static_cast<int>(q - nn * p.fd_rg.d);
    th = rg * p.chunk_rows + static_cast<int>(jr);
    n = static_cast<int>(nn);
  };
  auto issue = [&](int t, int stage) {  // one elected thread
    int cb, n, th, tw, rg;
    decode(t, cb, n, th, tw, rg);
    const uint32_t bar = s_bar + 8 * stage;
    mbar_arrive_expect_tx(bar, static_cast<uint32_t>(Cfg::IH * IW * PIX));
    tma_load_4d(s_stage + stage * Cfg::STAGE, &tm_in, bar, cb * CB, tw * Cfg::TW * S - p.pad_l,
                th * Cfg::TH * S - p.pad_t, n);
  };
  if (tid == 0)
    for (int i = 0; i < NST - 1 && i < n_local; ++i) issue(i, i);

  // swish(x) = h*tanh(h) + h with h = x/2: the halving is folded into the filters and the bias (exact: a
  // power of two), so the accumulators hold h and the activation is one FFMA2 + two MUFU per pair
  const float wscale = p.act == OCTSEG_ACT_SWISH ? 0.5f : 1.f;
  const uint32_t pix_bytes = static_cast<uint32_t>(p.C) * 2u;
  const size_t row_bytes = static_cast<size_t>(p.Wo) * pix_bytes;
  int cur_cb = -1, cur_n = -1, cur_rg = -1;
  float2 bias2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
  float2 ps[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
  bool cvalid = false;

  // SE sums of the finished chunk (image, row group, channel block): registers -> warp shuffle -> shared -> ONE plain
  // store per channel into the chunk's own slot (every slot is written exactly once per launch)
  auto flush_pool = [&](int n, int rg, int cb) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
#pragma unroll
      for (int o = LANES; o < 32; o <<= 1) {
        ps[e].x += __shfl_xor_sync(0xffffffffu, ps[e].x, o);
        ps[e].y += __shfl_xor_sync(0xffffffffu, ps[e].y, o);
      }
    }
    if ((tid & 31) < LANES) {
      float* d = part + (tid >> 5) * CB + lane_c * 4;
      d[0] = ps[0].x;
      d[1] = ps[0].y;
      d[2] = ps[1].x;
      d[3] = ps[1].y;
    }
    __syncthreads();
    if (tid < CB && cb * CB + tid < p.C) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kDwThreads / 32; ++w) s += part[w * CB + tid];
      p.pool_sum[(static_cast<size_t>(n) * p.pool_slots + rg) * p.C + cb * CB + tid] = s;
    }
    __syncthreads();
    ps[0] = ps[1] = make_float2(0.f, 0.f);
  };

  for (int it = 0; it < n_local; ++it) {
    int cb, n, th, tw, rg;
    decode(it, cb, n, th, tw, rg);
    if (tid == 0 && it + NST - 1 < n_local) issue(it + NST - 1, (it + NST - 1) % NST);
    if (p.pool_sum && cur_cb >= 0 && (cb != cur_cb || n != cur_n || rg != cur_rg)) flush_pool(cur_n, cur_rg, cur_cb);
    if (cb != cur_cb) {
      // the previous iteration ended with __syncthreads(): nobody still reads the old filters
      for (int i = tid; i < K * K * CB; i += kDwThreads) {
        const int tap = i / CB, cl = i - tap * CB, c = cb * CB + cl;
        wsm[i] = c < p.C ? wscale * __bfloat162float(p.weight[static_cast<size_t>(tap) * p.C + c]) : 0.f;
      }
      const int c = cb * CB + lane_c * 4;
      cvalid = c < p.C;
      if (cvalid) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + c));
        bias2[0] = make_float2(wscale * b.x, wscale * b.y);
        bias2[1] = make_float2(wscale * b.z, wscale * b.w);
      }
      __syncthreads();
      cur_cb = cb;
    }
    cur_n = n;
    cur_rg = rg;

    const int stage = it % NST;
    mbar_wait(s_bar + 8 * stage, static_cast<uint32_t>((it / NST) & 1));
    const uint32_t base = s_stage + stage * Cfg::STAGE + in_off;

    float2 acc[R][P][2];
    dw_patch<K, S, CB, IW, PIX>(base, w_off, bias2, p.act, acc);

    // bf16 store (8 bytes per pixel per thread; 16 lanes = one pixel's 128 bytes), SE sums
    const int oy0 = th * Cfg::TH + sy * R, ox0 = tw * Cfg::TW + sx * P;
    uint8_t* o0 = reinterpret_cast<uint8_t*>(p.out) +
                  static_cast<size_t>((n * p.Ho + oy0) * p.Wo + ox0) * pix_bytes + (cb * CB + lane_c * 4) * 2;
    if (cvalid && oy0 + R <= p.Ho && ox0 + P <= p.Wo) {  // interior patch: no per-pixel checks
#pragma unroll
      for (int r = 0; r < R; ++r) {
        uint8_t* orow = o0 + r * row_bytes;
#pragma unroll
        for (int q = 0; q < P; ++q) {
          *reinterpret_cast<uint2*>(orow + q * pix_bytes) =
              make_uint2(dw_cvt_bf16x2(acc[r][q][0]), dw_cvt_bf16x2(acc[r][q][1]));
          ps[0] = __fadd2_rn(ps[0], acc[r][q][0]);
          ps[1] = __fadd2_rn(ps[1], acc[r][q][1]);
        }
      }
    } else if (cvalid) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
#pragma unroll
        for (int q = 0; q < P; ++q) {
          if (oy0 + r < p.Ho && ox0 + q < p.Wo) {
            *reinterpret_cast<uint2*>(o0 + r * row_bytes + q * pix_bytes) =
                make_uint2(dw_cvt_bf16x2(acc[r][q][0]), dw_cvt_bf16x2(acc[r][q][1]));
            ps[0] = __fadd2_rn(ps[0], acc[r][q][0]);
            ps[1] = __fadd2_rn(ps[1], acc[r][q][1]);
          }
        }
      }
    }
    __syncthreads();  // every thread is done with this stage (and with `part`) before it is refilled
  }
  if (p.pool_sum) flush_pool(cur_n, cur_rg, cur_cb);
}

template <int K, int S, int CB, int SH, int SW>
static int launch_dw(const CUtensorMap& tm, DwParams p, int N, int cblocks, cudaStream_t st) {
  using Cfg = DwCfg<K, S, CB, SH, SW>;
  const int tiles_w = cdiv(p.Wo, Cfg::TW), tiles_h = cdiv(p.Ho, Cfg::TH);
  p.tiles_w = tiles_w;
  p.chunk_rows = tiles_w >= 4 ? 1 : tiles_h;          // a row of tiles, or the whole plane on small maps
  p.chunk_tiles = p.chunk_rows * tiles_w;
  const int row_groups = tiles_h / p.chunk_rows;
  if (p.pool_sum && p.pool_slots != row_groups)
    return fail(OCTSEG_EINVAL, "dwconv: pool_slots=%d but this shape writes %d slots (octseg_dwconv_pool_slots)", p.pool_slots, row_groups);
  const long long chunks = static_cast<long long>(row_groups) * N * cblocks;
  if (chunks * p.chunk_tiles >= (1ll << 24)) return fail(OCTSEG_EINVAL, "dwconv: too many tiles (%lld)", chunks * p.chunk_tiles);
  p.n_chunks = static_cast<int>(chunks);
  p.fd_chunk_tiles = make_fastdiv(static_cast<uint32_t>(p.chunk_tiles));
  p.fd_tw = make_fastdiv(static_cast<uint32_t>(tiles_w));
  p.fd_cb = make_fastdiv(static_cast<uint32_t>(cblocks));
  p.fd_rg = make_fastdiv(static_cast<uint32_t>(row_groups));
  const int sms = octseg_sm_count();
  if (sms <= 0) return sms;
  const int ctas = sms * Cfg::CTAS;
  const int grid = p.n_chunks < ctas ? p.n_chunks : ctas;
  static bool attr_set = false;
  if (!attr_set) {
    OCTSEG_CUDA(cudaFuncSetAttribute(dwconv_tma_kernel<K, S, CB, SH, SW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     Cfg::SMEM));
    attr_set = true;
  }
  dwconv_tma_kernel<K, S, CB, SH, SW><<<grid, kDwThreads, Cfg::SMEM, st>>>(tm, p);
  return check_launch("dwconv_tma_kernel");
}

}  // namespace octseg

using namespace octseg;

// tile geometry of octseg_dwconv for a shape: channel block, small-map flag, tile extent
static void dw_tile_config(int C, int Ho, int Wo, int& cb, bool& small, int& TH, int& TW) {
  cb = C <= 32 ? 32 : 64;
  small = cb == 64 && Ho <= 32 && Wo <= 32;  // 4 x 32 tiles waste less of 28 x 28 maps than 8 x 16
  const int sh = cb == 32 ? 4 : (small ? 2 : 4), sw = cb == 32 ? 8 : (small ? 8 : 4);
  TH = sh * kDwR;
  TW = sw * kDwP;
}

extern "C" int octseg_dwconv_pool_slots(int32_t C, int32_t Ho, int32_t Wo) {
  int cb, TH, TW;
  bool small;
  dw_tile_config(C, Ho, Wo, cb, small, TH, TW);
  const int tiles_w = cdiv(Wo, TW), tiles_h = cdiv(Ho, TH);
  return tiles_w >= 4 ? tiles_h : 1;
}

extern "C" int octseg_dwconv(const void* in, const void* weight, const float* bias, void* out, int32_t N, int32_t H,
                             int32_t W, int32_t C, int32_t k, int32_t stride, int32_t pad_t, int32_t pad_l,
                             int32_t Ho, int32_t Wo, int32_t act, float* pool_sum, int32_t pool_slots, void* stream) {
  if (C % 8) return fail(OCTSEG_EINVAL, "dwconv: C must be a multiple of 8 (C=%d)", C);
  if ((reinterpret_cast<uintptr_t>(in) & 15) || (reinterpret_cast<uintptr_t>(out) & 15) ||
      (reinterpret_cast<uintptr_t>(bias) & 15))
    return fail(OCTSEG_EINVAL, "dwconv: in/out/bias must be 16-byte aligned");
  if (act != OCTSEG_ACT_NONE && act != OCTSEG_ACT_RELU && act != OCTSEG_ACT_SWISH)
    return fail(OCTSEG_EINVAL, "dwconv: unsupported activation %d", act);
  const int cb = C <= 32 ? 32 : 64;
  const bool small = cb == 64 && Ho <= 32 && Wo <= 32;  // 4 x 32 tiles waste less of 28 x 28 maps than 8 x 16
  const int sh = cb == 32 ? 4 : (small ? 2 : 4), sw = cb == 32 ? 8 : (small ? 8 : 4);
  const int TH = sh * kDwR, TW = sw * kDwP;
  const int IH = (TH - 1) * stride + k, IW = (TW - 1) * stride + k;
  CUtensorMap tm;
  {
    const uint64_t dims[4] = {static_cast<uint64_t>(C), static_cast<uint64_t>(W), static_cast<uint64_t>(H),
                              static_cast<uint64_t>(N)};
    const uint64_t strides[3] = {static_cast<uint64_t>(C) * 2, static_cast<uint64_t>(W) * C * 2,
                                 static_cast<uint64_t>(H) * W * C * 2};
    const uint32_t box[4] = {static_cast<uint32_t>(cb), static_cast<uint32_t>(IW), static_cast<uint32_t>(IH), 1u};
    const uint32_t estr[4] = {1u, 1u, 1u, 1u};
    if (IW > 256 || IH > 256) return fail(OCTSEG_EINVAL, "dwconv: input tile %dx%d exceeds the TMA box limit", IH, IW);
    const int rc = encode_tensor_map_bf16(&tm, in, 4, dims, strides, box, estr, 0, 128, "dwconv input");
    if (rc) return rc;
  }
  DwParams p;
  p.weight = static_cast<const __nv_bfloat16*>(weight);
  p.bias = bias;
  p.out = static_cast<__nv_bfloat16*>(out);
  p.pool_sum = pool_sum;
  p.pool_slots = pool_slots;
  p.C = C;
  p.Ho = Ho;
  p.Wo = Wo;
  p.pad_t = pad_t;
  p.pad_l = pad_l;
  p.act = act;
  const int cblocks = cdiv(C, cb);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define OCTSEG_DW_SHAPE(KK, SS)                                                                   \
  (cb == 32 ? launch_dw<KK, SS, 32, 4, 8>(tm, p, N, cblocks, st)                                  \
            : (small ? launch_dw<KK, SS, 64, 2, 8>(tm, p, N, cblocks, st) : launch_dw<KK, SS, 64, 4, 4>(tm, p, N, cblocks, st)))
  if (k == 3 && stride == 1) return OCTSEG_DW_SHAPE(3, 1);
  if (k == 3 && stride == 2) return OCTSEG_DW_SHAPE(3, 2);
  if (k == 5 && stride == 1) return OCTSEG_DW_SHAPE(5, 1);
  if (k == 5 && stride == 2) return OCTSEG_DW_SHAPE(5, 2);
#undef OCTSEG_DW_SHAPE
  return fail(OCTSEG_EINVAL, "dwconv: unsupported kernel %d / stride %d", k, stride);
}
