// Fused MBConv front half (backbones/efficientnet.py:110-173, stride 1, expand_ratio != 1), bf16 tensor-core mode:
//
//     e = SiLU(BN0(conv1x1(x)))          x: [B,H,W,Cin] bf16 NHWC, e: Cexp channels (never leaves the SM)
//     y = SiLU(BN1(dwconv3x3(e)))        written to HBM (bf16)
//     pooled[b][c] = mean_hw y[b,:,:,c]  squeeze-excitation squeeze, fp32
//
// as ONE persistent tcgen05 kernel for 16x16 and 8x8 maps.  A tile holds whole crops (16x16: one crop = 256 pixels = two
// M = 128 accumulators sharing B; 8x8: two crops = 128 pixels), so the depthwise halo is only the zero padding: it is kept as a
// zero ring in the shared-memory patch, written once.
//
//   warp 8       TMA producer: the tile's [pixels x Cin] input block once per tile (stays resident for all Cexp chunks), then
//                per 64-channel chunk the weight k-blocks through a ring of 8 KB stages (128B-swizzled, as tc_conv_kernel)
//   warp 9       TMEM allocator + single-thread tcgen05.mma issuer, accumulators double-buffered: chunk c+1's MMAs run while
//                the CUDA-core warps work on chunk c
//   warps 0-7    per chunk: TMEM -> halved bias + SiLU (the FFMA2 arithmetic of tc_conv_kernel's epilogue) -> bf16 -> patch;
//                depthwise strips over the patch (dw_strip, shared with dw3x3s1_tma_kernel) -> bf16 stores; SE sums.
//
// Work unit = (tile, chunk) job; CTA i runs one contiguous range of jobs (balanced to within one job), reloading the input block
// when its range crosses into the next tile.  The expanded tensor's HBM round trip of the two-launch path (expand GEMM write,
// depthwise read) is gone.  Results are bit-identical to tc_conv_kernel + dw3x3s1_tma_kernel: the same MMA K order (64-wide
// k-blocks zero-padded past Cin, K = 16 steps), the same epilogue and depthwise arithmetic, the same strip and crop sum orders.
#pragma once
#include "dw_tma.cuh"

namespace mtb {

constexpr int XD_THREADS = 320;           // warps 0-7 epilogue + depthwise, 8 TMA producer, 9 TMEM + MMA issuer
constexpr int XD_NC = 64;                 // expanded channels per chunk (MMA N)
constexpr int XD_B_BYTES = XD_NC * 128;   // one weight k-block of a chunk: 64 rows x 64 bf16
constexpr int XD_A_BLOCK = 128 * 128;     // one input k-block of 128 pixel rows
constexpr int XD_MAX_A = 128 * 1024;      // resident input budget (larger inputs would leave too few weight stages)
constexpr int XD_MAX_STAGES = 8;
constexpr int XD_SMEM_BUDGET = 226 * 1024;  // + 1 KB alignment slack = the 227 KB opt-in limit

struct ExpdwParams {
  __nv_bfloat16* out;   // depthwise output [B][H][W][Cexp]
  float* pooled;        // SE means [B][Cexp]
  const float* bias1;   // expand bias [Cexp] (BN folded)
  const float* wdw;     // depthwise weights [9][Cexp] (BN folded)
  const float* bdw;     // depthwise bias [Cexp]
  int B, Cexp, kchunks, nch, jobs;
  int nstages, ring_off, patch_off, red_off, bar_off;
  float inv_hw;
};

struct ExpdwPlan {  // shared-memory plan (byte offsets from the 1024-aligned base; the resident input block sits at offset 0)
  bool ok = false;
  int crops = 0, pixels = 0, a_bytes = 0, nstages = 0, ring_off = 0, patch_off = 0, red_off = 0, bar_off = 0, smem_bytes = 0;
};

inline ExpdwPlan expdw_plan(int H, int W, int Cin, int Cexp) {
  ExpdwPlan pl;
  if (H != W || (H != 16 && H != 8) || Cin < 16 || Cin % 8 != 0 || Cexp < XD_NC || Cexp % 8 != 0) return pl;
  const int nh = H == 16 ? 2 : 1;
  pl.crops = H == 16 ? 1 : 2;
  pl.pixels = 128 * nh;
  pl.a_bytes = nh * ((Cin + 63) / 64) * XD_A_BLOCK;
  if (pl.a_bytes > XD_MAX_A) return pl;
  const int patch = (pl.crops * (H + 2) * (W + 2) * 128 + 1023) / 1024 * 1024;
  const int red = pl.crops * (H * W / 16) * XD_NC * 4;
  const int ns = std::min(XD_MAX_STAGES, (XD_SMEM_BUDGET - pl.a_bytes - patch - red - 256) / XD_B_BYTES);
  if (ns < 3) return pl;
  pl.nstages = ns;
  pl.ring_off = pl.a_bytes;
  pl.patch_off = pl.ring_off + ns * XD_B_BYTES;
  pl.red_off = pl.patch_off + patch;
  pl.bar_off = pl.red_off + red;
  pl.smem_bytes = pl.bar_off + 256 + 1024;
  pl.ok = true;
  return pl;
}

template <bool MAP16>
__global__ void __launch_bounds__(XD_THREADS, 1)
expdw_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const ExpdwParams p) {
  constexpr int S = MAP16 ? 16 : 8;         // map side
  constexpr int G = MAP16 ? 1 : 2;          // crops per tile
  constexpr int NH = MAP16 ? 2 : 1;         // M = 128 accumulators per chunk
  constexpr int PW = S + 2;                 // patch side
  constexpr int SPC = S * S / 16;           // 4x4 strips per crop
  constexpr int NV = MAP16 ? 2 : 1;         // depthwise: fp32 pairs per thread (16x16: 4 channels, 8x8: 2), 256 threads busy
  constexpr int NVEC = XD_NC / (2 * NV);
  static_assert(NVEC * G * SPC == 256, "one depthwise strip job per epilogue thread");
  extern __shared__ uint8_t tc_smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)tc_smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + p.bar_off);
  uint64_t* full = bars;             // [8] weight stage landed
  uint64_t* empty = bars + 8;        // [8] weight stage consumed (commit)
  uint64_t* a_full = bars + 16;      // input block landed
  uint64_t* a_empty = bars + 17;     // input block consumed by the tile's last MMAs (commit)
  uint64_t* acc_full = bars + 18;    // [2]
  uint64_t* acc_empty = bars + 20;   // [2] one arrive per epilogue warp
  uint32_t* tmem_slot = (uint32_t*)(bars + 22);
  uint8_t* patch = smem + p.patch_off;
  float* red = (float*)(smem + p.red_off);  // [G * SPC strips][64 channels]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
  }
  if (warp == 9 && lane == 0) {
    for (int i = 0; i < 8; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    mbar_init(a_full, 1); mbar_init(a_empty, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], TCV_EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 9) tmem_alloc(tmem_slot, 256);
  // the halo ring of the patch is the conv's zero padding: zero the whole patch once, the interior is rewritten per chunk
  for (int i = threadIdx.x; i < G * PW * PW * 8; i += XD_THREADS) reinterpret_cast<uint4*>(patch)[i] = make_uint4(0u, 0u, 0u, 0u);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  pdl_trigger();
  pdl_wait();

  const int per = p.jobs / (int)gridDim.x, extra = p.jobs % (int)gridDim.x;
  const int j0 = (int)blockIdx.x * per + min((int)blockIdx.x, extra);
  const int j1 = j0 + per + ((int)blockIdx.x < extra ? 1 : 0);
  const int nch = p.nch, kchunks = p.kchunks;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty);
  const int nstages = p.nstages;

  if (warp == 8) {
    // ===== TMA producer =====
    uint32_t stage = 0, phase = 0, a_phase = 0;
    int cur_tile = -1;
    for (int j = j0; j < j1; ++j) {
      const int tile = j / nch, c = j - tile * nch;
      if (tile != cur_tile) {
        if (cur_tile >= 0) { mbar_wait_a(smem_u32(a_empty), a_phase); a_phase ^= 1; }
        if (elect_one()) {
          mbar_expect_tx_a(smem_u32(a_full), (uint32_t)(NH * kchunks * XD_A_BLOCK));
          for (int h = 0; h < NH; ++h)
            for (int kb = 0; kb < kchunks; ++kb)
              tma_load_2d_a(smem_base + (uint32_t)((h * kchunks + kb) * XD_A_BLOCK), &tmA, smem_u32(a_full), kb * 64, tile * (NH * 128) + h * 128);
        }
        __syncwarp();
        cur_tile = tile;
      }
#pragma unroll 1
      for (int kb = 0; kb < kchunks; ++kb) {
        mbar_wait_a(empty0 + stage * 8, phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx_a(full0 + stage * 8, (uint32_t)XD_B_BYTES);
          tma_load_2d_a(smem_base + (uint32_t)p.ring_off + stage * XD_B_BYTES, &tmB, full0 + stage * 8, kb * 64, c * XD_NC);
        }
        __syncwarp();
        if (++stage == (uint32_t)nstages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 9) {
    // ===== MMA issuer: per chunk, k-block by k-block, the four K = 16 steps of each of the NH accumulators =====
    constexpr uint32_t hi_sw = (uint32_t)((8 * 64 * 2) >> 4) | (1u << 14) | (2u << 29);  // SBO 1024 B | version | SWIZZLE_128B
    const uint32_t idesc = umma_idesc_bf16(XD_NC);
    const uint32_t a16 = smem_base >> 4, ring16 = (smem_base + (uint32_t)p.ring_off) >> 4;
    uint32_t stage = 0, phase = 0, a_phase = 0;
    int cur_tile = -1, l = 0;
    for (int j = j0; j < j1; ++j, ++l) {
      const int tile = j / nch;
      if (tile != cur_tile) { mbar_wait_a(smem_u32(a_full), a_phase); a_phase ^= 1; cur_tile = tile; }
      const uint32_t buf = (uint32_t)l & 1u;
      mbar_wait_a(smem_u32(&acc_empty[buf]), (((uint32_t)l >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d = tmem_base + buf * (NH * XD_NC);
#pragma unroll 1
      for (int kb = 0; kb < kchunks; ++kb) {
        mbar_wait_a(full0 + stage * 8, phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t b16 = ring16 + stage * (XD_B_BYTES >> 4);
#pragma unroll
          for (int h = 0; h < NH; ++h) {
            const uint32_t ah = a16 + (uint32_t)((h * kchunks + kb) * (XD_A_BLOCK >> 4));
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(d + h * XD_NC, make_desc(ah + 2 * k, hi_sw), make_desc(b16 + 2 * k, hi_sw), idesc, (uint32_t)(kb | k));
          }
          umma_commit_a(empty0 + stage * 8);
        }
        __syncwarp();
        if (++stage == (uint32_t)nstages) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) {
        umma_commit_a(smem_u32(&acc_full[buf]));
        if (j + 1 < j1 && (j + 1) / nch != tile) umma_commit_a(smem_u32(a_empty));  // the producer may load the next tile's input
      }
      __syncwarp();
    }
  } else {
    // ===== epilogue + depthwise warps (256 threads) =====
    const int tid = threadIdx.x;
    const int q = warp & 3, wg = warp >> 2;
    // expand epilogue: thread = one pixel (TMEM lane) of the tile; 16x16: warp group wg takes accumulator wg, all 64 columns;
    // 8x8: one accumulator, warp group wg takes columns [32 wg, +32)
    const int pt = (MAP16 ? wg * 128 : 0) + q * 32 + lane;
    const int pg = pt / (S * S), py = (pt / S) % S, px = pt % S;
    const int ppix = (pg * PW + py + 1) * PW + px + 1;
    const int col0 = MAP16 ? 0 : wg * 32;
    constexpr int NCOL = MAP16 ? 64 : 32;
    const uint32_t lane_taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(MAP16 ? wg * XD_NC : 0) + (uint32_t)col0;
    uint8_t* prow = patch + (size_t)ppix * 128;
    // depthwise: thread = (channel vector vj, strip slot sidx); slots run crop-major, band-major within a crop
    const int vj = tid % NVEC, sidx = tid / NVEC;
    const int sg = sidx / SPC, srem = sidx % SPC, band = srem / (S / 4), ow0 = (srem % (S / 4)) * 4;
    const int spix0 = (sg * PW + band * 4) * PW + ow0;
    const int Cexp = p.Cexp;
    int l = 0;
    for (int j = j0; j < j1; ++j, ++l) {
      const int tile = j / nch, cch = j - tile * nch;
      const int c = cch * XD_NC + vj * 2 * NV;  // this thread's first depthwise channel
      const bool c_ok = c < Cexp;
      // (1) accumulator -> bias + SiLU -> bf16 -> this pixel's row of the patch
      const uint32_t buf = (uint32_t)l & 1u;
      mbar_wait_a(smem_u32(&acc_full[buf]), ((uint32_t)l >> 1) & 1u);
      tc_fence_after();
      const uint32_t taddr = lane_taddr + buf * (NH * XD_NC);
      const float* b1 = p.bias1 + cch * XD_NC + col0;
#pragma unroll
      for (int hf = 0; hf < NCOL / 32; ++hf) {
        uint32_t v[32];
        tmem_ld16_issue(taddr + hf * 32, v);
        tmem_ld16_issue(taddr + hf * 32 + 16, v + 16);
        tmem_ld_wait();
#pragma unroll
        for (int gq = 0; gq < 4; ++gq) {
          const int ch8 = col0 + hf * 32 + gq * 8;  // first channel of this 16-byte chunk, inside the 64-channel chunk
          float4 bl = make_float4(0.f, 0.f, 0.f, 0.f), bh = bl;
          if (cch * XD_NC + ch8 < Cexp) {
            bl = __ldg(reinterpret_cast<const float4*>(b1 + hf * 32 + gq * 8));
            bh = __ldg(reinterpret_cast<const float4*>(b1 + hf * 32 + gq * 8 + 4));
          }
          // bias HALVED: SiLU(v + b) = h + h tanh(h), h = 0.5 v + 0.5 b (scaling by 0.5 is exact) - tc_conv_kernel's epilogue
          const f32x2 hb[4] = {f2_pack(0.5f * bl.x, 0.5f * bl.y), f2_pack(0.5f * bl.z, 0.5f * bl.w), f2_pack(0.5f * bh.x, 0.5f * bh.y),
                               f2_pack(0.5f * bh.z, 0.5f * bh.w)};
          const f32x2 half2 = f2_pack(0.5f, 0.5f);
          uint4 ov;
          __nv_bfloat162* o2 = reinterpret_cast<__nv_bfloat162*>(&ov);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const f32x2 h = f2_fma(f2_pack(__uint_as_float(v[gq * 8 + 2 * e]), __uint_as_float(v[gq * 8 + 2 * e + 1])), half2, hb[e]);
            float h0, h1, x0, x1;
            f2_unpack(h, h0, h1);
            f2_unpack(f2_fma(h, f2_pack(tanh_approx(h0), tanh_approx(h1)), h), x0, x1);
            o2[e] = __floats2bfloat162_rn(x0, x1);
          }
          *reinterpret_cast<uint4*>(prow + ((((ch8 >> 3) ^ (ppix & 7))) << 4)) = ov;
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);
      // this thread's depthwise taps + bias (loaded here, not earlier: live across the conversion they would spill)
      f32x2 w[9][NV], bias[NV];
#pragma unroll
      for (int t = 0; t < 9; ++t) {
        if constexpr (NV == 2) {
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (c_ok) v = __ldg(reinterpret_cast<const float4*>(p.wdw + (size_t)t * Cexp + c));
          w[t][0] = f2_pack(v.x, v.y); w[t][1] = f2_pack(v.z, v.w);
        } else {
          float2 v = make_float2(0.f, 0.f);
          if (c_ok) v = __ldg(reinterpret_cast<const float2*>(p.wdw + (size_t)t * Cexp + c));
          w[t][0] = f2_pack(v.x, v.y);
        }
      }
      if constexpr (NV == 2) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c_ok) v = __ldg(reinterpret_cast<const float4*>(p.bdw + c));
        bias[0] = f2_pack(v.x, v.y); bias[1] = f2_pack(v.z, v.w);
      } else {
        float2 v = make_float2(0.f, 0.f);
        if (c_ok) v = __ldg(reinterpret_cast<const float2*>(p.bdw + c));
        bias[0] = f2_pack(v.x, v.y);
      }

      asm volatile("bar.sync 1, 256;" ::: "memory");  // patch complete

      // (2) depthwise strip + its activated sums
      f32x2 psum[NV];
#pragma unroll
      for (int k = 0; k < NV; ++k) psum[k] = f2_pack(0.f, 0.f);
      const int b = tile * G + sg;
      if (c_ok && b < p.B) {
        __nv_bfloat16* obase = p.out + ((size_t)(b * S + band * 4) * S + ow0) * Cexp + c;
        dw_strip<ACT_SILU, __nv_bfloat16, NV, true>(patch, spix0, PW, vj * 4 * NV, DWT_RUN, DWT_OW, obase, (size_t)S * Cexp, (size_t)Cexp, w,
                                                    bias, psum);
      }
      float* rs = red + sidx * XD_NC + vj * 2 * NV;
#pragma unroll
      for (int k = 0; k < NV; ++k) f2_unpack(psum[k], rs[2 * k], rs[2 * k + 1]);
      asm volatile("bar.sync 1, 256;" ::: "memory");  // strip sums complete, patch free

      // (3) SE means: owner thread (crop, channel) adds its crop's strips in slot order: ((0 + s0) + s1) + ...
      if (tid < G * XD_NC) {
        const int g = tid / XD_NC, ch = tid % XD_NC;
        const int bb = tile * G + g, cc = cch * XD_NC + ch;
        float t = 0.f;
#pragma unroll
        for (int s = 0; s < SPC; ++s) t += red[(g * SPC + s) * XD_NC + ch];
        if (bb < p.B && cc < Cexp) p.pooled[(size_t)bb * Cexp + cc] = t * p.inv_hw;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ------------------------------------------------------------------------------------------------ host side
struct ExpdwWeights {
  bool ready = false;
  ExpdwPlan plan;
  int H = 0, W = 0, Cin = 0, Cexp = 0;
  const float *bias1 = nullptr, *wdw = nullptr, *bdw = nullptr;
  CUtensorMap mapB;
  mutable CUtensorMap mapA;
  mutable const void* cached_in = nullptr;
  mutable int cached_B = -1;
};

inline bool expdw_enabled() {  // MTB_EXPDW=0: the expand GEMM and the depthwise op run as two launches (A/B runs, tests)
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MTB_EXPDW");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

// expand: tensor-core weights of the 1x1 expand conv ([Cexp][Cin] bf16 K-major + bias); wdw / bdw: depthwise weights [9][Cexp]
inline const char* expdw_prepare(ExpdwWeights& x, const TcWeights& expand, const float* wdw, const float* bdw, int H, int W) {
  x.ready = false;
  x.plan = expdw_plan(H, W, expand.Cin, expand.Cout);
  if (!x.plan.ok || expand.taps != 1) return nullptr;
  x.H = H; x.W = W; x.Cin = expand.Cin; x.Cexp = expand.Cout;
  x.bias1 = expand.d_bias; x.wdw = wdw; x.bdw = bdw;
  const char* e = make_tmap_2d(&x.mapB, expand.d_w, (uint64_t)x.Cexp, (uint64_t)x.Cin, (uint32_t)XD_NC);
  if (e) return e;
  x.cached_in = nullptr; x.cached_B = -1;
  x.ready = true;
  return nullptr;
}

template <bool MAP16>
inline cudaError_t expdw_launch_k(int grid, int smem, const CUtensorMap& a, const CUtensorMap& b, const ExpdwParams& p, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(expdw_kernel<MAP16>, cudaFuncAttributeMaxDynamicSharedMemorySize, XD_SMEM_BUDGET + 1024);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  launch_k(expdw_kernel<MAP16>, dim3(grid), dim3(XD_THREADS), (size_t)smem, st, a, b, p);
  return cudaGetLastError();
}

inline const char* expdw_launch(const ExpdwWeights& x, const void* in, void* out, float* pooled, int B, cudaStream_t st) {
  if (x.cached_in != in || x.cached_B != B) {
    const char* e = make_tmap_2d(&x.mapA, in, (uint64_t)B * x.H * x.W, (uint64_t)x.Cin, 128u);
    if (e) return e;
    x.cached_in = in; x.cached_B = B;
  }
  const ExpdwPlan& pl = x.plan;
  ExpdwParams p;
  p.out = (__nv_bfloat16*)out; p.pooled = pooled; p.bias1 = x.bias1; p.wdw = x.wdw; p.bdw = x.bdw;
  p.B = B; p.Cexp = x.Cexp;
  p.kchunks = (x.Cin + 63) / 64;
  p.nch = (x.Cexp + XD_NC - 1) / XD_NC;
  p.jobs = (B + pl.crops - 1) / pl.crops * p.nch;
  p.nstages = pl.nstages; p.ring_off = pl.ring_off; p.patch_off = pl.patch_off; p.red_off = pl.red_off; p.bar_off = pl.bar_off;
  p.inv_hw = 1.0f / (float)(x.H * x.W);
  const int grid = std::min(p.jobs, 148);
  const cudaError_t e = x.H == 16 ? expdw_launch_k<true>(grid, pl.smem_bytes, x.mapA, x.mapB, p, st)
                                  : expdw_launch_k<false>(grid, pl.smem_bytes, x.mapA, x.mapB, p, st);
  return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

}  // namespace mtb
