// Depthwise 3x3 stride-1 conv + bias + activation + squeeze-excitation pooling for bf16 NHWC tensors (the MBConv middle
// op, backbones/efficientnet.py:110-173), staged through shared memory by TMA.
//
// Why: the strip kernel (dwconv3x3_pool_bf16_kernel) ran at ~2 TB/s whatever the batch (so not HBM-bound): every thread
// lived for ONE strip - one global-load round trip, then compute, then a block reduction - and nothing overlapped the
// load latency.  Here a persistent CTA walks (crop group, 64-channel group, row band) items; the (rows+2) x (W+2) x 64ch
// input patch of the NEXT item is in flight (one 4D TMA box, out-of-image halo = TMA zero fill = the reference's explicit
// zero padding, efficientnet.py:1127-1161) while the current one is computed from shared memory, each input row is read
// and unpacked once per 4-row run (input-stationary: a row updates the three output rows it feeds), and the SE means are
// reduced in a fixed order inside the CTA.
#pragma once
#include "tc_gemm.cuh"

namespace mtb {

constexpr int DWT_THREADS = 128;   // 8 channel vectors (8 ch each) x 16 strips per pass
constexpr int DWT_CG = 64;         // channels per item (128-byte pixel rows in shared memory)
constexpr int DWT_RUN = 4;         // output rows per thread run (RUN + 2 input rows)
constexpr int DWT_OW = 4;          // output columns per thread (OW + 2 input columns)
constexpr int DWT_STAGES = 2;
constexpr int DWT_MAX_STAGE = 52 * 1024;
constexpr int DWT_MAX_G = 8;

struct DwTmaParams {
  void* out;           // bf16 or fp32 NHWC
  const float* w;      // [9][C] fp32 (BN folded)
  const float* bias;   // [C]
  float* pooled;       // [n_rb][B][C] partial means (nullptr: no squeeze-excitation behind this op)
  int B, H, W, C;
  int pad_t, pad_l;
  int G, BH;           // crops per item, output rows per item
  int n_cg, n_rb, items;
  int strips_w, bands, nstrips;  // per item: column strips, row runs per crop, G * bands * strips_w
  int stage_bytes;
  float inv_hw;
  int rev;             // walk the items last-to-first (see dw_tma_launch)
};

struct DwTmaPlan {
  bool ok = false;
  int G = 1, BH = 0, n_rb = 1;
};

// (crops per item, rows per item): maximise (busy strip slots) x (useful rows / staged rows) within the stage budget
inline DwTmaPlan dw_tma_plan(int H, int W) {
  DwTmaPlan best;
  double best_score = -1.0;
  const int PW = W + 2;
  const int strips_w = (W + DWT_OW - 1) / DWT_OW;
  if (PW > 256) return best;
  for (int BH = DWT_RUN; BH <= H + DWT_RUN - 1; BH += DWT_RUN) {
    const int bh = BH > H ? H : BH;
    if (bh + 2 > 256) break;
    const long patch = 128L * PW * (bh + 2);
    if (patch > DWT_MAX_STAGE) break;
    const int gmax = (int)std::min<long>(DWT_MAX_G, DWT_MAX_STAGE / patch);
    const int bands = (bh + DWT_RUN - 1) / DWT_RUN;
    const int n_rb = (H + bh - 1) / bh;
    for (int G = 1; G <= (n_rb == 1 ? gmax : 1); ++G) {
      const int nstrips = G * bands * strips_w;
      const double eff = (double)nstrips / (16.0 * ((nstrips + 15) / 16));
      const double score = eff * bh / (bh + 2.0) - 1e-3 * G;
      if (score > best_score) {
        best_score = score;
        best.ok = true; best.G = G; best.BH = bh; best.n_rb = n_rb;
      }
    }
  }
  return best;
}

// rank-4 NHWC tensor [B][H][W][C] (bf16: es = 2, fp32: es = 4); box = 128 bytes of channels (64 bf16 / 32 fp32) x (W+2) x
// (BH+2) x G, no swizzle (quarter-warps read whole 128-byte pixel rows: conflict-free as is)
inline const char* make_tmap_dw(CUtensorMap* m, const void* ptr, uint64_t B, uint64_t H, uint64_t W, uint64_t C, uint32_t pw,
                                uint32_t ph, uint32_t g, uint32_t es = 2) {
  tmap_encode_fn enc = get_tmap_encode();
  if (!enc) return "cuTensorMapEncodeTiled unavailable";
  cuuint64_t dims[4] = {C, W, H, B};
  cuuint64_t strides[3] = {C * es, W * C * es, H * W * C * es};
  cuuint32_t box[4] = {128 / es, pw, ph, g};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, es == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? nullptr : "cuTensorMapEncodeTiled(dw) failed";
}

// activation of a pair; SiLU(x) = h + h * tanh(h), h = x / 2 (same arithmetic as fast_act<ACT_SILU>)
template <int ACT>
__device__ __forceinline__ f32x2 f2_act(f32x2 x) {
  if constexpr (ACT == ACT_SILU) {
    const f32x2 h = f2_mul(x, f2_pack(0.5f, 0.5f));
    float h0, h1;
    f2_unpack(h, h0, h1);
    return f2_fma(h, f2_pack(fast_tanh(h0), fast_tanh(h1)), h);
  } else {
    float x0, x1;
    f2_unpack(x, x0, x1);
    return f2_pack(fast_act<ACT>(x0), fast_act<ACT>(x1));
  }
}

// n 32-bit words from / to shared or global memory as one vector access (n = 1, 2 or 4)
template <int N>
__device__ __forceinline__ void ld_words(const void* a, unsigned (&wd)[N]) {
  if constexpr (N == 4) { const uint4 r = *reinterpret_cast<const uint4*>(a); wd[0] = r.x; wd[1] = r.y; wd[2] = r.z; wd[3] = r.w; }
  else if constexpr (N == 2) { const uint2 r = *reinterpret_cast<const uint2*>(a); wd[0] = r.x; wd[1] = r.y; }
  else { wd[0] = *reinterpret_cast<const unsigned*>(a); }
}
template <int N>
__device__ __forceinline__ void st_words(void* a, const unsigned (&wd)[N]) {
  if constexpr (N == 4) *reinterpret_cast<uint4*>(a) = make_uint4(wd[0], wd[1], wd[2], wd[3]);
  else if constexpr (N == 2) *reinterpret_cast<uint2*>(a) = make_uint2(wd[0], wd[1]);
  else *reinterpret_cast<unsigned*>(a) = wd[0];
}

// One strip of the depthwise 3x3 stride-1 conv: rows_run (<= DWT_RUN) output rows x DWT_OW output columns x 2*NV channels,
// row-input-stationary (each of the rows_run + 2 input rows is read and unpacked once and updates the three output rows it
// feeds).  Every output starts its FMA chain from the bias and takes the taps in row-major order; then activation, store, and
// the activated fp32 values are added to psum in row-major order.  Shared by dw3x3s1_tma_kernel and expdw_kernel, so that
// both compute every output and every strip sum the same way.
//   patch: 128-byte pixel rows, PW pixels per patch row; pix0 = patch pixel of the strip's top-left input;
//   cbyte: byte offset of this thread's channels inside a pixel row; SWZ: 16-byte chunk k of patch pixel x sits at chunk
//   position k ^ (x & 7) (expdw_kernel: its TMEM-lane = pixel stores are bank-conflict free that way);
//   ncols: valid output columns of the strip; obase: output of (first row, first column, first channel).
template <int ACT, typename T, int NV, bool SWZ>
__device__ __forceinline__ void dw_strip(const uint8_t* patch, int pix0, int PW, int cbyte, int rows_run, int ncols, T* obase,
                                         size_t row_stride, size_t px_stride, const f32x2 (&w)[9][NV], const f32x2 (&bias)[NV],
                                         f32x2 (&psum)[NV]) {
  constexpr bool F32 = sizeof(T) == 4;
  constexpr int NW = F32 ? 2 * NV : NV;  // 32-bit words per pixel of this thread
  f32x2 acc[3][DWT_OW][NV];
#pragma unroll
  for (int pr = 0; pr < DWT_RUN + 2; ++pr) {
    if (pr < rows_run + 2) {
      // input row pr of the run is tap row r of output row pr - r (slot (pr - r) % 3); the first tap of an output row
      // (r = 0, s = 0) starts from the bias
#pragma unroll
      for (int x = 0; x < DWT_OW + 2; ++x) {
        const int pix = pix0 + pr * PW + x;
        const int off = SWZ ? ((((cbyte >> 4) ^ (pix & 7)) << 4) | (cbyte & 15)) : cbyte;
        unsigned wd[NW];
        ld_words<NW>(patch + (size_t)pix * 128 + off, wd);
        f32x2 v[NV];
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          if constexpr (F32) v[k] = f2_pack(__uint_as_float(wd[2 * k]), __uint_as_float(wd[2 * k + 1]));
          else v[k] = f2_pack(__uint_as_float(wd[k] << 16), __uint_as_float(wd[k] & 0xffff0000u));
        }
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const int o = pr - r;  // compile-time
          if (o < 0 || o >= DWT_RUN) continue;
#pragma unroll
          for (int i = 0; i < DWT_OW; ++i) {
            const int s_ = x - i;  // compile-time
            if (s_ >= 0 && s_ < 3) {
#pragma unroll
              for (int k = 0; k < NV; ++k)
                acc[o % 3][i][k] = f2_fma(v[k], w[r * 3 + s_][k], (r == 0 && s_ == 0) ? bias[k] : acc[o % 3][i][k]);
            }
          }
        }
      }
      // output row pr - 2 is complete
      if (pr >= 2 && pr - 2 < rows_run) {
        const int o = pr - 2, slot = o % 3;
        T* orow = obase + (size_t)o * row_stride;
#pragma unroll
        for (int i = 0; i < DWT_OW; ++i) {
          if (i < ncols) {
            unsigned ov[NW];
#pragma unroll
            for (int k = 0; k < NV; ++k) {
              if constexpr (F32) {
                float x0, x1;
                f2_unpack(acc[slot][i][k], x0, x1);
                const float a0 = act_t<ACT>(x0), a1 = act_t<ACT>(x1);  // exact activation: this is the parity mode
                psum[k] = f2_add(psum[k], f2_pack(a0, a1));
                ov[2 * k] = __float_as_uint(a0);
                ov[2 * k + 1] = __float_as_uint(a1);
              } else {
                const f32x2 a = f2_act<ACT>(acc[slot][i][k]);
                float a0, a1;
                f2_unpack(a, a0, a1);
                const __nv_bfloat162 b2 = __floats2bfloat162_rn(a0, a1);
                ov[k] = *reinterpret_cast<const unsigned*>(&b2);
                psum[k] = f2_add(psum[k], a);
              }
            }
            st_words<NW>(orow + (size_t)i * px_stride, ov);
          }
        }
      }
    }
  }
}

// T = __nv_bfloat16: 64 channels per item, 8 per thread (4 fp32 pairs), tanh.approx SiLU (the throughput mode);
// T = float (the 3xTF32 parity mode): 32 channels per item, 4 per thread (2 pairs), EXACT activation, fp32 in and out.
// Either way a pixel is 128 bytes of shared memory, so the tiling plan, the strips and the stages are the same.
template <int ACT, typename T = __nv_bfloat16>
__global__ void __launch_bounds__(DWT_THREADS, 2)
dw3x3s1_tma_kernel(const __grid_constant__ CUtensorMap tmIn, const DwTmaParams p) {
  constexpr bool F32 = sizeof(T) == 4;
  constexpr int NV = F32 ? 2 : 4;          // fp32 pairs per thread
  constexpr int CPT = 2 * NV;              // channels per thread
  constexpr int CG = F32 ? 32 : DWT_CG;    // channels per item
  extern __shared__ uint8_t dwt_smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)dwt_smem_raw + 127) & ~(uintptr_t)127);
  __shared__ uint64_t full[DWT_STAGES];
  __shared__ float red[16][DWT_CG];            // per pass: activated-output sums of each strip slot
  __shared__ float blocksum[DWT_MAX_G][DWT_CG];  // per item: sums per (crop of the group, channel), owner thread = channel

  const int tid = threadIdx.x;
  const int j = tid & 7;        // channel vector inside the 64-channel group
  const int sidx = tid >> 3;    // strip slot 0..15
  if (tid == 0) {
    tma_prefetch_desc(&tmIn);
    for (int i = 0; i < DWT_STAGES; ++i) mbar_init(&full[i], 1);
    fence_barrier_init();
  }
  __syncthreads();
  pdl_trigger();
  pdl_wait();

  const int PW = p.W + 2, PHB = p.BH + 2;
  const uint32_t stage_tx = (uint32_t)(128 * PW * PHB * p.G);
  const int strips_per_crop = p.bands * p.strips_w;
  constexpr int GSTEP = DWT_THREADS / CG;
  const int own_ch = tid & (CG - 1), own_g0 = tid / CG;  // blocksum owner: channel own_ch, crops own_g0, own_g0 + GSTEP, ...

  auto issue = [&](int it_, int stage) {
    const int it = p.rev ? p.items - 1 - it_ : it_;
    const int cg = it % p.n_cg;
    const int t2 = it / p.n_cg;
    const int rb = t2 % p.n_rb, bg = t2 / p.n_rb;
    mbar_expect_tx(&full[stage], stage_tx);
    tma_load_4d(smem + (size_t)stage * p.stage_bytes, &tmIn, &full[stage], cg * CG, -p.pad_l, rb * p.BH - p.pad_t, bg * p.G);
  };

  if (tid == 0 && (int)blockIdx.x < p.items) issue(blockIdx.x, 0);
  int li = 0;
  for (int it_ = blockIdx.x; it_ < p.items; it_ += gridDim.x, ++li) {
    const int stage = li & 1;
    if (tid == 0 && it_ + (int)gridDim.x < p.items) issue(it_ + gridDim.x, stage ^ 1);
    const int it = p.rev ? p.items - 1 - it_ : it_;
    const int cg = it % p.n_cg;
    const int t2 = it / p.n_cg;
    const int rb = t2 % p.n_rb, bg = t2 / p.n_rb;
    const int c = cg * CG + j * CPT;
    const bool c_ok = c < p.C;
    const int b0 = bg * p.G, row0 = rb * p.BH;
    const int rows_item = min(p.BH, p.H - row0);  // output rows of this item

    // this thread's 8 channels: 9 taps + bias, fp32 pairs (channels 2k, 2k+1), in registers for the whole item
    f32x2 w[9][NV], bias[NV];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
#pragma unroll
      for (int q = 0; q < NV / 2; ++q) {
        float4 w0 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c_ok) w0 = __ldg(reinterpret_cast<const float4*>(p.w + (size_t)t * p.C + c + 4 * q));
        w[t][2 * q] = f2_pack(w0.x, w0.y); w[t][2 * q + 1] = f2_pack(w0.z, w0.w);
      }
    }
#pragma unroll
    for (int q = 0; q < NV / 2; ++q) {
      float4 b0v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c_ok) b0v = __ldg(reinterpret_cast<const float4*>(p.bias + c + 4 * q));
      bias[2 * q] = f2_pack(b0v.x, b0v.y); bias[2 * q + 1] = f2_pack(b0v.z, b0v.w);
    }
    if (p.pooled) {
      for (int g = own_g0; g < p.G; g += GSTEP) blocksum[g][own_ch] = 0.f;
    }
    mbar_wait(&full[stage], (uint32_t)((li >> 1) & 1));
    const uint8_t* patch = smem + (size_t)stage * p.stage_bytes;

    for (int s0 = 0; s0 < p.nstrips; s0 += 16) {
      const int s = s0 + sidx;
      f32x2 psum[NV];
#pragma unroll
      for (int k = 0; k < NV; ++k) psum[k] = f2_pack(0.f, 0.f);
      if (s < p.nstrips && c_ok) {
        const int g = s / strips_per_crop;
        const int rem = s - g * strips_per_crop;
        const int band = rem / p.strips_w;
        const int ow0 = (rem - band * p.strips_w) * DWT_OW;
        const int b = b0 + g;
        const int orow0 = band * DWT_RUN;                       // first output row of the run, relative to the item
        const int rows_run = min(DWT_RUN, rows_item - orow0);   // >= 1 by construction of `bands`
        if (b < p.B && rows_run > 0) {
          T* obase = reinterpret_cast<T*>(p.out) + ((size_t)(b * p.H + row0 + orow0) * p.W + ow0) * p.C + c;
          dw_strip<ACT, T, NV, false>(patch, (g * PHB + orow0) * PW + ow0, PW, j * 16, rows_run, p.W - ow0, obase, (size_t)p.W * p.C,
                                      (size_t)p.C, w, bias, psum);
        }
      }
      if (p.pooled) {
        // fixed-order reduction of this pass: strip slots -> (crop, channel) owner threads
        *reinterpret_cast<ulonglong2*>(&red[sidx][j * CPT]) = make_ulonglong2(psum[0], psum[1]);
        if constexpr (!F32) *reinterpret_cast<ulonglong2*>(&red[sidx][j * CPT + 4]) = make_ulonglong2(psum[2], psum[3]);
        __syncthreads();
        for (int g = own_g0; g < p.G; g += GSTEP) {
          // strip slots of crop g in this pass: [g * strips_per_crop, (g + 1) * strips_per_crop) - s0, clipped
          const int qlo = max(g * strips_per_crop - s0, 0);
          const int qhi = min(min((g + 1) * strips_per_crop, p.nstrips) - s0, 16);
          float t = blocksum[g][own_ch];
          for (int q = qlo; q < qhi; ++q) t += red[q][own_ch];
          blocksum[g][own_ch] = t;
        }
        __syncthreads();
      }
    }
    if (p.pooled) {
      const int ch = cg * CG + own_ch;
      if (ch < p.C) {
        for (int g = own_g0; g < p.G; g += GSTEP) {
          if (b0 + g < p.B) p.pooled[((size_t)rb * p.B + b0 + g) * p.C + ch] = blocksum[g][own_ch] * p.inv_hw;
        }
      }
    }
    __syncthreads();  // every thread is done with `stage` (the next iteration's TMA may overwrite it) and with blocksum
  }
}

struct DwTmaCache {
  CUtensorMap map;
  const void* in = nullptr;
  int B = -1;
};

inline const char* dw_tma_launch(DwTmaCache& cache, const DwTmaPlan& plan, const void* in, void* out, const float* w, const float* bias,
                                 float* pooled, int B, int H, int W, int C, int pad_t, int pad_l, int act, cudaStream_t st,
                                 bool f32 = false) {
  DwTmaParams p;
  p.out = out; p.w = w; p.bias = bias; p.pooled = pooled;
  p.B = B; p.H = H; p.W = W; p.C = C; p.pad_t = pad_t; p.pad_l = pad_l;
  p.G = plan.G; p.BH = plan.BH; p.n_rb = plan.n_rb;
  const int cg_ch = f32 ? 32 : DWT_CG;
  p.n_cg = (C + cg_ch - 1) / cg_ch;
  const int n_bg = (B + plan.G - 1) / plan.G;
  p.items = n_bg * p.n_rb * p.n_cg;
  p.strips_w = (W + DWT_OW - 1) / DWT_OW;
  p.bands = (plan.BH + DWT_RUN - 1) / DWT_RUN;
  p.nstrips = plan.G * p.bands * p.strips_w;
  p.stage_bytes = 128 * (W + 2) * (plan.BH + 2) * plan.G;
  p.inv_hw = 1.0f / (float)(H * W);
  {
    // Serpentine traversal (MTB_DW_REV=0 disables; measured 22.47 vs 22.58 ms per step): the expand GEMM before this op wrote its output
    // first-crop-to-last, so the END of the tensor is what the L2 still holds; walking the items last-to-first reads that
    // part from L2, and leaves the BEGINNING of this op's output in L2 for the projection GEMM that follows.
    static int rev_env = -1;
    if (rev_env < 0) { const char* e = getenv("MTB_DW_REV"); rev_env = (e && e[0] == '0') ? 0 : 1; }
    p.rev = rev_env;
  }
  if (cache.in != in || cache.B != B) {
    const char* e = make_tmap_dw(&cache.map, in, (uint64_t)B, (uint64_t)H, (uint64_t)W, (uint64_t)C, (uint32_t)(W + 2),
                                 (uint32_t)(plan.BH + 2), (uint32_t)plan.G, f32 ? 4u : 2u);
    if (e) return e;
    cache.in = in;
    cache.B = B;
  }
  // + one pixel row of slack: the last strip of a ragged row may read (never use) a few pixels past the patch
  const size_t smem = (size_t)DWT_STAGES * p.stage_bytes + 128 + 8 * 128;
  const int grid = p.items < 2 * 148 ? p.items : 2 * 148;
#define MTB_DWT_LAUNCH_T(A, T)                                                                                             \
  {                                                                                                                        \
    static bool attr_set = false;                                                                                          \
    if (!attr_set) {                                                                                                       \
      if (cudaFuncSetAttribute(dw3x3s1_tma_kernel<A, T>, cudaFuncAttributeMaxDynamicSharedMemorySize,                       \
                               DWT_STAGES * DWT_MAX_STAGE + 128 + 8 * 128) != cudaSuccess)                                 \
        return "cannot raise dynamic shared memory for dw3x3s1_tma_kernel";                                                \
      attr_set = true;                                                                                                     \
    }                                                                                                                      \
    launch_k(dw3x3s1_tma_kernel<A, T>, dim3(grid), dim3(DWT_THREADS), smem, st, cache.map, p);                              \
  }
#define MTB_DWT_LAUNCH(A)                                                                                                  \
  {                                                                                                                        \
    if (f32) MTB_DWT_LAUNCH_T(A, float) else MTB_DWT_LAUNCH_T(A, __nv_bfloat16)                                             \
  }
  switch (act) {
    case ACT_SILU: MTB_DWT_LAUNCH(ACT_SILU); break;
    case ACT_RELU: MTB_DWT_LAUNCH(ACT_RELU); break;
    case ACT_HSWISH: MTB_DWT_LAUNCH(ACT_HSWISH); break;
    default: return "unsupported activation in dw3x3s1_tma_kernel";
  }
#undef MTB_DWT_LAUNCH
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

}  // namespace mtb
