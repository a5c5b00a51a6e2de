// Implicit-GEMM convolution for the IR-50 residual units on sm_100a.
//
//   D[m, co] = sum_{tap, ci} X[pixel(m) + tap, ci] * W[co, tap, ci]   (+ fused 1x1/s2 shortcut K-steps)
//
// GEMM view: M = frames*Hout*Wout output pixels, N = Cout, K = taps*Cin (+ Cin2).
//   A tile (128 pixels x 64 channels, bf16) : TMA *im2col* load from the NHWC activation; the halo
//                                             (zero padding) and frame boundaries are resolved by
//                                             the TMA unit, so a tile may start at any pixel.
//   B tile (BN couts x 64 k, bf16)          : TMA tiled load from the packed weight matrix [Cout][K].
//   D (128 x BN fp32)                       : TMEM accumulator, double buffered (2*BN columns).
// Warp roles (416 threads): warps 0-7 epilogue (warp w reads TMEM lanes 32*(w%4).., i.e. one output
// pixel per thread, and the column half w/4), warp 8 TMEM allocator + single-thread tcgen05.mma
// issuer, warps 9-10 TMA producers for A (even / odd k-steps), warps 11-12 TMA producers for B.  Four producer threads because one
// thread sustains only one TMA issue per ~410 cycles (mbarrier wait + expect_tx + issue; measured
// with tools/tma_probe.cu), while the TMA path itself delivers a 16 KB tile every ~200 cycles.
// Persistent: grid = min(#tiles, #SMs); tiles are walked n-tile-fastest so neighbouring CTAs
// share the same activation rows in L2.
//
// Epilogue (fused): + bias[class(pixel)][co]  -> PReLU(alpha[co]) -> + residual[m][co] -> bf16|fp32.
// `class(pixel)` is the 9-way border class (corner/edge/interior) that makes the pre-conv
// BatchNorm exact under zero padding (reference: models/arcface_model.py:52-55; DESIGN.md).
#pragma once
#include "ptx.cuh"

namespace cer {

struct alignas(64) ConvKernelParams {
  CUtensorMap tmap_a;    // im2col, main operand  [N,H,W,Cin]
  CUtensorMap tmap_a2;   // im2col, fused 1x1 shortcut operand [N,H2,W2,Cin2] (unused if ksteps2==0)
  CUtensorMap tmap_b;    // tiled, weights [Cout][Ktot]
  int M;                 // valid output pixels
  int Hout, Wout, Cout;
  int cin_chunks;        // Cin/64
  int cin_shift;         // log2(cin_chunks) when ksize == 3 (power of two there); unused for ksize == 1
  int ksize;             // 1 or 3
  int ksteps_main;       // ksize*ksize*cin_chunks
  int ksteps2;           // Cin2/64 or 0
  int stride, pad;       // main conv geometry (base coord = o*stride - pad)
  int stride2;           // shortcut stride
  int num_m_tiles, num_n_tiles;
  int bias_classes;      // 1 or 9
  int out_fp32;          // 0: bf16 output, 1: fp32 output
  int halo_frames, halo_bands, halo_cts;   // conv_halo_kernel only: frames, 16-row bands and 8-column tiles per frame
  int pool_xor;          // 0: no pooling; else fused MaxPool2d(2,2): the vertical pool partner is lane ^ pool_xor
                         // (8 or 16 = pixels per tile row), the horizontal one lane ^ 1; output is [M/4][Cout]
  int out_wp;            // 0: dense [M][Cout] output; else the output is a padded raster (conv_raster.cuh) of row pitch out_wp = Wout + 1
  int rs_wp, rs_P, rs_frames;   // conv_raster2_kernel only: input row pitch W + 1, positions per frame (H + 1) * (W + 1), frames
  int ctab_flags;        // bit 0: ctab holds the PReLU slopes, bit 1: ctab holds the (single-class) bias -- see kCtab*
  const float* bias;     // [bias_classes][Cout]
  const float* alpha;    // [Cout] PReLU slopes or nullptr
  const __nv_bfloat16* res;  // [M][Cout] residual or nullptr
  void* out;             // [M][Cout]
  // Per-channel epilogue constants as KERNEL PARAMETERS (constant bank): [0, 512) PReLU slopes, [512, 1024) bias.
  // A column's constant is the same for every lane of a warp, so the epilogue reads it as a uniform constant
  // operand instead of an LDS.128 per four columns.  That matters because the LSU's shared-memory wavefronts go
  // through the same port the tensor core reads its operands from: the table reads were 30 % of that port's
  // cycles in the N = 64 / N = 128 kernels, whose MMAs need 75-100 % of it (DESIGN.md section 5.14).
  float ctab[1024];
};
constexpr int kCtabAlpha = 1, kCtabBias = 2, kCtabMaxCout = 512;

constexpr int kConvThreads = 416;
constexpr int kEpiWarps = 8;
constexpr int kMmaWarp = 8;
constexpr int kProdWarp0 = 9;
constexpr int kProducersPerOperand = 2;
constexpr int kBlockM = 128;
constexpr int kBlockK = 64;           // 64 bf16 = 128 B = one swizzle row
constexpr int kABytes = kBlockM * 128;

constexpr int kPrefetchTiles = 2;      // L2 prefetch distance of the A producer, in tiles of this CTA
constexpr int kBresSteps = 9;          // weights-resident variant: all 9 taps of a Cin=64 layer stay in smem

// BRES = true: the whole weight matrix of the layer (9 k-steps x BN x 128 B) is loaded once per CTA
// and stays in shared memory; the ring stages then carry only the A operand.  Used for the
// Cin = 64 layers, where the TMA path (~80 B/cycle/SM) rather than the tensor pipe is the limit
// and B would otherwise be a third of the traffic.
template <int BN, int STAGES, bool BRES>
struct ConvSmem {
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kABytes + (BRES ? 0 : kBBytes);
  static constexpr int kBresOffset = STAGES * kStageBytes;
  static constexpr int kBarOffset = kBresOffset + (BRES ? kBresSteps * kBBytes : 0);
  static constexpr int kNumBars = 2 * STAGES + 5;                                   // full, empty, tfull[2], tempty[2], bres
  static constexpr int kTableOffset = (kBarOffset + kNumBars * 8 + 16 + 15) & ~15;  // bias table + PReLU slopes (float4 reads)
  static constexpr int kTableFloats = BN == 256 ? 8192 : 10 * BN;                   // [<=9][Cout] + [Cout]; 8192 = 2 x 4096 (VGGish FCs)
  static constexpr int kTotal = kTableOffset + kTableFloats * 4 + 1024 /*alignment slack*/;
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// One 256-bit global store (STG.256, sm_100): `p` must be 32-byte aligned.  The epilogue stores one pixel row per
// lane, so a 128-bit store covers only half of a 32 B sector in each of 32 rows; a 256-bit store writes whole
// sectors with half the instructions and no lane exchange (tools/epilogue_probe.cu, DESIGN.md section 5.12).
__device__ __forceinline__ void st_global_256(void* p, uint4 a, uint4 b) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
               : "memory");
}
__device__ __forceinline__ uint4 pack_bf16x8(const float* f) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}
__device__ __forceinline__ uint4 f32x4_bits(const float* f) {
  return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3]));
}

// One output tile of the fused epilogue, for one epilogue thread (warp 0-7):
//   + bias[class(pixel)][co] -> PReLU(alpha[co]) -> + residual[m][co] -> bf16 | fp32.
// `tmem_acc` is the accumulator's TMEM base column; `tfull` the barrier that says it is complete.
// The caller maps its TMEM lane to an output pixel: `valid`, its border class `cls` and the
// element offset `out_off` of (pixel, first channel of this thread's column half).
template <int BN>
__device__ __forceinline__ void conv_epilogue_core(const ConvKernelParams& p, const float* s_bias, const float* s_alpha,
                                                   uint32_t tmem_acc, int n0, int warp, uint32_t tfull, uint32_t parity,
                                                   bool valid, int cls, size_t out_off, uint32_t tempty,
                                                   bool pool_store = false, size_t pool_off = 0,
                                                   size_t res_off = ~size_t(0) /* = out_off */, bool zero_store = false);

template <int BN>
__device__ __forceinline__ void conv_epilogue_tile(const ConvKernelParams& p, const float* s_bias, const float* s_alpha,
                                                   uint32_t tmem_acc, int m_tile, int n_tile, int warp, int lane,
                                                   uint32_t tfull, uint32_t parity, uint32_t tempty) {
  constexpr int kHalf = BN / 2;                // columns per thread per tile
  const int quarter = warp & 3;                // TMEM lane quarter this warp may read
  const int half = warp >> 2;                  // column half
  const int row = quarter * 32 + lane;         // TMEM lane == row of the M tile
  const int hw = p.Hout * p.Wout;
  const int m = m_tile * kBlockM + row;
  const bool valid = m < p.M;
  const int n0 = n_tile * BN + half * kHalf;
  int cls = 0;
  if (p.bias_classes == 9) {
    const int rem = m % hw;
    const int oh = rem / p.Wout;
    const int ow = rem - oh * p.Wout;
    cls = (oh == 0 ? 0 : (oh == p.Hout - 1 ? 2 : 1)) * 3 + (ow == 0 ? 0 : (ow == p.Wout - 1 ? 2 : 1));
  }
  bool pool_store = false;
  size_t pool_off = 0;
  if (p.pool_xor) {      // fused 2x2 max-pool: the lane at even (oh, ow) stores the window's maximum
    const int rem = m % hw;
    const int oh = rem / p.Wout, ow = rem - oh * p.Wout;
    pool_store = valid && !(oh & 1) && !(ow & 1);
    pool_off = ((static_cast<size_t>(m / hw) * (p.Hout >> 1) + (oh >> 1)) * (p.Wout >> 1) + (ow >> 1)) * p.Cout + n0;
  }
  const size_t dense_off = static_cast<size_t>(m) * p.Cout + n0;
  size_t out_off = dense_off;
  if (p.out_wp) {        // the consumer reads a padded raster: one pad column per row, one pad row per frame
    const int n = m / hw, rem = m - n * hw;
    const int oh = rem / p.Wout, ow = rem - oh * p.Wout;
    out_off = ((static_cast<size_t>(n) * (p.Hout + 1) + oh) * p.out_wp + ow) * p.Cout + n0;
  }
  conv_epilogue_core<BN>(p, s_bias, s_alpha, tmem_acc, n0, warp, tfull, parity, valid, cls, out_off, tempty, pool_store,
                         pool_off, dense_off);
}

template <int BN>
__device__ __forceinline__ void conv_epilogue_core(const ConvKernelParams& p, const float* s_bias, const float* s_alpha,
                                                   uint32_t tmem_acc, int n0, int warp, uint32_t tfull, uint32_t parity,
                                                   bool valid, int cls, size_t out_off, uint32_t tempty, bool pool_store,
                                                   size_t pool_off, size_t res_off, bool zero_store) {
  constexpr int kHalf = BN / 2;
  if (res_off == ~size_t(0)) res_off = out_off;
  const int quarter = warp & 3;
  const int half = warp >> 2;
  const uint32_t lane_addr = (static_cast<uint32_t>(quarter * 32) << 16);
  const bool has_res = p.res != nullptr;
  const bool has_alpha = p.alpha != nullptr;
  const float* sb = s_bias + cls * p.Cout + n0;
  const float* sal = s_alpha + n0;
  const bool ld_res = has_res && valid;

  // residual of the first chunk is requested before the accumulator wait: its latency hides
  // behind the MMA of this tile
  uint4 rnext[4];
  if (ld_res) {
    const uint4* rp = reinterpret_cast<const uint4*>(p.res + res_off);
#pragma unroll
    for (int j = 0; j < 4; ++j) rnext[j] = __ldg(rp + j);
  }
  mbar_wait_a(tfull, parity);
  tc_fence_after();
#pragma unroll
  for (int c0 = 0; c0 < kHalf; c0 += 32) {
    uint32_t v[32];
    tmem_ld_32x32(tmem_acc + lane_addr + half * kHalf + c0, v);
    uint4 rres[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) rres[j] = rnext[j];
    if (c0 + 32 < kHalf && ld_res) {
      const uint4* rp = reinterpret_cast<const uint4*>(p.res + res_off + c0 + 32);
#pragma unroll
      for (int j = 0; j < 4; ++j) rnext[j] = __ldg(rp + j);
    }
    tmem_ld_wait();
    if (c0 + 32 >= kHalf) {
      // The accumulator is free as soon as its last tcgen05.ld has landed in registers (ld / wait::ld are
      // warp-collective, so lane 0 speaks for the warp).  Arriving HERE -- before the global stores, with
      // relaxed semantics -- keeps the MMA warp from waiting on this tile's stores and avoids the
      // MEMBAR.ALL.GPU + ERRBAR a release.cluster arrive after the stores costs (profiles/r01_full_pair128.txt).
      tc_fence_before();
      if ((threadIdx.x & 31) == 0) mbar_arrive_relaxed_cluster(tempty);
    }
    float f[32];
    if (p.ctab_flags & kCtabBias) {            // warp-uniform constant operands (kernel parameter space)
      const float* cb = p.ctab + 512 + n0 + c0;
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]) + cb[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = *reinterpret_cast<const float4*>(sb + c0 + 4 * j);
        f[4 * j + 0] = __uint_as_float(v[4 * j + 0]) + b.x;
        f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b.y;
        f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b.z;
        f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b.w;
      }
    }
    if (has_alpha) {
      if (p.ctab_flags & kCtabAlpha) {
        const float* ca = p.ctab + n0 + c0;
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = f[j] >= 0.f ? f[j] : f[j] * ca[j];
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 a = *reinterpret_cast<const float4*>(sal + c0 + 4 * j);
          f[4 * j + 0] = f[4 * j + 0] >= 0.f ? f[4 * j + 0] : f[4 * j + 0] * a.x;
          f[4 * j + 1] = f[4 * j + 1] >= 0.f ? f[4 * j + 1] : f[4 * j + 1] * a.y;
          f[4 * j + 2] = f[4 * j + 2] >= 0.f ? f[4 * j + 2] : f[4 * j + 2] * a.z;
          f[4 * j + 3] = f[4 * j + 3] >= 0.f ? f[4 * j + 3] : f[4 * j + 3] * a.w;
        }
      }
    }
    if (ld_res) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t w[4] = {rres[j].x, rres[j].y, rres[j].z, rres[j].w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const __nv_bfloat162 h = *reinterpret_cast<const __nv_bfloat162*>(&w[q]);
          f[8 * j + 2 * q + 0] += __bfloat162float(h.x);
          f[8 * j + 2 * q + 1] += __bfloat162float(h.y);
        }
      }
    }
    if (p.pool_xor) {
      // MaxPool2d(2,2) across the four lanes of the window (all 32 lanes take part in the shuffles);
      // max of the bf16-rounded values == bf16 rounding of the max, i.e. identical to pooling the stored tensor
      uint32_t h[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) h[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        uint32_t o = __shfl_xor_sync(0xffffffffu, h[j], 1);
        __nv_bfloat162 mx = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&h[j]), *reinterpret_cast<__nv_bfloat162*>(&o));
        h[j] = *reinterpret_cast<uint32_t*>(&mx);
        o = __shfl_xor_sync(0xffffffffu, h[j], p.pool_xor);
        mx = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&h[j]), *reinterpret_cast<__nv_bfloat162*>(&o));
        h[j] = *reinterpret_cast<uint32_t*>(&mx);
      }
      if (pool_store) {
        __nv_bfloat16* op = static_cast<__nv_bfloat16*>(p.out) + pool_off + c0;
#pragma unroll
        for (int j = 0; j < 2; ++j)
          st_global_256(op + 16 * j, make_uint4(h[8 * j], h[8 * j + 1], h[8 * j + 2], h[8 * j + 3]),
                        make_uint4(h[8 * j + 4], h[8 * j + 5], h[8 * j + 6], h[8 * j + 7]));
      }
    } else if (valid) {
      if (p.out_fp32) {
        float* op = static_cast<float*>(p.out) + out_off + c0;
#pragma unroll
        for (int j = 0; j < 4; ++j) st_global_256(op + 8 * j, f32x4_bits(f + 8 * j), f32x4_bits(f + 8 * j + 4));
      } else {
        __nv_bfloat16* op = static_cast<__nv_bfloat16*>(p.out) + out_off + c0;
#pragma unroll
        for (int j = 0; j < 2; ++j) st_global_256(op + 16 * j, pack_bf16x8(f + 16 * j), pack_bf16x8(f + 16 * j + 8));
      }
    } else if (zero_store) {                 // pad position of a padded-raster output (bf16): must read as the conv's zero padding
      __nv_bfloat16* op = static_cast<__nv_bfloat16*>(p.out) + out_off + c0;
#pragma unroll
      for (int j = 0; j < 2; ++j) st_global_256(op + 16 * j, make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u));
    }
  }
}

// ALIGNED = true: the host guarantees ksteps % STAGES == 0, so every tile walks the ring a whole
// number of times.  Stage indices are then compile-time inside the unrolled role loops: barrier,
// smem and descriptor addresses are base + immediate, which shrinks the MMA-issue loop from ~70 to
// ~20 instructions per k-step (at N = 64 a k-step is only 128 cycles of tensor work, so the
// issuing warp -- not memory -- was the limiter; profiles/r01_conv_v6_*).
template <int BN, int STAGES, bool BRES, bool ALIGNED>
__global__ void __launch_bounds__(kConvThreads, 1) conv_igemm_kernel(const __grid_constant__ ConvKernelParams p) {
  using L = ConvSmem<BN, STAGES, BRES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tfull_bar = empty_bar + STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* bres_bar = tempty_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres_bar + 1);
  float* s_bias = reinterpret_cast<float*>(smem + L::kTableOffset);     // [bias_classes][Cout]
  float* s_alpha = s_bias + p.bias_classes * p.Cout;                    // [Cout]

  // warp index broadcast from lane 0 so the compiler treats role dispatch and the role loops as
  // warp-uniform (descriptors and addresses then live in uniform registers)
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int total_tiles = p.num_m_tiles * p.num_n_tiles;
  const int ksteps = p.ksteps_main + p.ksteps2;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], BRES ? 1 : 2);   // one arrive.expect_tx per operand that travels through the ring
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], kEpiWarps);          // one arrival per epilogue warp
    }
    mbar_init(bres_bar, 1);
    fence_barrier_init();
  }
  if (warp == kProdWarp0 && lane == 0) {
    tma_prefetch_desc(&p.tmap_a);
    if (p.ksteps2 > 0) tma_prefetch_desc(&p.tmap_a2);
  }
  if (warp == kProdWarp0 + kProducersPerOperand && lane == 0) tma_prefetch_desc(&p.tmap_b);
  if (warp == kMmaWarp) {
    tmem_alloc(tmem_slot, 2 * BN);
    tmem_relinquish();
  }
  if (warp < kEpiWarps) {     // stage the epilogue constants once per CTA
    for (int i = threadIdx.x; i < p.bias_classes * p.Cout; i += kEpiWarps * 32) s_bias[i] = __ldg(p.bias + i);
    if (p.alpha != nullptr)
      for (int i = threadIdx.x; i < p.Cout; i += kEpiWarps * 32) s_alpha[i] = __ldg(p.alpha + i);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();     // everything above touched only constants: overlap it with the previous layer's tail
  pdl_wait();                  // the previous layer's activations are complete and visible from here on

  if (warp >= kProdWarp0) {
    // ===================== TMA producers (one lane each) =====================
    // first two: A operand of k-steps g = 0,1 (mod 2); next two: B operand likewise.  g counts
    // k-steps across all tiles of this CTA, so stage = g % STAGES and the phase flips per wrap.
    // Control flow is warp-uniform (all 32 lanes walk the loop and wait on the barrier); one
    // elected lane issues expect_tx + the TMA.  Barrier / stage addresses are running 32-bit
    // shared-memory addresses.
    const bool is_a = warp < kProdWarp0 + kProducersPerOperand;
    const int q = (warp - kProdWarp0) % kProducersPerOperand;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
    constexpr int kNPA = BRES ? 3 : 2;          // A producer warps in the aligned variant
    const int pw = warp - kProdWarp0;          // 0..3
    if (ALIGNED && !(BRES && pw == 3)) {
      // ---- stage-aligned producers: warp `pa` of kNP owns stages pa, pa+kNP, ... of every round ----
      const bool a_role = BRES ? true : pw < 2;
      const int kNP = a_role ? kNPA : 2;
      const int pa = a_role ? pw : pw - 2;
      const int hw = p.Hout * p.Wout;
      const int rounds = ksteps / STAGES;
      uint32_t phase = 0;
      const uint32_t sa0 = smem_base + pa * L::kStageBytes + (a_role ? 0 : kABytes);
      const uint32_t fb0 = full0 + pa * 8, eb0 = empty0 + pa * 8;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m_tile = tile / p.num_n_tiles;
        const int n_tile = tile - m_tile * p.num_n_tiles;
        const int n0 = n_tile * BN;
        int cw = 0, ch = 0, n_img = 0, cw2 = 0, ch2 = 0;
        if (a_role) {
          const int m0 = m_tile * kBlockM;
          n_img = m0 / hw;
          const int rem = m0 - n_img * hw;
          const int oh = rem / p.Wout;
          const int ow = rem - oh * p.Wout;
          cw = ow * p.stride - p.pad; ch = oh * p.stride - p.pad;
          cw2 = ow * p.stride2; ch2 = oh * p.stride2;
          if (pa == 0 && n_tile == 0) {          // L2 prefetch of the tile this CTA reaches kPrefetchTiles from now
            const int step = gridDim.x / p.num_n_tiles > 0 ? gridDim.x / p.num_n_tiles : 1;
            const int ptile_m = m_tile + kPrefetchTiles * step;
            if (ptile_m < p.num_m_tiles && elect_one()) {
              const int pm0 = ptile_m * kBlockM;
              const int pn = pm0 / hw;
              const int prem = pm0 - pn * hw;
              const int poh = prem / p.Wout;
              const int pow_ = prem - poh * p.Wout;
              const uint16_t mid = p.ksize == 3 ? 1 : 0;
              for (int c = 0; c < p.cin_chunks; ++c)
                tma_prefetch_im2col_4d(&p.tmap_a, c * kBlockK, pow_ * p.stride - p.pad, poh * p.stride - p.pad, pn, mid, mid);
            }
            __syncwarp();
          }
        }
        for (int r = 0; r < rounds; ++r) {
#pragma unroll
          for (int j = 0; j < STAGES; ++j) {
            if (j % (BRES ? 3 : 2) != 0) continue;            // j walks this warp's stages: pa + j (j multiple of kNP)
            if (j + pa >= STAGES) continue;
            const int ks = r * STAGES + pa + j;
            mbar_wait_a(eb0 + j * 8, phase ^ 1);
            if (a_role) {
              int tap = 0, chunk = ks;
              if (p.ksize == 3) { tap = ks >> p.cin_shift; chunk = ks & (p.cin_chunks - 1); }
              const int rr = (tap * 11) >> 5;
              const int ss = tap - rr * 3;
              if (elect_one()) {
                mbar_expect_tx_a(fb0 + j * 8, kABytes);
                if (ks < p.ksteps_main)
                  tma_load_im2col_4d_a(&p.tmap_a, fb0 + j * 8, sa0 + j * L::kStageBytes, chunk * kBlockK, cw, ch, n_img,
                                       (uint16_t)ss, (uint16_t)rr);
                else
                  tma_load_im2col_4d_a(&p.tmap_a2, fb0 + j * 8, sa0 + j * L::kStageBytes, (ks - p.ksteps_main) * kBlockK,
                                       cw2, ch2, n_img, 0, 0);
              }
            } else {
              if (elect_one()) {
                mbar_expect_tx_a(fb0 + j * 8, L::kBBytes);
                tma_load_2d_a(&p.tmap_b, fb0 + j * 8, sa0 + j * L::kStageBytes, ks * kBlockK, n0);
              }
            }
            __syncwarp();
          }
          phase ^= 1;
        }
      }
      (void)kNP;
    } else if (BRES && !is_a) {
      // resident weights: one producer warp loads every k-step's B tile once, then retires
      if ((ALIGNED ? pw == 3 : q == 0) && elect_one()) {
        const uint32_t bar = smem_u32(bres_bar);
        mbar_expect_tx_a(bar, ksteps * L::kBBytes);
        for (int ks = 0; ks < ksteps; ++ks)
          tma_load_2d_a(&p.tmap_b, bar, smem_base + L::kBresOffset + ks * L::kBBytes, ks * kBlockK, 0);
      }
      __syncwarp();
    } else {
      const int hw = p.Hout * p.Wout;
      uint32_t stage = q % STAGES;
      uint32_t phase = (q / STAGES) & 1;
      int ks_carry = q;                       // first k-step of this producer inside the current tile
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m_tile = tile / p.num_n_tiles;
        const int n_tile = tile - m_tile * p.num_n_tiles;
        int cw = 0, ch = 0, n_img = 0, cw2 = 0, ch2 = 0;
        if (is_a) {
          const int m0 = m_tile * kBlockM;
          n_img = m0 / hw;
          const int rem = m0 - n_img * hw;
          const int oh = rem / p.Wout;
          const int ow = rem - oh * p.Wout;
          cw = ow * p.stride - p.pad; ch = oh * p.stride - p.pad;
          cw2 = ow * p.stride2; ch2 = oh * p.stride2;
        }
        const int n0 = n_tile * BN;
        // The first tap of a tile misses L2 (every later tap re-reads almost the same pixels), and
        // the ring is too shallow to cover HBM latency, so the tile this CTA will process
        // kPrefetchTiles iterations from now is prefetched into L2 here (centre tap, all chunks).
        if (is_a && q == 0 && n_tile == 0) {
          const int ptile_m = m_tile + kPrefetchTiles * (gridDim.x / p.num_n_tiles > 0 ? gridDim.x / p.num_n_tiles : 1);
          if (ptile_m < p.num_m_tiles && elect_one()) {
            const int pm0 = ptile_m * kBlockM;
            const int pn = pm0 / hw;
            const int prem = pm0 - pn * hw;
            const int poh = prem / p.Wout;
            const int pow_ = prem - poh * p.Wout;
            const uint16_t mid = p.ksize == 3 ? 1 : 0;
            for (int c = 0; c < p.cin_chunks; ++c)
              tma_prefetch_im2col_4d(&p.tmap_a, c * kBlockK, pow_ * p.stride - p.pad, poh * p.stride - p.pad, pn, mid, mid);
            for (int c = 0; c < p.ksteps2; ++c)
              tma_prefetch_im2col_4d(&p.tmap_a2, c * kBlockK, pow_ * p.stride2, poh * p.stride2, pn, 0, 0);
          }
          __syncwarp();
        }
        int ks = ks_carry;
        for (; ks < ksteps; ks += kProducersPerOperand) {
          mbar_wait_a(empty0 + stage * 8, phase ^ 1);
          const uint32_t sa = smem_base + stage * L::kStageBytes;
          const uint32_t fb = full0 + stage * 8;
          if (is_a) {
            int tap = 0, chunk = ks;
            if (p.ksize == 3) { tap = ks >> p.cin_shift; chunk = ks & (p.cin_chunks - 1); }
            const int r = (tap * 11) >> 5;          // tap / 3 for tap in [0, 9)
            const int s = tap - r * 3;
            const bool main_op = ks < p.ksteps_main;
            if (elect_one()) {
              mbar_expect_tx_a(fb, kABytes);
              if (main_op) {
                tma_load_im2col_4d_a(&p.tmap_a, fb, sa, chunk * kBlockK, cw, ch, n_img, (uint16_t)s, (uint16_t)r);
              } else {
                tma_load_im2col_4d_a(&p.tmap_a2, fb, sa, (ks - p.ksteps_main) * kBlockK, cw2, ch2, n_img, 0, 0);
              }
            }
          } else {
            if (elect_one()) {
              mbar_expect_tx_a(fb, L::kBBytes);
              tma_load_2d_a(&p.tmap_b, fb, sa + kABytes, ks * kBlockK, n0);
            }
          }
          __syncwarp();
          stage += kProducersPerOperand;
          if (stage >= STAGES) { stage -= STAGES; phase ^= 1; }
        }
        ks_carry = ks - ksteps;                 // keeps the global even/odd split across tiles
      }
    }
  } else if (warp == kMmaWarp) {
    // ===================== MMA issuer (warp-uniform loop, one elected lane issues) =====================
    {
      constexpr uint32_t idesc = umma_idesc(kBlockM, BN, /*bf16*/ 1);
      constexpr uint32_t kStageLo = L::kStageBytes >> 4;     // descriptor address field counts 16 B units
      const uint32_t smem_base = smem_u32(smem);
      const uint32_t full0 = smem_u32(full_bar), empty0 = smem_u32(empty_bar);
      const uint32_t tfull0 = smem_u32(tfull_bar), tempty0 = smem_u32(tempty_bar);
      const uint32_t a_lo0 = umma_desc_lo(smem_base);
      const uint32_t bres_lo0 = umma_desc_lo(smem_base + L::kBresOffset);
      if (BRES) mbar_wait_a(smem_u32(bres_bar), 0);
      uint32_t stage = 0, phase = 0;
      int it = 0;
      if (ALIGNED) {
        const int rounds = ksteps / STAGES;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
          const uint32_t acc = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          mbar_wait_a(tempty0 + acc * 8, acc_phase ^ 1);
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + acc * BN;
          for (int r = 0; r < rounds; ++r) {
            const uint32_t b_round = bres_lo0 + r * STAGES * (L::kBBytes >> 4);
#pragma unroll
            for (int sidx = 0; sidx < STAGES; ++sidx) {
              mbar_wait_a(full0 + sidx * 8, phase);
              tc_fence_after();
              if (elect_one()) {
                const uint32_t a_lo = a_lo0 + sidx * kStageLo;
                const uint32_t b_lo = BRES ? b_round + sidx * (L::kBBytes >> 4) : a_lo + (kABytes >> 4);
                umma_f16(tmem_d, umma_desc_from_lo(a_lo), umma_desc_from_lo(b_lo), idesc, (r | sidx) != 0 ? 1u : 0u);
                umma_f16(tmem_d, umma_desc_from_lo(a_lo + 2), umma_desc_from_lo(b_lo + 2), idesc, 1u);
                umma_f16(tmem_d, umma_desc_from_lo(a_lo + 4), umma_desc_from_lo(b_lo + 4), idesc, 1u);
                umma_f16(tmem_d, umma_desc_from_lo(a_lo + 6), umma_desc_from_lo(b_lo + 6), idesc, 1u);
                umma_commit_a(empty0 + sidx * 8);
                if (sidx == STAGES - 1 && r == rounds - 1) umma_commit_a(tfull0 + acc * 8);
              }
              __syncwarp();
            }
            phase ^= 1;
          }
        }
      } else
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
        const uint32_t acc = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait_a(tempty0 + acc * 8, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int ks = 0; ks < ksteps; ++ks) {
          mbar_wait_a(full0 + stage * 8, phase);
          tc_fence_after();
          const uint32_t a_lo = a_lo0 + stage * kStageLo;
          const uint32_t b_lo = BRES ? bres_lo0 + ks * (L::kBBytes >> 4) : a_lo + (kABytes >> 4);
          if (elect_one()) {
            // +32 bytes along K inside the 128 B swizzle row == +2 in the descriptor address field
            umma_f16(tmem_d, umma_desc_from_lo(a_lo), umma_desc_from_lo(b_lo), idesc, ks != 0 ? 1u : 0u);
            umma_f16(tmem_d, umma_desc_from_lo(a_lo + 2), umma_desc_from_lo(b_lo + 2), idesc, 1u);
            umma_f16(tmem_d, umma_desc_from_lo(a_lo + 4), umma_desc_from_lo(b_lo + 4), idesc, 1u);
            umma_f16(tmem_d, umma_desc_from_lo(a_lo + 6), umma_desc_from_lo(b_lo + 6), idesc, 1u);
            umma_commit_a(empty0 + stage * 8);                      // frees the smem slot once these MMAs retire
            if (ks == ksteps - 1) umma_commit_a(tfull0 + acc * 8);  // accumulator complete -> epilogue
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== Epilogue (warps 0-7, 256 threads) =====================
    const uint32_t tfull0 = smem_u32(tfull_bar), tempty0 = smem_u32(tempty_bar);
    int it = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int m_tile = tile / p.num_n_tiles;
      const int n_tile = tile - m_tile * p.num_n_tiles;
      conv_epilogue_tile<BN>(p, s_bias, s_alpha, tmem_base + acc * BN, m_tile, n_tile, warp, lane, tfull0 + acc * 8, acc_phase,
                             tempty0 + acc * 8);          // arrives on tempty once the accumulator is in registers
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * BN);
  }
}

}  // namespace cer
