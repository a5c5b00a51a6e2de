// TemporalBlock on the tensor cores (tcgen05 kind::tf32, fp32 operands, fp32 accumulate in TMEM).
//
// Reference: TemporalBlock.forward, models/temporal_convolutional_model.py:21-54 (+ the eval
// BatchNorm1d of models/model.py:515 as a trailing affine).  A block is two launches of one kernel:
//   launch 1:  h1 = LReLU(conv1(x) + b1)
//   launch 2:  y  = post( LReLU( LReLU(conv2(h1) + b2) + res ) ),  res = x  or  Wd*x + bd
// Each launch is an implicit GEMM  D[m, co] = sum_{j, ci} X[b, t-(k-1-j)d, ci] * W[co, j, ci]:
//   M = B*T rows (time-major, channels contiguous), N = C_out, K = k*C_in.
//   A tile (128 rows x 32 fp32)  : TMA im2col over the [B, T, 1, C] tensor with bounding-box lower
//                                  corner -(k-1)d and tap offset j*d -- the causal left padding
//                                  (Conv1d padding + Chomp1d) and the batch boundaries come out of
//                                  the TMA unit as zeros, no padded copy exists.
//   B tile (BN couts x 32 fp32)  : tiled TMA from the packed weight [C_out][k*C_in (+ C_in_ds)].
//   The 1x1 downsample of launch 2 accumulates into a second TMEM accumulator (it is added AFTER
//   conv2's LeakyReLU, so it cannot share conv2's accumulator).
// One CTA = one 128 x BN tile (the head has only B*T/128 * C_out/BN <= ~80 tiles).  BN = 64 when C_out is a
// multiple of 64, else 32, so every C_out % 32 == 0 is covered by whole N tiles.
// Causal halo limit: the A map is a rank-4 im2col map, whose bounding-box corners cuTensorMapEncodeIm2col
// accepts only in [-128, 127]; the lower corner is -(k-1)d, so (k-1)d <= 128 (checked before any encode).
// The full range holds on a B200: a k = 5, d = 32 block (halo 128) matches its fp64 reference.
// Why TF32 and not bf16: SURVEY.md H4 -- argmax parity of the head is marginal in bf16
// (99.7-99.8 %) and safe in TF32 (1.5e-3 max-abs logit error, 100 % agreement).
#include <cuda_runtime.h>
#include <cuda.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/cer_b200.h"
#include "common.h"
#include "ptx.cuh"

namespace cer {

int make_im2col_map_generic(CUtensorMap* map, CUtensorMapDataType dt, int elem_bytes, const void* base, int N, int H,
                            int W, int C, const int lower[2], const int upper[2], int stride, int channels_per_pixel);
int make_tiled2d_map_generic(CUtensorMap* map, CUtensorMapDataType dt, int elem_bytes, const void* base, int rows,
                             int cols, int box_rows, int box_cols);

struct alignas(64) TcnKernelParams {
  CUtensorMap tmap_a;     // im2col over the main operand [B,T,1,C_main]
  CUtensorMap tmap_a2;    // im2col over x for the 1x1 downsample (unused if ksteps2 == 0)
  CUtensorMap tmap_b;     // weights [C_out][k*C_main + C_ds]
  int M, T, Cout;
  int chunks;             // C_main / 32
  int taps, dilation;
  int ksteps_main;        // taps * chunks
  int ksteps2;            // C_ds / 32 or 0
  int num_n_tiles;
  int mode;               // 0: LReLU(acc+bias)   1: post(LReLU(LReLU(acc+bias) + res))
  const float* bias;      // [Cout]
  const float* bias2;     // [Cout] downsample bias (mode 1 with ksteps2 > 0)
  const float* res;       // [M][Cout] identity residual (mode 1 with ksteps2 == 0)
  const float* post_scale;
  const float* post_shift;
  float* out;             // [M][Cout]
};

constexpr int kTcThreads = 256;       // warps 0-3 epilogue, 4 MMA, 5 A producer, 6 B producer, 7 spare
constexpr int kTcBlockM = 128;
constexpr int kTcBlockK = 32;         // 32 fp32 = 128 B = one swizzle row; 4 MMAs of K = 8 per k-step
constexpr int kTcABytes = kTcBlockM * 128;
constexpr float kLeakyTc = 0.01f;
constexpr int kTcMaxHalo = 128;

// The instantiations launch_tcn_tc can run (cer_head_last_variant reports the one a launch used).
static const char* const kHeadVariantNames[] = {"tcn_igemm_kernel<64,8>", "tcn_igemm_kernel<32,8>"};

template <int BN, int STAGES>
struct TcnSmem {
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kTcABytes + kBBytes;
  static constexpr int kBarOffset = STAGES * kStageBytes;
  static constexpr int kTotal = kBarOffset + (2 * STAGES + 2) * 8 + 16 + 1024;
};

__device__ __forceinline__ float lrelu_tc(float v) { return v >= 0.f ? v : v * kLeakyTc; }

template <int BN, int STAGES>
__global__ void __launch_bounds__(kTcThreads, 1) tcn_igemm_kernel(const __grid_constant__ TcnKernelParams p) {
  using L = TcnSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* done_bar = empty_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 2);
  constexpr uint32_t kTmemCols = (2 * BN < 32) ? 32 : 2 * BN;

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int m_tile = blockIdx.x / p.num_n_tiles;
  const int n_tile = blockIdx.x - m_tile * p.num_n_tiles;
  const int ksteps = p.ksteps_main + p.ksteps2;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 2);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&done_bar[0], 1);
    fence_barrier_init();
  }
  if (warp == 5 && lane == 0) {
    tma_prefetch_desc(&p.tmap_a);
    if (p.ksteps2 > 0) tma_prefetch_desc(&p.tmap_a2);
  }
  if (warp == 6 && lane == 0) tma_prefetch_desc(&p.tmap_b);
  if (warp == 4) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 5 || warp == 6) {
    // ---------------- TMA producers: warp 5 = A (im2col), warp 6 = B (weights) ----------------
    const bool is_a = warp == 5;
    const int m0 = m_tile * kTcBlockM;
    const int b_img = m0 / p.T;
    const int t0 = m0 - b_img * p.T;
    const int ch = t0 - (p.taps - 1) * p.dilation;       // base coordinate inside the bounding box
    int stage = 0;
    uint32_t phase = 0;
    int tap = 0, chunk = 0;
    for (int ks = 0; ks < ksteps; ++ks) {
      mbar_wait(&empty_bar[stage], phase ^ 1);
      uint8_t* sa = smem + stage * L::kStageBytes;
      if (is_a) {
        if (elect_one()) {
          mbar_expect_tx(&full_bar[stage], kTcABytes);
          if (ks < p.ksteps_main) {
            tma_load_im2col_4d(&p.tmap_a, &full_bar[stage], sa, chunk * kTcBlockK, 0, ch, b_img, 0,
                               (uint16_t)(tap * p.dilation));
          } else {
            tma_load_im2col_4d(&p.tmap_a2, &full_bar[stage], sa, (ks - p.ksteps_main) * kTcBlockK, 0, ch, b_img, 0,
                               (uint16_t)((p.taps - 1) * p.dilation));
          }
        }
      } else {
        if (elect_one()) {
          mbar_expect_tx(&full_bar[stage], L::kBBytes);
          tma_load_2d(&p.tmap_b, &full_bar[stage], sa + kTcABytes, ks * kTcBlockK, n_tile * BN);
        }
      }
      __syncwarp();
      if (++chunk == p.chunks) { chunk = 0; ++tap; }
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 4) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc = umma_idesc(kTcBlockM, BN, /*tf32*/ 2);
    const uint32_t smem_base = smem_u32(smem);
    int stage = 0;
    uint32_t phase = 0;
    for (int ks = 0; ks < ksteps; ++ks) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      const uint32_t a_addr = smem_base + stage * L::kStageBytes;
      const uint64_t adesc = umma_desc_sw128(a_addr);
      const uint64_t bdesc = umma_desc_sw128(a_addr + kTcABytes);
      const bool ds = ks >= p.ksteps_main;                 // downsample k-steps go to accumulator 1
      const uint32_t tmem_d = tmem_base + (ds ? BN : 0);
      const bool first = (ks == 0) || (ks == p.ksteps_main);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          umma_tf32(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
        umma_commit(&empty_bar[stage]);
        if (ks == ksteps - 1) umma_commit(&done_bar[0]);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp < 4) {
    // ---------------- Epilogue: one row per thread ----------------
    const int row = warp * 32 + lane;
    const uint32_t lane_addr = (static_cast<uint32_t>(warp * 32) << 16);
    const int m = m_tile * kTcBlockM + row;
    const bool valid = m < p.M;
    const int n0 = n_tile * BN;
    const size_t off = static_cast<size_t>(m) * p.Cout + n0;
    mbar_wait(&done_bar[0], 0);
    tc_fence_after();
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t v[32];
      tmem_ld_32x32(tmem_base + lane_addr + c0, v);
      tmem_ld_wait();
      float f[32];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c0) + j);
        f[4 * j + 0] = lrelu_tc(__uint_as_float(v[4 * j + 0]) + b.x);
        f[4 * j + 1] = lrelu_tc(__uint_as_float(v[4 * j + 1]) + b.y);
        f[4 * j + 2] = lrelu_tc(__uint_as_float(v[4 * j + 2]) + b.z);
        f[4 * j + 3] = lrelu_tc(__uint_as_float(v[4 * j + 3]) + b.w);
      }
      if (p.mode == 1) {
        if (p.ksteps2 > 0) {
          uint32_t r[32];
          tmem_ld_32x32(tmem_base + lane_addr + BN + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias2 + n0 + c0) + j);
            f[4 * j + 0] += __uint_as_float(r[4 * j + 0]) + b.x;
            f[4 * j + 1] += __uint_as_float(r[4 * j + 1]) + b.y;
            f[4 * j + 2] += __uint_as_float(r[4 * j + 2]) + b.z;
            f[4 * j + 3] += __uint_as_float(r[4 * j + 3]) + b.w;
          }
        } else if (valid) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 x = __ldg(reinterpret_cast<const float4*>(p.res + off + c0) + j);
            f[4 * j + 0] += x.x; f[4 * j + 1] += x.y; f[4 * j + 2] += x.z; f[4 * j + 3] += x.w;
          }
        }
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = lrelu_tc(f[j]);
        if (p.post_scale != nullptr) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 s = __ldg(reinterpret_cast<const float4*>(p.post_scale + n0 + c0) + j);
            const float4 t = __ldg(reinterpret_cast<const float4*>(p.post_shift + n0 + c0) + j);
            f[4 * j + 0] = fmaf(f[4 * j + 0], s.x, t.x); f[4 * j + 1] = fmaf(f[4 * j + 1], s.y, t.y);
            f[4 * j + 2] = fmaf(f[4 * j + 2], s.z, t.z); f[4 * j + 3] = fmaf(f[4 * j + 3], s.w, t.w);
          }
        }
      }
      if (valid) {
        float4* op = reinterpret_cast<float4*>(p.out + off + c0);
#pragma unroll
        for (int j = 0; j < 8; ++j) op[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <int BN, int STAGES>
static int launch_tcn_tc(const TcnKernelParams& p, int grid, cudaStream_t st) {
  using L = TcnSmem<BN, STAGES>;
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(tcn_igemm_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
  }
  static_assert((BN == 64 || BN == 32) && STAGES == 8, "kHeadVariantNames lists <64,8> and <32,8> only");
  set_head_variant(kHeadVariantNames[BN == 64 ? 0 : 1]);
  tcn_igemm_kernel<BN, STAGES><<<grid, kTcThreads, L::kTotal, st>>>(p);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

// One conv launch of a block.  main: [B,T,C_main] fp32; ds_x: x for the 1x1 downsample or null.
static int run_tcn_conv(const float* main_in, int c_main, const float* ds_x, int c_ds, const float* weight, int ktot,
                        const float* bias, const float* bias2, const float* res, const float* post_scale,
                        const float* post_shift, float* out, int mode, int B, int T, int cout, int taps, int dilation,
                        cudaStream_t st) {
  TcnKernelParams p;
  memset(&p, 0, sizeof p);
  const int halo = (taps - 1) * dilation;
  const int lower[2] = {0, -halo};
  const int upper[2] = {0, -halo};
  int rc = make_im2col_map_generic(&p.tmap_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, main_in, B, T, 1, c_main, lower, upper,
                                   1, kTcBlockK);
  if (rc) return rc;
  if (ds_x != nullptr) {
    rc = make_im2col_map_generic(&p.tmap_a2, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, ds_x, B, T, 1, c_ds, lower, upper, 1,
                                 kTcBlockK);
    if (rc) return rc;
  } else {
    p.tmap_a2 = p.tmap_a;
  }
  const int bn = cout % 64 == 0 ? 64 : 32;
  rc = make_tiled2d_map_generic(&p.tmap_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, weight, cout, ktot, bn, kTcBlockK);
  if (rc) return rc;
  p.M = B * T; p.T = T; p.Cout = cout;
  p.chunks = c_main / kTcBlockK;
  p.taps = taps; p.dilation = dilation;
  p.ksteps_main = taps * p.chunks;
  p.ksteps2 = ds_x ? c_ds / kTcBlockK : 0;
  p.num_n_tiles = cout / bn;
  p.mode = mode;
  p.bias = bias; p.bias2 = bias2; p.res = res; p.post_scale = post_scale; p.post_shift = post_shift; p.out = out;
  const int grid = ((p.M + kTcBlockM - 1) / kTcBlockM) * p.num_n_tiles;
  return bn == 64 ? launch_tcn_tc<64, 8>(p, grid, st) : launch_tcn_tc<32, 8>(p, grid, st);
}

}  // namespace cer

// Tensor-core TemporalBlock.  Weight layout differs from the fp32 kernel: K-major rows,
//   w1: [c_out][k*c_in] with K = (tap j, ci);  w2: [c_out][k*c_out (+ c_in)], the 1x1 downsample
//   weights appended as the last c_in columns.  `workspace` holds h1: B*T*c_out floats.
extern "C" size_t cer_tcn_block_tc_workspace_bytes(const cer_tcn_block* blk, int64_t batch, int64_t length) {
  if (!blk || batch <= 0 || length <= 0) return 0;
  return (size_t)batch * length * blk->c_out * sizeof(float);
}

extern "C" int cer_tcn_block_tc_forward(const cer_tcn_block* blk, const float* x, float* y, int64_t batch,
                                        int64_t length, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace cer;
  if (!blk || !x || !y || batch <= 0 || length <= 0) return set_error(CER_ERR_INVALID, "cer_tcn_block_tc_forward: bad argument");
  if (blk->c_in % 32 || blk->c_out % 32) return set_error(CER_ERR_INVALID, "tcn_tc: channels must be multiples of 32");
  if (blk->kernel_size < 1 || blk->kernel_size > 8) return set_error(CER_ERR_INVALID, "tcn_tc: kernel_size out of range");
  if ((blk->kernel_size - 1) * blk->dilation > kTcMaxHalo)
    return set_error(CER_ERR_INVALID, "tcn_tc: causal halo (kernel_size-1)*dilation must be at most 128 "
                                      "(rank-4 im2col bounding-box corner limit)");
  if (!blk->w1 || !blk->b1 || !blk->w2 || !blk->b2) return set_error(CER_ERR_INVALID, "tcn_tc: null weight");
  const bool has_ds = blk->wd != nullptr;     // here `wd` only flags that w2 carries the downsample columns
  if (!has_ds && blk->c_in != blk->c_out) return set_error(CER_ERR_INVALID, "tcn_tc: identity residual needs c_in == c_out");
  if (has_ds && !blk->bd) return set_error(CER_ERR_INVALID, "tcn_tc: downsample bias missing");
  if (workspace_bytes < cer_tcn_block_tc_workspace_bytes(blk, batch, length) || !workspace)
    return set_error(CER_ERR_WORKSPACE, "tcn_tc: workspace too small");
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(workspace)) % 16)
    return set_error(CER_ERR_INVALID, "tcn_tc: pointers must be 16B aligned");
  int rc = cer_check_device();
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* h1 = static_cast<float*>(workspace);
  const int B = (int)batch, T = (int)length, k = blk->kernel_size;
  rc = run_tcn_conv(x, blk->c_in, nullptr, 0, blk->w1, k * blk->c_in, blk->b1, nullptr, nullptr, nullptr, nullptr, h1, 0,
                    B, T, blk->c_out, k, blk->dilation, st);
  if (rc) return rc;
  return run_tcn_conv(h1, blk->c_out, has_ds ? x : nullptr, blk->c_in, blk->w2, k * blk->c_out + (has_ds ? blk->c_in : 0),
                      blk->b2, blk->bd, has_ds ? nullptr : x, blk->post_scale, blk->post_shift, y, 1, B, T, blk->c_out, k,
                      blk->dilation, st);
}
