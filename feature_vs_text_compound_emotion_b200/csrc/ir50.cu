// IR frame encoder plan (IR-50/100/152, plain or with SE units): stem kernel, tcgen05 implicit-GEMM residual
// units, SE tails (se.cu), FC head, L2 norm.  C-ABI: cer_ir50_* in include/cer_b200.h.  Reference semantics:
// models/arcface_model.py:23-84, :120-151 and models/backbone.py:99-103 (see DESIGN.md for the BN folding algebra).
#include <cuda_runtime.h>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/cer_b200.h"
#include "common.h"
#include "conv_plan.h"
#include "conv_igemm2.cuh"
#include "conv_halo.cuh"
#include "stem_tc.cuh"
#include "conv_strip.cuh"
#include "conv_raster.cuh"
#include "se.h"
#include <cstdlib>

namespace cer {

// ------------------------------------------------------------------------------------------
// Stem: conv3x3(3->64, pad 1) + BN + PReLU, fp32 NCHW in -> bf16 NHWC out.  K = 27 is not a
// tensor-core shape; the kernel is bound by fp32 FMA issue (1728 FMAs per pixel), not by its
// 128 B/pixel output stream (ncu: DRAM 10 %).  Weights [27][64] are broadcast from smem.
// Reference: Backbone.input_layer, models/arcface_model.py:130-132.
// ------------------------------------------------------------------------------------------
// v2: one thread = TWO horizontally adjacent output pixels (a 3 x 4 x 3 input patch in registers,
// duplicated into {x, x} pairs once), channel PAIRS on packed fp32 FMAs (fma.rn.f32x2): per tap and
// 8 channels, 2 x LDS.128 of weights feed 8 FFMA2 = 16 FMAs (v1: 2 x LDS.128 per 8 FMAs).
__device__ __forceinline__ void stem_ffma2(unsigned long long& d, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}
__device__ __forceinline__ unsigned long long stem_dup(float x) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %1};" : "=l"(r) : "f"(x));
  return r;
}
struct alignas(16) StemW2 { unsigned long long p0, p1; };     // channels (c, c+1), (c+2, c+3)

__global__ void __launch_bounds__(128) stem_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                   const float* __restrict__ bias, const float* __restrict__ alpha,
                                                   __nv_bfloat16* __restrict__ out, int n_frames, int H, int W) {
  __shared__ __align__(16) float ws[27 * 64];
  __shared__ __align__(16) float bs[64];
  __shared__ __align__(16) float as[64];
  for (int i = threadIdx.x; i < 27 * 64; i += blockDim.x) ws[i] = w[i];
  if (threadIdx.x < 64) {
    bs[threadIdx.x] = bias[threadIdx.x];
    as[threadIdx.x] = alpha[threadIdx.x];
  }
  __syncthreads();
  const int hw = H * W;
  const int W2 = (W + 1) >> 1;
  const long long total = static_cast<long long>(n_frames) * H * W2;           // pixel pairs
  for (long long pp = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; pp < total;
       pp += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int n = static_cast<int>(pp / (H * W2));
    const int rem = static_cast<int>(pp - static_cast<long long>(n) * H * W2);
    const int oh = rem / W2, ow = (rem - oh * W2) * 2;
    const bool has_b = ow + 1 < W;
    // patch[r][cc][c], cc = 0..3 <-> input column ow - 1 + cc, duplicated for the packed FMAs
    unsigned long long in2[3][4][3];
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int ih = oh + r - 1;
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        const int iw = ow + cc - 1;
        const bool ok = ih >= 0 && ih < H && iw >= 0 && iw < W;
#pragma unroll
        for (int c = 0; c < 3; ++c)
          in2[r][cc][c] = stem_dup(ok ? __ldg(x + (static_cast<size_t>(n) * 3 + c) * hw + ih * W + iw) : 0.f);
      }
    }
    const size_t pix = (static_cast<size_t>(n) * H + oh) * W + ow;
    uint4* opa = reinterpret_cast<uint4*>(out + pix * 64);
    uint4* opb = reinterpret_cast<uint4*>(out + (pix + 1) * 64);
#pragma unroll
    for (int cg = 0; cg < 8; ++cg) {
      unsigned long long accA[4], accB[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned long long b2 = *reinterpret_cast<const unsigned long long*>(&bs[cg * 8 + 2 * j]);
        accA[j] = b2; accB[j] = b2;
      }
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s2 = 0; s2 < 3; ++s2)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const int t = (r * 3 + s2) * 3 + c;
            const StemW2 w01 = *reinterpret_cast<const StemW2*>(&ws[t * 64 + cg * 8]);
            const StemW2 w23 = *reinterpret_cast<const StemW2*>(&ws[t * 64 + cg * 8 + 4]);
            const unsigned long long ia = in2[r][s2][c], ib = in2[r][s2 + 1][c];
            stem_ffma2(accA[0], ia, w01.p0); stem_ffma2(accA[1], ia, w01.p1);
            stem_ffma2(accA[2], ia, w23.p0); stem_ffma2(accA[3], ia, w23.p1);
            stem_ffma2(accB[0], ib, w01.p0); stem_ffma2(accB[1], ib, w01.p1);
            stem_ffma2(accB[2], ib, w23.p0); stem_ffma2(accB[3], ib, w23.p1);
          }
      uint32_t pa[4], pb[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float a0, a1, b0, b1;
        asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(accA[j]));
        asm("mov.b64 {%0, %1}, %2;" : "=f"(b0), "=f"(b1) : "l"(accB[j]));
        const float s0 = as[cg * 8 + 2 * j], s1 = as[cg * 8 + 2 * j + 1];
        a0 = a0 >= 0.f ? a0 : a0 * s0; a1 = a1 >= 0.f ? a1 : a1 * s1;
        b0 = b0 >= 0.f ? b0 : b0 * s0; b1 = b1 >= 0.f ? b1 : b1 * s1;
        pa[j] = pack_bf16x2(a0, a1);
        pb[j] = pack_bf16x2(b0, b1);
      }
      opa[cg] = make_uint4(pa[0], pa[1], pa[2], pa[3]);
      if (has_b) opb[cg] = make_uint4(pb[0], pb[1], pb[2], pb[3]);
    }
  }
}

// Row-wise L2 normalisation, one warp per row (l2_norm, models/arcface_model.py:17-20; no eps).
__global__ void l2norm_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int dim) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* ip = reinterpret_cast<const float4*>(in + static_cast<size_t>(row) * dim);
  float4* op = reinterpret_cast<float4*>(out + static_cast<size_t>(row) * dim);
  float ss = 0.f;
  for (int i = lane; i < dim / 4; i += 32) {
    const float4 v = ip[i];
    ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float inv = 1.0f / sqrtf(ss);
  for (int i = lane; i < dim / 4; i += 32) {
    float4 v = ip[i];
    v.x *= inv; v.y *= inv; v.z *= inv; v.w *= inv;
    op[i] = v;
  }
}

// ------------------------------------------------------------------------------------------
// Host side: tensor maps + launch descriptors
// ------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                     const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled g_encode_tiled = nullptr;
static PFN_encodeIm2col g_encode_im2col = nullptr;
static int g_driver_version = 0;

int load_driver_entry_points() {
  if (g_encode_tiled && g_encode_im2col) return CER_OK;
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  CER_CUDA(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &q));
  if (q != cudaDriverEntryPointSuccess || !fn) return set_error(CER_ERR_CUDA, "cuTensorMapEncodeTiled not found");
  g_encode_tiled = reinterpret_cast<PFN_encodeTiled>(fn);
  CER_CUDA(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeIm2col", &fn, 12000, cudaEnableDefault, &q));
  if (q != cudaDriverEntryPointSuccess || !fn) return set_error(CER_ERR_CUDA, "cuTensorMapEncodeIm2col not found");
  g_encode_im2col = reinterpret_cast<PFN_encodeIm2col>(fn);
  CER_CUDA(cudaDriverGetVersion(&g_driver_version));
  return CER_OK;
}

// NHWC bf16 activation [N][H][W][C], im2col traversal of a k x k / stride / pad convolution.
static int make_im2col_map(CUtensorMap* map, const void* base, int N, int H, int W, int C, int ksize, int stride,
                           int pad) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  int lower[2] = {-pad, -pad};
  int upper[2] = {pad - (ksize - 1), pad - (ksize - 1)};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = g_encode_im2col(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides,
                               lower, upper, /*channelsPerPixel*/ kBlockK, /*pixelsPerColumn*/ kBlockM, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[160];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeIm2col failed (%d) N=%d H=%d W=%d C=%d k=%d s=%d", (int)r, N, H, W, C,
             ksize, stride);
    return set_error(CER_ERR_CUDA, buf);
  }
  // Driver quirk (same guard as CUTLASS' im2col descriptor builder): small tensors need bit 21 of
  // descriptor word 1 cleared on drivers <= 13.1.
  if (g_driver_version <= 13010 && (size_t)N * H * W * C * 2 < 131072)
    reinterpret_cast<uint64_t*>(map)[1] &= ~(1ull << 21);
  return CER_OK;
}

// Packed weights [Cout][K] bf16 (rows of ld >= K elements; 0: ld = K), box = 64 (k) x BN (cout), 128B swizzle.
static int make_weight_map(CUtensorMap* map, const void* base, int Cout, int K, int BN, int ld = 0) {
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)Cout};
  cuuint64_t strides[1] = {(cuuint64_t)(ld > 0 ? ld : K) * 2};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)BN};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                              estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[128];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (%d) Cout=%d K=%d BN=%d", (int)r, Cout, K, BN);
    return set_error(CER_ERR_CUDA, buf);
  }
  return CER_OK;
}

// NHWC bf16 activation as a tiled 4-D map whose box is the (16+2) x (8+2) pixel halo of one output
// tile, 64 channels deep (conv_halo_kernel).  Out-of-bounds pixels read as zero = the conv padding.
static int make_halo_map(CUtensorMap* map, const void* base, int N, int H, int W, int C) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)(kHaloTileW + 2), (cuuint32_t)(kHaloTileH + 2), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[128];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled (halo) failed (%d) N=%d H=%d W=%d C=%d", (int)r, N, H, W, C);
    return set_error(CER_ERR_CUDA, buf);
  }
  return CER_OK;
}

// The same activation with an 8-row x (8+2)-pixel box: one half tile of one filter row of conv_strip_kernel.
static int make_strip_map(CUtensorMap* map, const void* base, int N, int H, int W, int C) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)(kHaloTileW + 2), (cuuint32_t)kStripBoxRows, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[128];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled (strip) failed (%d) N=%d H=%d W=%d C=%d", (int)r, N, H, W, C);
    return set_error(CER_ERR_CUDA, buf);
  }
  return CER_OK;
}

// Generic helpers shared with the TCN tensor-core path (tcn_tc.cu).
int make_im2col_map_generic(CUtensorMap* map, CUtensorMapDataType dt, int elem_bytes, const void* base, int N, int H,
                            int W, int C, const int lower[2], const int upper[2], int stride, int channels_per_pixel) {
  int rc = load_driver_entry_points();
  if (rc) return rc;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * elem_bytes, (cuuint64_t)W * C * elem_bytes, (cuuint64_t)H * W * C * elem_bytes};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = g_encode_im2col(map, dt, 4, const_cast<void*>(base), dims, strides, lower, upper, channels_per_pixel,
                               kBlockM, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[160];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeIm2col failed (%d) N=%d H=%d W=%d C=%d elem=%d", (int)r, N, H, W, C, elem_bytes);
    return set_error(CER_ERR_CUDA, buf);
  }
  if (g_driver_version <= 13010 && (size_t)N * H * W * C * elem_bytes < 131072)
    reinterpret_cast<uint64_t*>(map)[1] &= ~(1ull << 21);
  return CER_OK;
}

int make_tiled2d_map_generic(CUtensorMap* map, CUtensorMapDataType dt, int elem_bytes, const void* base, int rows,
                             int cols, int box_rows, int box_cols) {
  int rc = load_driver_entry_points();
  if (rc) return rc;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(map, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[128];
    snprintf(buf, sizeof buf, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d", (int)r, rows, cols);
    return set_error(CER_ERR_CUDA, buf);
  }
  return CER_OK;
}

static int pick_bn(int cout) { return cout % 256 == 0 ? 256 : (cout % 128 == 0 ? 128 : 64); }

// Fused pooling needs every 2x2 window inside one warp of the epilogue: 32 consecutive tile rows must
// cover whole pairs of map rows (halo tiles: always; im2col tiles: W in {8, 16}, H*W a multiple of 32
// so that frames start on even rows of a 128-pixel tile).
bool conv_can_pool(int H, int W, int Cin, int Cout) {
  if ((H & 1) || (W & 1) || Cout % 64) return false;
  if (Cin == 64) return W % kHaloTileW == 0 && (Cout == 64 || Cout == 128);
  return (W == 8 || W == 16) && (H * W) % 32 == 0 && Cin % 64 == 0;
}

// Copies the per-channel epilogue constants to the host so that they travel as kernel parameters (ConvKernelParams::ctab).
// Synchronous device-to-host copies: plan creation only (cer_conv_forward builds its op per call and keeps the
// shared-memory tables).
static int fill_ctab(ConvKernelParams* kp, const ConvGeom& g) {
  kp->ctab_flags = 0;
  if (g.Cout > kCtabMaxCout) return CER_OK;
  if (g.alpha) {
    CER_CUDA(cudaMemcpy(kp->ctab, g.alpha, (size_t)g.Cout * sizeof(float), cudaMemcpyDeviceToHost));
    kp->ctab_flags |= kCtabAlpha;
  }
  if (g.bias_classes == 1 && g.bias) {
    CER_CUDA(cudaMemcpy(kp->ctab + 512, g.bias, (size_t)g.Cout * sizeof(float), cudaMemcpyDeviceToHost));
    kp->ctab_flags |= kCtabBias;
  }
  return CER_OK;
}

// CER_CTAB=0 keeps every epilogue constant in shared memory (A/B timing); read when a plan is created.
static bool ctab_enabled() {
  const char* e = getenv("CER_CTAB");
  return !(e && e[0] == '0');
}

int build_conv_op(ConvOp* op, const ConvGeom& g, int n_cap, bool host_tables) {
  if (g.Cin % kBlockK || g.Cin2 % kBlockK || g.Cout % 64) return set_error(CER_ERR_INVALID, "channels must be multiples of 64");
  memset(op, 0, sizeof *op);
  const int Hout = (g.H + 2 * g.pad - g.ksize) / g.stride + 1;
  const int Wout = (g.W + 2 * g.pad - g.ksize) / g.stride + 1;
  op->bn = pick_bn(g.Cout);
  {
    // few output rows (the 12800 -> 512 FC: M = frames): 128 x 256 tiles would occupy a quarter of the SMs;
    // narrower N tiles trade L2 re-reads of A for parallelism
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long m_tiles = ((long long)n_cap * Hout * Wout + kBlockM - 1) / kBlockM;
    while (op->bn > 64 && m_tiles * (g.Cout / op->bn) < sms / 2 && (g.bias_classes + 1) * g.Cout <= 10 * (op->bn / 2))
      op->bn /= 2;          // the epilogue table of the narrower instantiation must still hold [classes + 1][Cout]
  }
  op->hw_out = Hout * Wout;
  ConvKernelParams& p = op->kp;
  int rc = make_im2col_map(&p.tmap_a, g.src, n_cap, g.H, g.W, g.Cin, g.ksize, g.stride, g.pad);
  if (rc) return rc;
  if (g.Cin2 > 0) {
    rc = make_im2col_map(&p.tmap_a2, g.src2, n_cap, g.H2, g.W2, g.Cin2, 1, g.stride2, 0);
    if (rc) return rc;
    if ((g.H2 - 1) / g.stride2 + 1 != Hout || (g.W2 - 1) / g.stride2 + 1 != Wout)
      return set_error(CER_ERR_INVALID, "shortcut geometry mismatch");
  } else {
    p.tmap_a2 = p.tmap_a;
  }
  const int ktot = g.ksize * g.ksize * g.Cin + g.Cin2;
  rc = make_weight_map(&p.tmap_b, g.weight, g.Cout, ktot, op->bn, g.wld);
  if (rc) return rc;
  rc = make_weight_map(&op->tmap_b_half, g.weight, g.Cout, ktot, op->bn / 2, g.wld);
  if (rc) return rc;
  p.Hout = Hout; p.Wout = Wout; p.Cout = g.Cout;
  p.cin_chunks = g.Cin / kBlockK;
  p.cin_shift = 0;
  while ((1 << p.cin_shift) < p.cin_chunks) ++p.cin_shift;
  if (g.ksize == 3 && (1 << p.cin_shift) != p.cin_chunks)
    return set_error(CER_ERR_INVALID, "3x3 conv needs Cin/64 to be a power of two");
  p.ksize = g.ksize;
  p.ksteps_main = g.ksize * g.ksize * p.cin_chunks;
  p.ksteps2 = g.Cin2 / kBlockK;
  p.stride = g.stride; p.pad = g.pad; p.stride2 = g.stride2 > 0 ? g.stride2 : 1;
  p.num_n_tiles = g.Cout / op->bn;
  p.bias_classes = g.bias_classes;
  p.out_fp32 = g.out_fp32;
  p.bias = g.bias; p.alpha = g.alpha; p.res = g.res; p.out = g.dst;
  p.pool_xor = 0;
  if (g.pool) {
    if (!conv_can_pool(g.H, g.W, g.Cin, g.Cout) || g.ksize != 3 || g.stride != 1 || g.pad != 1 || g.res || g.out_fp32 || g.Cin2)
      return set_error(CER_ERR_INVALID, "conv: this layer cannot fuse the max-pool");
    p.pool_xor = (g.Cin == 64) ? kHaloTileW : g.W;        // halo tiles are 8 pixels wide; im2col tiles follow the map width
  }
  op->halo_ok = g.ksize == 3 && g.stride == 1 && g.pad == 1 && g.Cin == 64 && g.Cin2 == 0 && (g.Cout == 64 || g.Cout == 128) &&
                g.W % kHaloTileW == 0 && !g.out_fp32;
  if (op->halo_ok) {
    rc = make_halo_map(&op->tmap_halo, g.src, n_cap, g.H, g.W, g.Cin);
    if (rc) return rc;
  }
  op->strip_ok = op->halo_ok && g.Cout == 64 && g.H % kStripBoxRows == 0 && !g.pool;
  if (op->strip_ok) {
    rc = make_strip_map(&op->tmap_strip, g.src, n_cap, g.H, g.W, g.Cin);
    if (rc) return rc;
  }
  if (host_tables && ctab_enabled()) return fill_ctab(&p, g);
  return CER_OK;
}

// CER_PDL=0 disables programmatic dependent launch (A/B timing).
static bool pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CER_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// All conv launches go through here: optional 2-CTA cluster, programmatic stream serialization so
// that the next layer's prologue overlaps this layer's tail (the kernels call griddepcontrol.wait
// before touching activations).
template <typename Kernel>
static int launch_conv_kernel(Kernel kernel, int grid, int threads, size_t smem, cudaStream_t st, int cluster,
                              const ConvKernelParams& p) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cluster; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr; cfg.numAttrs = na;
  CER_CUDA(cudaLaunchKernelEx(&cfg, kernel, p));
  return CER_OK;
}

template <int BN>
static int launch_halo_inst(const ConvKernelParams& p, int num_sms, cudaStream_t st) {
  using L = HaloSmem<BN>;
  static_assert(L::kTotal <= 232448, "halo conv kernel shared memory exceeds 227 KB");
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(conv_halo_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
  }
  const int tiles = p.halo_frames * p.halo_bands * p.halo_cts;
  return launch_conv_kernel(conv_halo_kernel<BN>, std::min(tiles, num_sms), kHaloThreads, L::kTotal, st, 1, p);
}

static int launch_strip_inst(const ConvKernelParams& p, int num_sms, cudaStream_t st) {
  using L = StripSmem;
  static_assert(L::kTotal <= 232448, "strip conv kernel shared memory exceeds 227 KB");
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(conv_strip_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
  }
  const long long vrows = (long long)p.halo_frames * p.halo_cts * p.Hout;
  const int tiles = (int)((vrows + 15) / 16);
  return launch_conv_kernel(conv_strip_kernel, std::min(tiles, num_sms), kHaloThreads, L::kTotal, st, 1, p);
}

// CER_STRIP=0: keep the halo kernel for the 64 -> 64 layers (A/B timing).
static bool strip_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CER_STRIP"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

// CER_HALO: unset/1 = halo kernel for the Cin = 64 layers, 0 = im2col kernel (A/B timing).
static int halo_mode() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CER_HALO"); v = e ? atoi(e) : 1; }
  return v;
}

template <int BN, int STAGES, bool BRES, bool ALIGNED>
static int launch_conv_inst(const ConvKernelParams& p, int grid, cudaStream_t st) {
  using L = ConvSmem<BN, STAGES, BRES>;
  static_assert(L::kTotal <= 232448, "conv kernel shared memory exceeds 227 KB");
  static_assert(!ALIGNED || (BRES ? STAGES % 3 == 0 : STAGES % 2 == 0), "aligned variant: producers must divide the ring");
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<BN, STAGES, BRES, ALIGNED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  L::kTotal));
  }
  if ((p.bias_classes + 1) * p.Cout > L::kTableFloats) return set_error(CER_ERR_INVALID, "conv: Cout too large for the epilogue table");
  return launch_conv_kernel(conv_igemm_kernel<BN, STAGES, BRES, ALIGNED>, grid, kConvThreads, L::kTotal, st, 1, p);
}

template <int BN, int STAGES>
static int launch_conv2_inst(const ConvKernelParams& p, int num_sms, cudaStream_t st) {
  using L = Conv2Smem<BN, STAGES>;
  static_assert(L::kTotal <= 232448, "pair conv kernel shared memory exceeds 227 KB");
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(conv_igemm2_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
  }
  if ((p.bias_classes + 1) * p.Cout > L::kTableFloats) return set_error(CER_ERR_INVALID, "conv: Cout too large for the epilogue table");
  const int ptiles = ((p.num_m_tiles + 1) / 2) * p.num_n_tiles;
  const int pairs = std::min(ptiles, num_sms / 2);
  return launch_conv_kernel(conv_igemm2_kernel<BN, STAGES>, 2 * pairs, kConvThreads, L::kTotal, st, 2, p);
}

template <int BN, int STAGES, int KSTEPS>
static int launch_conv2_bres_inst(const ConvKernelParams& p, int num_sms, cudaStream_t st) {
  using L = Conv2BresSmem<BN, STAGES, KSTEPS>;
  static_assert(L::kTotal <= 232448, "resident-weights pair conv kernel shared memory exceeds 227 KB");
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(conv_igemm2_bres_kernel<BN, STAGES, KSTEPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::kTotal));
  }
  if ((p.bias_classes + 1) * p.Cout > L::kTableFloats) return set_error(CER_ERR_INVALID, "conv: Cout too large for the epilogue table");
  const int pairs = std::min((p.num_m_tiles + 1) / 2, num_sms / 2);
  return launch_conv_kernel(conv_igemm2_bres_kernel<BN, STAGES, KSTEPS>, 2 * pairs, kConvThreads, L::kTotal, st, 2, p);
}

// CER_PAIR_BRES=0 disables the weights-resident pair variant (A/B timing).
static bool pair_bres_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CER_PAIR_BRES"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

static bool pair_mode_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CER_NO_PAIR"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

// Which kernel instantiation a layer runs at a given number of frames.  Selection is separate from
// launching so that the plan can REPORT its choice (cer_ir50_op_variant / cer_conv_last_variant):
// bench.py labels its roofline line with the variant that actually ran.
enum ConvVariant {
  kVarNone = 0, kVarStrip64, kVarHalo64, kVarHalo128, kVarPairBres128, kVarPairBres128Proj, kVarPair256, kVarPair128,
  kVar256Aligned, kVar256, kVar128Bres, kVar128Aligned, kVar128, kVar64Bres9, kVar64Aligned, kVar64
};
static const char* const kVariantNames[] = {
  "none", "conv_strip_kernel", "conv_halo_kernel<64>", "conv_halo_kernel<128>", "conv_igemm2_bres_kernel<128,4,18>",
  "conv_igemm2_bres_kernel<128,4,19>",
  "conv_igemm2_kernel<256,6>", "conv_igemm2_kernel<128,6>", "conv_igemm_kernel<256,4,0,1>", "conv_igemm_kernel<256,4,0,0>",
  "conv_igemm_kernel<128,4,1,0>", "conv_igemm_kernel<128,6,0,1>", "conv_igemm_kernel<128,6,0,0>",
  "conv_igemm_kernel<64,9,1,1>", "conv_igemm_kernel<64,8,0,1>", "conv_igemm_kernel<64,8,0,0>"};

static ConvVariant select_conv_variant(const ConvOp& op, int frames, int num_sms) {
  const ConvKernelParams& p = op.kp;
  const int num_m_tiles = (frames * op.hw_out + kBlockM - 1) / kBlockM;
  const int tiles = num_m_tiles * p.num_n_tiles;
  if (tiles == 0) return kVarNone;
  if (op.halo_ok && ((halo_mode() != 0 && tiles >= 2 * num_sms) || (p.pool_xor && p.cin_chunks == 1))) {
    if (op.strip_ok && !p.pool_xor && strip_enabled() && halo_mode() != 0 && tiles >= 2 * num_sms) return kVarStrip64;
    return op.bn == 64 ? kVarHalo64 : kVarHalo128;
  }
  const int grid = std::min(tiles, num_sms);
  const int ksteps = p.ksteps_main + p.ksteps2;
  // the 128 -> 128 stride-2 conv with its fused 64-channel projection (18 + 1 k-steps): weights resident, CTA pair
  if (pair_mode_enabled() && pair_bres_enabled() && op.bn == 128 && p.num_n_tiles == 1 && p.ksize == 3 && p.ksteps_main == 18 &&
      p.ksteps2 == 1 && tiles >= 4 * num_sms && !p.pool_xor)
    return kVarPairBres128Proj;
  // CTA-pair (cta_group::2) variant: plain 3x3 / 1x1 layers whose k-steps fill the 6-stage ring a whole
  // number of times and that have at least two waves of pair tiles
  if (pair_mode_enabled() && p.ksteps2 == 0 && ksteps % 6 == 0 && tiles >= 4 * num_sms && op.bn >= 128) {
    if (op.bn == 128 && p.num_n_tiles == 1 && ksteps == 18 && pair_bres_enabled()) return kVarPairBres128;   // stage 2: weights stay in smem
    return op.bn == 256 ? kVarPair256 : kVarPair128;
  }
  // weights-resident variants when the whole layer's B fits (Cin = 64 layers: 9 k-steps, one n-tile)
  const bool bres = p.num_n_tiles == 1 && ksteps <= kBresSteps && tiles >= 4 * grid;
  switch (op.bn) {
    case 256: return ksteps % 4 == 0 ? kVar256Aligned : kVar256;
    case 128: return bres ? kVar128Bres : (ksteps % 6 == 0 ? kVar128Aligned : kVar128);
    default:  return (bres && ksteps == 9) ? kVar64Bres9 : (ksteps % 8 == 0 ? kVar64Aligned : kVar64);
  }
}

const char* conv_variant_name(const ConvOp& op, int frames, int num_sms) {
  return kVariantNames[select_conv_variant(op, frames, num_sms)];
}

static thread_local const char* g_last_variant = "none";
const char* conv_last_variant() { return g_last_variant; }
static void g_last_variant_set(const char* v) { g_last_variant = v; }

int launch_conv(const ConvOp& op, int frames, int num_sms, cudaStream_t st, int out_wp) {
  ConvKernelParams p = op.kp;
  p.out_wp = out_wp;
  p.M = frames * op.hw_out;
  p.num_m_tiles = (p.M + kBlockM - 1) / kBlockM;
  const int tiles = p.num_m_tiles * p.num_n_tiles;
  const ConvVariant var = select_conv_variant(op, frames, num_sms);
  g_last_variant = kVariantNames[var];
  const int grid = std::min(tiles, num_sms);
  if (out_wp && (var == kVarStrip64 || var == kVarHalo64 || var == kVarHalo128))
    return set_error(CER_ERR_INVALID, "launch_conv: the halo / strip kernels cannot store a padded raster");
  switch (var) {
    case kVarNone: return CER_OK;
    case kVarStrip64:
      p.tmap_a = op.tmap_strip;
      p.halo_frames = frames;
      p.halo_cts = p.Wout / kHaloTileW;
      return launch_strip_inst(p, num_sms, st);
    case kVarHalo64:
    case kVarHalo128:
      p.tmap_a = op.tmap_halo;
      p.halo_frames = frames;
      p.halo_bands = (p.Hout + kHaloTileH - 1) / kHaloTileH;
      p.halo_cts = p.Wout / kHaloTileW;
      return var == kVarHalo64 ? launch_halo_inst<64>(p, num_sms, st) : launch_halo_inst<128>(p, num_sms, st);
    case kVarPairBres128: p.tmap_b = op.tmap_b_half; return launch_conv2_bres_inst<128, 4, 18>(p, num_sms, st);
    case kVarPairBres128Proj: p.tmap_b = op.tmap_b_half; return launch_conv2_bres_inst<128, 4, 19>(p, num_sms, st);
    case kVarPair256:     p.tmap_b = op.tmap_b_half; return launch_conv2_inst<256, 6>(p, num_sms, st);
    case kVarPair128:     p.tmap_b = op.tmap_b_half; return launch_conv2_inst<128, 6>(p, num_sms, st);
    case kVar256Aligned:  return launch_conv_inst<256, 4, false, true>(p, grid, st);
    case kVar256:         return launch_conv_inst<256, 4, false, false>(p, grid, st);
    case kVar128Bres:     return launch_conv_inst<128, 4, true, false>(p, grid, st);
    case kVar128Aligned:  return launch_conv_inst<128, 6, false, true>(p, grid, st);
    case kVar128:         return launch_conv_inst<128, 6, false, false>(p, grid, st);
    case kVar64Bres9:     return launch_conv_inst<64, 9, true, true>(p, grid, st);
    case kVar64Aligned:   return launch_conv_inst<64, 8, false, true>(p, grid, st);
    case kVar64:          return launch_conv_inst<64, 8, false, false>(p, grid, st);
  }
  return set_error(CER_ERR_INVALID, "launch_conv: unknown variant");
}

// ------------------------------------------------------------------------------------------
// Padded-raster stage (conv_raster.cuh): plan-level helpers.
// ------------------------------------------------------------------------------------------
static const char* const kRasterName128 = "conv_raster2_kernel<128,3,18,176>";
static const int kRasterBoxRows128 = 176;

// CER_RASTER=0 keeps the im2col / strip kernels for the identity stages (A/B timing); read when a plan is created.
bool raster_enabled() {
  const char* e = getenv("CER_RASTER");
  return !(e && e[0] == '0');
}

// can a 3x3/s1/p1 identity unit with these channels over an H x W map run on the raster kernel?
bool raster_unit_ok(int H, int W, int cin, int depth, int stride, int has_proj) {
  if (has_proj || stride != 1 || cin != depth || H < 2 || W < 2) return false;
  // 64 -> 64 stages stay on the strip kernel: the <64,6,9,216> instantiation of the raster kernel (pair MMAs of
  // N = 64, the stem storing the padded raster) was measured at 2.21 ms for IR-50 stage 1 against 2.07 ms
  return cin == 128 && kBlockM + 2 * (W + 2) <= kRasterBoxRows128;
}

// kernel parameters of one raster conv: src / res are padded rasters [n_cap][(H+1)][(W+1)][C], dst too unless
// out_padded == 0 (dense NHWC for a consumer that is not a raster kernel)
int build_raster_op(ConvKernelParams* kp, CUtensorMap* tmap_b_half, const ConvGeom& g, int n_cap, int out_padded) {
  memset(kp, 0, sizeof *kp);
  const int wp = g.W + 1, P = (g.H + 1) * wp;
  int rc = make_tiled2d_map_generic(&kp->tmap_a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, g.src, n_cap * P, g.Cin,
                                    kBlockM + 2 * (wp + 1), kBlockK);
  if (rc) return rc;
  rc = make_weight_map(tmap_b_half, g.weight, g.Cout, 9 * g.Cin, g.Cout / 2);
  if (rc) return rc;
  kp->tmap_b = *tmap_b_half;
  kp->tmap_a2 = kp->tmap_a;
  kp->Hout = g.H; kp->Wout = g.W; kp->Cout = g.Cout;
  kp->cin_chunks = g.Cin / kBlockK; kp->cin_shift = kp->cin_chunks == 2 ? 1 : 0; kp->ksize = 3;
  kp->ksteps_main = 9 * kp->cin_chunks; kp->ksteps2 = 0;
  kp->stride = 1; kp->pad = 1; kp->stride2 = 1;
  kp->num_n_tiles = 1;
  kp->bias_classes = g.bias_classes;
  kp->out_fp32 = 0;
  kp->bias = g.bias; kp->alpha = g.alpha; kp->res = g.res; kp->out = g.dst;
  kp->rs_wp = wp; kp->rs_P = P;
  kp->out_wp = out_padded ? wp : 0;
  if (ctab_enabled()) return fill_ctab(kp, g);
  return CER_OK;
}

template <int BN, int SLOTS, int KSTEPS, int BOX_ROWS_MAX>
static int launch_raster_inst(const ConvKernelParams& p, int ptiles, int num_sms, cudaStream_t st) {
  using L = RasterSmem<BN, SLOTS, KSTEPS, BOX_ROWS_MAX>;
  static_assert(L::kTotal <= 232448, "raster conv kernel shared memory exceeds 227 KB");
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured))
    CER_CUDA(cudaFuncSetAttribute(conv_raster2_kernel<BN, SLOTS, KSTEPS, BOX_ROWS_MAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  L::kTotal));
  return launch_conv_kernel(conv_raster2_kernel<BN, SLOTS, KSTEPS, BOX_ROWS_MAX>, 2 * std::min(ptiles, num_sms / 2), kConvThreads,
                            L::kTotal, st, 2, p);
}

static const char* raster_variant_name(const ConvKernelParams&) { return kRasterName128; }

int launch_raster(const ConvKernelParams& kp, int frames, int num_sms, cudaStream_t st) {
  ConvKernelParams p = kp;
  p.rs_frames = frames;
  p.M = frames * p.Hout * p.Wout;
  const long long pos = (long long)frames * p.rs_P;
  const int ptiles = (int)((pos + 2 * kBlockM - 1) / (2 * kBlockM));
  if (ptiles == 0) return CER_OK;
  g_last_variant_set(raster_variant_name(kp));
  return launch_raster_inst<128, 3, 18, kRasterBoxRows128>(p, ptiles, num_sms, st);
}

// CER_STEM_TC=0 keeps the CUDA-core stem (A/B timing, exact-fp32 first layer).
static bool stem_tc_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("CER_STEM_TC"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}

int launch_stem(const float* x, const float* w, const float* bias, const float* alpha, __nv_bfloat16* out,
                const CUtensorMap& tmap_out, int frames, int H, int W, int num_sms, cudaStream_t st) {
  if (frames <= 0) return CER_OK;
  if (stem_tc_enabled()) {
    static unsigned long long configured = 0;
    if (first_use_on_device(&configured))
      CER_CUDA(cudaFuncSetAttribute(stem_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, StemSmem::kTotal));
    ConvKernelParams p;
    memset(&p, 0, sizeof p);
    p.M = frames * H * W;
    p.Hout = H; p.Wout = W; p.Cout = 64;
    p.num_m_tiles = (p.M + kBlockM - 1) / kBlockM; p.num_n_tiles = 1;
    p.bias_classes = 1; p.bias = bias; p.alpha = alpha; p.out = out;
    stem_tc_kernel<<<std::min(p.num_m_tiles, num_sms), kStemThreads, StemSmem::kTotal, st>>>(p, tmap_out, x, w);
  } else {
    const long long pix = (long long)frames * H * ((W + 1) / 2);      // one thread per pixel pair
    const int blocks = (int)std::min<long long>((pix + 127) / 128, (long long)num_sms * 16);
    stem_kernel<<<blocks, 128, 0, st>>>(x, w, bias, alpha, out, frames, H, W);
  }
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

}  // namespace cer

using namespace cer;

struct cer_ir50 {
  cer_ir50_weights w;
  std::vector<cer_ir_unit> units;
  int64_t cap;            // frames per pass
  int n_cap;              // cap + padding frames (tensor-map N extent)
  int num_sms;
  uint8_t* buf[3];
  float* fc_out;          // [cap][emb_dim] pre-norm
  size_t act_bytes;       // per activation buffer
  std::vector<ConvOp> ops;          // 2 per unit, then FC
  // Padded-raster mode (conv_raster.cuh), used by a pass with enough frames (raster_pass): per op, the raster
  // kernel's parameters when the op runs on it (rast_ok) and whether the op's OUTPUT is then stored as a padded
  // raster (out_padded; for an im2col producer the pad positions are zeroed by raster_zero_pads_kernel).
  struct RasterOp { int rast_ok; int out_padded; ConvKernelParams kp; CUtensorMap tmap_b_half; };
  std::vector<RasterOp> rops;       // 2 per unit
  int raster_hw;                    // smallest map (pixels per frame) among the raster stages (0: none in this plan)
  struct ActInfo { const void* ptr; int H, W, C; };
  std::vector<ActInfo> unit_out;    // where each unit's output lives
  ActInfo stem_out;
  CUtensorMap stem_out_map;         // stem output [pixels][64] bf16 for the TMA store of stem_tc_kernel
  // IR-SE units (cer_ir50_create_se): conv2 stores the pre-gate r; the projection conv (ops[proj_op], after the FC)
  // writes the shortcut into the conv1 buffer; then squeeze-excite into `gate` and r * gate + shortcut over r.
  struct SeTail {
    int on, hidden;
    const float* fc1; const float* fc2;
    int proj_op;                    // -1: identity shortcut read from the unit input at stride sc_stride
    const __nv_bfloat16* sc; int sc_h, sc_w, sc_stride;
    __nv_bfloat16* r; int Ho, Wo, C;
  };
  std::vector<SeTail> se;           // per unit (all off for an IR plan)
  float* gate;                      // [cap][512] fp32, SE plans only
};

static const int kPadFrames = 8;   // a 128-pixel tile may run at most 127 pixels (<= 6 frames of 5x5) past the end

static size_t max_act_bytes_per_frame(const cer_ir50_weights* w) {
  int H = w->in_h, W = w->in_w;
  size_t mx = (size_t)H * W * 64 * 2;
  for (int i = 0; i < w->n_units; ++i) {
    const cer_ir_unit& u = w->units[i];
    mx = std::max(mx, (size_t)H * W * u.depth * 2);
    H = (H - 1) / u.stride + 1;
    W = (W - 1) / u.stride + 1;
    mx = std::max(mx, (size_t)H * W * u.depth * 2);
  }
  return mx;
}

// Marks the run of identity units that can use the raster kernel and builds their parameters.  The buffer
// rotation of cer_ir50_create is replayed so that every op sees the same src / res / dst pointers.
static int build_raster_stage(cer_ir50* p) {
  const int n_units = (int)p->units.size();
  p->rops.assign(2 * n_units, cer_ir50::RasterOp{});
  p->raster_hw = 0;
  if (!raster_enabled()) return CER_OK;
  int H = p->w.in_h, W = p->w.in_w;
  int cur = 0, tb = 1, nxt = 2;
  std::vector<int> ok(n_units + 1, 0);
  {
    int h = H, w2 = W;
    for (int i = 0; i < n_units; ++i) {
      const cer_ir_unit& u = p->units[i];
      // an SE unit runs on the im2col kernels; its tail stores dense NHWC, so the unit after it cannot start a run
      ok[i] = raster_unit_ok(h, w2, u.cin, u.depth, u.stride, u.has_proj) && !p->se[i].on && !(i > 0 && p->se[i - 1].on);
      // the tensor a run starts from must be storable as a padded raster: by an im2col kernel (Cin >= 128: never
      // the halo / strip kernels), not by the stem
      if (ok[i] && (i == 0 || (!ok[i - 1] && p->units[i - 1].depth < 128))) ok[i] = 0;
      if (ok[i]) p->raster_hw = p->raster_hw ? std::min(p->raster_hw, h * w2) : h * w2;
      h = (h - 1) / u.stride + 1; w2 = (w2 - 1) / u.stride + 1;
    }
    if (!p->raster_hw) return CER_OK;
  }
  for (int i = 0; i < n_units; ++i) {
    const cer_ir_unit& u = p->units[i];
    if (ok[i]) {
      ConvGeom g1{};
      g1.src = p->buf[cur]; g1.H = H; g1.W = W; g1.Cin = u.cin; g1.ksize = 3; g1.stride = 1; g1.pad = 1;
      g1.weight = u.w1; g1.bias = u.bias1; g1.bias_classes = 9; g1.alpha = u.alpha; g1.res = nullptr;
      g1.dst = p->buf[tb]; g1.Cout = u.depth;
      cer_ir50::RasterOp& r1 = p->rops[2 * i];
      int rc = build_raster_op(&r1.kp, &r1.tmap_b_half, g1, p->n_cap, /*out_padded*/ 1);
      if (rc) return rc;
      r1.rast_ok = 1; r1.out_padded = 1;
      ConvGeom g2 = g1;
      g2.src = p->buf[tb]; g2.weight = u.w2; g2.bias = u.bias2; g2.bias_classes = 1; g2.alpha = nullptr;
      g2.res = reinterpret_cast<const __nv_bfloat16*>(p->buf[cur]); g2.dst = p->buf[nxt];
      cer_ir50::RasterOp& r2 = p->rops[2 * i + 1];
      rc = build_raster_op(&r2.kp, &r2.tmap_b_half, g2, p->n_cap, /*out_padded*/ ok[i + 1]);
      if (rc) return rc;
      r2.rast_ok = 1; r2.out_padded = ok[i + 1];
    } else if (ok[i + 1]) {
      p->rops[2 * i + 1].out_padded = 1;          // im2col producer in front of the stage
    }
    H = (H - 1) / u.stride + 1;
    W = (W - 1) / u.stride + 1;
    std::swap(cur, nxt);
  }
  return CER_OK;
}

// does a pass over `frames` frames run the raster stage?  (same two-waves-of-pair-tiles rule as the pair kernels)
static bool raster_pass(const cer_ir50* p, int frames) {
  return p->raster_hw > 0 && ((long long)frames * p->raster_hw + kBlockM - 1) / kBlockM >= 4LL * p->num_sms;
}

// the SE tail of unit i after its conv2: projection conv (transition units), squeeze-excite, scale + shortcut
static int launch_se_tail(cer_ir50* p, int i, int frames, cudaStream_t st) {
  const cer_ir50::SeTail& s = p->se[i];
  if (s.proj_op >= 0) {
    int rc = launch_conv(p->ops[s.proj_op], frames, p->num_sms, st);
    if (rc) return rc;
  }
  int rc = launch_se_squeeze(s.r, s.fc1, s.fc2, p->gate, frames, s.Ho * s.Wo, s.C, s.hidden, st);
  if (rc) return rc;
  return launch_se_scale(s.r, p->gate, s.sc, frames, s.Ho, s.Wo, s.C, s.sc_h, s.sc_w, s.sc_stride, p->num_sms, st);
}

// one op of a pass (op = 0 .. 2U-1 unit convs, 2U = FC); the conv2 op of an SE unit includes the unit's SE tail
static int launch_plan_op(cer_ir50* p, int op, int frames, bool rast, cudaStream_t st) {
  const int n_units = (int)p->units.size();
  if (op < 2 * n_units && (op & 1) && p->se[op >> 1].on) {
    int rc = launch_conv(p->ops[op], frames, p->num_sms, st);
    if (rc) return rc;
    return launch_se_tail(p, op >> 1, frames, st);
  }
  if (!rast || op >= 2 * n_units) return launch_conv(p->ops[op], frames, p->num_sms, st);
  const cer_ir50::RasterOp& r = p->rops[op];
  if (r.rast_ok) return launch_raster(r.kp, frames, p->num_sms, st);
  if (!r.out_padded) return launch_conv(p->ops[op], frames, p->num_sms, st);
  const ConvKernelParams& kp = p->ops[op].kp;
  const long long vecs = (long long)frames * (kp.Hout + kp.Wout + 1) * (kp.Cout / 8);
  raster_zero_pads_kernel<<<(int)std::min<long long>((vecs + 255) / 256, 4LL * p->num_sms), 256, 0, st>>>(
      static_cast<__nv_bfloat16*>(kp.out), frames, kp.Hout, kp.Wout, kp.Cout);
  CER_CUDA(cudaGetLastError());
  return launch_conv(p->ops[op], frames, p->num_sms, st, kp.Wout + 1);
}

static const int kSeMaxC = 512;     // gate buffer row: the widest unit
static size_t gate_bytes(int64_t frames_per_pass) { return ((size_t)frames_per_pass * kSeMaxC * 4 + 1023) & ~size_t(1023); }

extern "C" size_t cer_ir50_workspace_bytes_se(const cer_ir50_weights* w, const cer_ir_se* se, int64_t frames_per_pass) {
  if (!w || frames_per_pass <= 0) return 0;
  const size_t act = ((max_act_bytes_per_frame(w) * (frames_per_pass + kPadFrames)) + 1023) & ~size_t(1023);
  const size_t fc = (((size_t)frames_per_pass + kPadFrames) * w->emb_dim * 4 + 1023) & ~size_t(1023);
  return 3 * act + fc + 1024 + (se ? gate_bytes(frames_per_pass) : 0);
}

extern "C" size_t cer_ir50_workspace_bytes(const cer_ir50_weights* w, int64_t frames_per_pass) {
  return cer_ir50_workspace_bytes_se(w, nullptr, frames_per_pass);
}

extern "C" int cer_ir50_create(cer_ir50** out, const cer_ir50_weights* w, int64_t frames_per_pass,
                               void* workspace_dev, size_t workspace_bytes) {
  return cer_ir50_create_se(out, w, nullptr, frames_per_pass, workspace_dev, workspace_bytes);
}

extern "C" int cer_ir50_create_se(cer_ir50** out, const cer_ir50_weights* w, const cer_ir_se* se, int64_t frames_per_pass,
                                  void* workspace_dev, size_t workspace_bytes) {
  if (!out || !w || !workspace_dev || frames_per_pass <= 0 || w->n_units <= 0 || !w->units)
    return set_error(CER_ERR_INVALID, "cer_ir50_create: null/invalid argument");
  if (frames_per_pass + kPadFrames > (1 << 24)) return set_error(CER_ERR_INVALID, "frames_per_pass too large");
  int rc = cer_check_device();
  if (rc) return rc;
  rc = load_driver_entry_points();
  if (rc) return rc;
  if (workspace_bytes < cer_ir50_workspace_bytes_se(w, se, frames_per_pass))
    return set_error(CER_ERR_WORKSPACE, "cer_ir50_create: workspace too small");
  if (se) {
    for (int i = 0; i < w->n_units; ++i) {
      const int d = w->units[i].depth;
      if (!se[i].fc1 || !se[i].fc2 || se[i].hidden <= 0 || se[i].hidden > 64 || d > kSeMaxC || 256 % (d / 8))
        return set_error(CER_ERR_INVALID, "cer_ir50_create_se: SE unit needs fc1/fc2, 0 < hidden <= 64, depth in {64,128,256,512}");
    }
  }
  if (reinterpret_cast<uintptr_t>(workspace_dev) % 256) return set_error(CER_ERR_INVALID, "workspace must be 256B aligned");

  cer_ir50* p = new cer_ir50();
  p->w = *w;
  p->units.assign(w->units, w->units + w->n_units);
  p->w.units = p->units.data();
  p->cap = frames_per_pass;
  p->n_cap = (int)frames_per_pass + kPadFrames;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&p->num_sms, cudaDevAttrMultiProcessorCount, dev);
  p->act_bytes = ((max_act_bytes_per_frame(w) * p->n_cap) + 1023) & ~size_t(1023);
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace_dev) + 1023) & ~uintptr_t(1023));
  for (int i = 0; i < 3; ++i) p->buf[i] = base + i * p->act_bytes;
  p->fc_out = reinterpret_cast<float*>(base + 3 * p->act_bytes);
  const size_t fc_bytes = ((size_t)p->n_cap * w->emb_dim * 4 + 1023) & ~size_t(1023);
  p->gate = se ? reinterpret_cast<float*>(base + 3 * p->act_bytes + fc_bytes) : nullptr;
  p->se.assign(w->n_units, cer_ir50::SeTail{});
  std::vector<int> proj_units;

  int H = w->in_h, W = w->in_w;
  int cur = 0, tb = 1, nxt = 2;
  p->stem_out = {p->buf[cur], H, W, 64};
  rc = make_tiled2d_map_generic(&p->stem_out_map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, p->buf[cur], p->n_cap * H * W, 64, kBlockM, 64);
  if (rc) { delete p; return rc; }
  int C = 64;
  for (int i = 0; i < w->n_units; ++i) {
    const cer_ir_unit& u = p->units[i];
    if (u.cin != C) { delete p; return set_error(CER_ERR_INVALID, "unit cin does not match previous depth"); }
    const bool is_se = se != nullptr;
    if (!u.has_proj && (u.cin != u.depth || (u.stride != 1 && !is_se))) {
      delete p;
      return set_error(CER_ERR_INVALID,
                       "identity shortcut needs cin == depth and stride 1 (pass a MaxPool(1,2) shortcut as identity columns)");
    }
    ConvGeom g1{};
    g1.src = p->buf[cur]; g1.H = H; g1.W = W; g1.Cin = u.cin; g1.ksize = 3; g1.stride = 1; g1.pad = 1;
    g1.weight = u.w1; g1.bias = u.bias1; g1.bias_classes = 9; g1.alpha = u.alpha; g1.res = nullptr;
    g1.dst = p->buf[tb]; g1.Cout = u.depth; g1.out_fp32 = 0;
    ConvOp op1;
    rc = build_conv_op(&op1, g1, p->n_cap, true);
    if (rc) { delete p; return rc; }
    p->ops.push_back(op1);

    ConvGeom g2{};
    g2.src = p->buf[tb]; g2.H = H; g2.W = W; g2.Cin = u.depth; g2.ksize = 3; g2.stride = u.stride; g2.pad = 1;
    if (is_se) {
      // r = conv2 + BN shift only: the gate scales r, the shortcut is added after it (launch_se_tail)
      if (u.has_proj) { g2.wld = 9 * u.depth + u.cin; proj_units.push_back(i); }
    } else if (u.has_proj) {
      g2.src2 = p->buf[cur]; g2.H2 = H; g2.W2 = W; g2.Cin2 = u.cin; g2.stride2 = u.stride;
    } else {
      g2.res = reinterpret_cast<const __nv_bfloat16*>(p->buf[cur]);
    }
    g2.weight = u.w2; g2.bias = u.bias2; g2.bias_classes = 1; g2.alpha = nullptr;
    g2.dst = p->buf[nxt]; g2.Cout = u.depth; g2.out_fp32 = 0;
    ConvOp op2;
    rc = build_conv_op(&op2, g2, p->n_cap, true);
    if (rc) { delete p; return rc; }
    p->ops.push_back(op2);

    const int Hin = H, Win = W;
    H = (H - 1) / u.stride + 1;
    W = (W - 1) / u.stride + 1;
    C = u.depth;
    if (is_se) {
      cer_ir50::SeTail& t = p->se[i];
      t.on = 1; t.hidden = se[i].hidden; t.fc1 = se[i].fc1; t.fc2 = se[i].fc2; t.proj_op = -1;
      t.r = reinterpret_cast<__nv_bfloat16*>(p->buf[nxt]); t.Ho = H; t.Wo = W; t.C = C;
      if (u.has_proj) {      // the projection output lands in the conv1 buffer, which conv2 has consumed
        t.sc = reinterpret_cast<const __nv_bfloat16*>(p->buf[tb]); t.sc_h = H; t.sc_w = W; t.sc_stride = 1;
      } else {
        t.sc = reinterpret_cast<const __nv_bfloat16*>(p->buf[cur]); t.sc_h = Hin; t.sc_w = Win; t.sc_stride = u.stride;
      }
    }
    p->unit_out.push_back({p->buf[nxt], H, W, C});
    std::swap(cur, nxt);
  }
  if (H * W * C != w->fc_in || w->emb_dim % 64) { delete p; return set_error(CER_ERR_INVALID, "fc_in / emb_dim mismatch"); }
  rc = build_raster_stage(p);
  if (rc) { delete p; return rc; }
  ConvGeom gf{};
  gf.src = p->buf[cur]; gf.H = 1; gf.W = 1; gf.Cin = w->fc_in; gf.ksize = 1; gf.stride = 1; gf.pad = 0;
  gf.weight = w->fc_w; gf.bias = w->fc_bias; gf.bias_classes = 1; gf.dst = p->fc_out; gf.Cout = w->emb_dim;
  gf.out_fp32 = 1;
  ConvOp opf;
  rc = build_conv_op(&opf, gf, p->n_cap, true);
  if (rc) { delete p; return rc; }
  p->ops.push_back(opf);
  // projection convs of the SE transition units: op indices after the FC; K = the w2 columns after 9*depth, BN folded,
  // output into the conv1 buffer (smaller than conv1's output: stride 2, same depth)
  for (int i : proj_units) {
    const cer_ir_unit& u = p->units[i];
    const cer_ir50::ActInfo& x = i == 0 ? p->stem_out : p->unit_out[i - 1];
    ConvGeom gp{};
    gp.src = x.ptr; gp.H = x.H; gp.W = x.W; gp.Cin = u.cin; gp.ksize = 1; gp.stride = u.stride; gp.pad = 0;
    gp.weight = static_cast<const __nv_bfloat16*>(u.w2) + 9 * u.depth; gp.wld = 9 * u.depth + u.cin;
    gp.bias = u.bias2 + u.depth; gp.bias_classes = 1; gp.alpha = nullptr;
    gp.dst = const_cast<__nv_bfloat16*>(p->se[i].sc); gp.Cout = u.depth; gp.out_fp32 = 0;
    ConvOp opp;
    rc = build_conv_op(&opp, gp, p->n_cap, true);
    if (rc) { delete p; return rc; }
    p->se[i].proj_op = (int)p->ops.size();
    p->ops.push_back(opp);
  }
  *out = p;
  return CER_OK;
}

static int launch_plan_stem(cer_ir50* p, const float* x, int frames, cudaStream_t st) {
  return launch_stem(x, p->w.stem_w, p->w.stem_bias, p->w.stem_alpha, reinterpret_cast<__nv_bfloat16*>(p->buf[0]), p->stem_out_map,
                     frames, p->w.in_h, p->w.in_w, p->num_sms, st);
}

static int run_pass(cer_ir50* p, const float* x, int frames, int last_unit, float* emb_out, cudaStream_t st) {
  const int n_units = (int)p->units.size();
  const bool rast = raster_pass(p, frames);
  {
    int rc = launch_plan_stem(p, x, frames, st);
    if (rc) return rc;
  }
  for (int i = 0; i < n_units && i <= last_unit; ++i) {
    int rc = launch_plan_op(p, 2 * i, frames, rast, st);
    if (rc) return rc;
    rc = launch_plan_op(p, 2 * i + 1, frames, rast, st);
    if (rc) return rc;
  }
  if (last_unit >= n_units) {
    int rc = launch_plan_op(p, 2 * n_units, frames, rast, st);
    if (rc) return rc;
    const int wpb = 8;
    l2norm_kernel<<<(frames + wpb - 1) / wpb, wpb * 32, 0, st>>>(p->fc_out, emb_out, frames, p->w.emb_dim);
    CER_CUDA(cudaGetLastError());
  }
  return CER_OK;
}

extern "C" int cer_ir50_forward(cer_ir50* p, const float* x, int64_t n_frames, float* emb_out, void* stream) {
  if (!p || n_frames < 0 || (n_frames > 0 && (!x || !emb_out))) return set_error(CER_ERR_INVALID, "cer_ir50_forward: bad argument");
  if (reinterpret_cast<uintptr_t>(x) % 4 || reinterpret_cast<uintptr_t>(emb_out) % 16)
    return set_error(CER_ERR_INVALID, "cer_ir50_forward: emb_out must be 16B aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t frame_elems = (size_t)3 * p->w.in_h * p->w.in_w;
  for (int64_t f0 = 0; f0 < n_frames; f0 += p->cap) {
    const int frames = (int)std::min<int64_t>(p->cap, n_frames - f0);
    int rc = run_pass(p, x + f0 * frame_elems, frames, (int)p->units.size(), emb_out + f0 * p->w.emb_dim, st);
    if (rc) return rc;
  }
  return CER_OK;
}

extern "C" int64_t cer_ir50_debug_activation(cer_ir50* p, const float* x, int64_t frames, int32_t unit_index,
                                             void* dst_dev, void* stream) {
  if (!p || !x || !dst_dev || frames <= 0 || frames > p->cap || unit_index < -1 || unit_index >= (int)p->units.size())
    return set_error(CER_ERR_INVALID, "cer_ir50_debug_activation: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int rc = run_pass(p, x, (int)frames, unit_index, nullptr, st);
  if (rc) return rc;
  const cer_ir50::ActInfo& a = unit_index < 0 ? p->stem_out : p->unit_out[unit_index];
  const int64_t elems = frames * a.H * a.W * a.C;
  if (unit_index >= 0 && raster_pass(p, (int)frames) && p->rops[2 * unit_index + 1].out_padded) {
    const long long vecs = elems / 8;
    raster_unpad_kernel<<<(int)std::min<long long>((vecs + 255) / 256, 8LL * p->num_sms), 256, 0, st>>>(
        static_cast<const __nv_bfloat16*>(a.ptr), static_cast<__nv_bfloat16*>(dst_dev), (int)frames, a.H, a.W, a.C);
    CER_CUDA(cudaGetLastError());
    return elems;
  }
  CER_CUDA(cudaMemcpyAsync(dst_dev, a.ptr, (size_t)elems * 2, cudaMemcpyDeviceToDevice, st));
  return elems;
}

extern "C" int cer_ir50_op_variant(const cer_ir50* p, int32_t op_index, int64_t n_frames, char* buf, int32_t buflen) {
  if (!p || !buf || buflen <= 0 || op_index < 0 || op_index >= (int)p->ops.size() || n_frames <= 0)
    return set_error(CER_ERR_INVALID, "cer_ir50_op_variant: bad argument");
  const int frames = (int)std::min<int64_t>(p->cap, n_frames);
  const bool rast = raster_pass(p, frames) && op_index < (int)p->rops.size() && p->rops[op_index].rast_ok;
  const int n = snprintf(buf, (size_t)buflen, "%s",
                         rast ? raster_variant_name(p->rops[op_index].kp) : conv_variant_name(p->ops[op_index], frames, p->num_sms));
  return n < buflen ? n : buflen - 1;
}

extern "C" const char* cer_conv_last_variant(void) { return conv_last_variant(); }

// Profiling aid: ops [first_op, last_op] of one pass in plan order -- 0 = stem, 1 .. 2U = the unit convs
// (conv1, conv2 of unit 0, ...), 2U + 1 = FC.  The activation buffers must hold a previous forward of the
// same frames (every op then reads the same data it reads in a real pass).
extern "C" int cer_ir50_run_ops(cer_ir50* p, const float* x, int64_t frames, int32_t first_op, int32_t last_op, void* stream) {
  const int n_conv = p ? 2 * (int)p->units.size() + 1 : 0;     // unit convs + FC (projection convs run inside conv2 ops)
  if (!p || frames <= 0 || frames > p->cap || first_op < 0 || last_op < first_op || last_op > n_conv || (first_op == 0 && !x))
    return set_error(CER_ERR_INVALID, "cer_ir50_run_ops: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  for (int op = first_op; op <= last_op; ++op) {
    if (op == 0) {
      int rc = launch_plan_stem(p, x, (int)frames, st);
      if (rc) return rc;
    } else {
      int rc = launch_plan_op(p, op - 1, (int)frames, raster_pass(p, (int)frames), st);
      if (rc) return rc;
    }
  }
  return CER_OK;
}

extern "C" int64_t cer_ir50_launches(const cer_ir50* p, int64_t n_frames) {
  if (!p || n_frames <= 0) return 0;
  int64_t total = 0;
  for (int64_t f0 = 0; f0 < n_frames; f0 += p->cap) {
    const int frames = (int)std::min<int64_t>(p->cap, n_frames - f0);
    total += 1 + 2 * (int64_t)p->units.size() + 2;
    for (const cer_ir50::SeTail& t : p->se) total += t.on ? 2 + (t.proj_op >= 0) : 0;   // squeeze, scale (+ projection)
    if (raster_pass(p, frames))
      for (const cer_ir50::RasterOp& r : p->rops) total += (!r.rast_ok && r.out_padded) ? 1 : 0;   // raster_zero_pads_kernel
  }
  return total;
}

extern "C" void cer_ir50_destroy(cer_ir50* p) { delete p; }

// Single convolution through the same kernel (tests and per-layer-class roofline measurements;
// the plan above is the production path).  Builds its tensor maps per call.
extern "C" int cer_conv_forward(const void* src_nhwc, int32_t n_frames, int32_t n_alloc, int32_t h, int32_t w,
                                int32_t cin, const void* weight, int32_t cout, int32_t ksize, int32_t stride,
                                int32_t pad, const float* bias, int32_t bias_classes, const float* alpha,
                                const void* res, void* dst, int32_t out_fp32, void* stream) {
  if (!src_nhwc || !weight || !bias || !dst || n_frames <= 0 || n_alloc < n_frames || (ksize != 1 && ksize != 3) ||
      (bias_classes != 1 && bias_classes != 9))
    return set_error(CER_ERR_INVALID, "cer_conv_forward: bad argument");
  int rc = cer_check_device();
  if (rc) return rc;
  rc = load_driver_entry_points();
  if (rc) return rc;
  ConvGeom g{};
  g.src = src_nhwc; g.H = h; g.W = w; g.Cin = cin; g.ksize = ksize; g.stride = stride; g.pad = pad;
  g.weight = weight; g.bias = bias; g.bias_classes = bias_classes; g.alpha = alpha;
  g.res = static_cast<const __nv_bfloat16*>(res); g.dst = dst; g.Cout = cout; g.out_fp32 = out_fp32;
  ConvOp op;
  rc = build_conv_op(&op, g, n_alloc);
  if (rc) return rc;
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return launch_conv(op, n_frames, sms, static_cast<cudaStream_t>(stream));
}
