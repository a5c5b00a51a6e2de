// Fused TemporalBlock kernel (fp32):  y = LReLU( LReLU(conv2(LReLU(conv1(x)))) + res(x) ) [* s + t]
// where conv{1,2} are causal dilated k=5 convolutions (Conv1d(pad=(k-1)d, dil=d) + Chomp1d) with
// weight-norm already folded into the weights on the host.
// Reference: TemporalBlock.forward, models/temporal_convolutional_model.py:21-54; the trailing
// affine is the eval BatchNorm1d of models/model.py:515.
//
// Layout: x [B][T][C_in], y [B][T][C_out] (time-major rows, channel contiguous) -- the layout the
// features arrive in ([B,1,T,D]) and the fusion kernel consumes; the reference's transpose to
// [B,C,T] is never materialised.
//
// One CTA = one (batch, 32-step time tile).  Phase 1 computes conv1 for the tile plus its causal
// halo ((k-1)d earlier steps) into shared memory; phase 2 runs conv2 from shared memory, adds the
// identity / 1x1 residual, applies the activations and writes y.  Both phases are register-tiled
// SGEMMs whose K loop walks (16-channel chunk, tap); the x chunk is staged once per chunk and
// re-used by all taps through a row shift.
//
// The head is fp32 on purpose (SURVEY.md H4: argmax parity is marginal with a bf16 head).  At
// B*T = 600..2400 rows the block is bound by streaming its weights from L2 and by FMA issue,
// not by HBM: compulsory bytes are 20 MB of weights for the whole head.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>

#include "../../include/cer_b200.h"
#include "common.h"

namespace cer {

constexpr int kTT = 32;        // output time steps per CTA
constexpr int kKC = 16;        // channels per K chunk
constexpr int kTcnThreads = 256;
constexpr float kLeaky = 0.01f;

__device__ __forceinline__ float lrelu(float v) { return v >= 0.f ? v : v * kLeaky; }

// The instantiations launch_tcn can run, COUT-major (cer_head_last_variant reports the one a launch used).
static const char* const kHeadVariantNames[] = {
  "tcn_block_kernel<32,1,5>", "tcn_block_kernel<32,2,5>", "tcn_block_kernel<32,4,5>", "tcn_block_kernel<32,8,5>",
  "tcn_block_kernel<64,1,5>", "tcn_block_kernel<64,2,5>", "tcn_block_kernel<64,4,5>", "tcn_block_kernel<64,8,5>",
  "tcn_block_kernel<128,1,5>", "tcn_block_kernel<128,2,5>", "tcn_block_kernel<128,4,5>", "tcn_block_kernel<128,8,5>",
  "tcn_block_kernel<256,1,5>", "tcn_block_kernel<256,2,5>", "tcn_block_kernel<256,4,5>", "tcn_block_kernel<256,8,5>"};

constexpr int log2_small(int v) { return v <= 1 ? 0 : 1 + log2_small(v / 2); }

// COUT in {32,64,128,256}; DIL in {1,2,4,8}; KS = kernel size (5).
template <int COUT, int DIL, int KS>
struct TcnCfg {
  static constexpr int HALO = (KS - 1) * DIL;
  static constexpr int R1 = kTT + HALO;            // conv1 rows needed (tile + causal halo)
  static constexpr int RX = kTT + 2 * HALO;        // x rows needed
  static constexpr int COLS_T = COUT / 4;          // threads across channels (4 channels each)
  static constexpr int ROWS_T = kTcnThreads / COLS_T;
  static constexpr int NR1 = (R1 + ROWS_T - 1) / ROWS_T;
  static constexpr int NR2 = (kTT + ROWS_T - 1) / ROWS_T;
  static constexpr int XS_LD = kKC + 1;
  static constexpr int H1_LD = COUT + 4;           // +4 floats: rows of different ty hit different banks
  static constexpr size_t SMEM = (size_t)(R1 * H1_LD + RX * XS_LD + kKC * COUT) * sizeof(float);
};

template <int COUT, int DIL, int KS>
__global__ void __launch_bounds__(kTcnThreads) tcn_block_kernel(cer_tcn_block blk, const float* __restrict__ x,
                                                                float* __restrict__ y, int T) {
  using C = TcnCfg<COUT, DIL, KS>;
  extern __shared__ __align__(16) float smem_f[];
  float* h1s = smem_f;                       // [R1][H1_LD]  conv1 output (post LReLU), zero for t < 0
  float* xs = h1s + C::R1 * C::H1_LD;           // [RX][XS_LD]  x chunk
  float* ws = xs + C::RX * C::XS_LD;         // [kKC][COUT]  weight chunk

  const int cin = blk.c_in;
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * kTT;
  const int tx = threadIdx.x % C::COLS_T;
  const int ty = threadIdx.x / C::COLS_T;
  const int c0 = tx * 4;
  const float* xb = x + (size_t)b * T * cin;

  auto load_x_chunk = [&](int ci0) {
    // rows t0-2*HALO .. t0+kTT-1, channels ci0..ci0+15; zero outside [0,T)
    for (int i = threadIdx.x; i < C::RX * (kKC / 4); i += kTcnThreads) {
      const int r = i / (kKC / 4), q = i % (kKC / 4);
      const int t = t0 - 2 * C::HALO + r;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t >= 0 && t < T) v = __ldg(reinterpret_cast<const float4*>(xb + (size_t)t * cin + ci0) + q);
      float* d = xs + r * C::XS_LD + q * 4;
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
  };
  auto load_w_chunk = [&](const float* wsrc /* [kKC][COUT] contiguous rows of stride COUT */) {
    for (int i = threadIdx.x; i < kKC * COUT / 4; i += kTcnThreads)
      reinterpret_cast<float4*>(ws)[i] = __ldg(reinterpret_cast<const float4*>(wsrc) + i);
  };

  // ---------------- phase 1: h1 = LReLU(conv1(x) + b1) on rows t0-HALO .. t0+kTT-1 ----------------
  {
    float acc[C::NR1][4];
#pragma unroll
    for (int i = 0; i < C::NR1; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
    for (int ci0 = 0; ci0 < cin; ci0 += kKC) {
      __syncthreads();
      load_x_chunk(ci0);
      for (int j = 0; j < KS; ++j) {
        __syncthreads();
        load_w_chunk(blk.w1 + ((size_t)j * cin + ci0) * COUT);
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kKC; ++kk) {
          const float4 w = *reinterpret_cast<const float4*>(&ws[kk * COUT + c0]);
#pragma unroll
          for (int i = 0; i < C::NR1; ++i) {
            const int lr = ty + i * C::ROWS_T;
            if (lr < C::R1) {
              const float a = xs[(lr + j * DIL) * C::XS_LD + kk];
              acc[i][0] = fmaf(a, w.x, acc[i][0]); acc[i][1] = fmaf(a, w.y, acc[i][1]);
              acc[i][2] = fmaf(a, w.z, acc[i][2]); acc[i][3] = fmaf(a, w.w, acc[i][3]);
            }
          }
        }
      }
    }
    const float4 bb = __ldg(reinterpret_cast<const float4*>(blk.b1 + c0));
#pragma unroll
    for (int i = 0; i < C::NR1; ++i) {
      const int lr = ty + i * C::ROWS_T;
      if (lr < C::R1) {
        const int t = t0 - C::HALO + lr;
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);       // conv2 sees zero padding before t = 0
        if (t >= 0) o = make_float4(lrelu(acc[i][0] + bb.x), lrelu(acc[i][1] + bb.y), lrelu(acc[i][2] + bb.z),
                                    lrelu(acc[i][3] + bb.w));
        *reinterpret_cast<float4*>(&h1s[lr * C::H1_LD + c0]) = o;
      }
    }
  }

  // ---------------- phase 2: conv2 from smem, residual, activations ----------------
  float acc[C::NR2][4];
#pragma unroll
  for (int i = 0; i < C::NR2; ++i) { acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f; }
  for (int cc0 = 0; cc0 < COUT; cc0 += kKC) {
    for (int j = 0; j < KS; ++j) {
      __syncthreads();
      load_w_chunk(blk.w2 + ((size_t)j * COUT + cc0) * COUT);
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < kKC; ++kk) {
        const float4 w = *reinterpret_cast<const float4*>(&ws[kk * COUT + c0]);
#pragma unroll
        for (int i = 0; i < C::NR2; ++i) {
          const int lr = ty + i * C::ROWS_T;
          if (lr < kTT) {
            const float a = h1s[(lr + j * DIL) * C::H1_LD + cc0 + kk];
            acc[i][0] = fmaf(a, w.x, acc[i][0]); acc[i][1] = fmaf(a, w.y, acc[i][1]);
            acc[i][2] = fmaf(a, w.z, acc[i][2]); acc[i][3] = fmaf(a, w.w, acc[i][3]);
          }
        }
      }
    }
  }
  const float4 b2 = __ldg(reinterpret_cast<const float4*>(blk.b2 + c0));
#pragma unroll
  for (int i = 0; i < C::NR2; ++i) {
    acc[i][0] = lrelu(acc[i][0] + b2.x); acc[i][1] = lrelu(acc[i][1] + b2.y);
    acc[i][2] = lrelu(acc[i][2] + b2.z); acc[i][3] = lrelu(acc[i][3] + b2.w);
  }

  // residual
  if (blk.wd != nullptr) {
    float racc[C::NR2][4];
#pragma unroll
    for (int i = 0; i < C::NR2; ++i) { racc[i][0] = racc[i][1] = racc[i][2] = racc[i][3] = 0.f; }
    for (int ci0 = 0; ci0 < cin; ci0 += kKC) {
      __syncthreads();
      load_x_chunk(ci0);
      load_w_chunk(blk.wd + (size_t)ci0 * COUT);
      __syncthreads();
#pragma unroll
      for (int kk = 0; kk < kKC; ++kk) {
        const float4 w = *reinterpret_cast<const float4*>(&ws[kk * COUT + c0]);
#pragma unroll
        for (int i = 0; i < C::NR2; ++i) {
          const int lr = ty + i * C::ROWS_T;
          if (lr < kTT) {
            const float a = xs[(lr + 2 * C::HALO) * C::XS_LD + kk];
            racc[i][0] = fmaf(a, w.x, racc[i][0]); racc[i][1] = fmaf(a, w.y, racc[i][1]);
            racc[i][2] = fmaf(a, w.z, racc[i][2]); racc[i][3] = fmaf(a, w.w, racc[i][3]);
          }
        }
      }
    }
    const float4 bd = __ldg(reinterpret_cast<const float4*>(blk.bd + c0));
#pragma unroll
    for (int i = 0; i < C::NR2; ++i) {
      acc[i][0] += racc[i][0] + bd.x; acc[i][1] += racc[i][1] + bd.y;
      acc[i][2] += racc[i][2] + bd.z; acc[i][3] += racc[i][3] + bd.w;
    }
  } else {
#pragma unroll
    for (int i = 0; i < C::NR2; ++i) {
      const int lr = ty + i * C::ROWS_T;
      const int t = t0 + lr;
      if (lr < kTT && t < T) {
        const float4 r = __ldg(reinterpret_cast<const float4*>(xb + (size_t)t * cin + c0));
        acc[i][0] += r.x; acc[i][1] += r.y; acc[i][2] += r.z; acc[i][3] += r.w;
      }
    }
  }

  float4 ps = make_float4(1.f, 1.f, 1.f, 1.f), pt = make_float4(0.f, 0.f, 0.f, 0.f);
  if (blk.post_scale != nullptr) {
    ps = __ldg(reinterpret_cast<const float4*>(blk.post_scale + c0));
    pt = __ldg(reinterpret_cast<const float4*>(blk.post_shift + c0));
  }
  float* yb = y + (size_t)b * T * COUT;
#pragma unroll
  for (int i = 0; i < C::NR2; ++i) {
    const int lr = ty + i * C::ROWS_T;
    const int t = t0 + lr;
    if (lr < kTT && t < T) {
      float4 o;
      o.x = fmaf(lrelu(acc[i][0]), ps.x, pt.x); o.y = fmaf(lrelu(acc[i][1]), ps.y, pt.y);
      o.z = fmaf(lrelu(acc[i][2]), ps.z, pt.z); o.w = fmaf(lrelu(acc[i][3]), ps.w, pt.w);
      *reinterpret_cast<float4*>(yb + (size_t)t * COUT + c0) = o;
    }
  }
}

template <int COUT, int DIL>
static int launch_tcn(const cer_tcn_block& blk, const float* x, float* y, int B, int T, cudaStream_t st) {
  using C = TcnCfg<COUT, DIL, 5>;
  static unsigned long long configured = 0;
  if (first_use_on_device(&configured)) {
    CER_CUDA(cudaFuncSetAttribute(tcn_block_kernel<COUT, DIL, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
  }
  static_assert(COUT >= 32 && COUT <= 256 && DIL <= 8, "kHeadVariantNames covers COUT 32..256, DIL 1..8");
  set_head_variant(kHeadVariantNames[4 * log2_small(COUT / 32) + log2_small(DIL)]);
  dim3 grid((T + kTT - 1) / kTT, B);
  tcn_block_kernel<COUT, DIL, 5><<<grid, kTcnThreads, C::SMEM, st>>>(blk, x, y, T);
  CER_CUDA(cudaGetLastError());
  return CER_OK;
}

template <int COUT>
static int dispatch_dil(const cer_tcn_block& blk, const float* x, float* y, int B, int T, cudaStream_t st) {
  switch (blk.dilation) {
    case 1: return launch_tcn<COUT, 1>(blk, x, y, B, T, st);
    case 2: return launch_tcn<COUT, 2>(blk, x, y, B, T, st);
    case 4: return launch_tcn<COUT, 4>(blk, x, y, B, T, st);
    case 8: return launch_tcn<COUT, 8>(blk, x, y, B, T, st);
    default: return set_error(CER_ERR_INVALID, "tcn: dilation must be 1, 2, 4 or 8");
  }
}

}  // namespace cer

extern "C" size_t cer_tcn_block_workspace_bytes(const cer_tcn_block*, int64_t, int64_t) { return 0; }

extern "C" int cer_tcn_block_forward(const cer_tcn_block* blk, const float* x, float* y, int64_t batch, int64_t length,
                                     void* /*workspace*/, size_t /*workspace_bytes*/, void* stream) {
  using namespace cer;
  if (!blk || !x || !y || batch <= 0 || length <= 0 || batch > 65535)
    return set_error(CER_ERR_INVALID, "cer_tcn_block_forward: bad argument");
  if (blk->kernel_size != 5) return set_error(CER_ERR_INVALID, "tcn: only kernel_size 5 is built (configs.py:74)");
  if (blk->c_in % 16 || blk->c_in <= 0) return set_error(CER_ERR_INVALID, "tcn: c_in must be a multiple of 16");
  if (!blk->w1 || !blk->b1 || !blk->w2 || !blk->b2) return set_error(CER_ERR_INVALID, "tcn: null weight");
  if (!blk->wd && blk->c_in != blk->c_out) return set_error(CER_ERR_INVALID, "tcn: identity residual needs c_in == c_out");
  if ((blk->wd == nullptr) != (blk->bd == nullptr) || (blk->post_scale == nullptr) != (blk->post_shift == nullptr))
    return set_error(CER_ERR_INVALID, "tcn: wd/bd and post_scale/post_shift come in pairs");
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) % 16)
    return set_error(CER_ERR_INVALID, "tcn: x and y must be 16B aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = (int)batch, T = (int)length;
  switch (blk->c_out) {
    case 32:  return dispatch_dil<32>(*blk, x, y, B, T, st);
    case 64:  return dispatch_dil<64>(*blk, x, y, B, T, st);
    case 128: return dispatch_dil<128>(*blk, x, y, B, T, st);
    case 256: return dispatch_dil<256>(*blk, x, y, B, T, st);
    default:  return set_error(CER_ERR_INVALID, "tcn: c_out must be 32, 64, 128 or 256");
  }
}
